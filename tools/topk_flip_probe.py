"""GPU probe: how often, and by how much, does the fused similarity/top-k kernel pick a different top-30 than exact
arithmetic on REAL-image keys (example clip of tests/golden/config1_vos.*)?  Memory = keys of frame 0, queries = keys
of frame 1, both from the cuDNN fp32 engine; ground truth = fp64 similarity on the CPU.  For every query whose set
differs it reports delta = sim64(best excluded) - sim64(worst included): the similarity error that caused the swap."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tracking-anything-with-deva_b200'))
from deva import _native as nat  # noqa: E402
from deva.model.engine import Engine  # noqa: E402
from deva.model.param_spec import synthetic_state_dict  # noqa: E402
from deva.utils.tensor_utils import pad_divide_by  # noqa: E402
from oracle import fixtures  # noqa: E402
from oracle import memory_math as mm  # noqa: E402

torch.set_grad_enabled(False)
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False


def main():
    g, _ = fixtures.config1_vos()
    mean = torch.tensor([0.485, 0.456, 0.406]).view(3, 1, 1)
    std = torch.tensor([0.229, 0.224, 0.225]).view(3, 1, 1)
    eng = Engine({k: v.cuda() for k, v in synthetic_state_dict(seed=1).items()})
    keys = []
    for t in (0, 1):
        img = ((torch.from_numpy(g['frames_u8'][t]).permute(2, 0, 1).float() / 255 - mean) / std).cuda()
        img, _ = pad_divide_by(img, 16)
        _, feat = eng.encode_image(img.unsqueeze(0))
        keys.append([x[0].flatten(1).contiguous() for x in eng.transform_key(feat)])
    (mk, ms, _), (qk, _, qe) = keys
    ms = ms.reshape(-1).contiguous()
    n, q, ck = mk.shape[1], qk.shape[1], mk.shape[0]
    k_hi = torch.zeros(n, 2 * ck, dtype=torch.float16, device='cuda'); k_lo = torch.zeros_like(k_hi)
    neg_s, raw_shr, raw_key = torch.zeros(n, device='cuda'), torch.zeros(n, device='cuda'), torch.zeros(n, ck, device='cuda')
    nat.pack_keys(mk, None, n, 1, ms, ck, n, k_hi, k_lo, neg_s, raw_key, None, raw_shr)
    q_hi = torch.empty(q, 2 * ck, dtype=torch.float16, device='cuda'); q_lo = torch.empty_like(q_hi)
    bsq = torch.empty(q, device='cuda')
    nat.pack_query(qk, qe, q, 1, ck, q, q_hi, q_lo, bsq)
    ws = torch.empty(nat.simtopk_workspace_bytes(q), dtype=torch.uint8, device='cuda')
    idx = torch.empty(q, 32, dtype=torch.int32, device='cuda'); w = torch.empty(q, 32, device='cuda')
    sims = torch.empty(q, 32, device='cuda')
    nat.sim_topk(k_hi, k_lo, neg_s, n, 0, q_hi, q_lo, bsq, q, ck, 30, ws, idx, w, None, 0, None, None, 0, False, False,
                 out_sim=sims)
    torch.cuda.synchronize()
    sim64 = mm.similarity(mk.cpu().double(), ms.cpu().double(), qk.cpu().double(), qe.cpu().double())  # [N, Q]
    sim32 = mm.similarity(mk, ms, qk, qe).cpu().double()  # the reference's own fp32 formulation, on this GPU
    ref_idx = torch.topk(sim64, 30, dim=0)[1].t()
    got = idx[:, :30].long().cpu()
    got_sim = torch.gather(sim64.t(), 1, got)
    print(f'N={n} Q={q}: kernel similarity vs fp64 at the selected slots: max |d| = '
          f'{float((sims[:, :30].cpu().double() - got_sim).abs().max()):.2e}; reference fp32 formulation vs fp64: '
          f'{float((sim32 - sim64).abs().max()):.2e}')
    for name, sel in (('kernel', got), ('reference fp32 formulation (ATen on GPU)', torch.topk(sim32, 30, dim=0)[1].t())):
        deltas = []
        for i in range(q):
            a, b = set(sel[i].tolist()), set(ref_idx[i].tolist())
            if a != b:
                inc, exc = list(a - b), list(b - a)
                deltas.append(float(sim64[exc, i].max() - sim64[inc, i].min()))
        d = torch.tensor(deltas) if deltas else torch.zeros(1)
        print(f'{name:45s}: {len(deltas)} of {q} queries differ from the fp64 top-30; swap deltas: median '
              f'{float(d.median()):.2e}  max {float(d.max()):.2e}')


if __name__ == '__main__':
    main()
