"""Where does the native (fp16-operand) conv stack lose accuracy?  Runs each network stage of the golden clip's first
frames through the hand-written kernels and through the cuDNN-fp32 debug engine ON THE SAME INPUTS and prints the
max-abs / relative error per stage output (single step, no recurrence).  GPU only."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tracking-anything-with-deva_b200'))
from deva.model.engine import Engine  # noqa: E402
from deva.model.native_engine import NativeEngine  # noqa: E402
from deva.model.param_spec import synthetic_state_dict  # noqa: E402
from deva.utils.tensor_utils import pad_divide_by  # noqa: E402
from oracle import fixtures  # noqa: E402

torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
torch.set_grad_enabled(False)


def report(name, a, b):
    a, b = a.float(), b.float()
    err = float((a - b).abs().max())
    scale = float(b.abs().max())
    rms = float((a - b).pow(2).mean().sqrt())
    print(f'{name:34s} max|d| {err:9.3e}  rel-to-max {err / max(scale, 1e-30):9.3e}  rms {rms:9.3e}  (max|ref| {scale:.3g})',
          flush=True)


def main():
    dev = 'cuda'
    g = {k: torch.from_numpy(v) for k, v in fixtures.vos_steps()[0].items()}
    sd = {k: v.to(dev) for k, v in synthetic_state_dict(seed=1).items()}
    ref, nat = Engine(sd), NativeEngine(sd)
    image, _ = pad_divide_by(g['frames'][0].to(dev), 16)
    image = image.unsqueeze(0)
    mask0 = g['mask0'].to(dev)
    masks = torch.stack([(mask0 == i).float() for i in (1, 2)])
    masks, _ = pad_divide_by(masks, 16)
    masks = masks.unsqueeze(0)

    (r16, r8, r4), rkf = ref.encode_image(image)
    (n16, n8, n4), nkf = nat.encode_image(image)
    for name, a, b in (('encode_image.f16', n16, r16), ('encode_image.f8', n8, r8), ('encode_image.f4', n4, r4),
                       ('encode_image.key_feat', nkf, rkf)):
        report(name, a, b)
    rk, rs, re = ref.transform_key(rkf)
    nk, ns, ne = nat.transform_key(nkf)
    report('transform_key.key', nk, rk); report('transform_key.shrinkage', ns, rs); report('transform_key.selection', ne, re)

    h, w = rk.shape[-2:]
    k = masks.shape[1]
    cv = 512
    sens0 = torch.zeros(1, k, cv, h, w, device=dev)
    # value encoder on identical inputs (the reference engine's features)
    rv, rsens = ref.encode_mask(image, (r16, r8, r4), sens0, masks)
    nv, nsens = nat.encode_mask(image, (r16, r8, r4), sens0.half(), masks)
    report('encode_mask.value (same feats)', nv, rv); report('encode_mask.sensory', nsens, rsens)
    nv2, _ = nat.encode_mask(image, (n16, n8, n4), sens0.half(), masks)
    report('encode_mask.value (own feats)', nv2, rv)

    # decoder on identical inputs: readout := the value itself (right shape and statistics)
    rs2, rlog = ref.decode((r16, r8, r4), rv, rsens, masks)
    ns2, nlog = nat.decode((r16, r8, r4), rv, rsens.half(), masks)
    report('decode.logits (same inputs)', nlog, rlog); report('decode.sensory', ns2, rs2)
    ns3, nlog3 = nat.decode((n16, n8, n4), nv2, nsens, masks)
    report('decode.logits (own inputs)', nlog3, rlog)
    _, nprob = nat.probabilities(nlog.float().contiguous())
    _, rprob = nat.probabilities(rlog.float().contiguous())
    report('prob (same inputs)', nprob, rprob)
    _, nprob3 = nat.probabilities(nlog3.float().contiguous())
    report('prob (own inputs)', nprob3, rprob)

    # second step of the recurrence with each engine's own state
    rs4, rlog4 = ref.decode((r16, r8, r4), rv, rs2, masks)
    ns4, nlog4 = nat.decode((n16, n8, n4), nv2, ns3, masks)
    report('decode#2.logits (own state)', nlog4, rlog4)
    _, p4n = nat.probabilities(nlog4.float().contiguous()); _, p4r = nat.probabilities(rlog4.float().contiguous())
    report('prob#2 (own state)', p4n, p4r)


if __name__ == '__main__':
    main()
