"""GPU diagnostic: where does the product differ from the CPU oracle on the real-image clip (config 1)?  Steps the
product core (both conv backends) and oracle.core.CoreOracle side by side and compares, frame by frame: key / shrinkage /
selection, the memory read-out, the aggregated logits and the probabilities (each pipeline on its own state)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tracking-anything-with-deva_b200'))
from deva.inference.inference_core import DEVAInferenceCore  # noqa: E402
from deva.model.network import DEVA  # noqa: E402
from deva.model.param_spec import synthetic_state_dict  # noqa: E402
from oracle import fixtures  # noqa: E402
from oracle import network as onet  # noqa: E402
from oracle.core import CoreOracle  # noqa: E402

torch.set_grad_enabled(False)
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False


def rel(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return f'max {float((a - b).abs().max()):.2e} (rel-to-max {float((a - b).abs().max() / b.abs().max()):.2e}, rms {float((a - b).pow(2).mean().sqrt()):.2e})'


def main():
    g, meta = fixtures.config1_vos()
    mean = torch.tensor([0.485, 0.456, 0.406]).view(3, 1, 1)
    std = torch.tensor([0.229, 0.224, 0.225]).view(3, 1, 1)
    frames = [((torch.from_numpy(g['frames_u8'][t]).permute(2, 0, 1).float() / 255) - mean) / std for t in range(4)]
    mask0 = torch.from_numpy(g['mask0'].astype(np.int64))
    sd = synthetic_state_dict(seed=1)

    cap = {}
    o_read, o_seg, o_key = CoreOracle._segment, onet.segment, onet.transform_key

    def seg_spy(sd_, ms, readout, sensory, last_mask, update_sensory=True):
        out = o_seg(sd_, ms, readout, sensory, last_mask, update_sensory=update_sensory)
        cap['o_readout'], cap['o_logits'], cap['o_sensory'] = readout.clone(), out[1].clone(), out[0].clone()
        return out

    def key_spy(sd_, feat):
        out = o_key(sd_, feat)
        cap['o_key'] = [x.clone() for x in out]
        return out

    onet.segment, onet.transform_key = seg_spy, key_spy
    np.random.seed(42)
    oracle = CoreOracle(sd, meta['config'])
    cores = {}
    for backend in ('torch', 'native'):
        net = DEVA(meta['config'])
        net.conv_backend = backend
        net = net.cuda().eval()
        net.load_weights({k: v.cuda() for k, v in sd.items()})
        core = DEVAInferenceCore(net, meta['config'])
        mm_, seg_, key_ = core.memory.match_memory, net.segment, net.transform_key

        def mm_spy(k, s, _f=mm_, _b=backend):
            out = _f(k, s)
            cap[_b + '_readout'] = torch.stack([out[o].float() for o in sorted(out)]).unsqueeze(0)
            return out

        def sg_spy(*a, _f=seg_, _b=backend, **kw):
            out = _f(*a, **kw)
            cap[_b + '_logits'], cap[_b + '_sensory'] = out[1].float(), out[0].float()
            return out

        def ky_spy(feat, _f=key_, _b=backend, **kw):
            out = _f(feat, **kw)
            cap[_b + '_key'] = [x.float() for x in out]
            return out

        core.memory.match_memory, net.segment, net.transform_key = mm_spy, sg_spy, ky_spy
        cores[backend] = core
    for t in range(4):
        po = oracle.step(frames[t], mask0 if t == 0 else None, meta['labels'] if t == 0 else None, end=(t == 3))
        print(f'frame {t}: oracle vs fixture lattice {float((po[:, 1::4, 2::4] - torch.from_numpy(g[f"prob_lattice_{t}"])).abs().max()):.2e}')
        for backend, core in cores.items():
            p = core.step(frames[t].cuda(), mask0.cuda() if t == 0 else None, meta['labels'] if t == 0 else None, end=(t == 3))
            print(f'  [{backend}] prob {rel(p, po)}')
            for i, name in enumerate(('key', 'shrinkage', 'selection')):
                print(f'  [{backend}]   {name:10s} {rel(cap[backend + "_key"][i], cap["o_key"][i])}')
            if t > 0:
                print(f'  [{backend}]   readout    {rel(cap[backend + "_readout"], cap["o_readout"])}')
                print(f'  [{backend}]   logits     {rel(cap[backend + "_logits"], cap["o_logits"])}')
                print(f'  [{backend}]   sensory    {rel(cap[backend + "_sensory"], cap["o_sensory"])}')
                d = (p.float().cpu() - po).abs()
                print(f'  [{backend}]   pixels with |d| > 3e-4: {int((d > 3e-4).sum())} of {d.numel()};  > 6e-4: {int((d > 6e-4).sum())}')


if __name__ == '__main__':
    main()
