"""Yardstick for the real-image parity test: the UNMODIFIED reference (oracle/_ref, staged by oracle/build_ref.py) run on
the GPU in fp32 with TF32 forbidden, compared with the fixture that the same code minted on the CPU
(tests/golden/config1_vos.*).  The memory read keeps the top-30 of ~1600 similarities per query; on a real image many
of them are nearly tied, and fp32 rounding that differs between devices (summation order of the GEMMs) swaps members
across the cut - the reference does not reproduce ITSELF bit for bit across devices.  Prints one JSON line:
{"max_abs": [per frame], "worst": ..., "device": ..., "power_limit_w": ..., "torch": ...}, which is stored as
tests/golden/config1_ref_on_gpu.json for tests/test_config1_gpu.py.  Own process: the reference's package is also called
``deva``."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import fixtures, ref_loader  # noqa: E402


def power_limit_w():
    try:
        out = subprocess.run(['nvidia-smi', '--id=0', '--query-gpu=power.limit', '--format=csv,noheader,nounits'],
                             capture_output=True, text=True, timeout=30).stdout
        return float(out.strip().splitlines()[0])
    except Exception:
        return None


def main():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.set_grad_enabled(False)
    DEVA, Core, synth = ref_loader.load()
    g, meta = fixtures.config1_vos(HERE)
    net = DEVA(meta['config']).cuda().eval()
    net.load_weights({k: v.cuda() for k, v in synth(seed=1).items()})
    np.random.seed(42)
    core = Core(net, meta['config'])
    mean = torch.tensor([0.485, 0.456, 0.406]).view(3, 1, 1)
    std = torch.tensor([0.229, 0.224, 0.225]).view(3, 1, 1)
    errs = []
    T = g['frames_u8'].shape[0]
    for t in range(T):
        img = ((torch.from_numpy(g['frames_u8'][t]).permute(2, 0, 1).float() / 255 - mean) / std).cuda()
        if t == 0:
            p = core.step(img, torch.from_numpy(g['mask0'].astype(np.int64)).cuda(), meta['labels'])
        else:
            p = core.step(img, end=(t == T - 1))
        errs.append(float((p.float().cpu()[:, 1::4, 2::4] - torch.from_numpy(g[f'prob_lattice_{t}'])).abs().max()))
    print(json.dumps({'max_abs': errs, 'worst': max(errs), 'device': torch.cuda.get_device_name(0),
                      'power_limit_w': power_limit_w(), 'torch': torch.__version__}))


if __name__ == '__main__':
    main()
