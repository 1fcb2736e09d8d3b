"""How far is the reference's OWN stock GPU path from its fp32 CPU path?  PyTorch's default lets cuDNN run fp32
convolutions on TF32 tensor cores (10-bit mantissa, like fp16).  Replays the golden clip through the cuDNN debug
backend (identical graphs, reference memory-read semantics through our kernels) with TF32 allowed / forbidden and
through the native fp16 stack, and prints max |prob - golden| for each.  GPU only."""
import json
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

torch.set_grad_enabled(False)


def run(backend, tf32):
    torch.backends.cudnn.allow_tf32 = tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    arrays, meta = fixtures.vos_steps()
    g = {k: torch.from_numpy(v) for k, v in arrays.items()}
    np.random.seed(42)
    net = DEVA(meta['config'])
    net.conv_backend = backend
    net = net.cuda().eval()
    net.load_weights({k: v.cuda() for k, v in synthetic_state_dict(seed=1).items()})
    core = DEVAInferenceCore(net, meta['config'])
    T = g['frames'].shape[0]
    worst, per_frame = 0.0, []
    for t in range(T):
        img = g['frames'][t].cuda()
        if t == 0:
            p = core.step(img, g['mask0'].cuda(), [1, 2])
        elif t == 6:
            p = core.step(img, g['mask6'].cuda(), [7])
        else:
            p = core.step(img, end=(t == T - 1))
        e = float((p.cpu() - g[f'prob_{t:02d}']).abs().max())
        per_frame.append(e)
        worst = max(worst, e)
    return worst, per_frame


if __name__ == '__main__':
    out = {}
    for name, backend, tf32 in (('cudnn fp32 (TF32 forbidden)', 'torch', False),
                                ('cudnn fp32, PyTorch default (TF32 allowed)', 'torch', True),
                                ('native sm_100a kernels (fp16 operands, fp32 accumulate)', 'native', False)):
        worst, per_frame = run(backend, tf32)
        out[name] = {'max_abs_prob_err': worst, 'per_frame': per_frame}
        print(f'{name:60s} max |prob - golden| = {worst:.3e}', flush=True)
    print(json.dumps(out))
