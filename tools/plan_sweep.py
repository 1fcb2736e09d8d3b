"""GPU experiment: max / rms |prob - reference| over the golden clip under different per-layer precision plans
(DEVA_B200_PLAN overrides on top of the default 'parity' plan).  Calibrates tools/precision_plan.py's CPU emulation
against the kernels.   python tools/plan_sweep.py [plan ...]   (a plan is a DEVA_B200_PLAN string; '' = default)"""
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
_ARRAYS, META = fixtures.vos_steps()
G = {k: torch.from_numpy(v) for k, v in _ARRAYS.items()}
SD = {k: v.cuda() for k, v in synthetic_state_dict(seed=1).items()}

DEFAULT_PLANS = [
    ('fast', None),
    ('parity (default)', ''),
    ('+ up_16_8 c1/c2 act_lo', 'up_16_8.out_conv.c=act_lo'),
    ('+ up_8_4 precise', 'up_8_4=precise'),
    ('+ up_8_4, up_16_8 precise', 'up_8_4=precise,up_16_8=precise'),
    ('+ fuser act_lo', 'mask_decoder.fuser.b1.c=act_lo,mask_decoder.fuser.b2=act_lo'),
    ('+ whole decoder precise (GRU single)', 'mask_decoder=precise'),
    ('+ mask encoder precise (GRU single)', 'mask_encoder=precise'),
    ('parity, key projection in fp32 ATen', 'hybrid:keyproj_fp32'),
    ('parity, encoder trunk in fp32 ATen', 'hybrid:trunk_fp32'),
    ('parity, whole key path in fp32 ATen', 'hybrid:keypath_fp32'),
]


def install_hybrid(eng, kind):
    """Swap parts of the native key path for plain fp32 ATen ops (TF32 off) to locate what the top-k read is sensitive to."""
    import torch.nn.functional as F
    from deva.model.engine import Engine
    from deva.model.native_engine import _api, _to_nhwc
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    ref = Engine(SD)

    def pair_api(x):  # fp32 NCHW -> API view of NHWC fp16 hi with the lo part riding along
        nhwc = x.permute(0, 2, 3, 1).contiguous()
        hi = nhwc.half()
        v = _api(hi)
        v._b200_lo = (nhwc - hi.float()).half()
        return v

    if kind in ('trunk_fp32', 'keypath_fp32'):
        def encode_image(image):
            (f16, f8, f4), feat = ref.encode_image(image.float())
            a16 = pair_api(f16)
            a16._b200_relu = torch.relu(_to_nhwc(a16))
            a16._b200_relu_lo = None
            kf = pair_api(feat)
            kf._fp32 = feat
            return (a16, pair_api(f8), pair_api(f4)), kf
        eng.encode_image = encode_image
    if kind in ('keyproj_fp32', 'keypath_fp32'):
        def transform_key(feat, need_sk=True, need_ek=True):
            x = getattr(feat, '_fp32', None)
            if x is None:
                hi = _to_nhwc(feat)
                x = (hi.float() + feat._b200_lo.float()).permute(0, 3, 1, 2).contiguous()
            return ref.transform_key(x, need_sk, need_ek)
        eng.transform_key = transform_key


def run(tag, plan):
    hybrid = None
    if plan and plan.startswith('hybrid:'):
        hybrid, plan = plan.split(':', 1)[1], ''
    os.environ.pop('DEVA_B200_PLAN', None)
    os.environ['DEVA_B200_PRECISION'] = 'fast' if plan is None else 'parity'
    if plan:
        os.environ['DEVA_B200_PLAN'] = plan
    np.random.seed(42)
    net = DEVA(META['config'])
    net.conv_backend = 'native'
    net = net.cuda().eval()
    net.load_weights(SD)
    core = DEVAInferenceCore(net, META['config'])
    if hybrid:
        install_hybrid(net.engine, hybrid)
    T = G['frames'].shape[0]
    worst, sq, n, per = 0.0, 0.0, 0, []
    for t in range(T):
        img = G['frames'][t].cuda()
        if t == 0:
            p = core.step(img, G['mask0'].cuda(), [1, 2])
        elif t == 6:
            p = core.step(img, G['mask6'].cuda(), [7])
        else:
            p = core.step(img, end=(t == T - 1))
        d = (p.float().cpu() - G[f'prob_{t:02d}'])
        per.append(float(d.abs().max()))
        worst = max(worst, per[-1])
        sq += float(d.pow(2).sum())
        n += d.numel()
    print(f'{tag:46s} max {worst:.3e}  rms {(sq / n) ** 0.5:.3e}  per-frame max ' + ' '.join(f'{e * 1e4:.1f}' for e in per), flush=True)


if __name__ == '__main__':
    plans = [(a, None if a == 'fast' else a) for a in sys.argv[1:]] or DEFAULT_PLANS
    for tag, plan in plans:
        try:
            run(tag, plan)
        except Exception as exc:
            print(f'{tag:46s} FAILED {type(exc).__name__}: {exc}', flush=True)
