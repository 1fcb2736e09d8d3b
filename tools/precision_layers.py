"""CPU study (test infrastructure, uses oracle/): per-layer sensitivity of the golden clip's probabilities to fp16
rounding of one conv's weights ('w') or of its input activations ('x').  Errors from independent roundings add in
quadrature, so `only layer L rounded` gives L's share of the error budget directly; the table ranks where a second MMA
pass (hi/lo weights) or a hi/lo activation operand buys the most.

  python tools/precision_layers.py scan            # one run per (layer, w|x)
  python tools/precision_layers.py plan a,b,c ...  # evaluate a named configuration
"""
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tracking-anything-with-deva_b200'))
from oracle import fixtures  # noqa: E402
from oracle import memory_math as mm  # noqa: E402
from oracle import network as net  # noqa: E402
from oracle.core import CoreOracle  # noqa: E402
from deva.model.param_spec import synthetic_state_dict  # noqa: E402

torch.set_grad_enabled(False)


def rh(x):
    return x.half().float()


# name -> set of {'w','x'}: what is rounded to fp16 for this conv.  '*' entry = default.
SPEC = {'*': set()}
SEEN = []
STATE = dict(sensory=False, values=False, readout=False, aff=False)


def spec_of(name):
    for k, v in SPEC.items():
        if k != '*' and name.startswith(k):
            return v
    return SPEC['*']


def conv(sd, name, x, stride=1, pad=0):
    if name not in SEEN:
        SEEN.append(name)
    s = spec_of(name)
    w = sd[name + '.weight']
    if 'w' in s:
        w = rh(w)
    if 'x' in s:
        x = rh(x)
    return F.conv2d(x, w, sd.get(name + '.bias'), stride=stride, padding=pad)


net._conv = conv
orig_gru, orig_encode_mask, orig_readout = net._gru, net.encode_mask, mm.readout


def gru(values, h, dim):
    if STATE['sensory']:
        return rh(orig_gru(values, rh(h), dim))
    return orig_gru(values, h, dim)


def encode_mask(*a, **k):
    v, s = orig_encode_mask(*a, **k)
    return (rh(v) if STATE['values'] else v), s


def readout(aff, mv):
    if STATE['aff']:
        aff = rh(aff)
    if STATE['values']:
        mv = rh(mv)
    out = orig_readout(aff, mv)
    return rh(out) if STATE['readout'] else out


net._gru = gru
net.encode_mask = encode_mask
mm.readout = readout

_ARRAYS, META = fixtures.vos_steps()
G = {k: torch.from_numpy(v) for k, v in _ARRAYS.items()}
SD = synthetic_state_dict(seed=1)
REF = None


def replay():
    np.random.seed(42)
    core = CoreOracle(SD, META['config'])
    T = G['frames'].shape[0]
    out = []
    for t in range(T):
        if t == 0:
            p = core.step(G['frames'][t], G['mask0'], [1, 2])
        elif t == 6:
            p = core.step(G['frames'][t], G['mask6'], [7])
        else:
            p = core.step(G['frames'][t], end=(t == T - 1))
        out.append(p.clone())
    return out


def run(tag):
    global REF
    out = replay()
    if REF is None:
        REF = out
        return
    worst = max(float((a - b).abs().max()) for a, b in zip(out, REF))
    sq = sum(float((a - b).pow(2).sum()) for a, b in zip(out, REF))
    n = sum(a.numel() for a in out)
    rms = (sq / n) ** 0.5
    print(f'{tag:58s} max {worst:.3e}  rms {rms:.3e}', flush=True)
    return worst, rms


NATIVE_PREFIXES = ('mask_encoder', 'mask_decoder')

if __name__ == '__main__':
    run('ref')  # fp32 oracle itself is the reference (isolates rounding from the fixture's 2e-5 noise)
    mode = sys.argv[1] if len(sys.argv) > 1 else 'scan'
    if mode == 'scan':
        names = [n for n in SEEN if n.startswith(NATIVE_PREFIXES) and not n.endswith('.pred')]
        SPEC.clear(); SPEC['*'] = set()
        for n in NATIVE_PREFIXES:
            SPEC[n] = {'w', 'x'}
        SPEC['mask_decoder.pred'] = set()
        run('all native layers w+x (states exact)')
        for what in ('w', 'x'):
            for n in names:
                SPEC.clear(); SPEC['*'] = set(); SPEC[n] = {what}
                run(f'only {what}: {n}')
        for st in STATE:
            SPEC.clear(); SPEC['*'] = set()
            for k in STATE:
                STATE[k] = k == st
            run(f'only state: {st}')
