"""CPU emulation of the native engine's rounding points (test infrastructure, uses oracle/).

The decoder / value encoder of ``deva.model.native_engine`` is restated on the oracle's fp32 ops with an explicit
rounding at every place the kernels store a tensor (fp16, or an fp16 hi/lo pair) and at every MMA operand.  A PLAN says
which tensors travel as hi/lo pairs and which convs consume the lo part of their input in a second MMA pass
(Xh.W + Xl.W).  Replays the golden clip and prints max / rms |prob - fp32 oracle|.

    python tools/precision_plan.py            # the plans listed in PLANS below
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

PLAN = dict(hl=set(), x2=set(), w2=set(), exact=False, w_exact=False)


def h(x):
    return x.half().float()


def hl(x):
    hi = x.half().float()
    return hi + (x - hi).half().float()


def S(name, x):
    """store tensor `name`: fp16, or an fp16 (hi, lo) pair when the plan says so"""
    if PLAN['exact']:
        return x
    for k in PLAN['hl']:
        if name.startswith(k):
            return hl(x)
    return h(x)


def conv(sd, name, x, stride=1, pad=0, tag=None):
    """MMA: operands are fp16 (weights always; activations unless the plan gives this conv a second pass)"""
    w = sd[name + '.weight']
    if not PLAN['exact']:
        if not PLAN['w_exact'] and not any((tag or name).startswith(k) for k in PLAN['w2']):
            w = h(w)
        two = any((tag or name).startswith(k) for k in PLAN['x2'])
        x = hl(x) if two else h(x)
    return F.conv2d(x, w, sd.get(name + '.bias'), stride=stride, padding=pad)


def gconv(sd, name, g, pad=0, tag=None):
    b, k = g.shape[:2]
    y = conv(sd, name, g.flatten(0, 1), pad=pad, tag=tag)
    return y.view(b, k, *y.shape[1:])


def resblock(sd, p, g, t):
    """GroupResBlock as the kernels run it: y = relu(c1(relu g)); short = ds(g) | g; out = c2(y) + short."""
    y = S(t + '.y', F.relu(gconv(sd, p + '.conv1', F.relu(g), pad=1, tag=t + '.c1')))
    if (p + '.downsample.weight') in sd:
        short = S(t + '.short', gconv(sd, p + '.downsample', g, tag=t + '.ds'))
    else:
        short = g
    return S(t + '.out', gconv(sd, p + '.conv2', y, pad=1, tag=t + '.c2') + short)


def fusion(sd, p, x, g, t):
    b, k = g.shape[:2]
    cat = torch.cat([x.unsqueeze(1).expand(-1, k, -1, -1, -1), g], 2)
    # block1 (the shared halves sx / dx are stored in fp16 too; emulated as part of the single rounding of y / short)
    g1 = resblock(sd, p + '.block1', cat, t + '.b1')
    r = net._cbam(sd, p + '.attention', g1.flatten(0, 1)).view_as(g1)
    gr = S(t + '.cbam', g1 + r)
    return resblock(sd, p + '.block2', gr, t + '.b2')


def resize(g, ratio, mode):
    return net._resize_groups(g, ratio, mode)


def segment(sd, ms_features, readout, sensory, last_mask, update_sensory=True):
    p = 'mask_decoder'
    f16, f8, f4 = ms_features
    f16, f8, f4 = S('f16', f16), S('f8', f8), S('f4', f4)
    b, k = readout.shape[:2]
    readout = S('readout', readout)
    sensory = S('sensory', sensory)
    last = F.interpolate(last_mask, size=readout.shape[-2:], mode='area').unsqueeze(2)
    skip8 = S('skip8', conv(sd, p + '.decoder_feat_proc.transforms.0', f8, tag='skipc8'))
    skip4 = S('skip4', conv(sd, p + '.decoder_feat_proc.transforms.1', f4, tag='skipc4'))
    # sensory_compress: the mask channel is a fp32 rank-1 term in the epilogue
    wn = p + '.sensory_compress'
    w = sd[wn + '.weight']
    sc = gconv({wn + '.weight': w[:, :-1], wn + '.bias': sd[wn + '.bias']}, wn, sensory, tag='compress')
    sc = sc + last * w[:, -1].view(1, 1, -1, 1, 1)
    p16 = S('p16in', readout + sc)
    p16 = fusion(sd, p + '.fuser', f16, p16, 'fuser')
    g8 = S('g8', skip8.unsqueeze(1) + resize(p16, 2, 'bilinear'))
    p8 = resblock(sd, p + '.up_16_8.out_conv', g8, 'up168')
    g4 = S('g4', skip4.unsqueeze(1) + resize(p8, 2, 'bilinear'))
    # the last block: p4 stays fp32 inside the epilogue for the logit head, its stored copy is fp16
    pq = p + '.up_8_4.out_conv'
    y = S('up84.y', F.relu(gconv(sd, pq + '.conv1', F.relu(g4), pad=1, tag='up84.c1')))
    p4_full = gconv(sd, pq + '.conv2', y, pad=1, tag='up84.c2') + g4
    logits = net._conv(sd, p + '.pred', F.relu(p4_full.flatten(0, 1)), pad=1)
    p4 = S('p4', p4_full)
    if update_sensory:
        su = p + '.sensory_update'
        g = S('su.g', gconv(sd, su + '.g16_conv', p16, tag='su.g16'))
        g = S('su.g', g + gconv(sd, su + '.g8_conv', S('su.p8d', resize(p8, 1 / 2, 'area')), tag='su.g8'))
        wn = su + '.g4_conv'
        w = sd[wn + '.weight']
        lg = logits.view(b, k, 1, *logits.shape[-2:])
        g4c = gconv({wn + '.weight': w[:, :-1], wn + '.bias': sd[wn + '.bias']}, wn, S('su.p4d', resize(p4, 1 / 4, 'area')),
                    tag='su.g4')
        g4c = g4c + resize(lg, 1 / 4, 'area') * w[:, -1].view(1, 1, -1, 1, 1)
        g = S('su.g', g + g4c)
        vals = gconv(sd, su + '.transform', torch.cat([g, sensory], 2), pad=1, tag='su.gru')
        sensory = S('sensory', net._gru(vals, sensory, sensory.shape[2]))
    logits = logits.view(b, k, *logits.shape[-2:])
    prob = torch.sigmoid(logits)
    logits = net.aggregate(prob, dim=1)
    logits = F.interpolate(logits, scale_factor=4, mode='bilinear', align_corners=False)
    return sensory, logits, F.softmax(logits, dim=1)


def basic_block(sd, p, x, stride, t):
    y = S(t + '.y', F.relu(net._bn(sd, p + '.bn1', conv(sd, p + '.conv1', x, stride=stride, pad=1, tag=t + '.c1'))))
    y = net._bn(sd, p + '.bn2', conv(sd, p + '.conv2', y, pad=1, tag=t + '.c2'))
    if (p + '.downsample.0.weight') in sd:
        x = S(t + '.short', net._bn(sd, p + '.downsample.1', conv(sd, p + '.downsample.0', x, stride=stride, tag=t + '.ds')))
    return S(t + '.out', F.relu(y + x))


def encode_mask(sd, image, ms_features, sensory, masks, deep_update=True):
    p = 'mask_encoder'
    b, k = masks.shape[:2]
    g = torch.cat([image.unsqueeze(1).expand(-1, k, -1, -1, -1), masks.unsqueeze(2)], 2)
    x = g.flatten(0, 1)
    x = net._bn(sd, p + '.bn1', conv(sd, p + '.conv1', x, stride=2, pad=3, tag='me.stem'))
    x = S('me.stem', F.relu(F.max_pool2d(S('me.stem0', x), 3, 2, 1)))
    for li, stride in ((1, 1), (2, 2), (3, 2)):
        for bi in range(2):
            x = basic_block(sd, f'{p}.layer{li}.{bi}', x, stride if bi == 0 else 1, f'me.l{li}.{bi}')
    f16 = S('f16', ms_features[0])
    g16 = fusion(sd, p + '.fuser', f16, x.view(b, k, *x.shape[1:]), 'me.fuser')
    sensory = S('sensory', sensory)
    if deep_update:
        vals = gconv(sd, p + '.sensory_update.transform', torch.cat([g16, sensory], 2), pad=1, tag='me.gru')
        sensory = S('sensory', net._gru(vals, sensory, sensory.shape[2]))
    return S('value', g16), sensory


orig_readout = mm.readout
orig_segment, orig_encode_mask = net.segment, net.encode_mask


def readout(aff, mv):
    # consolidation also routes through here (prototype values); prototype shrinkage is fp32 in the product, and it is
    # the [1, N] operand -> leave 1-row operands alone
    if PLAN['exact'] or mv.shape[0] == 1:
        return orig_readout(aff, mv)
    return orig_readout(h(aff), h(mv))


net.segment = segment
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


def run(tag, **plan):
    global REF
    PLAN.update(hl=set(), x2=set(), w2=set(), exact=False, w_exact=False)
    PLAN.update(plan)
    out = replay()
    if REF is None:
        REF = out
        fix = max(float((a - G[f'prob_{t:02d}']).abs().max()) for t, a in enumerate(out))
        print(f'restated graph in fp32 vs reference fixture: {fix:.2e}')
        return
    worst = max(float((a - b).abs().max()) for a, b in zip(out, REF))
    sq = sum(float((a - b).pow(2).sum()) for a, b in zip(out, REF))
    n = sum(a.numel() for a in out)
    print(f'{tag:70s} max {worst:.3e}  rms {(sq / n) ** 0.5:.3e}', flush=True)


STREAM = {'p16in', 'fuser.b1.short', 'fuser.b1.out', 'fuser.cbam', 'fuser.b2.out', 'g8', 'up168.short', 'up168.out',
          'g4'}

if __name__ == '__main__':
    run('ref', exact=True)
    run('product today (everything fp16)')
    run('weights exact (bound on what hi/lo weights could buy)', w_exact=True)
    run('residual stream hi/lo (DEVA_B200_RESIDUAL_LO=1)', hl=STREAM)
    ds = {'fuser.b1.ds', 'up168.ds'}
    run('stream hi/lo + 2-pass shortcut convs', hl=STREAM, x2=ds)
    run('stream hi/lo + 2-pass shortcuts + up84.c1/c2', hl=STREAM | {'up84.y'}, x2=ds | {'up84.c1', 'up84.c2'})
    run('stream hi/lo + 2-pass shortcuts + up168.c1/c2', hl=STREAM | {'up168.y'}, x2=ds | {'up168.c1', 'up168.c2'})
    run('stream hi/lo + 2-pass all of up168/up84/shortcuts', hl=STREAM | {'up168.y', 'up84.y'},
        x2=ds | {'up168.c1', 'up168.c2', 'up84.c1', 'up84.c2'})
    run('whole decoder hi/lo + 2-pass', hl=STREAM | {'up168', 'up84', 'fuser', 'skip', 'readout', 'su', 'f'},
        x2={'fuser', 'up168', 'up84', 'compress', 'su', 'mask_decoder'})
