"""Convolution epilogue features on the launch paths the 1080p workloads take them on.

launch_conv (csrc/conv.cu) picks one of three kernels by shape - one CTA per tile, a two-CTA cluster that shares the
weight tile by TMA multicast (shallow K loop), a tcgen05 CTA pair (deep K loop) - and runs split-K chains without
clusters.  Each case below states the path it is meant to take; a mirror of the rule checks the shape still selects it
and the profiler checks the pair / single-CTA kernel really ran.  References are float64 on the operands the kernel
sees; every output lives inside a sentinel-filled buffer whose guard bands are checked bit for bit afterwards.
"""
import math
import os
import re

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

SPLIT_TOL = 2e-5   # split-precision modes: x max|ref| against float64 (as test_precision_gpu.py)
PLAIN_TOL = 1e-2   # single-pass fp16 outputs (as test_conv_gpu.py)
HEAD_TOL = 2e-3    # fused logit head after head_gather3x3, against the two-convolution reference


@pytest.fixture(autouse=True)
def _release_cached_memory():
    """The GPU is shared: hand each test's 1080p-sized buffers back to the device instead of keeping them cached."""
    yield
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------ guard bands
GUARD = 256  # sentinel elements on either side; 256 elements of a 1-, 2- or 4-byte type keep 256-byte alignment
_SENTINEL = {torch.float16: (torch.int16, 0x7E5A), torch.float32: (torch.int32, 0x7FA5A5A5), torch.uint8: (torch.uint8, 0xFF)}


class Guarded:
    """An output tensor inside a larger buffer filled with a NaN bit pattern: elements the kernel never writes stay NaN
    (and fail any value check), stores past either end show up in the guard bands."""

    def __init__(self, shape, dtype):
        self.n = math.prod(shape)
        ity, self.val = _SENTINEL[dtype]
        self.buf = torch.empty(self.n + 2 * GUARD, dtype=dtype, device='cuda')
        self.buf.view(ity).fill_(self.val)
        self.ity = ity
        self.t = self.buf[GUARD:GUARD + self.n].view(shape)

    def check(self, what):
        bits = self.buf.view(self.ity)
        assert bool((bits[:GUARD] == self.val).all()), f'{what}: store before the tensor'
        assert bool((bits[GUARD + self.n:] == self.val).all()), f'{what}: store past the tensor'


def _err(got, want):
    e = float((got.double() - want).abs().max())
    return math.inf if math.isnan(e) else e


# ------------------------------------------------------------------------------------------ launch-path mirror
def launch_path(b, ho, wo, cout_pad, nt, taps, cin_pad, head, ksplit, sms):
    """Mirror of the kernel choice in launch_conv: 'single' (one CTA per tile), 'multicast' (two-CTA cluster sharing the
    weight tile), 'pair' (tcgen05 cta_group::2) or 'splitk' (fp32 partial sums, one CTA per unit).  `taps` counts the
    filter taps of every MMA pass (x3 for `precise`, x2 for two-pass modes, +k*k for the fp8 correction pass)."""
    from deva.model.native_ops import choose_tile
    if ksplit > 1:
        return 'splitk'
    th, tw = choose_tile(ho, wo)
    tiles = b * -(-ho // th) * -(-wo // tw) * (cout_pad // nt)
    max_cs = int(os.environ.get('DEVA_B200_CONV_CLUSTER', 2))
    cs, c = 1, max_cs
    while c >= 2:
        if c in (2, 4) and (nt // c) % 8 == 0 and tiles >= 2 * sms and sms % c == 0:
            cs = c
            break
        c >>= 1
    pair = (int(os.environ.get('DEVA_B200_CONV_PAIR', 1)) != 0 and cs >= 2 and (nt // 2) % 16 == 0
            and taps * (cin_pad // 64) >= 16 and (not head or int(os.environ.get('DEVA_B200_CONV_PAIR_HEAD', 1)) != 0))
    return 'pair' if pair else ('multicast' if cs > 1 else 'single')


def _taps(pc):
    kk = pc.k * pc.k
    passes = 3 if pc.precise else (2 if (pc.act_lo or pc.w_lo or pc.two_inputs) else 1)
    return kk * passes + (kk if pc.act_lo8 else 0)


def _k_iters(pc):
    return _taps(pc) * (pc.cin_pad // 64)


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _path_of(pc, b, h, w, head=False, ksplit=0):
    ho, wo = pc.out_hw(h, w)
    return launch_path(b, ho, wo, pc.cout_pad, pc.nt, _taps(pc), pc.cin_pad, head, ksplit, _sms())


def _tiles(pc, b, h, w):
    from deva.model.native_ops import choose_tile
    ho, wo = pc.out_hw(h, w)
    th, tw = choose_tile(ho, wo)
    return b * -(-ho // th) * -(-wo // tw)


def _kernels_of(fn):
    """Runs fn under the profiler -> (its result, names of the CUDA kernels it launched)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, [e.name for e in prof.events()]


def _assert_ran(names, path, head):
    """The conv kernel that ran has the template arguments of `path`: conv_kernel<PAIR, EPI>."""
    got = {m.groups() for m in (re.search(r'conv_kernel<(true|false), (\d)>', n) for n in names) if m}
    want = ('true' if path == 'pair' else 'false', '1' if head else '0')
    assert got == {want}, (path, head, got, sorted(set(names))[:20])


# ------------------------------------------------------------------------------------------ operands and references
def _ops():
    from deva import _native
    from deva.model import native_ops
    _native.require_device()
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return native_ops


def _split(x):
    hi = x.half()
    return hi, (x - hi.float()).half()


def conv64(x, wgt, bias=None):
    """Stride-1 'same' convolution in float64: x NHWC [B,H,W,Cin], wgt [Cout,Cin,k,k] -> NHWC [B,H,W,Cout] float64.
    One image and one tap at a time (a DGEMM each), so a 1080p layer fits in a few hundred MB."""
    b, h, w, _ = x.shape
    cout, _, k, _ = wgt.shape
    p = k // 2
    wt = wgt.double()
    out = torch.empty(b, h, w, cout, dtype=torch.float64, device=x.device)
    for i in range(b):
        xp = F.pad(x[i].double(), (0, 0, p, p, p, p))
        acc = torch.zeros(h, w, cout, dtype=torch.float64, device=x.device)
        for ky in range(k):
            for kx in range(k):
                acc += xp[ky:ky + h, kx:kx + w] @ wt[:, :, ky, kx].t()
        if bias is not None:
            acc += bias.double()
        out[i] = acc
    return out


def _run(pc, x, *, outs, x_lo=None, x_lo8=None, res=None, res_lo=None, rank1_x=None, head_w=None, ksplit=0, nparts=1):
    """nat.conv2d (the call conv_ex makes) with every requested output guard-banded -> {name: Guarded}."""
    from deva import _native as nat
    from deva.model.native_ops import choose_tile
    b, h, w, _ = x.shape
    ho, wo = pc.out_hw(h, w)
    th, tw = choose_tile(ho, wo)
    shape = (b, ho, wo, pc.cout)
    o = {}
    for name in outs:
        dtype = {'f32': torch.float32, 'relu_lo8': torch.uint8}.get(name, torch.float16)
        o[name] = Guarded(((nparts,) if name == 'f32' and ksplit > 1 else ()) + shape, dtype)
    if head_w is not None:
        o['head'] = Guarded((b, ho, wo, head_w.shape[0]), torch.float32)
    t = lambda n: o[n].t if n in o else None  # noqa: E731
    nat.conv2d(x, b, h, w, pc.cin_pad, pc.w_packed, pc.k, pc.stride, pc.cout, pc.cout_pad, pc.nt, th, tw, pc.bias,
               x_lo=x_lo, res=res, res_lo=res_lo, res_broadcast=res is not None and res.shape[0] == 1 and b > 1,
               rank1_w=pc.rank1_w, rank1_x=rank1_x, out_raw=t('raw'), out_relu=t('relu'), out_f32=t('f32'),
               out_raw_lo=t('raw_lo'), out_relu_lo=t('relu_lo'), head_w=head_w, head_out=t('head'),
               head_n=0 if head_w is None else head_w.shape[0], split_mode=pc.split_mode, ksplit=ksplit, x_lo8=x_lo8,
               w8_packed=pc.w8_packed, acc_scale=pc.acc_scale, out_relu_lo8=t('relu_lo8'))
    return o


def _check_guards(o):
    for name, g in o.items():
        g.check(name)


def _check_split_outputs(o, ref, tol=SPLIT_TOL):
    """(hi, lo) pairs and fp32 against a float64 reference of the pre-activation result."""
    scale = float(ref.abs().max())
    if 'f32' in o:
        assert _err(o['f32'].t, ref) < tol * scale, ('f32', _err(o['f32'].t, ref) / scale)
    if 'raw' in o:
        assert _err(o['raw'].t.double() + o['raw_lo'].t.double(), ref) < tol * scale, 'raw + raw_lo'
    if 'relu' in o:
        assert _err(o['relu'].t.double() + o['relu_lo'].t.double(), ref.clamp_min(0)) < tol * scale, 'relu + relu_lo'


def _rand(g, *shape, scale=1.0):
    return torch.randn(*shape, device='cuda', generator=g) * scale


# ------------------------------------------------------------------------------------------ the cases
# name: (feature, b, h, w, cin, cout, k, expected path) - shapes are the 1080p layers (136 x 240 = stride 4, 67/68 x 120 =
# stride 16); b = objects.  Odd tile counts on a pair leave one CTA with a clamped "phantom" tile that must store nothing.
CASES = {
    'head_lo8_odd': ('fused head, act_lo8 + res + res_lo (up_8_4.c2)', 3, 136, 240, 256, 256, 3, 'pair'),
    'head_plain': ('fused head, plain', 2, 136, 240, 256, 256, 3, 'pair'),
    'head_shallow': ('fused head, plain, shallow K', 2, 136, 240, 256, 256, 1, 'multicast'),
    'rank1_wlo_odd': ('rank-1 + w_lo + res (sensory_compress)', 3, 67, 120, 512, 512, 1, 'pair'),
    'precise_pair': ('precise 3-pass, res + res_lo, raw/relu hi+lo', 3, 136, 240, 128, 256, 3, 'pair'),
    'precise_shallow': ('precise 3-pass, res + res_lo, raw/relu hi+lo', 2, 136, 240, 256, 256, 1, 'multicast'),
    'bcast_pair': ('broadcast residual +- res_lo (precise)', 2, 136, 240, 128, 256, 3, 'pair'),
    'bcast_shallow': ('broadcast residual +- res_lo (precise)', 2, 136, 240, 256, 256, 1, 'multicast'),
    'chain_3x3': ('conv_ex chain split -> sum_parts (precise)', 1, 68, 120, 256, 256, 3, 'splitk'),
    'chain_1x1': ('conv_ex chain split -> sum_parts (precise)', 1, 68, 120, 1024, 512, 1, 'splitk'),
}


def _packed(name, g):
    """The PackedConv of a case, with its float32 weights and bias."""
    ops = _ops()
    _, b, h, w, cin, cout, k, _ = CASES[name]
    wgt = _rand(g, cout, cin + (1 if name.startswith('rank1') else 0), k, k, scale=1 / math.sqrt(cin * k * k))
    bias = _rand(g, cout)
    if name.startswith('head_lo8'):
        pc = ops.PackedConv(wgt, bias, 1, act_lo8=True)
    elif name.startswith('head'):
        pc = ops.PackedConv(wgt, bias, 1)
    elif name.startswith('rank1'):
        pc = ops.PackedConv(wgt, bias, 1, rank1_in=cin, w_lo=True)
    else:
        pc = ops.PackedConv(wgt, bias, 1, precise=True)
    return pc, wgt, bias


def _case_path(name, pc):
    _, b, h, w, _, _, _, _ = CASES[name]
    head = name.startswith('head')
    ksplit = -(-_k_iters(pc) // _ops().CHAIN) if name.startswith('chain') else 0
    return _path_of(pc, b, h, w, head=head, ksplit=ksplit)


def test_launch_path_table():
    """Every case still selects the path it was written for; `pytest -s` prints the feature x path table."""
    _ops()
    g = torch.Generator(device='cuda').manual_seed(0)
    rows = []
    for name, (feature, b, h, w, cin, cout, k, want) in CASES.items():
        pc, _, _ = _packed(name, g)
        got = _case_path(name, pc)
        tiles = _tiles(pc, b, h, w)
        rows.append((feature, f'{b}x{h}x{w} {cin}->{cout} k{k}', tiles * (pc.cout_pad // pc.nt), tiles, got, want))
    print(f'\nconv launch paths on {torch.cuda.get_device_name()} ({_sms()} SMs)')
    print(f'{"feature":48s} {"shape":26s} {"tiles":>6s} {"pixel tiles":>11s}  path')
    for feature, shape, tiles, m_tiles, got, want in rows:
        odd = ' (odd)' if got == 'pair' and m_tiles % 2 else ''
        print(f'{feature:48s} {shape:26s} {tiles:6d} {m_tiles:11d}  {got}{odd}')
    assert [r[4] for r in rows] == [r[5] for r in rows]
    by_name = dict(zip(CASES, rows))
    assert by_name['head_lo8_odd'][3] % 2 == 1 and by_name['rank1_wlo_odd'][3] % 2 == 1  # phantom tile on a pair


@pytest.mark.parametrize('name', ['head_lo8_odd', 'head_plain', 'head_shallow'])
def test_fused_head_paths(name):
    """c2 + residual with the fused 9-tap logit head, then head_gather3x3 == pred(relu(c2(x) + res)) as two convolutions.
    head_lo8_odd is the production up_8_4.c2 of the parity plan (fp8 correction pass, residual hi/lo) with 765 pixel
    tiles on CTA pairs."""
    ops = _ops()
    from deva import _native as nat
    _, b, h, w, cin, cout, k, want_path = CASES[name]
    g = torch.Generator(device='cuda').manual_seed(100 + len(name))
    pc, wgt, bias = _packed(name, g)
    assert _case_path(name, pc) == want_path
    pw = _rand(g, 1, cout, 3, 3, scale=3 / math.sqrt(cout * 9))
    pb = 0.3
    head_w = pw[0].permute(1, 2, 0).reshape(9, cout).contiguous()
    lo8 = name.startswith('head_lo8')
    if lo8:
        x = _rand(g, b, h, w, cin, scale=2).relu()   # a ReLU'd activation, as the layer receives it
        xh = x.half()
        x_lo8 = ((x - xh.float()) * 4096.0).to(torch.float8_e4m3fn).view(torch.uint8).contiguous()
        res, res_lo = _split(_rand(g, b, h, w, cout))
    else:
        xh, x_lo8 = _rand(g, b, h, w, cin).half(), None
        res, res_lo = _rand(g, b, h, w, cout).half(), None
    o, names = _kernels_of(lambda: _run(pc, xh, x_lo8=x_lo8, res=res, res_lo=res_lo, head_w=head_w, outs=('raw',)))
    _assert_ran(names, want_path, head=True)
    logits = Guarded((b, h, w, 1), torch.float32)
    nat.head_gather3x3(o['head'].t, logits.t, pb, b, h, w)
    torch.cuda.synchronize()
    _check_guards(o)
    logits.check('logits')
    if lo8:  # the quantised operands: fp16(x) . fp16(W * 2^S) + e4m3 remainder . e4m3(W * 2^(S-12)), scaled by 2^-S
        w16 = pc.w_packed.float().view(pc.cout_pad, k, k, pc.cin_pad)[:cout, :, :, :cin].permute(0, 3, 1, 2)
        w8 = pc.w8_packed.view(torch.float8_e4m3fn).float().view(pc.cout_pad, k, k, pc.cin_pad)[:cout, :, :, :cin].permute(0, 3, 1, 2)
        p4 = conv64(xh, w16) + conv64(x_lo8.view(torch.float8_e4m3fn).float(), w8)
        p4 = p4 * pc.acc_scale + bias.double() + res.double() + res_lo.double()
        # fp16 output of a ~fp32 result: at most half an fp16 ulp from the reference
        bound = p4.abs() * 2.0 ** -11 + SPLIT_TOL * float(p4.abs().max())
        assert bool(((o['raw'].t.double() - p4).abs() <= bound).all()), 'raw vs quantised operands'
    else:
        p4 = conv64(xh, wgt.half()) + bias.double() + res.double()
        assert _err(o['raw'].t, p4) < PLAIN_TOL
    # the nine per-tap dot products, then the gathered logits
    z = torch.empty(b, h, w, 9, dtype=torch.float64, device='cuda')
    for i in range(b):
        z[i] = p4[i].clamp_min(0) @ head_w.double().t()
    assert _err(o['head'].t, z) < HEAD_TOL
    ref = conv64(p4.clamp_min(0), pw) + pb
    assert _err(logits.t, ref) < HEAD_TOL


def test_rank1_weight_lo_paths():
    """sensory_compress of the parity plan: X.Wh + X.Wl + w1 * x1 + res on CTA pairs with an odd pixel-tile count,
    written as raw and ReLU'd (hi, lo) pairs."""
    _ops()
    name = 'rank1_wlo_odd'
    _, b, h, w, cin, cout, k, want_path = CASES[name]
    g = torch.Generator(device='cuda').manual_seed(7)
    pc, wgt, bias = _packed(name, g)
    assert _case_path(name, pc) == want_path
    xh = _rand(g, b, h, w, cin).half()
    plane = torch.rand(b, h, w, device='cuda', generator=g)
    res = _rand(g, b, h, w, cout).half()
    o, names = _kernels_of(lambda: _run(pc, xh, rank1_x=plane, res=res, outs=('raw', 'raw_lo', 'relu', 'relu_lo')))
    _assert_ran(names, want_path, head=False)
    torch.cuda.synchronize()
    _check_guards(o)
    ref = conv64(torch.cat([xh.double(), plane.double().unsqueeze(-1)], -1), wgt, bias) + res.double()
    _check_split_outputs(o, ref)


@pytest.mark.parametrize('name', ['precise_pair', 'precise_shallow'])
def test_precise_epilogue_paths(name):
    """Three-pass split precision with residual (hi, lo) and every output the epilogue can write."""
    _ops()
    _, b, h, w, cin, cout, k, want_path = CASES[name]
    g = torch.Generator(device='cuda').manual_seed(11 + k)
    pc, wgt, bias = _packed(name, g)
    assert _case_path(name, pc) == want_path
    x = _rand(g, b, h, w, cin)
    xh, xl = _split(x)
    r = _rand(g, b, h, w, cout)
    rh, rl = _split(r)
    o, names = _kernels_of(lambda: _run(pc, xh, x_lo=xl, res=rh, res_lo=rl, outs=('raw', 'raw_lo', 'relu', 'relu_lo', 'f32')))
    _assert_ran(names, want_path, head=False)
    torch.cuda.synchronize()
    _check_guards(o)
    ref = conv64(x, wgt, bias) + rh.double() + rl.double()
    _check_split_outputs(o, ref)


@pytest.mark.parametrize('with_lo', [False, True])
@pytest.mark.parametrize('name', ['bcast_pair', 'bcast_shallow'])
def test_broadcast_residual_paths(name, with_lo):
    """One residual image added to every image of the batch (res_batch_stride 0), with and without its low part."""
    _ops()
    _, b, h, w, cin, cout, k, want_path = CASES[name]
    g = torch.Generator(device='cuda').manual_seed(13 + k)
    pc, wgt, bias = _packed(name, g)
    assert _case_path(name, pc) == want_path
    x = _rand(g, b, h, w, cin)
    xh, xl = _split(x)
    rh, rl = _split(_rand(g, 1, h, w, cout))
    rl = rl if with_lo else None
    o, names = _kernels_of(lambda: _run(pc, xh, x_lo=xl, res=rh, res_lo=rl, outs=('raw', 'raw_lo', 'f32')))
    _assert_ran(names, want_path, head=False)
    torch.cuda.synchronize()
    _check_guards(o)
    ref = conv64(x, wgt, bias) + rh.double() + (rl.double() if with_lo else 0)
    _check_split_outputs(o, ref)


@pytest.mark.parametrize('name', ['chain_3x3', 'chain_1x1'])
def test_conv_ex_chain_split(name, monkeypatch):
    """A deep split-precision K loop without want_f32: conv_ex runs it as chains of <= CHAIN k-iterations (split-K
    partial sums) and sum_parts adds them with the bias, the residual and the output conversions.  Checked directly
    (guard-banded partial sums and outputs) and through conv_ex, which must take that route and give the same bits."""
    ops = _ops()
    from deva import _native as nat
    _, b, h, w, cin, cout, k, want_path = CASES[name]
    g = torch.Generator(device='cuda').manual_seed(17 + k)
    pc, wgt, bias = _packed(name, g)
    nparts = -(-_k_iters(pc) // ops.CHAIN)
    assert _k_iters(pc) > ops.MAX_CHAIN and nparts > 1 and _case_path(name, pc) == want_path
    x = _rand(g, b, h, w, cin)
    xh, xl = _split(x)
    conv_ref = conv64(x, wgt, bias)
    parts, names = _kernels_of(lambda: _run(pc, xh, x_lo=xl, outs=('f32',), ksplit=nparts, nparts=nparts))
    _assert_ran(names, want_path, head=False)
    torch.cuda.synchronize()
    _check_guards(parts)
    pt = parts['f32'].t
    scale = float(conv_ref.abs().max())
    assert _err(pt.double().sum(0), conv_ref) < SPLIT_TOL * scale
    spy = []
    real_sum_parts = nat.sum_parts

    def sum_parts(*a, **kw):
        spy.append(a[1])
        return real_sum_parts(*a, **kw)

    monkeypatch.setattr(nat, 'sum_parts', sum_parts)
    r = _rand(g, b, h, w, cout)
    for res, res_lo in ((None, None), _split(r)):
        outs = {n: Guarded(tuple(pt.shape[1:]), torch.float16) for n in ('raw', 'raw_lo', 'relu', 'relu_lo')}
        real_sum_parts(pt, nparts, pt[0].numel(), pt[0].numel(), res=res, res_lo=res_lo,
                       **{n: gd.t for n, gd in outs.items()})
        spy.clear()
        o = ops.conv_ex(xh, pc, x_lo=xl, res=res, res_lo=res_lo, want_raw=True, want_relu=True, want_lo=True)
        torch.cuda.synchronize()
        assert spy == [nparts] and o.f32 is None
        _check_guards(outs)
        ref = conv_ref + (0 if res is None else res.double() + res_lo.double())
        _check_split_outputs(outs, ref)
        for n in outs:
            assert torch.equal(getattr(o, n), outs[n].t), n
