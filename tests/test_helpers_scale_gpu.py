"""Helper and bank kernels at the sizes of the 1080p workloads and at their edges.

The elementwise kernels cap their grid at 32 blocks per SM and the bank kernels at 16, so a grid-stride loop only runs
a second iteration past SMs x 32 x 256 work items; every capped case here asserts it is past that point.  References are
float64, or the kernel's own fp32 operation order where the result is claimed bit for bit.  Every output lives inside a
sentinel-filled buffer whose guard bands are checked bit for bit afterwards.
"""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

SPLIT_TOL = 2e-5  # (hi, lo) pairs: x max|ref| against float64


@pytest.fixture(autouse=True)
def _release_cached_memory():
    """The GPU is shared: hand each test's 1080p-sized buffers back to the device instead of keeping them cached."""
    yield
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------ guard bands
GUARD = 256  # sentinel elements on either side; 256 elements of a 1-, 2- or 4-byte type keep 256-byte alignment
_SENTINEL = {torch.float16: (torch.int16, 0x7E5A), torch.float32: (torch.int32, 0x7FA5A5A5), torch.uint8: (torch.uint8, 0xFF),
             torch.int32: (torch.int32, 0x7FA5A5A5)}


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

    def check(self, what=''):
        bits = self.buf.view(self.ity)
        assert bool((bits[:GUARD] == self.val).all()), f'{what}: store before the tensor'
        assert bool((bits[GUARD + self.n:] == self.val).all()), f'{what}: store past the tensor'

    def untouched(self):
        return bool((self.buf.view(self.ity) == self.val).all())


def _err(got, want):
    e = float((got.double() - want).abs().max())
    return math.inf if math.isnan(e) else e


def _within_half_ulp(got16, ref, scale):
    """An fp16 output of a ~fp32 result: at most half an fp16 ulp (plus a float32-arithmetic allowance) from float64."""
    return bool(((got16.double() - ref).abs() <= ref.abs() * 2.0 ** -11 + SPLIT_TOL * scale).all())


def _nat():
    from deva import _native
    _native.require_device()
    return _native


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _past_cap(work_items):
    """More grid-stride work items than the largest capped grid (32 blocks x 256 threads per SM) covers at once."""
    cap = _sms() * 32 * 256
    assert work_items > cap, (work_items, cap)


def _split(x):
    hi = x.half()
    return hi, (x - hi.float()).half()


def _rand(g, *shape, scale=1.0):
    return torch.randn(*shape, device='cuda', generator=g) * scale


def _nchw(x):
    return x.permute(0, 3, 1, 2)


def _nhwc(x):
    return x.permute(0, 2, 3, 1)


# ------------------------------------------------------------------------------------------ output tail
@pytest.mark.parametrize('with_logits', [False, True])
@pytest.mark.parametrize('k,h,w', [(1, 20, 36), (31, 20, 36), (32, 20, 36), (40, 20, 36), (16, 68, 120)])
def test_output_tail(k, h, w, with_logits):
    """Soft aggregation + bilinear x4 + softmax.  K + 1 <= 32 keeps the logits in registers; K >= 32 stashes them in
    `prob` and normalises in a third pass.  The last case is the 1080p stride-4 map (272 x 480)."""
    nat = _nat()
    g = torch.Generator(device='cuda').manual_seed(k * 100 + h)
    # |logit| <= 6: the kernel's fp32 log-odds of a sigmoid lose ~eps / (1 - p) to cancellation, under 3e-5 here
    logits = (_rand(g, k, h, w) * 2).clamp(-6, 6)
    agg = Guarded((k + 1, h, w), torch.float32)
    prob = Guarded((k + 1, 4 * h, 4 * w), torch.float32)
    lo = Guarded((k + 1, 4 * h, 4 * w), torch.float32) if with_logits else None
    nat.output_tail(logits, agg.t, prob.t, lo.t if with_logits else None, k, h, w)
    torch.cuda.synchronize()
    pr = torch.sigmoid(logits.double())
    full = torch.cat([torch.prod(1 - pr, 0, keepdim=True), pr], 0).clamp(1e-7, 1 - 1e-7)
    ref_agg = torch.log(full / (1 - full))
    ref_l = F.interpolate(ref_agg.unsqueeze(0), scale_factor=4, mode='bilinear', align_corners=False)[0]
    for gd, name in ((agg, 'agg'), (prob, 'prob'), (lo, 'logits')):
        if gd is not None:
            gd.check(name)
    assert _err(agg.t, ref_agg) < 1e-4
    assert _err(prob.t, torch.softmax(ref_l, 0)) < 1e-5
    if with_logits:
        assert _err(lo.t, ref_l) < 1e-4


# ------------------------------------------------------------------------------------------ CBAM
def _cbam_params(g, c, r):
    return dict(w1=_rand(g, r, c, scale=1 / c**0.5), b1=_rand(g, r, scale=0.1), w2=_rand(g, c, r, scale=1 / r**0.5),
                b2=_rand(g, c, scale=0.1), ws=_rand(g, 98, scale=0.1), bs=_rand(g, 1, scale=0.1))


def _cbam_ref(x_pool, x_val, p, i):
    """float64 x + CBAM(x) of image i: channel gate and spatial statistics from x_pool, applied to x_val."""
    d = {k: v.double() for k, v in p.items()}
    xp, xv = x_pool[i].double(), x_val[i].double()
    h, w, c = xp.shape

    def mlp(v):
        return F.relu(v @ d['w1'].t() + d['b1']) @ d['w2'].t() + d['b2']

    flat = xp.reshape(h * w, c)
    gate = torch.sigmoid(mlp(flat.mean(0)) + mlp(flat.amax(0)))
    xg = xp * gate
    stats = torch.stack([xg.amax(-1), xg.mean(-1)]).unsqueeze(0)  # [1, 2, h, w]
    sg = torch.sigmoid(F.conv2d(stats, d['ws'].view(1, 2, 7, 7), d['bs'], padding=3))[0, 0]
    return xv + xv * gate * sg.unsqueeze(-1)


CBAM_SHAPES = [
    (16, 68, 120, 512, 32),  # the 1080p stride-16 fusion: 128 pixels per pooling slice, four pixel lanes
    (2, 5, 9, 512, 32),      # 45 pixels: most of the 64 pooling slices are empty
    (2, 5, 13, 512, 32),     # 65 = 64 + 1 pixels: two per slice, the last slice holds one
    (3, 17, 31, 64, 4),      # C = 64: 32 pixel lanes
    (2, 20, 30, 2048, 128),  # C = 2048: a single pixel lane
]


@pytest.mark.parametrize('variant', ['plain', 'split_pool_lo', 'split_pool_hi'])
@pytest.mark.parametrize('b,h,w,c,r', CBAM_SHAPES)
def test_cbam(b, h, w, c, r, variant):
    """cbam (single fp16 input) and cbam_split (hi/lo input; with pool_lo=False the gate statistics - channel pooling
    and the per-pixel max / mean - come from the hi part only, the residual and the gated product use hi + lo)."""
    nat = _nat()
    from deva.model.native_ops import CBAM_POOL_SPLIT
    g = torch.Generator(device='cuda').manual_seed(b * 7 + c + h)
    # per-channel offsets make the channel means matter to the gate
    x = _rand(g, b, h, w, c) + _rand(g, c, scale=1.5)
    xh, xl = _split(x)
    p = _cbam_params(g, c, r)
    scratch = torch.empty((2 * CBAM_POOL_SPLIT + 1) * b * c + 2 * b * h * w, dtype=torch.float32, device='cuda')
    split = variant != 'plain'
    names = ('raw', 'raw_lo', 'relu', 'relu_lo') if variant == 'split_pool_lo' else (
        ('raw', 'raw_lo', 'relu') if split else ('raw', 'relu'))
    o = {n: Guarded((b, h, w, c), torch.float16) for n in names}
    t = lambda n: o[n].t if n in o else None  # noqa: E731
    if split:
        nat.cbam_split(xh, xl, p['w1'], p['b1'], p['w2'], p['b2'], p['ws'], p['bs'], scratch, t('raw'), t('raw_lo'),
                       t('relu'), b, h, w, c, r, relu_lo=t('relu_lo'), pool_lo=variant == 'split_pool_lo')
    else:
        nat.cbam(xh, p['w1'], p['b1'], p['w2'], p['b2'], p['ws'], p['bs'], scratch, t('raw'), t('relu'), b, h, w, c, r)
    torch.cuda.synchronize()
    for n, gd in o.items():
        gd.check(n)
    x_val = xh.double() + xl.double() if split else xh
    x_pool = x_val if variant == 'split_pool_lo' else xh
    for i in range(b):
        ref = _cbam_ref(x_pool, x_val, p, i)
        scale = float(ref.abs().max())
        if split:
            assert _err(o['raw'].t[i].double() + o['raw_lo'].t[i].double(), ref) < SPLIT_TOL * scale, ('raw', i)
            if 'relu_lo' in o:
                assert _err(o['relu'].t[i].double() + o['relu_lo'].t[i].double(), ref.clamp_min(0)) < SPLIT_TOL * scale
            else:
                assert _within_half_ulp(o['relu'].t[i], ref.clamp_min(0), scale), ('relu', i)
        else:
            assert _within_half_ulp(o['raw'].t[i], ref, scale), ('raw', i)
            assert _within_half_ulp(o['relu'].t[i], ref.clamp_min(0), scale), ('relu', i)


# ------------------------------------------------------------------------------------------ split-K finish
SUM_CASES = [  # n_parts, res, res_lo, raw, raw_lo, relu, relu_lo
    (1, 0, 0, 1, 0, 0, 0),
    (2, 1, 0, 1, 1, 0, 0),
    (3, 1, 1, 0, 0, 1, 1),
    (4, 0, 1, 1, 0, 1, 0),
    (5, 1, 1, 1, 1, 1, 1),
    (5, 0, 0, 0, 0, 1, 0),
]


@pytest.mark.parametrize('n_parts,res,res_lo,raw,raw_lo,relu,relu_lo', SUM_CASES)
def test_sum_parts(n_parts, res, res_lo, raw, raw_lo, relu, relu_lo):
    """sum_p parts[p] (+ res + res_lo) in fixed-order fp32 round-to-nearest adds, as fp16 (hi, lo): bit for bit."""
    nat = _nat()
    g = torch.Generator(device='cuda').manual_seed(n_parts * 64 + res * 2 + relu)
    shape = (1, 136, 240, 320)
    n = math.prod(shape)
    _past_cap(n // 8)
    parts = _rand(g, n_parts, *shape, scale=3)
    rs = _split(_rand(g, *shape))
    ins = dict(res=rs[0] if res else None, res_lo=rs[1] if res_lo else None)
    want = dict(raw=raw, raw_lo=raw and raw_lo, relu=relu, relu_lo=relu and relu_lo)
    o = {k: Guarded(shape, torch.float16) for k, on in want.items() if on}
    nat.sum_parts(parts, n_parts, n, n, **ins, **{k: (o[k].t if k in o else None) for k in want})
    torch.cuda.synchronize()
    v = parts[0].clone()
    for q in range(1, n_parts):
        v += parts[q]
    for k in ('res', 'res_lo'):
        if ins[k] is not None:
            v += ins[k].float()
    for name, val in (('raw', v), ('relu', v.clamp_min(0))):
        if name in o:
            o[name].check(name)
            hi = val.half()
            assert torch.equal(o[name].t, hi), name
            if name + '_lo' in o:
                o[name + '_lo'].check(name + '_lo')
                assert torch.equal(o[name + '_lo'].t, (val - hi.float()).half()), name + '_lo'


@pytest.mark.parametrize('q', [8160, 3 * 8160])
def test_key_tail_parts(q):
    """Key projection tail over 8 split-K partial sums [Q, ld = 129] = [key(64) | d | e(64)]: key bit for bit,
    shrinkage = d^2 + 1 and selection = sigmoid(e) of the fixed-order fp32 sums.  Q = 8160 is one 1080p frame."""
    nat = _nat()
    g = torch.Generator(device='cuda').manual_seed(q)
    ck, ld, n_parts = 64, 129, 8
    if q > 8160:
        _past_cap(q * ck)
    y = _rand(g, n_parts, q, ld)
    key, shr, sel = Guarded((q, ck), torch.float32), Guarded((q,), torch.float32), Guarded((q, ck), torch.float32)
    nat.key_tail(y, ld, q, ck, key.t, shr.t, sel.t, n_parts=n_parts, part_stride=q * ld)
    torch.cuda.synchronize()
    s = y[0].clone()
    for p in range(1, n_parts):
        s += y[p]
    for gd, name in ((key, 'key'), (shr, 'shrinkage'), (sel, 'selection')):
        gd.check(name)
    assert torch.equal(key.t, s[:, :ck])
    torch.testing.assert_close(shr.t.double(), s[:, ck].double()**2 + 1, rtol=1e-6, atol=0)
    torch.testing.assert_close(sel.t.double(), torch.sigmoid(s[:, ck + 1:].double()), rtol=1e-6, atol=1e-12)


# ------------------------------------------------------------------------------------------ x2 upsampling + skip
UP2_SHAPES = [(16, 68, 120, 512), (4, 136, 240, 256), (2, 1, 1, 8), (3, 1, 7, 8), (2, 5, 1, 8)]


def _up2_ref(gv, sv, i):
    """float64 bilinear x2 (align_corners=False) of image i + the broadcast skip image, NHWC."""
    return _nhwc(F.interpolate(_nchw(gv[i:i + 1].double()), scale_factor=2, mode='bilinear', align_corners=False))[0] + sv[0].double()


@pytest.mark.parametrize('variant', ['plain', 'split_relu_lo', 'split_relu_hi', 'split_relu_lo8'])
@pytest.mark.parametrize('b,h,w,c', UP2_SHAPES)
def test_up2_add(b, h, w, c, variant):
    """up2_add (fp16 in, raw / relu fp16 out) and up2_add_split (hi/lo in; raw as hi/lo, relu as hi/lo, hi, or hi + the
    e4m3 remainder operand of an fp8 correction pass)."""
    nat = _nat()
    g = torch.Generator(device='cuda').manual_seed(b + h * 3 + c)
    gh, gl = _split(_rand(g, b, h, w, c, scale=3))
    sh, sl = _split(_rand(g, 1, 2 * h, 2 * w, c))
    out = (b, 2 * h, 2 * w, c)
    if variant == 'plain':
        o = {'raw': Guarded(out, torch.float16), 'relu': Guarded(out, torch.float16)}
        nat.up2_add(gh, sh, o['raw'].t, o['relu'].t, b, h, w, c)
        gv, sv = gh, sh
    else:
        skip_lo = sl if variant != 'split_relu_hi' else None
        o = {n: Guarded(out, torch.float16) for n in ('raw', 'raw_lo', 'relu')}
        if variant == 'split_relu_lo':
            o['relu_lo'] = Guarded(out, torch.float16)
        if variant == 'split_relu_lo8':
            o['relu_lo8'] = Guarded(out, torch.uint8)
        t = lambda n: o[n].t if n in o else None  # noqa: E731
        nat.up2_add_split(gh, gl, sh, t('raw'), t('raw_lo'), t('relu'), b, h, w, c, skip_lo=skip_lo, relu_lo=t('relu_lo'),
                          relu_lo8=t('relu_lo8'))
        gv = gh.double() + gl.double()
        sv = sh.double() + (sl.double() if skip_lo is not None else 0)
    torch.cuda.synchronize()
    for n, gd in o.items():
        gd.check(n)
    for i in range(b):
        ref = _up2_ref(gv, sv, i)
        pos = ref.clamp_min(0)
        scale = float(ref.abs().max())
        if variant == 'plain':
            assert _within_half_ulp(o['raw'].t[i], ref, scale) and _within_half_ulp(o['relu'].t[i], pos, scale), i
            continue
        assert _err(o['raw'].t[i].double() + o['raw_lo'].t[i].double(), ref) < SPLIT_TOL * scale, ('raw', i)
        if 'relu_lo' in o:
            assert _err(o['relu'].t[i].double() + o['relu_lo'].t[i].double(), pos) < SPLIT_TOL * scale, ('relu', i)
            continue
        assert _within_half_ulp(o['relu'].t[i], pos, scale), ('relu', i)
        if 'relu_lo8' in o:
            # e4m3 of (relu - fp16(relu)) * 4096: 3 mantissa bits (<= 6.25 %) + the subnormal step, + the fp32
            # interpolation error scaled by 4096
            rem = (pos - o['relu'].t[i].double()) * 4096.0
            got = o['relu_lo8'].t[i].view(torch.float8_e4m3fn).double()
            bound = 0.0625 * rem.abs() + 2.0 ** -9 + 4096 * 2e-6 * (ref.abs() + 4)
            assert bool(((got - rem).abs() <= bound).all()), ('relu_lo8', i)


# ------------------------------------------------------------------------------------------ pooling / resampling
@pytest.mark.parametrize('with_lo', [False, True])
@pytest.mark.parametrize('b,h,w,c', [(2, 544, 960, 64), (3, 17, 31, 64), (2, 17, 31, 8)])
def test_maxpool(b, h, w, c, with_lo):
    """3x3 / stride 2 / pad 1 max pool of fp16 (or fp16 hi + lo) NHWC: bit for bit.  2 x 544 x 960 x 64 is the 1080p stem."""
    nat = _nat()
    g = torch.Generator(device='cuda').manual_seed(h + c + with_lo)
    xh, xl = _split(_rand(g, b, h, w, c, scale=4))
    ho, wo = (h + 1) // 2, (w + 1) // 2
    if h > 100:
        _past_cap(b * ho * wo * c // 8)
    y = Guarded((b, ho, wo, c), torch.float16)
    y_lo = Guarded((b, ho, wo, c), torch.float16) if with_lo else None
    nat.maxpool(xh, y.t, b, h, w, c, x_lo=xl if with_lo else None, y_lo=y_lo.t if with_lo else None)
    torch.cuda.synchronize()
    y.check('y')
    m = _nhwc(F.max_pool2d(_nchw(xh.float() + (xl.float() if with_lo else 0)), 3, 2, 1))
    assert torch.equal(y.t, m.half())
    if with_lo:
        y_lo.check('y_lo')
        assert torch.equal(y_lo.t, (m - m.half().float()).half())


def _area_sum(x, r):
    """r x r window sums of [..., H, W, (C)] in the kernel's order (row-major over the window, fp32 adds)."""
    acc = None
    for dy in range(r):
        for dx in range(r):
            s = x[:, dy::r, dx::r].float()
            acc = s.clone() if acc is None else acc.add_(s)
    return acc


@pytest.mark.parametrize('b,h,w,c,r', [(8, 136, 240, 256, 2), (8, 272, 480, 256, 4)])
def test_area_down(b, h, w, c, r):
    """r x r average pool of fp16 NHWC (the sensory update's p8 / p4 inputs at 1080p): bit for bit."""
    nat = _nat()
    g = torch.Generator(device='cuda').manual_seed(r)
    x = _rand(g, b, h, w, c).half()
    _past_cap(b * (h // r) * (w // r) * c // 8)
    y = Guarded((b, h // r, w // r, c), torch.float16)
    nat.area_down(x, y.t, b, h, w, c, r)
    torch.cuda.synchronize()
    y.check('y')
    assert torch.equal(y.t, (_area_sum(x, r) * (1.0 / (r * r))).half())


@pytest.mark.parametrize('b,h,w,r', [(40, 544, 960, 4), (160, 1088, 1920, 16)])
def test_area_down_plane(b, h, w, r):
    """r x r average pool of fp32 planes (mask / logit planes down to the stride-16 grid): bit for bit."""
    nat = _nat()
    g = torch.Generator(device='cuda').manual_seed(r + 1)
    x = torch.rand(b, h, w, device='cuda', generator=g)
    _past_cap(b * (h // r) * (w // r))
    y = Guarded((b, h // r, w // r), torch.float32)
    nat.area_down_plane(x, y.t, b, h, w, r)
    torch.cuda.synchronize()
    y.check('y')
    assert torch.equal(y.t, _area_sum(x, r) * (1.0 / (r * r)))


def test_head_gather3x3():
    """logits = bias + sum over the 3 x 3 neighbours of their per-tap head sums (zero padded), 16 objects at 1080p:
    bit for bit against the same fp32 additions in tap order."""
    nat = _nat()
    g = torch.Generator(device='cuda').manual_seed(9)
    b, h, w, bias = 16, 272, 480, -0.375
    _past_cap(b * h * w)
    z = _rand(g, b, h, w, 9)
    out = Guarded((b, h, w, 1), torch.float32)
    nat.head_gather3x3(z, out.t, bias, b, h, w)
    torch.cuda.synchronize()
    out.check('logits')
    zp = F.pad(z, (0, 0, 1, 1, 1, 1))
    a = torch.full((b, h, w), bias, device='cuda')
    for t in range(9):
        a += zp[:, t // 3:t // 3 + h, t % 3:t % 3 + w, t]
    assert torch.equal(out.t[..., 0], a)


# ------------------------------------------------------------------------------------------ layout / im2col / append
def test_layout_converters():
    """fp32 NCHW -> fp16 NHWC with zero channel padding (c_pad > c), and fp16 NHWC -> fp32 NCHW: bit for bit."""
    nat = _nat()
    g = torch.Generator(device='cuda').manual_seed(4)
    b, c, h, w, cp = 4, 100, 136, 240, 104
    _past_cap(b * h * w * cp)
    x = _rand(g, b, c, h, w, scale=10)
    d = Guarded((b, h, w, cp), torch.float16)
    nat.nchw_to_nhwc(x, d.t, b, c, h, w, cp)
    back = Guarded((b, cp, h, w), torch.float32)
    nat.nhwc_to_nchw(d.t, back.t, b, cp, h, w)
    torch.cuda.synchronize()
    d.check('nhwc')
    back.check('nchw')
    assert torch.equal(d.t[..., :c], _nhwc(x).half()) and bool((d.t[..., c:] == 0).all())
    assert torch.equal(back.t, _nchw(d.t).float())


@pytest.mark.parametrize('b,c,with_lo', [(16, 1, False), (1, 3, True)])
def test_stem_columns_1080p(b, c, with_lo):
    """im2col of the 7x7 stride-2 stems at 1088 x 1920 (16 mask planes; the image with its fp16 remainder): bit for bit
    against F.unfold."""
    nat = _nat()
    g = torch.Generator(device='cuda').manual_seed(c)
    h, w = 1088, 1920
    kp = (49 * c + 63) // 64 * 64
    x = _rand(g, b, c, h, w)
    out = Guarded((b, h // 2, w // 2, kp), torch.float16)
    lo = Guarded((b, h // 2, w // 2, kp), torch.float16) if with_lo else None
    nat.stem_im2col(x, out.t, b, c, h, w, kp, dst_lo=lo.t if with_lo else None)
    torch.cuda.synchronize()
    out.check('columns')
    if with_lo:
        lo.check('columns_lo')
    for i in range(b):
        cols = F.unfold(x[i:i + 1], 7, padding=3, stride=2).view(c, 49, h // 2, w // 2)
        ref = torch.zeros(h // 2, w // 2, kp, device='cuda')
        ref[..., :49 * c] = cols.permute(2, 3, 1, 0).reshape(h // 2, w // 2, 49 * c)
        assert torch.equal(out.t[i], ref.half()), i
        if with_lo:
            assert torch.equal(lo.t[i], (ref - ref.half().float()).half()), i


def test_transpose_append_offset():
    """Token-major [n, C] -> bank rows [C, ld] at a column offset (a value append behind 24 stored tokens): exactly the
    n x C block changes."""
    nat = _nat()
    g = torch.Generator(device='cuda').manual_seed(6)
    n, c, off, ld = 8161, 512, 24, 8200
    src = _rand(g, n, c).half()
    bank = Guarded((c, ld), torch.float16)
    nat.transpose_append(src, bank.t[:, off:], ld, n, c)
    torch.cuda.synchronize()
    bank.check('bank')
    assert torch.equal(bank.t[:, off:off + n], src.t())
    bits = bank.t.view(torch.int16)
    assert bool((bits[:, :off] == bank.val).all()) and bool((bits[:, off + n:] == bank.val).all())


# ------------------------------------------------------------------------------------------ bank kernels
@pytest.mark.parametrize('row_bytes', [16, 256, 512])
def test_gather_rows(row_bytes):
    nat = _nat()
    g = torch.Generator(device='cuda').manual_seed(row_bytes)
    vec = row_bytes // 16
    n = 1_500_000 // vec
    _past_cap(n * vec)
    src = torch.randint(-2**31, 2**31 - 1, (n * 2 // 3, row_bytes // 4), dtype=torch.int32, device='cuda', generator=g)
    idx = torch.randint(0, src.shape[0], (n,), dtype=torch.int32, device='cuda', generator=g)  # repeats included
    dst = Guarded((n, row_bytes // 4), torch.int32)
    nat.gather_rows(dst.t, src, idx, n, row_bytes)
    torch.cuda.synchronize()
    dst.check('rows')
    assert torch.equal(dst.t, src[idx.long()])


def test_gather_f32_cols_usage():
    """gather_f32, gather_cols_f16 (the value bank: 512 rows x 8160 columns, both pitched) and usage = use / life."""
    nat = _nat()
    g = torch.Generator(device='cuda').manual_seed(1)
    n = 2_000_000
    src = torch.randn(n // 2, device='cuda', generator=g)
    idx = torch.randint(0, n // 2, (n,), dtype=torch.int32, device='cuda', generator=g)
    dst = Guarded((n,), torch.float32)
    nat.gather_f32(dst.t, src, idx, n)
    rows, cols, ld_src, ld_dst = 512, 8160, 10000, 8192
    _past_cap(rows * cols)
    vals = torch.randn(rows, ld_src, device='cuda', generator=g).half()
    cidx = torch.randint(0, ld_src, (cols,), dtype=torch.int32, device='cuda', generator=g)
    bank = Guarded((rows, ld_dst), torch.float16)
    nat.gather_cols_f16(bank.t, ld_dst, vals, ld_src, cidx, rows, cols)
    use = torch.rand(n, device='cuda', generator=g) * 10
    life = 1 + torch.rand(n, device='cuda', generator=g) * 100
    usage = Guarded((n,), torch.float32)
    nat.usage(usage.t, use, life, n)
    torch.cuda.synchronize()
    for gd, name in ((dst, 'gather_f32'), (bank, 'gather_cols_f16'), (usage, 'usage')):
        gd.check(name)
    assert torch.equal(dst.t, src[idx.long()])
    assert torch.equal(bank.t[:, :cols], vals[:, cidx.long()])
    assert bool((bank.t[:, cols:].view(torch.int16) == bank.val).all())
    assert torch.equal(usage.t, use / life)


def test_bank_kernels_empty():
    """n = 0 launches nothing and leaves every destination untouched."""
    nat = _nat()
    src = torch.zeros(64, 32, dtype=torch.int32, device='cuda')
    idx = torch.zeros(0, dtype=torch.int32, device='cuda')
    rows, f32, cols, use = (Guarded((64, 32), torch.int32), Guarded((64,), torch.float32), Guarded((8, 64), torch.float16),
                            Guarded((64,), torch.float32))
    nat.gather_rows(rows.t, src, idx, 0, 128)
    nat.gather_f32(f32.t, src.view(torch.float32), idx, 0)
    nat.gather_cols_f16(cols.t, 64, src.view(torch.float16), 64, idx, 8, 0)
    nat.usage(use.t, src.view(torch.float32)[0], src.view(torch.float32)[1], 0)
    torch.cuda.synchronize()
    assert rows.untouched() and f32.untouched() and cols.untouched() and use.untouched()
