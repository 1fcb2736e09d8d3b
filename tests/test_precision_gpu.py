"""Kernels of the 'parity' precision plan (DESIGN "precision plan"): the residual stream as fp16 (hi, lo) pairs and the
two-pass convolution modes that remove either the activation-operand or the weight rounding."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


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


def _nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous()


def _nchw(x):
    return x.float().permute(0, 3, 1, 2).contiguous()


@pytest.mark.parametrize('with_skip_lo,with_relu_lo', [(False, False), (True, True)])
def test_up2_add_split_matches_torch(with_skip_lo, with_relu_lo):
    ops = _ops()
    g = torch.Generator(device='cuda').manual_seed(2)
    b, h, w, c = 3, 9, 13, 64
    x = torch.randn(b, h, w, c, device='cuda', generator=g) * 3
    skip = torch.randn(1, 2 * h, 2 * w, c, device='cuda', generator=g)
    hi, lo = _split(x)
    s_hi, s_lo = _split(skip)
    raw, raw_lo, relu, relu_lo = ops.up2_add_split(hi, lo, s_hi, s_lo if with_skip_lo else None,
                                                   want_relu_lo=with_relu_lo)
    s_true = s_hi.float() + (s_lo.float() if with_skip_lo else 0)
    ref = F.interpolate((hi.float() + lo.float()).permute(0, 3, 1, 2), scale_factor=2, mode='bilinear',
                        align_corners=False).permute(0, 2, 3, 1) + s_true
    torch.cuda.synchronize()
    assert float((raw.float() + raw_lo.float() - ref).abs().max()) < 2e-5
    if with_relu_lo:
        assert float((relu.float() + relu_lo.float() - ref.clamp_min(0)).abs().max()) < 2e-5
    else:
        assert relu_lo is None and float((relu.float() - ref.clamp_min(0)).abs().max()) < 4e-3


@pytest.mark.parametrize('b,h,w,cin,cout,k', [(2, 14, 18, 128, 256, 3), (5, 72, 121, 256, 256, 3), (3, 20, 33, 512, 512, 1)])
def test_conv_activation_lo_mode(b, h, w, cin, cout, k):
    """split_mode 1: D = Xh.W + Xl.W equals the convolution of the exact activations with the fp16 weights."""
    ops = _ops()
    g = torch.Generator(device='cuda').manual_seed(5 + cin + k)
    x = torch.randn(b, cin, h, w, device='cuda', generator=g)
    wgt = (torch.randn(cout, cin, k, k, device='cuda', generator=g) / (cin * k * k)**0.5).half().float()
    bias = torch.randn(cout, device='cuda', generator=g)
    pc = ops.PackedConv(wgt, bias, 1, act_lo=True)
    xh, xl = _split(_nhwc(x))
    ref = F.conv2d((xh.float() + xl.float()).permute(0, 3, 1, 2).double(), wgt.double(), bias.double(), padding=k // 2).float()
    o = ops.conv_ex(xh, pc, x_lo=xl, want_f32=True, want_relu=True, want_lo=True)
    torch.cuda.synchronize()
    scale = float(ref.abs().max())
    assert float((_nchw(o.f32) - ref).abs().max()) < 2e-5 * scale
    assert float((_nchw(o.relu) + _nchw(o.relu_lo) - ref.clamp_min(0)).abs().max()) < 2e-5 * scale
    # and it matters: the single-pass result on the same inputs is ~2^-11 off
    single = ops.conv_ex(xh, ops.PackedConv(wgt, bias, 1), want_f32=True)
    torch.cuda.synchronize()
    assert float((_nchw(single.f32) - ref).abs().max()) > 10 * float((_nchw(o.f32) - ref).abs().max())


def test_conv_weight_lo_mode_with_rank1_and_residual():
    """split_mode 2 (sensory_compress in the parity plan): D = X.Wh + X.Wl + w1*x1 + res."""
    ops = _ops()
    g = torch.Generator(device='cuda').manual_seed(9)
    b, h, w, cin, cout = 3, 17, 30, 512, 512
    x = torch.randn(b, cin, h, w, device='cuda', generator=g).half().float()
    plane = torch.rand(b, h, w, device='cuda', generator=g)
    wgt = torch.randn(cout, cin + 1, 1, 1, device='cuda', generator=g) / cin**0.5
    bias = torch.randn(cout, device='cuda', generator=g)
    res = torch.randn(b, cout, h, w, device='cuda', generator=g).half()
    pc = ops.PackedConv(wgt, bias, 1, rank1_in=cin, w_lo=True)
    ref = F.conv2d(torch.cat([x, plane.unsqueeze(1)], 1).double(), wgt.double(), bias.double()).float() + res.float()
    o = ops.conv_ex(_nhwc(x).half(), pc, rank1_x=plane.contiguous(), res=_nhwc(res), want_raw=True, want_relu=True,
                    want_lo=True, want_f32=True)
    torch.cuda.synchronize()
    scale = float(ref.abs().max())
    assert float((_nchw(o.f32) - ref).abs().max()) < 2e-5 * scale
    assert float((_nchw(o.raw) + _nchw(o.raw_lo) - ref).abs().max()) < 2e-5 * scale


def test_fast_plan_is_still_available(golden_dir, synthetic_sd, monkeypatch):
    """DEVA_B200_PRECISION=fast: single fp16 operands everywhere (the round-1 stack) stays within 2.5e-3."""
    import numpy as np
    from deva.inference.inference_core import DEVAInferenceCore
    from deva.model.network import DEVA
    from oracle import fixtures
    monkeypatch.setenv('DEVA_B200_PRECISION', 'fast')
    arrays, meta = fixtures.vos_steps(golden_dir)
    g = {k: torch.from_numpy(v) for k, v in arrays.items()}
    np.random.seed(42)
    net = DEVA(meta['config'])
    net.conv_backend = 'native'
    net = net.cuda().eval()
    net.load_weights({k: v.cuda() for k, v in synthetic_sd.items()})
    core = DEVAInferenceCore(net, meta['config'])
    assert net.engine.precision == 'fast'
    T, worst = g['frames'].shape[0], 0.0
    for t in range(T):
        img = g['frames'][t].cuda()
        if t == 0:
            p = core.step(img, g['mask0'].cuda(), [1, 2])
        elif t == 6:
            p = core.step(img, g['mask6'].cuda(), [7])
        else:
            p = core.step(img, end=(t == T - 1))
        worst = max(worst, float((p.cpu() - g[f'prob_{t:02d}']).abs().max()))
    print('fast plan: max |prob - reference| =', worst)
    assert worst < 2.5e-3, worst


@pytest.mark.parametrize('ksplit', [1, 4, 8])
def test_conv_split_k_partial_sums(ksplit):
    """ksplit: the K loop runs as short accumulation chains whose fp32 partial sums the consumer adds - the result
    must equal the convolution (and, for a deep split-precision K loop, be closer to fp64 than one long chain: the tensor
    core's accumulator rounds toward zero at every step)."""
    ops = _ops()
    g = torch.Generator(device='cuda').manual_seed(31)
    b, h, w, cin, cout, k = 1, 30, 43, 512, 129, 3   # the key projection's shape: ragged Cout, one channel tile
    x = torch.randn(b, cin, h, w, device='cuda', generator=g)
    wgt = torch.randn(cout, cin, k, k, device='cuda', generator=g) / (cin * k * k)**0.5
    bias = torch.randn(cout, device='cuda', generator=g)
    pc = ops.PackedConv(wgt, bias, 1, precise=True)
    xh, xl = _split(_nhwc(x))
    ref = F.conv2d(x.double(), wgt.double(), bias.double(), padding=1)
    o = ops.conv_ex(xh, pc, x_lo=xl, want_f32=True, ksplit=ksplit)
    torch.cuda.synchronize()
    parts = o.f32 if ksplit > 1 else o.f32.unsqueeze(0)
    assert parts.shape[0] == max(ksplit, 1)
    got = parts.double().sum(0).permute(0, 3, 1, 2)
    scale = float(ref.abs().max())
    err = float((got - ref).abs().max()) / scale
    print(f'split-K {ksplit}: max rel err {err:.2e}')
    assert err < (5e-5 if ksplit == 1 else 5e-6), err  # one chain: the accumulator's round-toward-zero shows


def _e4m3_bytes(x):
    return x.to(torch.float8_e4m3fn).view(torch.uint8)


def _from_e4m3(b):
    return b.view(torch.float8_e4m3fn).float()


@pytest.mark.parametrize('b,h,w,cin,cout,k', [(2, 14, 18, 128, 256, 3), (5, 72, 121, 256, 256, 3), (3, 20, 33, 256, 128, 1)])
def test_conv_fp8_correction_mode(b, h, w, cin, cout, k):
    """split_mode 3: D = (Xh.W16 + Xlo8.W8) * 2^-S on mixed kind::f16 / kind::f8f6f4 MMAs into one accumulator.  Checked
    (a) against the same quantised operands in fp64 (the kernel adds nothing to their error) and (b) against the exact
    activations: the e4m3 correction pass must remove most of the single-pass operand rounding."""
    ops = _ops()
    g = torch.Generator(device='cuda').manual_seed(7 + cin + k)
    x = torch.randn(b, cin, h, w, device='cuda', generator=g).relu() * 2
    wgt = (torch.randn(cout, cin, k, k, device='cuda', generator=g) / (cin * k * k)**0.5).half().float()
    bias = torch.randn(cout, device='cuda', generator=g)
    pc = ops.PackedConv(wgt, bias, 1, act_lo8=True)
    xn = _nhwc(x)
    xh = xn.half()
    lo8 = _e4m3_bytes((xn - xh.float()) * 4096.0).contiguous()
    w16 = pc.w_packed.float().view(pc.cout_pad, k, k, pc.cin_pad)[:cout, :, :, :cin].permute(0, 3, 1, 2).double()
    w8 = _from_e4m3(pc.w8_packed).view(pc.cout_pad, k, k, pc.cin_pad)[:cout, :, :, :cin].permute(0, 3, 1, 2).double()
    quant = (F.conv2d(xh.double().permute(0, 3, 1, 2), w16, padding=k // 2) +
             F.conv2d(_from_e4m3(lo8).double().permute(0, 3, 1, 2), w8, padding=k // 2)) * pc.acc_scale + bias.double().view(1, -1, 1, 1)
    exact = F.conv2d(x.double(), wgt.double(), bias.double(), padding=k // 2)
    o = ops.conv_ex(xh, pc, x_lo8=lo8, want_f32=True, want_relu=True, want_relu_lo8=True)
    single = ops.conv_ex(xh, ops.PackedConv(wgt, bias, 1), want_f32=True)
    torch.cuda.synchronize()
    scale = float(exact.abs().max())
    e_quant = float((_nchw(o.f32).double() - quant).abs().max()) / scale
    e_exact = float((_nchw(o.f32).double() - exact).abs().max()) / scale
    e_single = float((_nchw(single.f32).double() - exact).abs().max()) / scale
    print(f'fp8 correction: vs quantised operands {e_quant:.2e}, vs exact {e_exact:.2e}, single pass vs exact {e_single:.2e}')
    assert e_quant < 2e-5, e_quant
    assert e_exact < 0.25 * e_single, (e_exact, e_single)
    # the e4m3 remainder of the ReLU'd output, as the next layer's low-order operand
    want = _nchw(o.f32).clamp_min(0)
    rem = (want - want.half().float()) * 4096.0
    got = _from_e4m3(o.relu_lo8).permute(0, 3, 1, 2)
    assert float((got - rem).abs().max()) <= 0.07 * float(rem.abs().max()) + 2 ** -9  # 3-bit mantissa: <= 6.25 % + subnormal step


def test_up2_add_split_e4m3_remainder():
    ops = _ops()
    g = torch.Generator(device='cuda').manual_seed(12)
    b, h, w, c = 2, 11, 17, 128
    x = torch.randn(b, h, w, c, device='cuda', generator=g) * 3
    skip = torch.randn(1, 2 * h, 2 * w, c, device='cuda', generator=g)
    hi, lo = _split(x)
    s_hi, s_lo = _split(skip)
    raw, raw_lo, relu, relu_lo8 = ops.up2_add_split(hi, lo, s_hi, s_lo, want_relu_lo8=True)
    ref = F.interpolate((hi.float() + lo.float()).permute(0, 3, 1, 2), scale_factor=2, mode='bilinear',
                        align_corners=False).permute(0, 2, 3, 1) + s_hi.float() + s_lo.float()
    torch.cuda.synchronize()
    assert relu_lo8.dtype == torch.uint8
    want = ref.clamp_min(0)
    assert float((relu.float() - want).abs().max()) < 4e-3
    rem = (want - relu.float()) * 4096.0
    got = _from_e4m3(relu_lo8)
    assert float((got - rem).abs().max()) <= 0.07 * float(rem.abs().max()) + 2 ** -9 + 0.1  # + fp32 interpolation order
    assert float((raw.float() + raw_lo.float() - ref).abs().max()) < 2e-5
