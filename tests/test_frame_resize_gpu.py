"""Frames and first-frame palette masks resized to the evaluation size on the device (frame_io.frame_from_rgb8(size=),
frame_io.mask_from_palette), against the reference's own CPU transforms.

Reader mode is compared with VideoReader's im_transform (torchvision ToTensor, Normalize, Resize(bilinear,
antialias=True)) and with the same resize in float64.  torch's fp32 resize is 1.0e-4 (1080p -> 480), 1.5e-4 (720p) and
2.5e-4 (481x853 -> 480x851) away from float64 on normalised noise in [-2.1, 2.7]: its fp32 scale and center move the
taps by up to an fp32 ulp of the source coordinate.  The kernel computes the very same fp32 taps, so it must be no
farther from torch's fp32 result than that result is from float64 (in practice a few fp32 ulps).  Demo mode is
compared with CUDA F.interpolate(bilinear, align_corners=False), masks with Pillow's NEAREST bit for bit.  Every
output lives inside a NaN-patterned buffer whose 256-element guard bands are checked bit for bit.
"""
import functools
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from PIL import Image
from torchvision import transforms
from torchvision.transforms import InterpolationMode

from deva import _native as nat
from deva.inference.frame_io import IMAGENET_MEAN, IMAGENET_STD, frame_from_rgb8, mask_from_palette, prob_to_ids, \
    resized_shape

pytestmark = pytest.mark.gpu

SHAPES = [(1080, 1920), (720, 1280), (481, 853), (1920, 1080), (240, 427), (17, 23), (2160, 3840), (480, 640)]
SIZES = [480, 360, -1]
ULPS = 1e-6  # a few fp32 ulps of the largest normalised value (2.64; one ulp is 2.4e-7)


@pytest.fixture(autouse=True)
def _release_cached_memory():
    yield
    torch.cuda.empty_cache()


GUARD = 256
_SENTINEL = {torch.float32: (torch.int32, 0x7FA5A5A5), torch.int64: (torch.int64, 0x7FF5A5A5A5A5A5A5)}


class Guarded:
    """An output inside a buffer filled with a NaN bit pattern (for int64, a value no label takes): elements never
    written keep it, stores past either end show up in the 256 guard elements."""

    def __init__(self, shape, dtype):
        self.n = math.prod(shape)
        self.ity, self.val = _SENTINEL[dtype]
        self.buf = torch.empty(self.n + 2 * GUARD, dtype=dtype, device='cuda')
        self.buf.view(self.ity).fill_(self.val)
        self.t = self.buf[GUARD:GUARD + self.n].view(shape)

    def check(self, what=''):
        bits = self.buf.view(self.ity)
        assert bool((bits[:GUARD] == self.val).all()), f'{what}: store before the tensor'
        assert bool((bits[GUARD + self.n:] == self.val).all()), f'{what}: store past the tensor'
        assert not bool((bits[GUARD:GUARD + self.n] == self.val).any()), f'{what}: unwritten elements'


def _frame(h, w, seed=0):
    g = torch.Generator().manual_seed(seed * 100003 + h * 7 + w)
    return torch.randint(0, 256, (h, w, 3), generator=g, dtype=torch.uint8)


def _normalised(frame):
    return transforms.Compose([transforms.ToTensor(), transforms.Normalize(IMAGENET_MEAN, IMAGENET_STD)])(frame.numpy())


@functools.lru_cache(maxsize=4)
def _reader_refs(h, w, size):
    """(VideoReader's im_transform on the CPU, the same resize in float64) for the seeded frame."""
    frame = _frame(h, w)
    im_transform = transforms.Compose([transforms.ToTensor(), transforms.Normalize(IMAGENET_MEAN, IMAGENET_STD),
                                       transforms.Resize(size, interpolation=InterpolationMode.BILINEAR,
                                                         antialias=True)])
    ref = im_transform(frame.numpy())
    oh, ow = ref.shape[1:]
    ref64 = F.interpolate(_normalised(frame).double()[None], size=(oh, ow), mode='bilinear', antialias=True,
                          align_corners=False)[0]
    return ref, ref64


def _max_err(a, b):
    e = float((a.double().cpu() - b.double().cpu()).abs().max())
    return math.inf if math.isnan(e) else e


def _resize_guarded(frame_dev, h, w, oh, ow, mode):
    out = Guarded((3, oh, ow), torch.float32)
    ws_bytes = nat.resize_rgb8_workspace_bytes(h, w, oh, ow, mode)
    ws = Guarded((ws_bytes // 4,), torch.float32) if ws_bytes else None
    nat.resize_rgb8(frame_dev, out.t, ws.t if ws else None, h, w, oh, ow, mode, IMAGENET_MEAN, IMAGENET_STD)
    torch.cuda.synchronize()
    out.check(f'resize_rgb8 {mode} {h}x{w}->{oh}x{ow}')
    if ws:
        ws.check('resize_rgb8 workspace')
    return out.t


@pytest.mark.parametrize('size', SIZES)
@pytest.mark.parametrize('h,w', SHAPES)
def test_reader_mode(h, w, size):
    frame = _frame(h, w)
    oh, ow = resized_shape(h, w, size, 'reader')
    got = frame_from_rgb8(frame.cuda(), size=size, mode='reader')
    assert tuple(got.shape) == (3, oh, ow)
    if (oh, ow) == (h, w):  # torchvision returns the frame unresized: the ingest path, bit-exact
        assert torch.equal(got.cpu(), _normalised(frame))
        assert torch.equal(got, frame_from_rgb8(frame.cuda()))
        return
    ref, ref64 = _reader_refs(h, w, size)
    assert torch.equal(_resize_guarded(frame.cuda(), h, w, oh, ow, 'reader'), got)
    err, err64, gap = _max_err(got, ref), _max_err(got, ref64), _max_err(ref, ref64)
    print(f'reader {h}x{w} -> {oh}x{ow}: |gpu - torchvision cpu| {err:.2e}, |gpu - fp64| {err64:.2e}, '
          f'|torchvision cpu - fp64| {gap:.2e}')
    assert err <= max(gap, ULPS), (err, gap)
    assert err64 <= gap + ULPS, (err64, gap)


@pytest.mark.parametrize('size', SIZES)
@pytest.mark.parametrize('h,w', SHAPES)
def test_demo_mode(h, w, size):
    frame = _frame(h, w)
    oh, ow = resized_shape(h, w, size, 'demo')
    got = frame_from_rgb8(frame.cuda(), size=size, mode='demo')
    assert tuple(got.shape) == (3, oh, ow)
    norm = _normalised(frame).cuda()
    if size < 0:
        assert torch.equal(got, norm)
        return
    # get_input_frame_for_deva: /255, normalise, then F.interpolate(bilinear, align_corners=False)
    ref = F.interpolate(norm[None], (oh, ow), mode='bilinear', align_corners=False)[0]
    assert torch.equal(_resize_guarded(frame.cuda(), h, w, oh, ow, 'demo'), got)
    err = _max_err(got, ref)
    print(f'demo {h}x{w} -> {oh}x{ow}: |gpu - F.interpolate cuda| {err:.2e}')
    assert err <= ULPS, err


def _palette_mask(h, w, seed=0):
    """A label map with a few large objects (ids 1, 2, 7, 200) and scattered single pixels of id 9."""
    g = torch.Generator().manual_seed(seed + h * 31 + w)
    yy, xx = torch.meshgrid(torch.arange(h), torch.arange(w), indexing='ij')
    m = torch.zeros(h, w, dtype=torch.uint8)
    for label in (1, 2, 7, 200):
        cy, cx = torch.rand(2, generator=g) * torch.tensor([h, w])
        ry, rx = (0.1 + 0.25 * torch.rand(2, generator=g)) * torch.tensor([h, w])
        m[((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 < 1] = label
    m[torch.rand(h, w, generator=g) < 0.01] = 9
    return m


def _pil_reference(mask, size):
    """VideoReader: Image 'P' -> mask_transform (Resize(size, NEAREST), or nothing for size < 0) -> LongTensor."""
    img = Image.fromarray(mask.numpy(), mode='P')
    if size >= 0:
        img = transforms.Resize(size, interpolation=InterpolationMode.NEAREST)(img)
    ref = torch.LongTensor(np.array(img))
    labels = torch.unique(ref)
    return ref, labels[labels != 0]


@pytest.mark.parametrize('size', SIZES)
@pytest.mark.parametrize('h,w', SHAPES)
def test_mask_nearest(h, w, size):
    mask = _palette_mask(h, w)
    ref, ref_labels = _pil_reference(mask, size)
    got, labels = mask_from_palette(mask.cuda(), size)
    assert got.dtype == torch.long and got.is_cuda
    assert torch.equal(got.cpu(), ref)
    assert torch.equal(labels.cpu(), ref_labels)
    oh, ow = ref.shape
    if (oh, ow) != (h, w):
        from deva.inference.frame_io import pil_nearest_index
        out = Guarded((oh, ow), torch.int64)
        src_y = torch.tensor(pil_nearest_index(h, oh), dtype=torch.int32, device='cuda')
        src_x = torch.tensor(pil_nearest_index(w, ow), dtype=torch.int32, device='cuda')
        nat.resize_labels(mask.cuda(), out.t, h, w, oh, ow, src_y, src_x)
        torch.cuda.synchronize()
        out.check(f'resize_labels {h}x{w}->{oh}x{ow}')
        assert torch.equal(out.t.cpu(), ref)


def _host(t, kind):
    return {'host': lambda: t, 'pinned': lambda: t.pin_memory(), 'device': lambda: t.cuda()}[kind]()


@pytest.mark.parametrize('kind', ['host', 'pinned', 'device'])
def test_inputs_and_streams(kind):
    """Host, pinned and device inputs, on the default and on a side stream, give the same bits."""
    h, w, size = 1080, 1920, 480
    frame, mask = _frame(h, w, seed=1), _palette_mask(h, w, seed=1)
    want = {m: frame_from_rgb8(frame.cuda(), size=size, mode=m) for m in ('reader', 'demo')}
    want_mask, want_labels = mask_from_palette(mask.cuda(), size)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    for stream in (torch.cuda.current_stream(), side):
        with torch.cuda.stream(stream):
            got = {m: frame_from_rgb8(_host(frame, kind), size=size, mode=m) for m in ('reader', 'demo')}
            got_mask, got_labels = mask_from_palette(_host(mask, kind), size)
            ids = got_mask.clone()
        stream.synchronize()
        for m in ('reader', 'demo'):
            assert torch.equal(got[m], want[m]), (kind, m, stream)
        assert torch.equal(got_mask, want_mask) and torch.equal(ids, want_mask)
        assert torch.equal(got_labels, want_labels)


def test_bad_arguments():
    with pytest.raises(RuntimeError):
        nat.resize_rgb8(torch.zeros(4, 4, 3, dtype=torch.uint8, device='cuda'), torch.empty(3, 2, 2, device='cuda'),
                        None, 4, 4, 2, 2, 'reader', IMAGENET_MEAN, IMAGENET_STD)  # reader mode needs its workspace
    with pytest.raises(ValueError):
        frame_from_rgb8(torch.zeros(4, 4, 3, dtype=torch.uint8), size=2, mode='bicubic')


def test_bmx_trees_at_360_matches_cpu_resize(golden_dir, synthetic_sd):
    """The example clip at --size 360: step on device-resized inputs against step on the reference's CPU transforms
    (torchvision for the frames, Pillow for the first-frame mask), then prob_to_ids back to the original size."""
    from oracle import fixtures
    from deva.inference.inference_core import DEVAInferenceCore
    from deva.model.network import DEVA
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    g, meta = fixtures.config1_vos(golden_dir)
    frames = torch.from_numpy(g['frames_u8'])
    T, (H, W) = frames.shape[0], frames.shape[1:3]
    size = 360
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing='ij')
    mask0 = torch.zeros(H, W, dtype=torch.uint8)
    mask0[((yy - 0.55 * H) / (0.3 * H)) ** 2 + ((xx - 0.3 * W) / (0.15 * W)) ** 2 < 1] = 1
    mask0[(yy > 0.2 * H) & (yy < 0.6 * H) & (xx > 0.6 * W) & (xx < 0.85 * W)] = 2
    im_transform = transforms.Compose([transforms.ToTensor(), transforms.Normalize(IMAGENET_MEAN, IMAGENET_STD),
                                       transforms.Resize(size, interpolation=InterpolationMode.BILINEAR,
                                                         antialias=True)])

    def run(device_resize):
        net = DEVA(meta['config']).cuda().eval()
        net.load_weights({k: v.cuda() for k, v in synthetic_sd.items()})
        np.random.seed(42)
        core = DEVAInferenceCore(net, meta['config'])
        probs, ids = [], []
        for t in range(T):
            if device_resize:
                img = frame_from_rgb8(frames[t].pin_memory(), size=size)
            else:
                img = im_transform(frames[t].numpy()).cuda()
            if t == 0:
                if device_resize:
                    m, labels = mask_from_palette(mask0, size)
                else:
                    m, labels = _pil_reference(mask0, size)
                    m = m.cuda()
                p = core.step(img, m, labels.tolist())
            else:
                p = core.step(img, end=(t == T - 1))
            probs.append(p.float().cpu())
            ids.append(prob_to_ids(p.float(), core.object_manager, size=(H, W)).cpu())
        return probs, ids

    got_p, got_ids = run(True)
    ref_p, ref_ids = run(False)
    oh, ow = resized_shape(H, W, size)
    worst, over = 0.0, 0.0
    for t in range(T):
        assert tuple(got_p[t].shape) == (3, oh, ow)
        d = (got_p[t] - ref_p[t]).abs()
        worst, over = max(worst, float(d.max())), max(over, float((d > 1e-3).float().mean()))
        up = F.interpolate(ref_p[t][None], (H, W), mode='bilinear', align_corners=False)[0]
        top2 = torch.topk(up, 2, dim=0)[0]
        confident = (top2[0] - top2[1]) > 2 * max(1e-3, float(d.max()))
        assert float(confident.float().mean()) > 0.5 or t > 0
        assert bool((got_ids[t][confident] == ref_ids[t][confident]).all()), t
    print(f'bmx-trees at size {size}: max |prob(device resize) - prob(cpu resize)| {worst:.2e}, '
          f'fraction over 1e-3 {over:.2e}')
    assert over <= 5e-4, (over, worst)
