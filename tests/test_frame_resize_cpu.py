"""Host side of the resize to the evaluation size (deva.inference.frame_io): output shapes, Pillow's NEAREST index
tables and the antialiased tap tables the frame kernel computes, all without a GPU."""
import random

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from PIL import Image
from torchvision import transforms
from torchvision.transforms import InterpolationMode
from torchvision.transforms.functional import _compute_resized_output_size

from deva import _native as nat
from deva.inference.frame_io import pil_nearest_index, resized_shape


def _random_shapes(n, seed):
    rng = random.Random(seed)
    shapes = [(1080, 1920), (720, 1280), (481, 853), (1920, 1080), (240, 427), (17, 23), (2160, 3840), (480, 640),
              (640, 480), (480, 480), (360, 1000)]
    while len(shapes) < n:
        h, w = rng.randint(1, 4000), rng.randint(1, 4000)
        shapes.append((h, w) if rng.random() < 0.7 else (min(h, w), min(h, w) * rng.randint(1, 3)))
    return shapes


@pytest.mark.parametrize('size', [480, 360, 1, 2000])
def test_resized_shape_reader_matches_torchvision(size):
    for h, w in _random_shapes(300, size):
        assert resized_shape(h, w, size, 'reader') == tuple(_compute_resized_output_size((h, w), [size])), (h, w)
        assert resized_shape(h, w, -1, 'reader') == (h, w)
    assert resized_shape(480, 853, 480, 'reader') == (480, 853)  # the unresized shortcut
    assert resized_shape(240, 427, 480, 'reader') == (480, 854)  # upscale


@pytest.mark.parametrize('size', [480, 360, 1, 2000])
def test_resized_shape_demo_matches_demo_utils(size):
    for h, w in _random_shapes(300, 7 + size):
        scale = size / min(h, w)  # deva/inference/demo_utils.py: get_input_frame_for_deva
        assert resized_shape(h, w, size, 'demo') == (int(h * scale), int(w * scale)), (h, w)
    assert resized_shape(100, 200, 0, 'demo') == (100, 200)
    with pytest.raises(ValueError):
        resized_shape(100, 200, 0, 'reader')
    with pytest.raises(ValueError):
        resized_shape(100, 200, 480, 'nearest')


@pytest.mark.parametrize('hw,size', [((1080, 1920), 480), ((720, 1280), 480), ((577, 1023), 480), ((481, 853), 480),
                                     ((1920, 1080), 360), ((240, 427), 480), ((17, 23), 480), ((333, 91), 50)])
def test_nearest_tables_reproduce_pillow(hw, size):
    h, w = hw
    rng = np.random.default_rng(h * 7 + w)
    mask = rng.integers(0, 256, (h, w), dtype=np.uint8)
    img = Image.fromarray(mask, mode='P')
    oh, ow = resized_shape(h, w, size)
    want = np.array(transforms.Resize(size, interpolation=InterpolationMode.NEAREST)(img))  # video_reader.py's path
    assert want.shape == (oh, ow)
    assert np.array_equal(want, np.array(img.resize((ow, oh), Image.NEAREST)))
    ys, xs = np.array(pil_nearest_index(h, oh)), np.array(pil_nearest_index(w, ow))
    assert ys.min() >= 0 and xs.min() >= 0 and ys.max() < h and xs.max() < w
    assert np.array_equal(mask[np.ix_(ys, xs)], want)


def _aa_weights_fp64(n_in, n_out):
    """torch's _compute_weights_aa restated in float64 throughout, as a dense [n_out, n_in] matrix."""
    scale = n_in / n_out
    support = scale if scale >= 1 else 1.0
    inv = 1 / scale if scale >= 1 else 1.0
    out = np.zeros((n_out, n_in))
    for i in range(n_out):
        center = scale * (i + 0.5)
        x0 = max(int(center - support + 0.5), 0)
        x1 = min(int(center + support + 0.5), n_in)
        t = np.maximum(0.0, 1.0 - np.abs((np.arange(x0, x1) - center + 0.5) * inv))
        out[i, x0:x1] = t / t.sum() if t.sum() else t
    return out


def _dense(n_in, n_out):
    x0, n, w = nat.resize_aa_weights(n_in, n_out)
    m = torch.zeros(n_out, n_in)
    for i in range(n_out):
        m[i, x0[i]:x0[i] + n[i]] = w[i, :n[i]]
    return m


# the axes of the GPU test shapes at sizes 480 and 360: downscales, near-identity, upscales, 4K, a 1-pixel output
AA_AXES = [(1920, 853), (1080, 480), (1280, 853), (720, 480), (853, 851), (481, 480), (427, 853), (240, 480),
           (3840, 853), (2160, 480), (17, 480), (23, 649), (5, 1)]


@pytest.mark.parametrize('n_in,n_out', AA_AXES)
def test_aa_weight_tables(n_in, n_out):
    got = _dense(n_in, n_out)
    # bit-identical to the taps torch uses for a float32 CPU tensor: resizing the identity along one axis reads them out
    eye = torch.eye(n_in)[None, None]
    torch_w = F.interpolate(eye, size=(n_in, n_out), mode='bilinear', antialias=True, align_corners=False)[0, 0].T
    assert torch.equal(got, torch_w)
    # and close to fp64: the fp32 scale and center shift the window by up to an fp32 ulp of the source coordinate
    # (~1.2e-4 at 1920), which is the whole of the ~1e-4 gap between torch's fp32 resize and an fp64 one
    ref = _aa_weights_fp64(n_in, n_out)
    err = float(np.abs(got.double().numpy() - ref).max())
    assert err < 2e-4 * max(1.0, n_out / n_in), err
    rows = got.sum(1)
    assert float((rows - 1).abs().max()) < 1e-5


def test_aa_weight_tables_random_axes():
    rng = random.Random(5)
    for _ in range(60):
        n_in, n_out = rng.randint(1, 4000), rng.randint(1, 1500)
        eye = torch.eye(n_in)[None, None]
        torch_w = F.interpolate(eye, size=(n_in, n_out), mode='bilinear', antialias=True)[0, 0].T
        assert torch.equal(_dense(n_in, n_out), torch_w), (n_in, n_out)


def test_aa_weight_tables_reject_short_rows():
    x0, n, w = torch.empty(480, dtype=torch.int32), torch.empty(480, dtype=torch.int32), torch.empty(480, 5)
    rc = nat.lib().deva_b200_resize_aa_weights(1080, 480, 5, x0.data_ptr(), n.data_ptr(), w.data_ptr())
    assert rc != 0 and b'max_taps' in nat.lib().deva_b200_last_error()
