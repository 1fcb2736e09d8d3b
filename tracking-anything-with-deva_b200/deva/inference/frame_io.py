"""Frame ingest / egress around ``DEVAInferenceCore.step`` (SURVEY 8f-3): the two per-frame host<->device hops of a
real pipeline, each as one kernel.

* ``frame_from_rgb8``: the decoded uint8 frame is uploaded as is (3 bytes / pixel instead of 12) and ToTensor +
  Normalize (deva/inference/data/video_reader.py:146-150, IMAGENET mean/std) run on the device - bit-exact.
* ``frame_from_rgb8(size=...)`` / ``mask_from_palette``: the resize to the evaluation size (``--size``, 480 by
  default) on the device too - torchvision's Resize(bilinear, antialias=True) of the reader or the demos'
  F.interpolate for frames, Pillow's NEAREST for the first-frame palette mask.
* ``prob_to_ids``: the driver's post-step (evaluation/eval_vos.py:169-181) - bilinear resize to the original size,
  optional flip, argmax, ``ObjectManager.tmp_to_obj_cls`` - fused into a single pass that writes the id map.
"""
from typing import List, Optional, Sequence, Tuple

import torch

from deva import _native as nat

IMAGENET_MEAN = (0.485, 0.456, 0.406)
IMAGENET_STD = (0.229, 0.224, 0.225)


def resized_shape(h: int, w: int, size: int, mode: str = 'reader') -> Tuple[int, int]:
    """(out_h, out_w) of an h x w frame evaluated at ``size`` (< 0: no resize).

    ``reader``: torchvision Resize(size) - the shorter side becomes ``size``, the longer ``int(size * long / short)``
    (``_compute_resized_output_size``).  ``demo``: ``scale = size / min(h, w)``, ``int(h * scale), int(w * scale)``
    (deva/inference/demo_utils.py)."""
    if mode not in ('reader', 'demo'):
        raise ValueError(f'unknown resize mode {mode!r}')
    if size < 0 or (mode == 'demo' and size == 0):  # the demos resize only for min_side > 0
        return h, w
    if size == 0 or h <= 0 or w <= 0:
        raise ValueError(f'cannot resize {h} x {w} to size {size}')
    if mode == 'demo':
        scale = size / min(h, w)
        return int(h * scale), int(w * scale)
    short, long = (w, h) if w <= h else (h, w)
    new_long = int(size * long / short)
    return (new_long, size) if w <= h else (size, new_long)


def frame_from_rgb8(frame: torch.Tensor, mean: Sequence[float] = IMAGENET_MEAN, std: Sequence[float] = IMAGENET_STD,
                    device: Optional[torch.device] = None, size: int = -1, mode: str = 'reader') -> torch.Tensor:
    """uint8 [H, W, 3] RGB (host - ideally pinned - or device) -> normalised float32 [3, H', W'] on the device.

    ``size`` < 0 keeps H x W.  Otherwise the frame is resized to ``resized_shape(H, W, size, mode)`` after the
    normalisation: ``mode='reader'`` equals VideoReader's ``im_transform`` (torchvision Resize(bilinear,
    antialias=True); a frame already at that shape is returned unresized, as torchvision does), ``mode='demo'``
    equals ``get_input_frame_for_deva`` (F.interpolate(bilinear, align_corners=False), always applied)."""
    assert frame.dtype == torch.uint8 and frame.dim() == 3 and frame.shape[2] == 3
    h, w = frame.shape[:2]
    oh, ow = resized_shape(h, w, size, mode)
    if not frame.is_cuda:
        frame = frame.to(device or torch.device('cuda', torch.cuda.current_device()), non_blocking=True)
    frame = frame.contiguous()
    out = torch.empty(3, oh, ow, dtype=torch.float32, device=frame.device)
    if size <= 0 or (mode == 'reader' and (oh, ow) == (h, w)):
        nat.ingest_rgb8(frame, out, h, w, mean, std)
        return out
    ws_bytes = nat.resize_rgb8_workspace_bytes(h, w, oh, ow, mode)
    ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=frame.device) if ws_bytes else None
    nat.resize_rgb8(frame, out, ws, h, w, oh, ow, mode, mean, std)
    return out


def pil_nearest_index(n_in: int, n_out: int) -> List[int]:
    """Source index of each of n_out outputs of Pillow's NEAREST resize along one axis (-1: none, left 0).

    Pillow (ImagingScaleAffine) starts at ``a[2] + a[0] * 0.5`` with ``a[0] = n_in / n_out`` and adds ``a[0]`` per
    output, all in double, truncating each position to an index; Python floats are the same doubles."""
    step = n_in / n_out
    pos = 0.0 + step * 0.5
    idx = []
    for _ in range(n_out):
        i = -1 if pos < 0.0 else int(pos)
        idx.append(i if i < n_in else -1)
        pos += step
    return idx


def mask_from_palette(mask: torch.Tensor, size: int = -1,
                      device: Optional[torch.device] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """uint8 palette (index) mask [H, W] (host or device) -> (int64 [H', W'] on the device, valid_labels).

    Equals VideoReader's first-frame mask: ``transforms.Resize(size, NEAREST)`` on the 'P' image (Pillow's nearest,
    not torch's ``nearest``), ``torch.LongTensor``, and the sorted unique non-zero ids as ``valid_labels``
    (video_reader.py:211-217).  ``size`` < 0 keeps H x W."""
    assert mask.dtype == torch.uint8 and mask.dim() == 2
    h, w = mask.shape
    oh, ow = resized_shape(h, w, size, 'reader')
    if not mask.is_cuda:
        mask = mask.to(device or torch.device('cuda', torch.cuda.current_device()), non_blocking=True)
    mask = mask.contiguous()
    if (oh, ow) == (h, w):
        out = mask.long()
    else:
        src_y = torch.tensor(pil_nearest_index(h, oh), dtype=torch.int32, device=mask.device)
        src_x = torch.tensor(pil_nearest_index(w, ow), dtype=torch.int32, device=mask.device)
        out = torch.empty(oh, ow, dtype=torch.long, device=mask.device)
        nat.resize_labels(mask, out, h, w, oh, ow, src_y, src_x)
    labels = torch.unique(out)
    return out, labels[labels != 0]


def id_lut(object_manager, channels: int, device) -> torch.Tensor:
    """int32 [channels]: temporary id (prob channel) -> object id; channel 0 and unknown channels -> 0."""
    lut = [0] * channels
    for tmp_id, obj in object_manager.tmp_id_to_obj.items():
        if 0 < tmp_id < channels:
            lut[tmp_id] = int(obj.id)
    return torch.tensor(lut, dtype=torch.int32, device=device)


def prob_to_ids(prob: torch.Tensor, object_manager=None, size: Optional[Tuple[int, int]] = None, flip: bool = False,
                dtype: torch.dtype = torch.long, lut: Optional[torch.Tensor] = None) -> torch.Tensor:
    """prob float32 [K+1, H, W] from ``step`` -> id map [H0, W0] (``size`` or H, W), dtype long or uint8.

    Equals ``tmp_to_obj_cls(argmax(flip(interpolate(prob, size, 'bilinear', align_corners=False))))``."""
    assert prob.is_cuda and prob.dtype == torch.float32 and prob.dim() == 3 and dtype in (torch.long, torch.uint8)
    prob = prob.contiguous()
    c, h, w = prob.shape
    oh, ow = (h, w) if size is None else (int(size[0]), int(size[1]))
    if lut is None and object_manager is not None:
        lut = id_lut(object_manager, c, prob.device)
    out = torch.empty(oh, ow, dtype=dtype, device=prob.device)
    nat.prob_to_ids(prob, c, h, w, oh, ow, flip, lut, out if dtype == torch.uint8 else None,
                    out if dtype == torch.long else None)
    return out
