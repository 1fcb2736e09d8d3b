"""Frame and mask resize to the evaluation size on the device (frame_io.frame_from_rgb8(size=), mask_from_palette)
against the host transform it replaces (VideoReader's torchvision im_transform / PIL mask_transform).

Device times are CUDA events over --iters calls on device-resident uint8 inputs (the upload is the same 3 bytes / pixel
with or without the resize and is not included), rotating over enough distinct input and output buffers that every
pass reads from HBM rather than from the 126 MB L2.  Bytes are the algorithmic ones: the uint8 frame read once and the
fp32 output written once (the reader mode's [3, H, out_w] fp32 intermediate is extra traffic and is not counted).
The host transforms are timed on the same machine with time.perf_counter over --host-iters calls.

    python tools/bench_ingest.py [--iters 200] [--host-iters 5] [--out profiles/<name>.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tracking-anything-with-deva_b200'))
from deva import _native as nat  # noqa: E402
from deva.inference.frame_io import IMAGENET_MEAN, IMAGENET_STD, frame_from_rgb8, mask_from_palette, \
    pil_nearest_index, resized_shape  # noqa: E402

L2_BYTES = 126e6


def device_ms(fn, per_call_bytes, iters):
    """Mean device time of iters calls of fn(k) (k selects the buffer set) between two events, after a warm-up pass.
    A sleep kernel ahead of the first event holds the stream while the host enqueues every call, so the window
    measures the device, not the Python launch rate."""
    n_sets = max(2, int(np.ceil(3 * L2_BYTES / per_call_bytes)))
    for k in range(n_sets):
        fn(k)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(200_000_000)  # ~0.1 s at the B200's clock
    e0.record()
    for i in range(iters):
        fn(i % n_sets)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters, n_sets


def host_ms(fn, iters):
    fn()
    t0 = time.perf_counter()
    for _ in range(iters):
        fn()
    return (time.perf_counter() - t0) * 1e3 / iters


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        q = 'nvidia-smi unavailable'
    return dict(device=torch.cuda.get_device_name(0), nvidia_smi=q)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=200)
    ap.add_argument('--host-iters', type=int, default=5)
    ap.add_argument('--size', type=int, default=480)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    nat.require_device()
    from PIL import Image
    from torchvision import transforms
    from torchvision.transforms import InterpolationMode
    g = torch.Generator().manual_seed(0)
    rows = []
    for h, w in [(1080, 1920), (720, 1280)]:
        host_frame = torch.randint(0, 256, (h, w, 3), generator=g, dtype=torch.uint8)
        im_transform = transforms.Compose([
            transforms.ToTensor(), transforms.Normalize(IMAGENET_MEAN, IMAGENET_STD),
            transforms.Resize(a.size, interpolation=InterpolationMode.BILINEAR, antialias=True)])
        pil = Image.fromarray(host_frame.numpy())
        host_reader = host_ms(lambda: im_transform(pil), a.host_iters)
        for mode in ('reader', 'demo'):
            oh, ow = resized_shape(h, w, a.size, mode)
            bytes_alg = h * w * 3 + 3 * oh * ow * 4
            n_sets = max(2, int(np.ceil(3 * L2_BYTES / bytes_alg)))
            frames = [host_frame.cuda() for _ in range(n_sets)]
            ms, n_sets = device_ms(lambda k: frame_from_rgb8(frames[k], size=a.size, mode=mode), bytes_alg, a.iters)
            row = dict(what=f'frame {mode}', src=[h, w], dst=[oh, ow], device_ms=round(ms, 4),
                       MB_read=round(h * w * 3 / 1e6, 2), MB_written=round(3 * oh * ow * 4 / 1e6, 2),
                       GBps=round(bytes_alg / ms / 1e6, 1), buffer_sets=n_sets)
            if mode == 'reader':
                row.update(host_ms=round(host_reader, 2), host_transform='torchvision ToTensor+Normalize+Resize(aa)')
            rows.append(row)
            print(json.dumps(row), flush=True)
            del frames
        mask = torch.randint(0, 3, (h, w), generator=g, dtype=torch.uint8)
        oh, ow = resized_shape(h, w, a.size)
        pil_mask = Image.fromarray(mask.numpy(), mode='P')
        mask_transform = transforms.Resize(a.size, interpolation=InterpolationMode.NEAREST)
        host_mask = host_ms(lambda: torch.LongTensor(np.array(mask_transform(pil_mask))), a.host_iters)
        bytes_alg = h * w + oh * ow * 8
        masks = [mask.cuda() for _ in range(max(2, int(np.ceil(3 * L2_BYTES / bytes_alg))))]
        ms, n_sets = device_ms(lambda k: mask_from_palette(masks[k], a.size), bytes_alg, a.iters)
        row = dict(what='mask nearest + valid_labels', src=[h, w], dst=[oh, ow], device_ms=round(ms, 4),
                   MB_read=round(h * w / 1e6, 2), MB_written=round(oh * ow * 8 / 1e6, 2), host_ms=round(host_mask, 2),
                   host_transform='PIL Resize(NEAREST) + LongTensor', buffer_sets=n_sets,
                   note='device_ms includes the host-built index tables, their upload and torch.unique')
        rows.append(row)
        print(json.dumps(row), flush=True)
        src_y = torch.tensor(pil_nearest_index(h, oh), dtype=torch.int32, device='cuda')
        src_x = torch.tensor(pil_nearest_index(w, ow), dtype=torch.int32, device='cuda')
        outs = [torch.empty(oh, ow, dtype=torch.long, device='cuda') for _ in masks]
        ms, n_sets = device_ms(lambda k: nat.resize_labels(masks[k], outs[k], h, w, oh, ow, src_y, src_x), bytes_alg,
                               a.iters)
        row = dict(what='mask resize_labels kernel', src=[h, w], dst=[oh, ow], device_ms=round(ms, 4),
                   GBps=round(bytes_alg / ms / 1e6, 1), buffer_sets=n_sets)
        rows.append(row)
        print(json.dumps(row), flush=True)
        del masks, outs
    res = dict(gpu_info(), size=a.size, iters=a.iters, host_threads=torch.get_num_threads(), host_cpus=os.cpu_count(),
               torch=torch.__version__, rows=rows)
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
