"""Loaders of the two clip fixtures under ``tests/golden/``, which are stored compactly to keep every file small.

Both return ``(arrays, meta)``: a dict of numpy arrays with the keys and dtypes the fixtures were minted with by
``tests/golden/make_golden.py``, and the fixture's JSON record.

* ``vos_steps``: the 16 synthetic input frames are not stored; they are regenerated from the seed they were drawn with
  and checked against the SHA-256 recorded at minting time.  The reference's probabilities are stored as 16-bit fixed
  point (``round(p * 65535)``), so a loaded probability is within 7.7e-6 of the reference's fp32 value.
* ``config1_vos``: the four frames are the reference's own example JPEGs, decoded with PIL exactly as the reference's
  video reader does and checked against the SHA-256 of the decoded frames recorded at minting time.  Probabilities
  stay fp32.
"""
import hashlib
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')
PROB_SCALE = 65535


def sha256(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def vos_frames(seed: int, t: int, h: int, w: int) -> np.ndarray:
    """The synthetic clip of ``vos_steps``: one random base image plus small per-frame noise, [t, 3, h, w] fp32."""
    import torch
    g = torch.Generator().manual_seed(seed)
    base = torch.randn(3, h, w, generator=g)
    return torch.stack([base + 0.2 * torch.randn(3, h, w, generator=g) for _ in range(t)]).numpy()


def vos_steps(golden_dir: str = GOLDEN):
    meta = json.load(open(os.path.join(golden_dir, 'vos_steps.json')))
    f = meta['frames']
    arrays = {'frames': vos_frames(f['seed'], *f['shape'])}
    if sha256(arrays['frames']) != f['sha256']:
        raise RuntimeError('vos_steps: the regenerated frames differ from the ones the fixture was minted with '
                           '(torch.randn no longer draws the same numbers for this seed)')
    with np.load(os.path.join(golden_dir, 'vos_steps.npz')) as z:
        for k in z.files:
            arrays[k] = (z[k] / np.float32(PROB_SCALE)).astype(np.float32) if k.startswith('prob_') else \
                z[k].astype(np.int64)
    return arrays, meta


def config1_vos(golden_dir: str = GOLDEN):
    from PIL import Image
    meta = json.load(open(os.path.join(golden_dir, 'config1_vos.json')))
    frames = np.stack([np.array(Image.open(os.path.join(golden_dir, meta['video'], n)).convert('RGB'))
                       for n in meta['frames']])
    if sha256(frames) != meta['frames_u8_sha256']:
        raise RuntimeError('config1_vos: the decoded JPEG frames differ from the ones the fixture was minted with '
                           '(a different JPEG decoder?)')
    with np.load(os.path.join(golden_dir, 'config1_vos.npz')) as z:
        arrays = {k: z[k] for k in z.files}
    arrays['frames_u8'] = frames
    return arrays, meta
