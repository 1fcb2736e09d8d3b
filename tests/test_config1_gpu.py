"""BASELINE configs[0] through the drop-in: the reference's own example clip (example/vos/bmx-trees, 4 frames 854x480 ->
padded 480x864, first-frame ids {1, 2}) driven like evaluation/eval_vos.py:133-198 - uint8 frame -> ToTensor/Normalize
(on the device, bit-exact) -> DEVAInferenceCore.step -> argmax + tmp_to_obj_cls (prob_to_ids) - against outputs of the
unmodified reference recorded by tests/golden/make_golden.py::golden_config1.  The only real-image, real-size case in
the suite (everything else is <= 100x150 synthetic frames)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import fixtures

pytestmark = pytest.mark.gpu


def _reference_cross_device_deviation(golden_dir):
    """max |prob(reference on a B200, fp32, no TF32) - prob(reference on the CPU, the fixture)| on the lattice, as
    measured by tests/golden/ref_on_gpu.py and stored next to the fixture, with the device it was measured on."""
    return json.load(open(os.path.join(golden_dir, 'config1_ref_on_gpu.json')))


@pytest.mark.parametrize('backend,tol', [('native', 1e-3), ('torch', 1e-3)])
def test_example_vos_clip_matches_reference(golden_dir, synthetic_sd, backend, tol):
    from deva.inference.frame_io import frame_from_rgb8, prob_to_ids
    from deva.inference.inference_core import DEVAInferenceCore
    from deva.model.network import DEVA
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    g, meta = fixtures.config1_vos(golden_dir)
    net = DEVA(meta['config'])
    net.conv_backend = backend
    net = net.cuda().eval()
    net.load_weights({k: v.cuda() for k, v in synthetic_sd.items()})
    np.random.seed(42)
    core = DEVAInferenceCore(net, meta['config'])
    frames = torch.from_numpy(g['frames_u8'])
    T, (H, W) = frames.shape[0], frames.shape[1:3]
    worst, over = 0.0, 0.0
    for t in range(T):
        img = frame_from_rgb8(frames[t].pin_memory())
        if t == 0:
            p = core.step(img, torch.from_numpy(g['mask0'].astype(np.int64)).cuda(), meta['labels'])
        else:
            p = core.step(img, end=(t == T - 1))
        assert tuple(p.shape) == (len(meta['labels']) + 1, H, W)
        ids = prob_to_ids(p.float(), core.object_manager, dtype=torch.uint8).cpu()
        ref_ids = torch.from_numpy(g[f'ids_{t}'])
        assert set(ids.unique().tolist()) <= {0, *meta['labels']}
        # object-id indexing: bit-exact on every confident pixel of the full-resolution map ...
        confident = torch.from_numpy(np.unpackbits(g[f'confident_{t}'])[:H * W].reshape(H, W).astype(bool))
        assert bool((ids[confident] == ref_ids[confident]).all()), t
        # ... and, on the stride-4 lattice where the reference probabilities are stored, everywhere the reference's top-2
        # margin exceeds twice the tolerance (random-init outputs are near-uniform: most margins are tiny)
        lat = torch.from_numpy(g[f'prob_lattice_{t}'])
        got = p.float().cpu()[:, 1::4, 2::4]
        d = (got - lat).abs()
        worst = max(worst, float(d.max()))
        over = max(over, float((d > tol).float().mean()))
        top2 = torch.topk(lat, 2, dim=0)[0]
        decided = (top2[0] - top2[1]) > 2 * max(tol, float(d.max()))
        assert bool((got.argmax(0)[decided] == lat.argmax(0)[decided]).all()), t
        assert bool((ids[1::4, 2::4][decided] == ref_ids[1::4, 2::4][decided]).all()), t
        assert float(decided.float().mean()) > 0.5 or t > 0
    floor = _reference_cross_device_deviation(golden_dir)
    print(f'[{backend}] example/vos clip: max |prob - reference| on the lattice = {worst:.3e}, fraction of lattice points '
          f'over {tol:g}: {over:.2e}; unmodified reference on {floor["device"]} ({floor["power_limit_w"]} W limit) vs '
          f'its own CPU run: {floor["worst"]:.3e}')
    # Real-image keys put the top-30 cut of the memory read (memory_utils.py:56-64) through nearly tied similarities:
    # on this clip 12 % of the queries have their 30th and 31st similarity within 1e-4, some within the ~4e-6 rounding
    # noise of the fp32 similarity itself, and the 30th member still carries 1/30 of the softmax weight.  Which member
    # of such a tie survives depends on summation order; one swap moves the read-out of that query by ~3e-2 and the
    # probabilities of the ~100 pixels around it by ~1e-3 (tools/config1_stage_probe.py shows exactly one such event,
    # in frame 3, identical for the cuDNN-fp32 and the native conv stacks: it comes from the tie, not from precision;
    # tools/topk_flip_probe.py: the kernel's similarity is within 3e-6 of fp64 and agrees with the fp64 top-30 on 1619 of
    # 1620 queries).  So: the contract tolerance must hold on all but a vanishing fraction of the lattice, and nothing
    # may be further off than a single tie swap explains.
    assert over <= 5e-4, (over, worst)
    assert worst < 3e-3, worst
