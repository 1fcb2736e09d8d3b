"""GPU parity of the full DEVAInferenceCore.step path against reference-minted golden frames."""
import numpy as np
import pytest
import torch

from oracle import fixtures

pytestmark = pytest.mark.gpu


def _core(cfg, sd, backend):
    from deva.inference.inference_core import DEVAInferenceCore
    from deva.model.network import DEVA
    net = DEVA(cfg)
    net.conv_backend = backend
    net = net.cuda().eval()
    net.load_weights({k: v.cuda() for k, v in sd.items()})
    return DEVAInferenceCore(net, cfg)


# 'native': every layer on the hand-written sm_100a kernels (fp16 MMA operands, fp32 accumulate, the default 'parity'
# precision plan); 'torch': the same graphs through cuDNN fp32 (isolates the memory-read kernels).
# Both are held to north_star's 1e-3 max-abs against the fp32 reference.
@pytest.mark.parametrize('backend,tol', [('native', 1e-3), ('torch', 1e-3)])
def test_vos_clip_matches_reference(golden_dir, synthetic_sd, backend, tol):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    arrays, meta = fixtures.vos_steps(golden_dir)
    g = {k: torch.from_numpy(v) for k, v in arrays.items()}
    np.random.seed(42)
    core = _core(meta['config'], synthetic_sd, backend)
    T = g['frames'].shape[0]
    worst = 0.0
    for t in range(T):
        img = g['frames'][t].cuda()
        if t == 0:
            p = core.step(img, g['mask0'].cuda(), [1, 2])
        elif t == 6:
            p = core.step(img, g['mask6'].cuda(), [7])
        else:
            p = core.step(img, end=(t == T - 1))
        ref = g[f'prob_{t:02d}']
        assert tuple(p.shape) == tuple(ref.shape)
        err = float((p.cpu() - ref).abs().max())
        worst = max(worst, err)
        sizes = {str(b): [core.memory.work_mem.size(b), core.memory.long_mem.size(b)]
                 for b in core.memory.work_mem.buckets}
        assert sizes == meta['sizes'][t], (t, sizes, meta['sizes'][t])
        # object-id indexing: confident pixels must agree exactly
        top2 = torch.topk(ref, 2, dim=0)[0]
        confident = (top2[0] - top2[1]) > 0.05
        assert bool((p.cpu().argmax(0)[confident] == ref.argmax(0)[confident]).all()), t
    print(f'[{backend}] max |prob - reference| over the clip:', worst)
    assert worst < tol, worst  # north_star target: 1e-3 max-abs vs the fp32 reference
    om = core.object_manager
    assert {t: o.id for t, o in om.tmp_id_to_obj.items()} == {1: 1, 2: 2, 3: 7}
    ids = om.tmp_to_obj_cls(torch.tensor([[0, 1], [2, 3]]).cuda())
    assert ids.cpu().tolist() == [[0, 1], [2, 7]]


def _run_clip(core, frames, mask, ids, n=5):
    out = []
    for t in range(n):
        out.append(core.step(frames[t], mask if t == 0 else None, ids if t == 0 else None).float().cpu())
    return out


def test_chunked_objects_and_odd_frame_size(synthetic_sd):
    """chunk_size only splits the object batch (reference quirk Q11) and padding/unpadding handles sizes that are not
    multiples of 16: native == native(chunked) exactly, native ~ cuDNN-fp32 backend within the fp16 budget."""
    cfg = dict(key_dim=64, value_dim=512, pix_feat_dim=512, mem_every=2, enable_long_term=True, chunk_size=-1, top_k=30,
               enable_long_term_count_usage=True, max_mid_term_frames=10, min_mid_term_frames=5, num_prototypes=128,
               max_long_term_elements=10000)
    g = torch.Generator().manual_seed(3)
    H, W = 100, 150  # -> padded to 112 x 160
    base = torch.randn(3, H, W, generator=g)
    frames = [(base + 0.2 * torch.randn(3, H, W, generator=g)).cuda() for _ in range(5)]
    mask = torch.zeros(H, W, dtype=torch.long)
    mask[5:45, 10:70] = 4
    mask[50:95, 60:140] = 9
    mask[20:60, 100:145] = 2
    mask = mask.cuda()
    ids = [2, 4, 9]
    a = _run_clip(_core(cfg, synthetic_sd, 'native'), frames, mask, ids)
    b = _run_clip(_core(dict(cfg, chunk_size=2), synthetic_sd, 'native'), frames, mask, ids)
    c = _run_clip(_core(cfg, synthetic_sd, 'torch'), frames, mask, ids)
    for t in range(5):
        assert a[t].shape == (4, H, W)
        assert float((a[t] - b[t]).abs().max()) < 1e-6, t       # same kernels per object -> same numbers
        assert float((a[t] - c[t]).abs().max()) < 4e-3, t       # fp16 conv stack vs fp32 cuDNN
        assert float((a[t].sum(0) - 1).abs().max()) < 1e-5
