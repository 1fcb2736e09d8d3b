"""Pin the CPU oracle against fixtures minted from the reference (tests/golden/make_golden.py)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import fixtures
from oracle import memory_math as mm
from oracle import network as net
from oracle.core import CoreOracle
from oracle.memory_bank import MemoryOracle

torch.set_grad_enabled(False)


def _load(golden_dir, name):
    return {k: torch.from_numpy(v) for k, v in np.load(os.path.join(golden_dir, name)).items()}


def test_checkpoint_spec_matches_reference(golden_dir):
    from deva.model.param_spec import checkpoint_spec
    ref = json.load(open(os.path.join(golden_dir, 'checkpoint_spec.json')))
    mine = {k: list(shape) for k, (shape, _) in checkpoint_spec().items()}
    assert list(mine.keys()) == list(ref.keys())
    assert mine == ref


def test_memory_math_matches_reference(golden_dir):
    g = _load(golden_dir, 'memory_read.npz')
    sim = mm.similarity(g['mk'], g['ms'].reshape(-1), g['qk'], g['qe'])
    torch.testing.assert_close(sim, g['sim'], rtol=1e-5, atol=1e-5)
    idx, w = mm.topk_softmax(sim, 30)
    assert torch.equal(idx, g['topk_idx'])
    aff = mm.dense_affinity(sim, 30)
    torch.testing.assert_close(aff, g['affinity'], rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(mm.usage_of(aff), g['usage'], rtol=1e-5, atol=1e-8)
    out = mm.readout(aff, g['mv'].flatten(0, 1)).view_as(g['readout'])
    torch.testing.assert_close(out, g['readout'], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(mm.dense_affinity(sim, None), g['affinity_full'], rtol=1e-5, atol=1e-7)


def test_network_stages_match_reference(golden_dir, synthetic_sd):
    g = _load(golden_dir, 'network_stages.npz')
    sd = synthetic_sd
    ms, feat = net.encode_image(sd, g['image'])
    for a, b in zip(ms, (g['f16'], g['f8'], g['f4'])):
        torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(feat, g['feat'], rtol=1e-4, atol=1e-5)
    key, shr, sel = net.transform_key(sd, feat)
    torch.testing.assert_close(key, g['key'], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(shr, g['shrinkage'], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(sel, g['selection'], rtol=1e-4, atol=1e-5)
    value, s1 = net.encode_mask(sd, g['image'], ms, g['sensory0'], g['masks'])
    torch.testing.assert_close(value, g['value'], rtol=1e-4, atol=2e-5)
    torch.testing.assert_close(s1, g['sensory1'], rtol=1e-4, atol=2e-5)
    s2, logits, prob = net.segment(sd, ms, g['readout'], g['sensory1'], g['masks'])
    torch.testing.assert_close(s2, g['sensory2'], rtol=1e-4, atol=2e-5)
    torch.testing.assert_close(logits, g['logits'], rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(prob, g['prob'], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(net.aggregate(g['masks'][0] * 0.9, dim=0), g['aggregate'])


def test_vos_steps_match_reference(golden_dir, synthetic_sd):
    arrays, meta = fixtures.vos_steps(golden_dir)
    g = {k: torch.from_numpy(v) for k, v in arrays.items()}
    np.random.seed(42)
    core = CoreOracle(synthetic_sd, meta['config'])
    T = g['frames'].shape[0]
    for t in range(T):
        if t == 0:
            p = core.step(g['frames'][t], g['mask0'], [1, 2])
        elif t == 6:
            p = core.step(g['frames'][t], g['mask6'], [7])
        else:
            p = core.step(g['frames'][t], end=(t == T - 1))
        ref = g[f'prob_{t:02d}']
        assert p.shape == ref.shape
        assert float((p - ref).abs().max()) < 2e-4, t
        assert {str(b): list(s) for b, s in core.memory.sizes().items()} == meta['sizes'][t], t
    assert core.objects.tmp_to_id == {1: 1, 2: 2, 3: 7}


def test_bank_trace_matches_reference(golden_dir):
    """Weight-independent known answer for the bank bookkeeping (SURVEY.md 8c)."""
    meta = json.load(open(os.path.join(golden_dir, 'bank_trace.json')))
    cfg, hw = meta['config'], meta['hw']
    torch.manual_seed(3)
    mem = MemoryOracle(cfg)
    h = w = 6
    objs = []
    for t, want in enumerate(meta['trace']):
        if t == 0:
            objs += [1, 2]
        if t == 12:
            objs += [7]
        key, shr = torch.randn(1, 64, h, w), 1 + torch.rand(1, 1, h, w)
        sel = torch.sigmoid(torch.randn(1, 64, h, w))
        if t > 0:
            mem.read(key, sel)
        mem.add(key, shr, torch.randn(1, len(objs), 8, h, w), list(objs), selection=sel)
        assert {str(b): list(s) for b, s in mem.sizes().items()} == want, t


# ---------------------------------------------------------------------------- in-clip consensus (SURVEY 8f-1)
def _scenario(golden_dir):
    import importlib.util
    spec = importlib.util.spec_from_file_location('consensus_scenario', os.path.join(golden_dir, 'consensus_scenario.py'))
    sc = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(sc)
    return sc


def test_consensus_alignment_matches_reference(golden_dir, synthetic_sd):
    from oracle import consensus as oc
    from oracle.core import pad_to_multiple
    sc = _scenario(golden_dir)
    g = _load(golden_dir, 'consensus.npz')
    meta = json.load(open(os.path.join(golden_dir, 'consensus.json')))
    cfg, data = meta['config'], sc.frames()
    img0, _ = pad_to_multiple(data[0][0], 16)
    img1, _ = pad_to_multiple(data[1][0], 16)
    m0, _ = pad_to_multiple(torch.stack([data[0][1] == 3, data[0][1] == 5]).float(), 16)
    prob = oc.spatial_alignment(synthetic_sd, img0, m0, img1, cfg)[0]
    torch.testing.assert_close(prob, g['align_prob'], rtol=1e-4, atol=2e-5)
    pick = [(0, (3, 5)), (1, (1, 4)), (3, (7, 8))]
    for key, scores in (('established_mask', None), ('established_mask_scored', [0.2, 0.9, 0.5])):
        kti, total = oc.established_association(
            synthetic_sd, [sc.TIMES[i] for i, _ in pick], [data[i][0] for i, _ in pick],
            [torch.stack([data[i][1] == a, data[i][1] == b]).float() for i, (a, b) in pick], cfg, scores=scores)
        assert kti == meta['established_keyframe' + ('_scored' if scores else '')]
        torch.testing.assert_close(total, g[key], rtol=1e-4, atol=2e-5)


def test_consensus_voting_matches_reference(golden_dir, synthetic_sd):
    """Matching (IoU > 0.5, same isthing), exact selection, meta merging and painting order: bit-exact ids."""
    from oracle import consensus as oc
    sc = _scenario(golden_dir)
    g = _load(golden_dir, 'consensus.npz')
    meta = json.load(open(os.path.join(golden_dir, 'consensus.json')))
    data = sc.frames()

    def frames():
        return [(ti, image, ids, [oc.Segment(sid, cat, thing, score) for sid, _, cat, thing, score in dets])
                for ti, (image, ids), dets in zip(sc.TIMES, data, sc.DETECTIONS)]

    for keyframe in ('first', 'last', 'middle'):
        kti, mask, infos = oc.auto_association(frames(), keyframe, sc.shifted_alignment)
        want = meta['auto']['shifted_' + keyframe]
        assert kti == want['keyframe']
        assert [list(i) for i in infos] == want['segments']
        assert torch.equal(mask, g[f'auto_shifted_{keyframe}_mask'])
    kti, mask, infos = oc.auto_association(
        frames(), 'first', lambda sti, si, sm, tti, tim: oc.spatial_alignment(synthetic_sd, si, sm, tim, meta['config']))
    want = meta['auto']['real_first']
    assert kti == want['keyframe'] and [list(i) for i in infos] == want['segments']
    assert torch.equal(mask, g['auto_real_first_mask'])


def test_detection_session_matches_reference(golden_dir, synthetic_sd):
    """incorporate_detection (match & merge, poke / purge, new buckets, memory purge) interleaved with step():
    probabilities to fp32 round-off, ids / poke counts / merged meta / bank sizes exact."""
    from oracle.detections import DetectionCoreOracle, Tracked
    sc = _scenario(golden_dir)
    g = _load(golden_dir, 'detections.npz')
    meta = json.load(open(os.path.join(golden_dir, 'detections.json')))
    np.random.seed(42)
    core = DetectionCoreOracle(synthetic_sd, meta['config'])
    frames = sc.detect_frames()
    for t, (frame, dets) in enumerate(zip(frames, sc.DETECT_SESSION)):
        if dets is None:
            p = core.step(frame, end=(t == len(frames) - 1))
        else:
            ids = sc.merge_masks({d[0]: d[1] for d in dets}, sc.DETECT_HW)
            p = core.incorporate_detection(frame, ids, [Tracked(d[0], d[2], d[3], d[4]) for d in dets])
        want = meta['states'][t]
        objects = [[tt, o.id, o.poke_count, list(o.category_ids), list(o.scores)] for tt, o in core.objects.by_tmp.items()]
        assert objects == want['objects'], (t, objects, want['objects'])
        sizes = {str(b): list(s) for b, s in core.memory.sizes().items()}
        assert sizes == want['sizes'], (t, sizes, want['sizes'])
        torch.testing.assert_close(p, g[f'prob_{t:02d}'], rtol=1e-4, atol=2e-5)
