"""Mint golden fixtures by running the UNMODIFIED reference on CPU.

    DEVA_REFERENCE_ROOT=<checkout of hkchengrex/Tracking-Anything-with-DEVA @ 404a112> python tests/golden/make_golden.py

Imports the reference read-only from that checkout with the three shims of SURVEY.md section 8(c):
a stub ``pulp`` module, ``pretrained=False`` ResNets, nothing else.  Writes small fixtures next to
this file; they pin ``oracle/`` (tests/test_oracle_golden.py) and, through it, the CUDA path.
Nothing at test/bench time runs this script: the tests need only what it wrote.
"""
import json
import os
import shutil
import sys
import types
import zipfile

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.modules['pulp'] = types.ModuleType('pulp')
REF = os.environ['DEVA_REFERENCE_ROOT']
sys.path.insert(0, REF)

import numpy as np
import torch

import deva.model.resnet as _R  # the reference's deva package

_r18, _r50 = _R.resnet18, _R.resnet50
_R.resnet18 = lambda pretrained=True, extra_dim=0: _r18(pretrained=False, extra_dim=extra_dim)
_R.resnet50 = lambda pretrained=True, extra_dim=0: _r50(pretrained=False, extra_dim=extra_dim)
from deva.inference.inference_core import DEVAInferenceCore
from deva.inference.memory_manager import MemoryManager
from deva.model.memory_utils import do_softmax, get_similarity
from deva.model.network import DEVA

# the product's checkpoint synthesiser (pure python, no CUDA needed) - loaded by path because
# the package directory shadows the reference's ``deva`` name
import importlib.util

_spec = importlib.util.spec_from_file_location(
    'b200_param_spec', os.path.join(ROOT, 'tracking-anything-with-deva_b200', 'deva', 'model', 'param_spec.py'))
param_spec = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(param_spec)
sys.path.append(ROOT)
from oracle import fixtures  # noqa: E402  (the compact storage of the two clip fixtures)

CFG = dict(key_dim=64, value_dim=512, pix_feat_dim=512, mem_every=5, enable_long_term=True,
           chunk_size=-1, top_k=30, enable_long_term_count_usage=True, max_mid_term_frames=10,
           min_mid_term_frames=5, num_prototypes=128, max_long_term_elements=10000)
torch.set_grad_enabled(False)


def save(name, **arrays):
    """np.savez_compressed's layout at the strongest deflate level (keeps every fixture under 1 MB)."""
    with zipfile.ZipFile(os.path.join(HERE, name), 'w', zipfile.ZIP_DEFLATED, compresslevel=9) as zf:
        for k, v in arrays.items():
            with zf.open(k + '.npy', 'w', force_zip64=True) as f:
                np.lib.format.write_array(f, np.asarray(v.numpy() if torch.is_tensor(v) else v), allow_pickle=False)
    print('wrote', name, {k: tuple(v.shape) for k, v in arrays.items() if hasattr(v, 'shape')})


def golden_spec():
    sd = DEVA(CFG).state_dict()
    json.dump({k: list(v.shape) for k, v in sd.items()}, open(os.path.join(HERE, 'checkpoint_spec.json'), 'w'),
              indent=0)
    print('wrote checkpoint_spec.json', len(sd))


def golden_memory_read():
    """get_similarity -> do_softmax(top_k, usage) -> _readout on seeded inputs (BASELINE.md section 4)."""
    torch.manual_seed(0)
    CK, N, Q, K, CV = 64, 600, 80, 2, 32
    mk, ms = torch.randn(CK, N), 1 + torch.rand(1, N)
    qk, qe = torch.randn(CK, Q), torch.sigmoid(torch.randn(CK, Q))
    mv = torch.randn(K, CV, N)
    sim = get_similarity(mk, ms, qk, qe, add_batch_dim=True)
    vals, idx = torch.topk(sim, k=30, dim=1)
    aff, usage = do_softmax(sim.clone(), top_k=30, inplace=True, return_usage=True)
    mm = MemoryManager(CFG)
    out = mm._readout(aff[0], mv)
    # full-softmax branch used by consolidation (memory_utils.py:66-71)
    aff_full = do_softmax(sim.clone())
    save('memory_read.npz', mk=mk, ms=ms, qk=qk, qe=qe, mv=mv, sim=sim[0], topk_idx=idx[0], topk_val=vals[0],
         affinity=aff[0], usage=usage[0], readout=out, affinity_full=aff_full[0])


def golden_bank_trace():
    """Weight-independent (work,long) size trace, SURVEY.md section 8(c)."""
    torch.manual_seed(0)
    cfg = dict(CFG, mem_every=1, max_long_term_elements=400)
    net = DEVA(cfg).eval()
    core = DEVAInferenceCore(net, cfg)
    H = W = 96
    trace = []
    for t in range(40):
        img = torch.randn(3, H, W)
        if t == 0:
            m = torch.zeros(H, W, dtype=torch.long); m[8:40, 8:40] = 1; m[50:90, 50:90] = 2
            core.step(img, m, [1, 2])
        elif t == 12:
            m = torch.zeros(H, W, dtype=torch.long); m[8:30, 60:90] = 7
            core.step(img, m, [7])
        else:
            core.step(img)
        mem = core.memory
        trace.append({str(b): [mem.work_mem.size(b), mem.long_mem.size(b)] for b in mem.work_mem.buckets})
    json.dump({'config': cfg, 'hw': 36, 'trace': trace, 'tmp_ids': {str(o.id): t for o, t in
                                                                     core.object_manager.obj_to_tmp_id.items()}},
              open(os.path.join(HERE, 'bank_trace.json'), 'w'))
    print('wrote bank_trace.json', trace[9], trace[24], trace[36])


def golden_network():
    """Stage outputs of the reference network with the synthetic checkpoint (seed 1)."""
    sd = param_spec.synthetic_state_dict(seed=1)
    net = DEVA(CFG).eval()
    net.load_weights(sd)
    g = torch.Generator().manual_seed(5)
    H, W, K = 64, 80, 2
    image = torch.randn(1, 3, H, W, generator=g)
    masks = torch.zeros(1, K, H, W); masks[0, 0, 5:30, 5:40] = 1; masks[0, 1, 30:60, 30:75] = 1
    ms, feat = net.encode_image(image)
    key, shr, sel = net.transform_key(feat)
    h, w = key.shape[-2:]
    sensory0 = 0.5 * torch.randn(1, K, 512, h, w, generator=g)
    value, sensory1 = net.encode_mask(image, ms, sensory0, masks, is_deep_update=True)
    readout = torch.randn(1, K, 512, h, w, generator=g)
    sensory2, logits, prob = net.segment(ms, readout, sensory1, masks, update_sensory=True)
    agg = net.aggregate(masks[0] * 0.9, dim=0)
    save('network_stages.npz', image=image, masks=masks, f16=ms[0], f8=ms[1], f4=ms[2], feat=feat, key=key,
         shrinkage=shr, selection=sel, sensory0=sensory0, value=value, sensory1=sensory1, readout=readout,
         sensory2=sensory2, logits=logits, prob=prob, aggregate=agg)
    for n, t in dict(f16=ms[0], f8=ms[1], f4=ms[2], key=key, shr=shr, value=value, sensory2=sensory2,
                     logits=logits).items():
        print(f'  {n}: mean {t.mean():.3f} std {t.std():.3f} absmax {t.abs().max():.3f}')


def golden_vos():
    """DEVAInferenceCore.step over a 16-frame synthetic clip (objects {1,2}, new object 7 at t=6)."""
    sd = param_spec.synthetic_state_dict(seed=1)
    cfg = dict(CFG, mem_every=1, max_long_term_elements=300)
    net = DEVA(cfg).eval()
    net.load_weights(sd)
    np.random.seed(42)
    core = DEVAInferenceCore(net, cfg)
    H, W, T = 80, 96, 16
    frames = torch.from_numpy(fixtures.vos_frames(11, T, H, W))
    m0 = torch.zeros(H, W, dtype=torch.long); m0[6:40, 6:44] = 1; m0[44:76, 40:90] = 2
    m6 = torch.zeros(H, W, dtype=torch.long); m6[10:34, 56:92] = 7
    probs, sizes = [], []
    for t in range(T):
        if t == 0:
            p = core.step(frames[t], m0, [1, 2])
        elif t == 6:
            p = core.step(frames[t], m6, [7])
        else:
            p = core.step(frames[t], end=(t == T - 1))
        probs.append(p.clone())
        mem = core.memory
        sizes.append({str(b): [mem.work_mem.size(b), mem.long_mem.size(b)] for b in mem.work_mem.buckets})
    # frames are regenerated from their seed by oracle.fixtures.vos_steps; probabilities as 16-bit fixed point
    arrays = {f'prob_{t:02d}': (p.double() * fixtures.PROB_SCALE).round().to(torch.int32).numpy().astype(np.uint16)
              for t, p in enumerate(probs)}
    save('vos_steps.npz', mask0=m0.to(torch.uint8), mask6=m6.to(torch.uint8), **arrays)
    json.dump({'config': cfg, 'sizes': sizes,
               'frames': {'seed': 11, 'shape': [T, H, W], 'sha256': fixtures.sha256(frames.numpy())}},
              open(os.path.join(HERE, 'vos_steps.json'), 'w'))
    print('  sizes', sizes[-1], 'prob range', float(probs[-1].min()), float(probs[-1].max()))


def golden_consensus():
    """In-clip consensus (consensus_associated.py / consensus_automatic.py) on the seeded scenario of
    consensus_scenario.py.  `pulp` is absent: the reference's fallback-solver hook `solve_with_pulp` gets an exact
    enumeration of its own integer program (ascending bitmask order, first strictly better selection wins)."""
    sys.path.insert(0, HERE)
    import consensus_scenario as sc
    import deva.inference.consensus_automatic as CA
    from deva.inference.consensus_associated import find_consensus_with_established_association, spatial_alignment
    from deva.inference.frame_utils import FrameInfo
    from deva.inference.image_feature_store import ImageFeatureStore
    from deva.inference.object_info import ObjectInfo
    from deva.utils.tensor_utils import pad_divide_by

    def brute(pairwise_iou, indicator, total):
        w = [float(pairwise_iou[:, i].sum() * 2) - 1.0 for i in range(total)]
        conflicts = [(i, j) for i in range(total) for j in range(i + 1, total) if indicator[i, j]]
        best_v, best_x = 0.0, 0
        for x in range(1, 1 << total):
            if any((x >> i) & 1 and (x >> j) & 1 for i, j in conflicts):
                continue
            v = sum(w[i] for i in range(total) if (x >> i) & 1)
            if v > best_v + 1e-9:
                best_v, best_x = v, x
        return [bool((best_x >> i) & 1) for i in range(total)]

    CA.use_gurobi = False
    CA.solve_with_pulp = brute
    sd = param_spec.synthetic_state_dict(seed=1)
    net = DEVA(CFG).eval()
    net.load_weights(sd)
    data = sc.frames()

    def frame_infos():
        out = []
        for ti, (image, ids), dets in zip(sc.TIMES, data, sc.DETECTIONS):
            infos = [ObjectInfo(sid, category_id=cat, isthing=thing, score=score) for sid, _, cat, thing, score in dets]
            out.append(FrameInfo(image, ids, infos, ti, {}))
        return out

    arrays, meta = {}, {'config': CFG, 'auto': {}}
    # (1) spatial_alignment frame 0 -> frame 1, two objects
    store = ImageFeatureStore(net, no_warning=True)
    img0, pads = pad_divide_by(data[0][0], 16)
    img1, _ = pad_divide_by(data[1][0], 16)
    m0, _ = pad_divide_by(torch.stack([data[0][1] == 3, data[0][1] == 5]).float(), 16)
    arrays['align_prob'] = spatial_alignment(10, img0, m0, 11, img1, net, store, CFG)[0]
    # (2) established association over frames 0, 1, 3 (channels: object A, object B)
    store = ImageFeatureStore(net, no_warning=True)
    pick = [(0, (3, 5)), (1, (1, 4)), (3, (7, 8))]
    images = [data[i][0].clone() for i, _ in pick]
    masks = [torch.stack([data[i][1] == a, data[i][1] == b]).float() for i, (a, b) in pick]
    kti, total = find_consensus_with_established_association([sc.TIMES[i] for i, _ in pick], images, masks, net, store, CFG)
    arrays['established_mask'] = total
    meta['established_keyframe'] = kti
    kti, total = find_consensus_with_established_association([sc.TIMES[i] for i, _ in pick],
                                                            [data[i][0].clone() for i, _ in pick],
                                                            [torch.stack([data[i][1] == a, data[i][1] == b]).float()
                                                             for i, (a, b) in pick], net,
                                                            ImageFeatureStore(net, no_warning=True), CFG,
                                                            scores=[0.2, 0.9, 0.5])
    arrays['established_mask_scored'] = total
    meta['established_keyframe_scored'] = kti

    # (3) automatic association, the real projection
    def run(tag, keyframe):
        kti, mask, infos = CA.find_consensus_auto_association(frame_infos(), keyframe, network=net,
                                                              store=ImageFeatureStore(net, no_warning=True), config=CFG)
        arrays[f'auto_{tag}_mask'] = mask
        meta['auto'][tag] = {'keyframe': kti, 'segments': [[o.id, o.category_ids, o.scores] for o in infos]}
        print('  consensus', tag, kti, [o.id for o in infos], 'ids in mask', mask.unique().tolist())

    run('real_first', 'first')
    # (4) automatic association on prescribed projections: pins matching / selection / merging / painting
    real = CA.spatial_alignment
    CA.spatial_alignment = lambda *a: sc.shifted_alignment(*a[:5])
    for keyframe in ('first', 'last', 'middle'):
        run('shifted_' + keyframe, keyframe)
    CA.spatial_alignment = real
    save('consensus.npz', **arrays)
    json.dump(meta, open(os.path.join(HERE, 'consensus.json'), 'w'))


def golden_match_and_merge():
    """segment_merging.match_and_merge over three detection rounds (plain / incremental / object cap)."""
    sys.path.insert(0, HERE)
    import consensus_scenario as sc
    import warnings
    from deva.inference.object_info import ObjectInfo
    from deva.inference.object_manager import ObjectManager
    from deva.inference.segment_merging import match_and_merge
    np.random.seed(5)
    om = ObjectManager()
    om.add_new_objects([ObjectInfo(i, category_id=c, isthing=t, score=s) for i, c, t, s in sc.MERGE_TRACKED])
    our_boxes = dict(sc.MERGE_OUR_BOXES)
    arrays, rounds = {}, []
    for r, (dets, incremental, cap, override) in enumerate(sc.MERGE_ROUNDS):
        if override is not None:
            our_boxes = dict(override)
        our = sc.merge_masks(our_boxes)
        new = sc.merge_masks({d[0]: d[1] for d in dets})
        infos = [ObjectInfo(d[0], category_id=d[2], isthing=d[3], score=d[4]) for d in dets]
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            one_hot = match_and_merge(our, new, om, infos, max_num_objects=cap, incremental_mode=incremental)
        arrays[f'merge_{r}'] = one_hot.to(torch.uint8)
        rounds.append([[t, o.id, o.poke_count, list(o.category_ids), list(o.scores)] for t, o in om.tmp_id_to_obj.items()])
        print('  merge round', r, [(t, o.id, o.poke_count) for t, o in om.tmp_id_to_obj.items()])
    save('match_and_merge.npz', **arrays)
    json.dump({'rounds': rounds}, open(os.path.join(HERE, 'match_and_merge.json'), 'w'))


def golden_object_manager():
    """ObjectManager / ObjectInfo bookkeeping script (ids, random re-ids, deletion, purging, votes): integer-exact."""
    sys.path.insert(0, HERE)
    import consensus_scenario as sc
    from deva.inference.object_info import ObjectInfo
    from deva.inference.object_manager import ObjectManager
    log = sc.object_manager_script(ObjectManager, ObjectInfo)
    json.dump(log, open(os.path.join(HERE, 'object_manager.json'), 'w'))
    print('wrote object_manager.json', len(log), 'snapshots; final', log[-2]['tmp_to_obj'])


def golden_eval_args():
    from argparse import ArgumentParser
    from deva.inference.eval_args import add_common_eval_args
    p = ArgumentParser()
    add_common_eval_args(p)
    ref = {a.dest: [a.default, type(a).__name__, (a.type.__name__ if a.type else None)] for a in p._actions if a.dest != 'help'}
    json.dump(ref, open(os.path.join(HERE, 'eval_args.json'), 'w'), indent=0)
    print('wrote eval_args.json', len(ref))


def golden_detections():
    """incorporate_detection + step over a semi-online session (inference_core.py:137-290): probabilities, object
    manager state (ids, poke counts, merged meta) and bank sizes after every call."""
    sys.path.insert(0, HERE)
    import consensus_scenario as sc
    from deva.inference.object_info import ObjectInfo
    sd = param_spec.synthetic_state_dict(seed=1)
    cfg = dict(CFG, **sc.DETECT_CONFIG_EXTRA)
    net = DEVA(cfg).eval()
    net.load_weights(sd)
    np.random.seed(42)
    core = DEVAInferenceCore(net, cfg)
    frames = sc.detect_frames()
    arrays, states = {}, []
    # also record what the reference's detection frames see internally: the forward prediction (inference_core.py:163-167)
    # and its argmax - random-init probabilities are near-uniform, so that argmax is ill-conditioned; the product test
    # checks its own forward prediction against these and continues on the reference's forward mask
    import deva.inference.inference_core as ic
    seen = {}
    real_merge, real_segment = ic.match_and_merge, core._segment

    def merge_spy(forward_mask, *a, **k):
        seen['fwd'] = forward_mask.clone()
        return real_merge(forward_mask, *a, **k)

    def segment_spy(*a, **k):
        seen['prob'] = real_segment(*a, **k)
        return seen['prob']

    ic.match_and_merge, core._segment = merge_spy, segment_spy
    for t, (frame, dets) in enumerate(zip(frames, sc.DETECT_SESSION)):
        seen.clear()
        if dets is None:
            p = core.step(frame, end=(t == len(frames) - 1))
        else:
            ids = sc.merge_masks({d[0]: d[1] for d in dets}, sc.DETECT_HW)
            infos = [ObjectInfo(d[0], category_id=d[2], isthing=d[3], score=d[4]) for d in dets]
            p = core.incorporate_detection(frame, ids, infos)
            arrays[f'fwd_{t:02d}'] = seen['fwd'].to(torch.int16)
            if 'prob' in seen:
                arrays[f'fwdprob_{t:02d}'] = seen['prob'].clone()
        arrays[f'prob_{t:02d}'] = p.clone()
        mem = core.memory
        states.append({'objects': [[tt, o.id, o.poke_count, list(o.category_ids), list(o.scores)]
                                   for tt, o in core.object_manager.tmp_id_to_obj.items()],
                       'sizes': {str(b): [mem.work_mem.size(b), mem.long_mem.size(b)] for b in mem.work_mem.buckets}})
        print('  detections t', t, 'prob', tuple(p.shape), states[-1]['objects'], states[-1]['sizes'])
    ic.match_and_merge = real_merge
    save('detections.npz', **arrays)
    json.dump({'config': cfg, 'states': states}, open(os.path.join(HERE, 'detections.json'), 'w'))


def golden_read_memory():
    """DEVA.read_memory (network.py:72-92), the training-time read: full softmax over T*H*W memory tokens."""
    torch.manual_seed(5)
    B, K, CK, CV, T, H, W = 2, 2, 64, 128, 3, 6, 9
    net = DEVA(dict(CFG, value_dim=CV)).eval()
    qk, qe = torch.randn(B, CK, H, W), torch.sigmoid(torch.randn(B, CK, H, W))
    mk, ms = torch.randn(B, CK, T, H, W), 1 + torch.rand(B, 1, T, H, W)
    mv = torch.randn(B, K, CV, T, H, W)
    out = net.read_memory(qk, qe, mk, ms, mv)
    save('read_memory.npz', qk=qk, qe=qe, mk=mk, ms=ms, mv=mv, out=out)


def golden_config1():
    """BASELINE configs[0]: the reference's own example clip (example/vos/bmx-trees, 4 frames 854x480, first-frame ids
    {1, 2}) through DEVAInferenceCore.step exactly as evaluation/eval_vos.py:110-198 drives it (generic dataset, size 480,
    no flip): frames decoded and normalised like deva/inference/data/video_reader.py:146-170, per-video config like
    eval_vos.py:124-128.  Stored: the decoded uint8 frames, the annotation, and per frame the reference's id map, the
    confident-pixel mask (top-2 margin > 0.05, bit-packed) and the probabilities on a stride-4 lattice (fp16 storage of
    fp32 values is NOT used: kept fp32 so the 1e-3 contract can be checked)."""
    from PIL import Image
    from torchvision import transforms
    root = os.path.join(REF, 'example', 'vos')
    vid = 'bmx-trees'
    names = sorted(os.listdir(os.path.join(root, 'JPEGImages', vid)))
    norm = transforms.Compose([transforms.ToTensor(),
                               transforms.Normalize(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])])  # dataset/utils.py
    frames_u8 = np.stack([np.array(Image.open(os.path.join(root, 'JPEGImages', vid, n)).convert('RGB')) for n in names])
    mask0 = np.array(Image.open(os.path.join(root, 'Annotations', vid, names[0][:-4] + '.png')))
    labels = [int(v) for v in np.unique(mask0) if v != 0]
    cfg = dict(CFG)
    vid_length = len(names)
    cfg['enable_long_term_count_usage'] = bool(cfg['enable_long_term'] and (
        vid_length / (cfg['max_mid_term_frames'] - cfg['min_mid_term_frames']) * cfg['num_prototypes']) >= cfg['max_long_term_elements'])
    net = DEVA(cfg).eval()
    net.load_weights(param_spec.synthetic_state_dict(seed=1))
    np.random.seed(42)
    core = DEVAInferenceCore(net, cfg)
    arrays = dict(mask0=mask0.astype(np.uint8))  # the frames are stored as the example's JPEG files
    for t in range(vid_length):
        image = norm(Image.fromarray(frames_u8[t]))
        mask = torch.from_numpy(mask0.astype(np.int64)) if t == 0 else None
        prob = core.step(image, mask, labels if t == 0 else None, end=(t == vid_length - 1))
        ids = core.object_manager.tmp_to_obj_cls(torch.argmax(prob, dim=0))
        top2 = torch.topk(prob, 2, dim=0)[0]
        arrays[f'ids_{t}'] = ids.numpy().astype(np.uint8)
        arrays[f'confident_{t}'] = np.packbits(((top2[0] - top2[1]) > 0.05).numpy())
        arrays[f'prob_lattice_{t}'] = prob[:, 1::4, 2::4].contiguous().numpy()
        print('  config1 t', t, 'prob', tuple(prob.shape), 'ids', np.unique(arrays[f'ids_{t}']).tolist(),
              'confident', float(((top2[0] - top2[1]) > 0.05).float().mean()))
    save('config1_vos.npz', **arrays)
    os.makedirs(os.path.join(HERE, vid), exist_ok=True)
    for n in names:
        shutil.copyfile(os.path.join(root, 'JPEGImages', vid, n), os.path.join(HERE, vid, n))
    json.dump({'config': cfg, 'labels': labels, 'frames': names, 'video': vid,
               'frames_u8_sha256': fixtures.sha256(frames_u8)},
              open(os.path.join(HERE, 'config1_vos.json'), 'w'))


if __name__ == '__main__':
    golden_read_memory()
    golden_config1()
    golden_spec()
    golden_memory_read()
    golden_bank_trace()
    golden_network()
    golden_vos()
    golden_consensus()
    golden_match_and_merge()
    golden_object_manager()
    golden_eval_args()
    golden_detections()
