"""Bank-sharded single-video mode (BASELINE configs[4]): ShardedDEVAInferenceCore against the plain core.

* one rank (no process group): the sharded code path - candidate merge, scatter read-out into the peer buffer,
  object-partitioned decode, token-sliced append, distributed consolidation hooks - must reproduce the plain core;
* two ranks over NCCL (skipped on a 1-GPU box): every rank must return the same probabilities as the unsharded run;
  slots, objects and prototypes are really split (bank sizes are halves)."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _clip(golden_dir):
    from oracle import fixtures
    arrays, meta = fixtures.vos_steps(golden_dir)
    return {k: torch.from_numpy(v) for k, v in arrays.items()}, meta


def _run(core, g, device):
    T = g['frames'].shape[0]
    out, sizes = [], []
    for t in range(T):
        img = g['frames'][t].to(device)
        if t == 0:
            p = core.step(img, g['mask0'].to(device), [1, 2])
        elif t == 6:
            p = core.step(img, g['mask6'].to(device), [7])
        else:
            p = core.step(img, end=(t == T - 1))
        out.append(p.float().cpu())
        mem = core.memory
        sizes.append({str(b): [mem.work_mem.size(b), mem.long_mem.size(b)] for b in mem.work_mem.buckets})
    return out, sizes


def _net(meta, sd, device):
    from deva.model.network import DEVA
    net = DEVA(meta['config'])
    net.conv_backend = 'native'
    net = net.to(device).eval()
    net.load_weights({k: v.to(device) for k, v in sd.items()})
    return net


def test_sharded_core_on_one_rank_equals_plain_core(golden_dir, synthetic_sd):
    from deva.inference.inference_core import DEVAInferenceCore
    from deva.inference.sharded_core import ShardedDEVAInferenceCore
    g, meta = _clip(golden_dir)
    np.random.seed(42)
    plain, plain_sizes = _run(DEVAInferenceCore(_net(meta, synthetic_sd, 'cuda'), meta['config']), g, 'cuda')
    np.random.seed(42)
    shard, shard_sizes = _run(ShardedDEVAInferenceCore(_net(meta, synthetic_sd, 'cuda'), meta['config']), g, 'cuda')
    assert shard_sizes == plain_sizes == meta['sizes']
    worst = max(float((a - b).abs().max()) for a, b in zip(plain, shard))
    ref = max(float((a - g[f'prob_{t:02d}']).abs().max()) for t, a in enumerate(shard))
    print(f'sharded core on one rank: max |prob - plain core| = {worst:.2e}, vs reference {ref:.2e}')
    assert worst < 2e-5, worst  # same kernels; the read-out goes through fp32 red.add instead of a plain store
    assert ref < 1e-3, ref


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank, world, port, golden_dir, out_path):
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for p in (root, os.path.join(root, 'tracking-anything-with-deva_b200')):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch.distributed as dist
    from deva.inference.sharded_core import ShardedDEVAInferenceCore
    from deva.model.param_spec import synthetic_state_dict
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device('cuda', rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=dev)
    g, meta = _clip(golden_dir)
    cfg = dict(meta['config'], num_prototypes=128, max_long_term_elements=300 - 300 % world)
    np.random.seed(42)
    core = ShardedDEVAInferenceCore(_net(dict(config=cfg), synthetic_state_dict(seed=1), dev), cfg)
    probs, sizes = _run(core, g, dev)
    if rank == 0:
        torch.save({'probs': probs, 'sizes': sizes}, out_path)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs 2 GPUs')
def test_sharded_core_on_two_ranks_matches_reference(golden_dir, tmp_path):
    import torch.multiprocessing as mp
    g, meta = _clip(golden_dir)
    out_path = str(tmp_path / 'rank0.pt')
    mp.spawn(_worker, args=(2, _free_port(), golden_dir, out_path), nprocs=2, join=True)
    got = torch.load(out_path)
    worst = max(float((a - g[f'prob_{t:02d}']).abs().max()) for t, a in enumerate(got['probs']))
    print(f'sharded core on two ranks: max |prob - reference| = {worst:.2e}')
    assert worst < 1e-3, worst
    # the bank really is split: every rank holds half of every bucket
    want = [{b: [w // 2, l // 2] for b, (w, l) in s.items()} for s in meta['sizes']]
    assert got['sizes'] == want, (got['sizes'], want)
