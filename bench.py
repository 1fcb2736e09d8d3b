#!/usr/bin/env python
"""Benchmark of the DEVA propagation hot path on B200 (contract: see the task statement / DESIGN.md).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3|c2] [--dump-outputs DIR]

Workload (BASELINE.json configs[2], "c3"): synthetic 1080p frames (padded 1088x1920, Q = 8160 query
positions), 16 objects, memory bank pre-filled to 10 000 slots, full encode -> read -> decode per frame
through ``DEVAInferenceCore.step``; every 5th frame is a memory frame (value encoder + bank append,
``mem_every=5``) after which the bank is clamped back to 10 000 slots so the configuration stays the named
one.  One step = one frame.  Metric = propagation FPS (whole job, all ranks).  N > 1: one process per GPU,
each rank propagates its own clip (clip-parallel, weak scaling, NCCL barrier only - BASELINE configs[3]).

Printed JSON line: metric/value/unit/... plus
  roofline      fused affinity path (pack_query + similarity/top-k/softmax + readout GEMM), algorithmic
                FLOPs 2*N*Q*2CK + 2*K*CV*N*Q per frame / CUDA-event time per frame, vs measured bf16 peak;
                roofline_conv: the same for the convolution stack (algorithmic conv FLOPs / CUDA-event time);
  e2e           same FPS through the public API with host frames (pinned H2D of every frame, D2H of the id mask);
  cpu_baseline  the UNMODIFIED reference (oracle/_ref, staged by oracle/build_ref.py) on this box's host cores, on a
                bounded sample (all shared stages + `--ref-objects` of the K objects, linearly extrapolated and flagged);
  torch_gpu_baseline  the unmodified reference on the SAME B200 (all K objects): fp32 (PyTorch's TF32 default), fp32
                with TF32 off, and --amp (fp16 autocast, evaluation/eval_vos.py:137) - the real bar;
  clocks        SM clock / throttle reasons sampled with nvidia-smi during the timed region.
``--impl reference`` times the reference's own ``DEVAInferenceCore.step`` on the host cores (``oracle/_ref``; the
oracle port only when the staged copy is missing).
``--dump-outputs DIR`` writes what the last timed step returned (see dump_outputs) so that two builds can be compared
output for output: every input is seeded, so the same arguments give the same inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

sys.dont_write_bytecode = True  # the tree may be read-only; the bench writes nothing into it
ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, 'tracking-anything-with-deva_b200')
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

try:  # a baseline leg started by a pinned parent (see _run_leg) gets every host core back, before torch sizes its pools
    if os.environ.get('DEVA_B200_BENCH_CORES'):
        os.sched_setaffinity(0, {int(c) for c in os.environ['DEVA_B200_BENCH_CORES'].split(',')})
    ALL_CORES = os.sched_getaffinity(0)
except Exception:
    ALL_CORES = None

import torch  # noqa: E402

CK, CV, TOP_K = 64, 512, 30
WORKLOADS = {
    'c3': dict(name='c3: 1080p, 16 objects, 10k memory slots, full encode->read->decode', h=1080, w=1920, k=16,
               n=10000),
    'c2': dict(name='c2: 480p, 5 objects, 2k memory slots', h=480, w=854, k=5, n=2000),
    # BASELINE configs[3]: 64 independent 480p clips sharded round-robin over the ranks (clip-parallel; a step = one frame
    # of EVERY clip, total work fixed -> strong scaling)
    'c4': dict(name='c4: 64 independent 480p clips, 5 objects, 2k memory slots each, clip-parallel', h=480, w=854, k=5,
               n=2000, clips=64),
    # BASELINE configs[4]: ONE 1080p video, 32 objects, 50k memory slots: bank sharded over the ranks + object-parallel
    # decode (deva.inference.sharded_core); every rank sees every frame, total work fixed -> strong scaling
    'c5': dict(name='c5: single 1080p clip, 32 objects, 50k memory slots, bank-sharded + object-parallel', h=1080, w=1920,
               k=32, n=50000, sharded=True),
}
METRIC = 'propagation FPS @1080p, 10k-mem, 16 obj; affinity GEMM TFLOPS vs bf16 peak'


def base_config():
    return dict(key_dim=CK, value_dim=CV, pix_feat_dim=512, mem_every=5, enable_long_term=True, chunk_size=-1,
                top_k=TOP_K, enable_long_term_count_usage=True, max_mid_term_frames=10, min_mid_term_frames=5,
                num_prototypes=128, max_long_term_elements=10000)


def synth_frames(wl, count, seed):
    g = torch.Generator().manual_seed(seed)
    base = torch.randn(3, wl['h'], wl['w'], generator=g)
    return torch.stack([base + 0.2 * torch.randn(3, wl['h'], wl['w'], generator=g) for _ in range(count)])


def synth_mask(wl):
    """K rectangles on a grid, ids 1..K."""
    k, h, w = wl['k'], wl['h'], wl['w']
    cols = 4 if k > 4 else k
    rows = (k + cols - 1) // cols
    m = torch.zeros(h, w, dtype=torch.long)
    for i in range(k):
        r, c = divmod(i, cols)
        y0, x0 = int((r + 0.15) * h / rows), int((c + 0.15) * w / cols)
        m[y0:y0 + int(0.6 * h / rows), x0:x0 + int(0.6 * w / cols)] = i + 1
    return m


DUMP_LIMIT = 60 << 20  # bytes of array data in all files of --dump-outputs: the dump stays under 64 MB


def dump_outputs(path, outputs, limit=DUMP_LIMIT, seed=0):
    """Write ``outputs`` (name -> probabilities [C, H, W]) as float32 ``path/<name>.npy``.  When they exceed ``limit``
    bytes together, each is stored as [C, S] instead: the same S pixel positions of every output, drawn with a fixed seed
    and kept in raster order, S as large as the limit allows."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    per_pixel = sum(4 * t.shape[0] for t in outputs.values())
    sample = {}
    for name, t in outputs.items():
        x = t.detach().float()
        hw = x[0].numel()
        if per_pixel * max(u[0].numel() for u in outputs.values()) > limit:
            if hw not in sample:
                g = torch.Generator().manual_seed(seed)
                sample[hw] = torch.randperm(hw, generator=g)[:limit // per_pixel].sort().values
            x = x.reshape(x.shape[0], hw)[:, sample[hw].to(x.device)]
        np.save(os.path.join(path, name + '.npy'), x.cpu().numpy())


def read_flops(wl, q):
    return 2.0 * wl['n'] * q * 2 * CK + 2.0 * wl['k'] * CV * wl['n'] * q


class ClockSampler:
    QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
             'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(suffix='.csv')
        self.proc = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={gpu_index}', f'--query-gpu={self.QUERY}',
                                          '--format=csv,noheader,nounits', '-lms', '50'],
                                         stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def mark(self):
        """Samples written so far (start-up, warm-up) are dropped by stop()."""
        try:
            self.skip = sum(1 for _ in open(self.path))
        except Exception:
            self.skip = 0

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for n_line, line in enumerate(open(self.path)):
                if n_line < getattr(self, 'skip', 0):
                    continue
                f = [x.strip() for x in line.split(',')]
                if len(f) < 9:
                    continue
                sm.append(float(f[1])); mx.append(float(f[2]))
                for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'),
                                     f[5:9]):
                    if val.lower().startswith('active'):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------------------------------------ ours
def make_network(device):
    from deva.model.network import DEVA
    from deva.model.param_spec import synthetic_state_dict
    net = DEVA(base_config()).to(device).eval()
    net.load_weights({k: v.to(device) for k, v in synthetic_state_dict(seed=0).items()})
    return net


class Clip:
    """One clip on one GPU (or, for a sharded workload, this rank's share of the one clip): core + bank pre-filled to
    wl['n'] slots."""
    def __init__(self, wl, device, seed, net=None):
        from deva import _native as nat
        from deva.inference.inference_core import DEVAInferenceCore
        nat.require_device()
        self.nat, self.wl, self.device = nat, wl, device
        cfg = base_config()
        net = net or make_network(device)
        if wl.get('sharded'):
            from deva.inference.sharded_core import ShardedDEVAInferenceCore, token_bounds
            self.core = ShardedDEVAInferenceCore(net, cfg)
            world, rank = self.core.world, self.core.rank
        else:
            self.core = DEVAInferenceCore(net, cfg)
            world, rank = 1, 0
        self.frames_host = synth_frames(wl, 5, seed).pin_memory()
        self.frames_dev = self.frames_host.to(device)
        ids = list(range(1, wl['k'] + 1))
        self.core.step(self.frames_dev[0], synth_mask(wl).to(device), ids)  # first frame -> Q memory tokens
        mem = self.core.memory
        bank = next(iter(mem._banks.values()))
        self.q = (-(-wl['h'] // 16)) * (-(-wl['w'] // 16))
        extra = wl['n'] - self.q
        assert extra >= 0, 'bank already larger than the configured slot count'
        if extra > 0:  # random-init top-up to exactly n slots (BASELINE.md section 4 generator); every rank draws the
            # same tokens and keeps its slice
            lo, hi = (0, extra) if world == 1 else token_bounds(extra, world, rank)
            g = torch.Generator(device=device).manual_seed(seed + 1)
            key = torch.randn(1, CK, extra, 1, device=device, generator=g)[:, :, lo:hi]
            shr = (1 + torch.rand(1, 1, extra, 1, device=device, generator=g))[:, :, lo:hi]
            sel = torch.sigmoid(torch.randn(1, CK, extra, 1, device=device, generator=g))[:, :, lo:hi]
            val = torch.cat([torch.randn(1, 1, CV, extra, 1, device=device, generator=g)[:, :, :, lo:hi]
                             for _ in range(wl['k'])], 1)
            mem.add_memory(key.contiguous(), shr.contiguous(), val, ids, selection=sel.contiguous())
        self.bank, self.mark = bank, bank.hi
        total = torch.tensor([bank.work_size], device=device)
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(total)
        assert int(total) == wl['n'], (int(total), wl['n'])
        self.i = 0

    def clamp(self):
        if self.core.last_mem_ti == self.core.curr_ti:  # a memory frame was just appended
            self.bank.hi = self.mark

    def step_resident(self):
        p = self.core.step(self.frames_dev[self.i % 5])
        self.clamp()
        self.i += 1
        return p

    def step_e2e(self):
        """What a user of the public API does per frame (evaluation/eval_vos.py:138-198)."""
        img = self.frames_host[self.i % 5].to(self.device, non_blocking=True)
        p = self.core.step(img)
        ids = self.core.object_manager.tmp_to_obj_cls(torch.argmax(p, dim=0)).to(torch.uint8)
        host = ids.cpu()
        self.clamp()
        self.i += 1
        return host


    def step_e2e_fused_io(self):
        """Same, with the decoded uint8 frame uploaded as is and the ingest / egress kernels of SURVEY 8(f)-3
        (deva.inference.frame_io): normalise on the device, fused argmax + id remap -> uint8 id map."""
        from deva.inference.frame_io import frame_from_rgb8, prob_to_ids
        if not hasattr(self, 'frames_u8'):
            mean = torch.tensor([0.485, 0.456, 0.406]).view(1, 3, 1, 1)
            std = torch.tensor([0.229, 0.224, 0.225]).view(1, 3, 1, 1)
            u8 = ((self.frames_host * std + mean) * 255).round().clamp(0, 255).to(torch.uint8)
            self.frames_u8 = u8.permute(0, 2, 3, 1).contiguous().pin_memory()
        img = frame_from_rgb8(self.frames_u8[self.i % 5], device=self.device)
        p = self.core.step(img)
        host = prob_to_ids(p, self.core.object_manager, dtype=torch.uint8).cpu()
        self.clamp()
        self.i += 1
        return host


class ClipSet:
    """Workload c4: this rank's share (round-robin, deva.utils.dist_utils.assign_clips) of the independent clips, all
    driven through ONE network; a step advances every clip by one frame."""
    def __init__(self, wl, device, rank, world):
        from deva.utils.dist_utils import assign_clips
        net = make_network(device)
        self.ids = assign_clips(wl['clips'], world, rank)
        self.clips = [Clip(wl, device, seed=100 + i, net=net) for i in self.ids]
        self.nat, self.wl, self.q = self.clips[0].nat, wl, self.clips[0].q
        self.core = self.clips[0].core
        self.frames_host = self.clips[0].frames_host

    def step_resident(self):
        return [c.step_resident() for c in self.clips]

    def step_e2e(self):
        for c in self.clips:
            c.step_e2e()

    def step_e2e_fused_io(self):
        for c in self.clips:
            c.step_e2e_fused_io()


HOST_MS = []  # host time (enqueue only, no sync) of every timed step of the last timed() call: a stall of the launching
              # thread (GC, scheduler, allocator) longer than the GPU's queued work shows up in the event time as well


def timed(fn, steps, dist_on):
    import gc
    import torch.distributed as dist
    if dist_on:
        dist.barrier()
    torch.cuda.synchronize()
    gc.collect()
    gc.disable()  # no collector pause between two launches of the timed region
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    del HOST_MS[:]
    out = None
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        h0 = time.perf_counter()
        out = None  # keep the last step's result without extending the life of an earlier one into the next step
        out = fn()
        HOST_MS.append((time.perf_counter() - h0) * 1e3)
    e1.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3
    gc.enable()
    ms = max(e0.elapsed_time(e1), 0.0)
    if dist_on:
        t = torch.tensor([ms, wall], device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.barrier()
        ms, wall = float(t[0]), float(t[1])
    return ms, wall, out


def pin_to_gpu_numa_node(gpu_index):
    """Keep this rank's (single, launch-issuing) host thread on the cores next to its GPU: the 8-GPU boxes have two
    sockets (SCALE topology: GPU0-3 on NUMA 0, GPU4-7 on NUMA 1) and an unpinned rank may issue its ~115 launches per frame
    across the socket interconnect."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cores = {64 * i + b for i, wd in enumerate(words) for b in range(64) if (wd >> b) & 1}
        allowed = cores & set(os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
        return sorted(allowed)
    except Exception:
        return None


def run_ours(args):
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', 0)); world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    dist_on = world > 1
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    pin_to_gpu_numa_node(local)
    if dist_on:
        dist.init_process_group('nccl', device_id=device)
    torch.backends.cudnn.benchmark = True
    wl = WORKLOADS[args.workload]
    if 'clips' in wl:      # c4: fixed set of clips split over the ranks
        clip = ClipSet(wl, device, rank, world)
        frames_per_step, scaling, n_clips_rank = wl['clips'], 'strong', len(clip.clips)
    elif wl.get('sharded'):  # c5: one clip, every rank works on every frame
        clip = Clip(wl, device, seed=100)
        frames_per_step, scaling, n_clips_rank = 1, 'strong', 1
    else:                  # c3 / c2: one clip per rank
        clip = Clip(wl, device, seed=100 + rank)
        frames_per_step, scaling, n_clips_rank = world, 'weak', 1
    nat = clip.nat
    # the clock sampler starts BEFORE the warm-up: nvidia-smi's start-up (NVML initialisation takes driver locks) must not
    # fall into the timed region; only samples taken during the timed region are kept (ClockSampler.mark)
    sampler = ClockSampler(local) if rank == 0 else None
    # Setup steps + the requested warm-up together cover at least one full mem_every period (6 steps): the first regular
    # memory frame grows the allocator's pools, which must not happen inside the timed region.  `warmup` in the JSON line is
    # the requested W (at least 3); the untimed steps before it (clip initialisation + priming) are counted in `setup_steps`.
    n_warm = max(args.warmup, 3)
    n_prime = max(0, 6 - n_warm)
    for _ in range(n_prime + n_warm):
        clip.step_resident()
    torch.cuda.synchronize()
    if sampler:
        sampler.mark()
    clip.core.memory.read_events = []
    l0 = nat.launch_count()
    ms, wall, last = timed(clip.step_resident, args.steps, dist_on)
    launches = nat.launch_count() - l0
    ev = clip.core.memory.read_events
    clip.core.memory.read_events = None
    read_ms = sum(a.elapsed_time(b) for a, b in ev) / max(len(ev), 1)
    clocks = sampler.stop() if sampler else None
    host_ms = sorted(HOST_MS)
    if args.dump_outputs and rank == 0:  # this rank's clips
        dump_outputs(args.dump_outputs, {f'prob_clip{i:02d}': p for i, p in zip(clip.ids, last)} if 'clips' in wl
                     else {'prob': last})
    del last

    for _ in range(2):
        clip.step_e2e()
    ms_e2e, _, _ = timed(clip.step_e2e, args.steps, dist_on)
    ms_e2e_io = 0.0
    if not args.quick:
        for _ in range(2):
            clip.step_e2e_fused_io()
        ms_e2e_io, _, _ = timed(clip.step_e2e_fused_io, args.steps, dist_on)

    # conv-stack roofline: a separate short pass with CUDA events around every conv launch (not part of `value`)
    from deva.model import native_ops
    precision = getattr(clip.core.network.engine, 'precision', 'n/a')
    conv_roof = None
    if args.quick:
        conv_ms = conv_flops = mma_flops = 0.0
    elif rank == 0 or wl.get('sharded'):  # a sharded clip steps on every rank (collectives inside the step)
        if rank == 0:
            native_ops.PROFILE = []
        for _ in range(5):  # exactly one memory frame
            clip.step_resident()
        torch.cuda.synchronize()
    if rank == 0 and not args.quick:
        prof, native_ops.PROFILE = native_ops.PROFILE, None
        conv_ms = sum(a.elapsed_time(b) for a, b, _, _ in prof) / 5
        conv_flops = sum(f for _, _, f, _ in prof) / 5
        mma_flops = sum(f * n for _, _, f, n in prof) / 5

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        peak = peaks.get('bf16_tflops_sustained', 1400.0)
        peak_src = 'MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)' if peaks else \
            'fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)'
        flops = read_flops(wl, clip.q)
        achieved = flops / (read_ms * 1e-3) / 1e12
        if wl.get('sharded'):  # every rank multiplies 1/world of the slots: per-GPU rate against one GPU's peak
            achieved /= world
        traffic = conv_traffic = None
        try:
            tr = json.load(open(os.path.join(ROOT, 'profiles', 'roofline_traffic.json')))
            traffic = tr.get(args.workload)  # readout_sparse_kernel, per launch
            conv_traffic = tr.get(args.workload + '_conv')
        except Exception:
            pass
        conv_ach = conv_flops / (conv_ms * 1e-3) / 1e12 if not args.quick else 0.0
        conv_roof = None if args.quick else {'kernel': 'conv_kernel (tcgen05 implicit GEMM), all launches of a frame', 'bound': 'tensor',
                     'achieved': conv_ach, 'peak': peak, 'unit': 'TFLOP/s', 'frac': conv_ach / peak,
                     'traffic': conv_traffic, 'ms_per_frame': conv_ms, 'flops_per_frame': conv_flops,
                     'what': 'algorithmic FLOPs 2*B*Ho*Wo*Cout*k*k*Cin per layer (extra split-precision passes NOT counted) / '
                             'CUDA-event time of the conv launches, 5-frame pass incl. one memory frame',
                     'executed_tflops': mma_flops / (conv_ms * 1e-3) / 1e12}
        h2d = int(clip.frames_host[0].numel() * 4)
        d2h = int(wl['h'] * wl['w'])
        out = {
            'metric': METRIC, 'value': frames_per_step * args.steps / (ms * 1e-3), 'unit': 'frames/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': n_warm, 'ms_per_step': ms / args.steps,
            'higher_is_better': True, 'scaling': scaling, 'vs_baseline': None, 'dtype': 'f16 MMA operands / f32 accumulate '
            f'(tcgen05 memory read + conv stack), precision plan {precision!r}; key path split-f16x3 (~f32)', 'data': 'synthetic',
            'config': workload_config(wl, clip.q, world), 'setup_steps': 1 + n_prime,
            'roofline': {'kernel': 'fused affinity path: pack_query + sim_topk(tcgen05 fp16x3) + merge + bucket + readout_sparse(tcgen05, '
                                   'affinity tiles built in smem); traffic = DRAM bytes of readout_sparse_kernel (ncu, the fp16 '
                                   'token-major output variant the step runs)',
                         'bound': 'tensor', 'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s',
                         'frac': achieved / peak, 'traffic': traffic, 'peak_source': peak_src,
                         'ms_per_launch': read_ms, 'flops_per_launch': flops},
            'roofline_conv': conv_roof,
            'e2e': {'value': frames_per_step * args.steps / (ms_e2e * 1e-3), 'unit': 'frames/s',
                    'h2d_bytes_per_step': h2d * n_clips_rank, 'd2h_bytes_per_step': d2h * n_clips_rank},
            'e2e_fused_io': None if args.quick else {'value': frames_per_step * args.steps / (ms_e2e_io * 1e-3), 'unit': 'frames/s',
                             'h2d_bytes_per_step': int(wl['h'] * wl['w'] * 3) * n_clips_rank,
                             'd2h_bytes_per_step': d2h * n_clips_rank,
                             'what': 'uint8 frame upload + on-device normalise; fused argmax + id remap (deva.inference.frame_io)'},
            'gpu_launches': int(launches), 'wall_ms_per_step': wall / args.steps, 'clocks': clocks,
            'host_enqueue_ms_per_step': {'median': host_ms[len(host_ms) // 2], 'max': host_ms[-1]} if host_ms else None,
            'precision_plan': precision,
        }
    # everything below runs without the clip: give the legs the device
    del clip
    torch.cuda.empty_cache()
    c5 = None
    if dist_on and args.workload == 'c3' and not args.quick and not args.no_c5_leg:
        # BASELINE configs[4] on the same ranks: the bank-sharded single video (workload c5) as a second process group of
        # child processes, one per rank, so that a failure or a hang there can never take the c3 line with it.
        c5 = _run_dist_leg(['--workload', 'c5', '--quick', '--steps', '10', '--warmup', '3', '--no-c5-leg'], timeout=240)
    if rank == 0:
        if c5 is not None:
            out['bank_sharded_c5'] = c5 if 'error' in c5 else {
                k: c5.get(k) for k in ('value', 'unit', 'n_gpus', 'steps', 'ms_per_step', 'scaling', 'config', 'roofline', 'e2e',
                                       'gpu_launches', 'precision_plan')}
        if world == 1 and not args.no_cpu_baseline:
            try:  # bounded sample: 1 warm-up + 5 timed sample steps (exactly one memory frame: the right 1-in-5 weight)
                # of the unmodified reference on the host cores; reference_cpu shortens it on a slow box and says so
                leg = _run_leg(['--impl', 'reference', '--steps', '5', '--warmup', '1', '--workload', args.workload,
                                '--ref-objects', str(args.ref_objects)], timeout=900)
                out['cpu_baseline'] = leg['cpu_baseline']
            except Exception as exc:
                out['cpu_baseline'] = {'error': f'{type(exc).__name__}: {exc}'[:300]}
        if world == 1 and not args.no_torch_baseline:
            try:
                out['torch_gpu_baseline'] = _run_leg(['--impl', 'reference_gpu', '--workload', args.workload], timeout=900)
            except Exception as exc:  # reported extra, never fatal for the bench line
                out['torch_gpu_baseline'] = {'error': f'{type(exc).__name__}: {exc}'[:300]}
        print(json.dumps(out))
    if dist_on:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------ fallback: the oracle port, stage by stage
def _oracle_stages(wl, budget_s, device, k_s):
    """One frame of the reference algorithm (the oracle's fp32 PyTorch restatement) on ``device``, stage by stage.
    Returns wall-clock seconds per stage; per-object stages run on ``k_s`` objects."""
    from deva.model.param_spec import synthetic_state_dict
    from oracle import memory_math as mm
    from oracle import network as onet
    from oracle.core import pad_to_multiple
    cuda = torch.device(device).type == 'cuda'

    def clock():
        if cuda:
            torch.cuda.synchronize()
        return time.perf_counter()

    sd = {name: v.to(device) for name, v in synthetic_state_dict(seed=0).items()}
    t_all = time.perf_counter()
    with torch.no_grad():
        img, _ = pad_to_multiple(synth_frames(wl, 1, 7)[0], 16)
        img = img.unsqueeze(0).to(device)
        t0 = clock()
        ms, feat = onet.encode_image(sd, img)
        key, shr, sel = onet.transform_key(sd, feat)
        t_shared = clock() - t0
        h, w = key.shape[-2:]
        n = wl['n']
        g = torch.Generator().manual_seed(0)
        mk, msh = torch.randn(CK, n, generator=g).to(device), (1 + torch.rand(n, generator=g)).to(device)
        mv = torch.randn(k_s * CV, n, generator=g).to(device)
        t0 = clock()
        sim = mm.similarity(mk, msh, key[0].flatten(1), sel[0].flatten(1))
        aff = mm.dense_affinity(sim, TOP_K)
        t_aff = clock() - t0
        t0 = clock()
        ro = mm.readout(aff, mv)
        t_ro = clock() - t0
        del sim, aff
        masks = synth_mask(wl)
        masks = torch.stack([(masks == (i % wl['k']) + 1).float() for i in range(k_s)])
        masks, _ = pad_to_multiple(masks, 16)
        masks = masks.unsqueeze(0).to(device)
        sens = torch.zeros(1, k_s, CV, h, w, device=device)
        t0 = clock()
        onet.segment(sd, ms, ro.view(1, k_s, CV, h, w), sens, masks)
        t_seg = clock() - t0
        t_enc = None
        if time.perf_counter() - t_all < budget_s:
            t0 = clock()
            onet.encode_mask(sd, img, ms, sens, masks)
            t_enc = clock() - t0
    return {'encode': t_shared, 'affinity': t_aff, 'readout': t_ro, 'decode': t_seg, 'encode_mask': t_enc}


def _blend(st, scale):
    per_frame = st['encode'] + st['affinity'] + (st['readout'] + st['decode']) * scale
    if st['encode_mask'] is not None:
        per_frame += st['encode_mask'] * scale / 5.0
    return per_frame


def cpu_baseline_port(wl, budget_s):
    """Reference-algorithm frame rate on the host cores: the oracle's stages on a bounded sample.

    Object-independent stages run in full; per-object stages run on ``k_s`` of the K objects and are scaled by
    K/k_s (every per-object op is independent across objects, SURVEY quirk Q11)."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    k, k_s = wl['k'], 1
    st = _oracle_stages(wl, budget_s, 'cpu', k_s)
    scale = k / k_s
    return {'value': 1.0 / _blend(st, scale), 'unit': 'frames/s', 'cores': cores, 'kind': 'port',
            'sample': f'1 frame {wl["h"]}x{wl["w"]}, N={wl["n"]}: encode_image+transform_key and similarity/top-k in '
                      f'full; readout, decoder' + (', value encoder (1 frame in 5)' if st['encode_mask'] is not None else '') +
                      f' on {k_s} of {k} objects, scaled x{scale:g}; oracle = fp32 PyTorch-CPU port of the reference',
            'stage_s': {'encode': st['encode'], 'affinity': st['affinity'], 'readout_per_obj': st['readout'],
                        'decode_per_obj': st['decode'], 'encode_mask_per_obj': st['encode_mask']}}


# ---------------------------------------------------------------------- unmodified reference (oracle/_ref)
def workload_config(wl, q, world):
    """The `config` object of the JSON line - identical for the product arm and the reference arm."""
    return {'workload': wl['name'], 'frame': [wl['h'], wl['w']], 'query_positions': q, 'objects': wl['k'],
            'memory_slots': wl['n'], 'mem_every': 5, 'top_k': TOP_K,
            'parallelism': f'clip-parallel x{world}' if world > 1 else 'single clip',
            'l2': 'per-step working set (activations > 2 GB) exceeds the 126 MB L2; no explicit flush',
            'weights': 'synthetic_state_dict(seed=0), real architecture (69.2 M parameters)'}


class RefClip:
    """The same clip as ``Clip`` driven through the UNMODIFIED reference (DEVA + DEVAInferenceCore from oracle/_ref):
    same seeded frames, masks, checkpoint and random bank top-up; ``n_obj`` of the workload's objects."""
    def __init__(self, wl, device, n_obj, seed):
        from oracle import ref_loader
        DEVA, Core, synth = ref_loader.load()
        self.wl, self.device, self.n_obj = wl, device, n_obj
        cfg = base_config()
        net = DEVA(cfg).to(device).eval()
        net.load_weights({k: v.to(device) for k, v in synth(seed=0).items()})
        self.net = net
        self.core = Core(net, cfg)
        self.frames = synth_frames(wl, 5, seed).to(device)
        ids = list(range(1, n_obj + 1))
        mask = synth_mask(wl)
        mask[mask > n_obj] = 0
        self.core.step(self.frames[0], mask.to(device), ids)
        mem = self.core.memory
        self.bucket = next(iter(mem.work_mem.buckets))
        self.q = mem.HW
        extra = wl['n'] - mem.work_mem.size(self.bucket)
        assert extra >= 0
        if extra > 0:
            g = torch.Generator().manual_seed(seed + 1)
            key = torch.randn(1, CK, extra, 1, generator=g).to(device)
            shr = (1 + torch.rand(1, 1, extra, 1, generator=g)).to(device)
            sel = torch.sigmoid(torch.randn(1, CK, extra, 1, generator=g)).to(device)
            val = torch.randn(1, n_obj, CV, extra, 1, generator=g).to(device)
            mem.add_memory(key, shr, val, ids, selection=sel)
        assert mem.work_mem.size(self.bucket) == wl['n']
        self.i = 0

    def clamp(self):
        """Keep the configuration the named one: drop what a memory frame just appended (kv_memory_store.py:35-116)."""
        if self.core.last_mem_ti != self.core.curr_ti:
            return
        wm, b, n = self.core.memory.work_mem, self.bucket, self.wl['n']
        wm.k[b], wm.s[b], wm.e[b] = wm.k[b][:, :n], wm.s[b][:, :n], wm.e[b][:, :n]
        wm.use_cnt[b], wm.life_cnt[b] = wm.use_cnt[b][:n], wm.life_cnt[b][:n]
        for obj in wm.buckets[b]:
            wm.v[obj] = wm.v[obj][:, :n]

    def step(self):
        p = self.core.step(self.frames[self.i % 5])
        self.clamp()
        self.i += 1
        return p


class _SharedTimer:
    """Accumulates the wall time of the object-independent stages of a reference step (CPU: calls are synchronous):
    encode_image, transform_key (network.py:42-68) and get_similarity / do_softmax (memory_utils.py:6-76)."""
    def __init__(self, net):
        import deva.inference.memory_manager as mmod  # the reference's (oracle/_ref)
        self.total = 0.0
        self._undo = []
        for obj, name in ((net, 'encode_image'), (net, 'transform_key'), (mmod, 'get_similarity'), (mmod, 'do_softmax')):
            fn = getattr(obj, name)
            setattr(obj, name, self._wrap(fn))
            self._undo.append((obj, name, fn))

    def _wrap(self, fn):
        def timed_fn(*a, **k):
            t0 = time.perf_counter()
            try:
                return fn(*a, **k)
            finally:
                self.total += time.perf_counter() - t0
        return timed_fn

    def close(self):
        for obj, name, fn in self._undo:
            setattr(obj, name, fn)


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def reference_cpu(wl, steps, warmup, n_obj, budget_s=150.0):
    """The reference's own step() on the host cores.  A step of the sample is one full-resolution frame of the named
    workload with ``n_obj`` of its K objects; every per-object stage of DEVA is independent across objects (the
    reference's own note, docs/DEMO.md:41: run time is linear in the number of objects), so the full-frame time is
    shared + K * per_object with both terms MEASURED here.  Returns the cpu_baseline record."""
    cores = host_cores()
    torch.set_num_threads(cores)
    torch.set_grad_enabled(False)
    k = wl['k']
    n_obj = max(1, min(n_obj, k))
    t_build = time.perf_counter()
    clip = RefClip(wl, 'cpu', n_obj, seed=100)
    t_build = time.perf_counter() - t_build
    t_warm, warm_done, t_warm_all = 0.0, 0, time.perf_counter()
    for _ in range(warmup):  # at least one; no further ones once a minute has gone into warming up
        t0 = time.perf_counter()
        clip.step()
        t_warm = time.perf_counter() - t0
        warm_done += 1
        if time.perf_counter() - t_warm_all > 60.0:
            break
    # time budget of the timed region (a sample step is 4 s on a fast 64-core box, 30 s on a slow 128-core one): never fewer
    # than 2 steps, never more than requested; a shortened run is flagged and the value stays a per-step average
    requested = steps
    if t_warm > 0 and steps * t_warm > budget_s:
        steps = max(2, min(steps, int(budget_s / t_warm)))
    timer = _SharedTimer(clip.net)
    mem_frames = 0
    t0 = time.perf_counter()
    for _ in range(steps):
        clip.step()
        mem_frames += int(clip.core.last_mem_ti == clip.core.curr_ti)
    wall = time.perf_counter() - t0
    timer.close()
    t_step = wall / steps
    t_shared = timer.total / steps
    t_obj = max(t_step - t_shared, 0.0) / n_obj
    frame_s = t_shared + k * t_obj
    return {'value': 1.0 / frame_s, 'unit': 'frames/s', 'cores': cores, 'kind': 'reference',
            'extrapolated': n_obj < k, 'steps_requested': requested, 'steps_timed': steps, 'truncated': steps < requested,
            'warmup_requested': warmup, 'warmup_done': warm_done,
            'memory_frames_in_sample': mem_frames,  # a memory frame adds the value encoder; 0 of them = an optimistic CPU figure
            'sample': f'{steps} timed (+{warm_done} warm-up) steps of the unmodified reference DEVAInferenceCore.step (oracle/_ref, '
                      f'fp32, torch {torch.__version__}, {cores} threads) on full {wl["h"]}x{wl["w"]} frames, N={wl["n"]} slots, '
                      f'{n_obj} of {k} objects per step, every 5th step a memory frame; full-frame time = shared + {k} x per-object, '
                      f'both measured',
            'measured': {'objects_in_sample': n_obj, 's_per_sample_step': t_step, 's_shared_per_step': t_shared,
                         's_per_object': t_obj, 's_full_frame': frame_s, 'timed_wall_s': wall, 'setup_s': t_build},
            'q': clip.q}


def reference_gpu(wl, device, steps=5, warmup=2):
    """SURVEY 8(d) "GPU-side comparison": the UNMODIFIED reference on the same B200, all K objects, through its public
    step(): fp32 under PyTorch's default TF32 policy (what a user of the reference gets), fp32 with TF32 forbidden
    (the precision the 1e-3 parity contract is written against) and --amp (evaluation/eval_vos.py:137)."""
    torch.set_grad_enabled(False)
    out = {'kind': 'unmodified reference (oracle/_ref) on cuda', 'objects': wl['k'], 'steps': steps, 'warmup': warmup,
           'sample': f'{steps} frames {wl["h"]}x{wl["w"]} incl. one memory frame, N={wl["n"]}, all {wl["k"]} objects'}
    torch.backends.cudnn.benchmark = True
    for mode in ('fp32_tf32_default', 'fp32_strict', 'amp_fp16'):
        torch.backends.cudnn.allow_tf32 = mode != 'fp32_strict'
        torch.backends.cuda.matmul.allow_tf32 = mode != 'fp32_strict'  # eval scripts leave matmul at PyTorch's default (off)
        if mode == 'fp32_tf32_default':
            torch.backends.cuda.matmul.allow_tf32 = False
        try:
            with torch.autocast('cuda', dtype=torch.float16, enabled=(mode == 'amp_fp16')):
                clip = RefClip(wl, device, wl['k'], seed=100)
                for _ in range(warmup):
                    clip.step()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(steps):
                    clip.step()
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[mode] = {'value': 1e3 / ms, 'unit': 'frames/s', 'ms_per_step': ms,
                         'max_allocated_gb': torch.cuda.max_memory_allocated() / 2**30}
            del clip
        except Exception as exc:  # a reported extra, never fatal
            out[mode] = {'error': f'{type(exc).__name__}: {exc}'[:300]}
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
    return out


def _run_leg(args_list, timeout):
    """Run another leg of this script in its own process (the reference's package is also called `deva`)."""
    cmd = [sys.executable, os.path.abspath(__file__)] + args_list
    env = dict(os.environ)
    for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK', 'MASTER_ADDR', 'MASTER_PORT'):
        env.pop(k, None)
    if ALL_CORES:  # run_ours pinned this process to its GPU's NUMA node; a baseline leg may use every host core (the child
        env['DEVA_B200_BENCH_CORES'] = ','.join(str(c) for c in sorted(ALL_CORES))  # re-opens its mask before importing torch)
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
    for line in reversed(r.stdout.strip().splitlines()):
        if line.startswith('{'):
            return json.loads(line)
    raise RuntimeError(f'leg {args_list} printed no JSON (rc {r.returncode}): {r.stderr[-300:]}')


def _run_dist_leg(args_list, timeout):
    """Every rank of a torchrun launch calls this: each starts ONE child of this script with its own RANK / LOCAL_RANK /
    WORLD_SIZE and a rendezvous port of its own, so the children form their own process group (rank 0's child hosts the store:
    the elastic agent's variables are dropped).  Returns the child's JSON line on rank 0 ({'error': ...} when the leg
    failed or timed out), None elsewhere.  Never raises."""
    rank = int(os.environ.get('RANK', 0))
    env = {k: v for k, v in os.environ.items() if not k.startswith('TORCHELASTIC')}
    env['MASTER_ADDR'] = os.environ.get('MASTER_ADDR', '127.0.0.1')
    port = int(os.environ.get('MASTER_PORT', '29500'))
    # well away from the launcher's port: a driver that walks P, P+1, ... for its N = 1, 2, 4, 8 launches must not find
    # the children's store port in TIME_WAIT
    env['MASTER_PORT'] = str(port + 1537 if port + 1537 < 65000 else port - 1537)
    cmd = [sys.executable, os.path.abspath(__file__)] + args_list
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
    except subprocess.TimeoutExpired:
        return {'error': f'timed out after {timeout} s'} if rank == 0 else None
    except Exception as exc:
        return {'error': f'{type(exc).__name__}: {exc}'[:300]} if rank == 0 else None
    if rank != 0:
        return None
    for line in reversed(r.stdout.strip().splitlines()):
        if line.startswith('{'):
            try:
                return json.loads(line)
            except Exception:
                break
    return {'error': f'no JSON line (rc {r.returncode}): {r.stderr[-300:]}'}


def run_reference(args):
    rank = int(os.environ.get('RANK', 0)); world = int(os.environ.get('WORLD_SIZE', 1))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    from oracle import ref_loader
    if ref_loader.available():
        base = reference_cpu(wl, args.steps, max(args.warmup, 1), args.ref_objects)
        q = base.pop('q')
        ms_step = base['measured']['s_per_sample_step'] * 1e3
        steps_done, warm_done = base['steps_timed'], base['warmup_done']
    else:  # staged copy missing: the oracle port, stage by stage (kind 'port')
        base = cpu_baseline_port(wl, budget_s=40.0)
        q = (-(-wl['h'] // 16)) * (-(-wl['w'] // 16))
        ms_step = 1e3 / base['value']
        steps_done, warm_done = 1, 0
    out = {'impl': 'reference', 'metric': METRIC, 'value': base['value'], 'unit': 'frames/s', 'n_gpus': world,
           # the steps / warm-up actually EXECUTED (= the requested ones unless the time budget shortened the run, see
           # cpu_baseline.truncated): ms_per_step * steps is the timed wall
           'steps': steps_done, 'warmup': warm_done, 'ms_per_step': ms_step, 'higher_is_better': True,
           'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
           'extrapolated': bool(base.get('extrapolated', True)),
           'ms_per_step_is': 'measured time of one SAMPLE step (see cpu_baseline.sample); value = 1 / (shared + K x per-object)',
           'config': workload_config(wl, q, world), 'cpu_baseline': base, 'gpu_launches': 0,
           'e2e': {'value': base['value'], 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(out))


def run_reference_gpu(args):
    torch.cuda.set_device(0)
    print(json.dumps(reference_gpu(WORKLOADS[args.workload], torch.device('cuda', 0))))


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10, help='timed steps (frames) of the measured path')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference', 'reference_gpu'])
    ap.add_argument('--ref-objects', type=int, default=1,
                    help='objects per sample step of the CPU reference leg (the rest is extrapolated linearly and flagged)')
    ap.add_argument('--no-cpu-baseline', action='store_true', help='skip the host-cores reference leg')
    ap.add_argument('--quick', action='store_true', help='value + e2e only (no fused-io e2e, no conv roofline pass)')
    ap.add_argument('--workload', default='c3', choices=list(WORKLOADS))
    ap.add_argument('--no-torch-baseline', action='store_true', help='skip the stock-PyTorch-on-GPU comparison pass')
    ap.add_argument('--no-c5-leg', action='store_true',
                    help='N > 1 only: skip the bank-sharded single-video leg (workload c5 on the same ranks, key bank_sharded_c5)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs of the last timed step to DIR/<name>.npy '
                    '(float32, at most 64 MB in all: a fixed, seeded sample of the pixels of a larger output)')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.impl == 'reference':
        run_reference(a)
    elif a.impl == 'reference_gpu':
        run_reference_gpu(a)
    else:
        run_ours(a)
