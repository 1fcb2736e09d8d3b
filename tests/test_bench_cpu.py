"""Host-side plumbing of bench.py that the driver's launches rely on (no GPU): the clock-sample parser, the guarded
multi-rank leg, the launch-list summariser."""
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


class _Proc:
    def terminate(self):
        pass

    def wait(self, timeout=None):
        return 0

    def kill(self):
        pass


def test_clock_sampler_keeps_only_samples_after_mark():
    import bench
    s = object.__new__(bench.ClockSampler)
    s.proc = _Proc()
    fd, s.path = tempfile.mkstemp(suffix='.csv')
    os.close(fd)
    line = '0, {sm}, 1965, 900.0, 0x0, Not Active, Not Active, Not Active, {cap}\n'
    with open(s.path, 'w') as f:   # start-up / warm-up samples: idle clocks, must be dropped
        f.write(line.format(sm=345, cap='Not Active') * 3)
    s.mark()
    with open(s.path, 'a') as f:   # samples of the timed region
        f.write(line.format(sm=1600, cap='Active'))
        f.write(line.format(sm=1700, cap='Active'))
        f.write(line.format(sm=1650, cap='Not Active'))
        f.write('garbage\n')
    out = s.stop()
    assert out['samples'] == 3 and out['sm_mhz'] == 1650.0 and out['sm_max_mhz'] == 1965.0
    assert out['reasons'] == ['sw_power_cap']
    assert not os.path.exists(s.path)


def test_dist_leg_failure_is_contained(monkeypatch):
    """A child that dies (here: argparse rejects the arguments) must come back as an error record on rank 0 and as None
    on the other ranks - never as an exception: the clip-parallel numbers of the parent are already taken."""
    import bench
    monkeypatch.setenv('MASTER_ADDR', '127.0.0.1')
    monkeypatch.setenv('MASTER_PORT', '29533')
    monkeypatch.setenv('TORCHELASTIC_RUN_ID', 'x')  # must not reach the child (its rank 0 hosts the store itself)
    monkeypatch.setenv('RANK', '0')
    rec = bench._run_dist_leg(['--impl', 'no-such-implementation'], timeout=120)
    assert set(rec) == {'error'} and 'rc 2' in rec['error']
    monkeypatch.setenv('RANK', '1')
    assert bench._run_dist_leg(['--impl', 'no-such-implementation'], timeout=120) is None
    monkeypatch.setenv('RANK', '0')
    rec = bench._run_dist_leg(['--help'], timeout=0.001)   # the time-out path
    assert rec == {'error': 'timed out after 0.001 s'}


def test_launch_list_summary(tmp_path):
    csv = tmp_path / 'launches.csv'
    csv.write_text(
        '==PROF== Connected to process 1\n'
        '"ID","Process ID","Process Name","Host Name","Kernel Name","Context","Stream","Block Size","Grid Size","Device","CC",'
        '"Section Name","Metric Name","Metric Unit","Metric Value"\n'
        '"0","1","python","h","void b200::conv::conv_kernel<(bool)1, (int)0>(b200::conv::Maps, b200::conv::Params)","1","7",'
        '"(320, 1, 1)","(148, 1, 1)","0","10.0","s","gpu__time_duration.sum","ns","3,000,000"\n'
        '"1","1","python","h","ew::maxpool_kernel(const __half *, int)","1","7","(256, 1, 1)","(10, 1, 1)","0","10.0","s",'
        '"gpu__time_duration.sum","us","1000"\n')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'summarise_launches.py'), str(csv), 't'],
                         capture_output=True, text=True, check=True).stdout
    assert '2 consecutive launches, 4.0 ms' in out
    assert '| 3.00 | 75.0% | 1 | `conv::conv_kernel<' in out and '| 1.00 | 25.0% | 1 | `ew::maxpool_kernel` |' in out


def test_workload_table_matches_baseline_json():
    import bench
    base = json.load(open(os.path.join(ROOT, 'BASELINE.json')))
    assert bench.METRIC == base['metric']
    c3, c5 = bench.WORKLOADS['c3'], bench.WORKLOADS['c5']
    assert (c3['h'], c3['w'], c3['k'], c3['n']) == (1080, 1920, 16, 10000)     # configs[2]
    assert (c5['k'], c5['n'], c5.get('sharded')) == (32, 50000, True)          # configs[4]
    assert bench.WORKLOADS['c4']['clips'] == 64                                 # configs[3]


def test_dump_outputs_are_float32_bounded_and_repeatable(tmp_path):
    """--dump-outputs: a small output is written whole as float32; one over the limit becomes [C, S], S pixel positions
    in raster order, the same ones on every run."""
    import numpy as np
    import torch
    import bench
    small = torch.rand(3, 4, 5, dtype=torch.float16)
    bench.dump_outputs(str(tmp_path / 'a'), {'prob': small})
    got = np.load(tmp_path / 'a' / 'prob.npy')
    assert got.dtype == np.float32 and np.array_equal(got, small.float().numpy())
    big = torch.rand(17, 30, 40)
    limit = 17 * 4 * 500
    for d in ('b', 'c'):
        bench.dump_outputs(str(tmp_path / d), {'prob': big}, limit=limit)
    b, c = np.load(tmp_path / 'b' / 'prob.npy'), np.load(tmp_path / 'c' / 'prob.npy')
    assert b.dtype == np.float32 and b.shape == (17, 500) and b.nbytes <= limit and np.array_equal(b, c)
    column = {v: i for i, v in enumerate(big[0].flatten().tolist())}
    idx = [column[v] for v in b[0].tolist()]
    assert idx == sorted(set(idx))
    assert np.array_equal(b, big.reshape(17, -1).numpy()[:, idx])
