"""bench.py's reference arm runs without a GPU: check that it prints one JSON
line with the keys the driver reads (the GPU arm prints the same keys plus
`roofline`; it cannot run here).  Also the clocks sampler's parsing, the
files of --dump-outputs and, on a GPU, what --steps and --dump-outputs do."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_reference_arm_json_line():
    out = subprocess.run(
        [sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference',
         '--steps', '1', '--warmup', '1', '--cpu-rows', '20000',
         '--rows', '20000'],
        capture_output=True, check=True, text=True, timeout=600).stdout
    lines = [l for l in out.splitlines() if l.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup',
              'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline',
              'dtype', 'data', 'config', 'cpu_baseline', 'e2e', 'impl'):
        assert k in d, k
    assert d['impl'] == 'reference' and d['metric'] == 'json_records_per_sec'
    assert d['value'] > 0 and d['cpu_baseline']['kind'] in ('port', 'reference')
    assert d['e2e']['h2d_bytes_per_step'] == 0
    assert 'workload' in d['config']


def test_clock_sampler_summarises_what_it_saw():
    import bench
    s = bench.ClockSampler([0, 1])
    s.proc = object()            # pretend nvidia-smi is running
    s.lines = [(1.0, '0, 1965, 1965, 400.1, Not Active, Not Active, Not Active, Not Active'),
               (1.0, '1, 1950, 1965, 410.0, Not Active, Not Active, Not Active, Active'),
               (5.0, '0, 1800, 1965, 420.0, Not Active, Not Active, Not Active, Not Active'),
               (5.0, '1, 1965, 1965, 415.0, Not Active, Not Active, Active, Not Active')]
    s.t0 = 4.0
    r = s.since_mark()
    assert r['samples'] == 2 and r['sm_max_mhz'] == 1965.0
    assert r['reasons'] == ['sw_thermal_slowdown']
    s.t0 = 9.0                   # nothing since the mark: the latest lines
    r = s.since_mark()
    assert r['samples'] == 2 and r['sm_mhz'] in (1800.0, 1965.0)


def _load(d):
    return {n: np.load(os.path.join(str(d), n + '.npy'))
            for n in ('counters', 'points_count', 'points_key')}


def test_dump_outputs_files(tmp_path, monkeypatch):
    import bench
    from dragnet_b200 import native
    pts = [([b'GET', b'200'], 5), ([b'PUT', 404.0], 2), ([b'GET', b'20'], 7)]
    ctr = {n: i for i, n in enumerate(native.COUNTER_FIELDS)}
    bench.dump_outputs(str(tmp_path / 'a'), pts, ctr)
    a = _load(tmp_path / 'a')
    assert all(x.dtype == np.float64 for x in a.values())
    assert a['counters'].tolist() == list(range(len(native.COUNTER_FIELDS)))
    # in the order of the key bytes
    assert a['points_count'].tolist() == [7, 5, 2]
    keys = [bytes(int(b) for b in row if b >= 0) for row in a['points_key']]
    assert keys == [b'sGET\0s20', b'sGET\0s200', b'sPUT\0n404.0']

    # over the size limit: the same seeded sample every time, within it
    monkeypatch.setattr(bench, 'DUMP_LIMIT', 8192)
    many = [([b'k%05d' % i], i) for i in range(1000)]
    for d in ('b', 'c'):
        bench.dump_outputs(str(tmp_path / d), many, ctr)
    b, c = _load(tmp_path / 'b'), _load(tmp_path / 'c')
    assert sum(x.nbytes for x in b.values()) <= 8192
    assert 0 < len(b['points_count']) < 1000
    for n in b:
        assert np.array_equal(b[n], c[n])
    assert list(b['points_count']) == sorted(b['points_count'])


@pytest.mark.gpu
def test_steps_and_dump_outputs(tmp_path):
    """--steps sets the number of timed scans, and what --dump-outputs writes
    of the last one does not depend on it."""
    small = ['--rows', '300000', '--pool-rows', '100000', '--warmup', '1',
             '--stream-rows', '0', '--cpu-rows', '20000', '--cpu-seconds',
             '0.1', '--e2e-steps', '1', '--file-steps', '0', '--cfg-steps',
             '0']
    runs = []
    for steps in (1, 3):
        d = tmp_path / str(steps)
        out = subprocess.run(
            [sys.executable, os.path.join(ROOT, 'bench.py'), '--steps',
             str(steps), '--dump-outputs', str(d)] + small,
            capture_output=True, check=True, text=True, timeout=900).stdout
        line = json.loads([l for l in out.splitlines()
                           if l.startswith('{')][-1])
        assert line['steps'] == steps and line['parity'] == 'exact'
        runs.append((line, _load(d)))
    (one, a), (three, b) = runs
    assert three['scan_kernel_launches'] == 3 * one['scan_kernel_launches']
    assert three['gpu_launches'] == 3 * one['gpu_launches']
    for n in a:
        assert np.array_equal(a[n], b[n]), n
    from dragnet_b200 import native
    ctr = dict(zip(native.COUNTER_FIELDS, a['counters']))
    assert ctr['lines'] == 300000
    assert len(a['points_count']) == one['config']['points'] > 0
