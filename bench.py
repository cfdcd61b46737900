#!/usr/bin/env python
"""bench.py: the headline benchmark -- JSON records/s scanned+aggregated.

  python bench.py --gpus N --steps K --warmup W            (our CUDA path)
      [--dump-outputs DIR]     (+ the last timed step's outputs as .npy)
  python bench.py --impl reference --gpus N --steps K ...  (CPU reference arm)

Workload (BASELINE.json configs[2], the north star's own target shape): 100 M
rows of mktestdata-shaped NDJSON per GPU (~22.4 GB, generated on the device,
deterministic), `dn scan -b req.method,res.statusCode -f {"eq":["req.method",
"GET"]}`.  A step is one full scan of the shard (+ the NCCL merge of the tallies
when N > 1).  `value` = records of all ranks / device time with the input
resident in HBM; `e2e` = the same scan fed from pinned HOST buffers through the
public C ABI (dng_scan_feed_pinned: H2D inside the timed region), its tallies
checked against the oracle's, with the PCIe roofline from a pinned-copy probe of
the same run; `roofline` = algorithmic input bytes / scan-kernel time (CUDA
events on the launch stream) against the measured HBM copy peak; `configs` =
the other BASELINE configs (C2, C4, C5 resident; configs[3]'s 1 B rows streamed
from a cycled pinned pool with the expected counts); `cpu_baseline` =
oracle/dn_oracle.cpp (restated CPU reference: node + the reference's npm
dependencies do not exist in this image) on a bounded sample, 1 thread and all
host threads.  Inputs (22 GB) are far larger than L2 (126 MB), so no explicit
L2 flush is needed between iterations.

The scan compiles its matcher at run time (NVRTC + nvJitLink, cached per
process: dragnet_b200/csrc/jit.h); bench.py asks for the synchronous mode
(DNG_JIT=sync), so the compilation (about a second, once per query shape)
happens in the warm-up steps and every timed step includes the template
learning and the cache lookup a scan does.
"""

import argparse
import atexit
import ctypes
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

# torch is plumbing here (device buffers, NCCL): left alone it starts one OpenMP
# thread per CPU it sees (128 on the B200 hosts) and their spin-waiting eats the
# container's CPU quota (16-24 CPUs) -- the file readers of the e2e_file leg
# were throttled to a tenth of their speed by it
os.environ.setdefault('OMP_NUM_THREADS', '4')
os.environ.setdefault('MKL_NUM_THREADS', '4')

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

def _bd(*fields):
    return [dict(f) if isinstance(f, dict) else {'name': f, 'field': f}
            for f in fields]


# (query configuration as `dn scan` builds it from its arguments
# (bin/dn:696-724), datasource config, what BASELINE.json calls it, the
# arguments for the record)
QUERIES = {
    'C2': ({'breakdowns': _bd('req.method')}, None,
           'configs[1]: 100M-row synthetic NDJSON, -b req.method',
           '-b req.method'),
    'C3': ({'breakdowns': _bd('req.method', 'res.statusCode'),
            'filter': {'eq': ['req.method', 'GET']}}, None,
           'configs[2]: 100M rows, -b req.method,res.statusCode + krill eq',
           '-b req.method,res.statusCode -f {"eq":["req.method","GET"]}'),
    'C4': ({'breakdowns': _bd({'name': 'latency', 'field': 'latency',
                               'aggr': 'quantize'})}, None,
           'configs[3]: -b latency[aggr=quantize] numeric histogram',
           '-b latency[aggr=quantize]'),
    'C5': ({'breakdowns': _bd('operation', 'req.method', 'host')}, None,
           'configs[4]: 3-key breakdown, NCCL final reduce',
           '-b operation,req.method,host'),
}


def make_plan(qconf, ds=None):
    from dragnet_b200 import query as mod_query
    ds = ds or {}
    q = mod_query.queryLoad({'query': qconf})
    if isinstance(q, Exception):
        raise q
    return mod_query.scan_plan(q, ds_filter=ds.get('filter'),
                               time_field=ds.get('timeField'))


def kernel_sources_sha16():
    """What the library is built from (dragnet_b200/csrc), as a digest: ties a
    stored ncu capture (profiles/r2_traffic.json) to the kernel it was taken
    on."""
    import glob
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, 'dragnet_b200', 'csrc')
    for p in sorted(glob.glob(os.path.join(d, '*'))):
        if os.path.isfile(p) and (os.path.splitext(p)[1] in (
                '.cu', '.cuh', '.cpp', '.h', '.S') or p.endswith('Makefile')):
            h.update(os.path.basename(p).encode())
            h.update(open(p, 'rb').read())
    return h.hexdigest()[:16]


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured'
        except Exception:
            pass
    return 6650.0, 'fallback'


class ClockSampler(object):
    """nvidia-smi clocks/throttle reasons during the timed regions.

    ONE nvidia-smi process for the whole run, started before any warm-up (its
    start-up attaches to every GPU of the box and stalls CUDA calls for a
    while: eight of them starting inside an 8-rank timed region cost 150 ms
    per step), sampling all the GPUs of the job every 100 ms; a timed region
    is marked and what was sampled since the mark is summarised."""

    Q = ('index,clocks.sm,clocks.max.sm,power.draw,'
         'clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, indexes):
        self.indexes = list(indexes)
        self.proc = None
        self.lines = []          # (arrival time, text)
        self.t0 = 0.0

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', ','.join(str(i) for i in self.indexes),
                 '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                 '-lms', '100'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark(self):
        self.t0 = time.time()

    def since_mark(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [],
                    'samples': 0}
        lines = [l for t, l in self.lines if t >= self.t0]
        if not lines:            # region shorter than the sampling interval
            lines = [l for _, l in self.lines[-len(self.indexes):]]
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown',
                 'sw_power_cap']
        for l in lines:
            f = [x.strip() for x in l.split(',')]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None,
                'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
            self.proc = None


def host_cores():
    """-> (threads worth starting, description).  os.cpu_count() counts the
    machine's CPUs; a container may be allowed far fewer (affinity mask, cgroup
    CPU quota): 128 threads on a 2-CPU quota only add scheduling overhead, and
    a baseline that says "128 cores" for it misleads."""
    n = os.cpu_count() or 1
    why = ['os.cpu_count()=%d' % n]
    try:
        a = len(os.sched_getaffinity(0))
        why.append('affinity=%d' % a)
        n = min(n, a)
    except Exception:
        pass
    for path, parse in (
            ('/sys/fs/cgroup/cpu.max',
             lambda t: None if t.split()[0] == 'max' else
             float(t.split()[0]) / float(t.split()[1])),
            ('/sys/fs/cgroup/cpu/cpu.cfs_quota_us',
             lambda t: None if int(t) <= 0 else int(t) / float(
                 open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read()))):
        try:
            q = parse(open(path).read().strip())
        except Exception:
            continue
        if q:
            why.append('cgroup quota=%.1f' % q)
            n = min(n, max(1, int(q + 0.999)))
        break
    return max(1, n), ', '.join(why)


def canon(points):
    return sorted((tuple(repr(c) for c in cols), v) for cols, v in points)


DUMP_LIMIT = 64 << 20


def dump_outputs(d, points, counters):
    """--dump-outputs: what a caller of the timed scan receives, as float64
    .npy files under `d`, so that the outputs of two builds can be compared:

      counters.npy      [len(native.COUNTER_FIELDS)], in that order
      points_count.npy  [n]: each point's count
      points_key.npy    [n, width]: each point's key as bytes ('s' + the
                        bytes of a string column, 'n' + repr() of a number,
                        columns joined by NUL), -1 past its end

    Points are in the order of their key bytes.  Should they come to more
    than DUMP_LIMIT bytes, a fixed seeded sample of them is written."""
    import numpy as np
    from dragnet_b200 import native
    os.makedirs(d, exist_ok=True)
    keyed = sorted((b'\0'.join(b's' + c if isinstance(c, bytes)
                               else b'n' + repr(c).encode() for c in cols), v)
                   for cols, v in points or [])
    width = max([len(k) for k, _ in keyed] + [1])
    cap = max(1, (DUMP_LIMIT - 8 * len(native.COUNTER_FIELDS)) //
              (8 * (width + 1)))
    if len(keyed) > cap:
        pick = np.sort(np.random.default_rng(0).choice(len(keyed), cap,
                                                       replace=False))
        keyed = [keyed[i] for i in pick]
    key = np.full((len(keyed), width), -1.0)
    for i, (k, _) in enumerate(keyed):
        key[i, :len(k)] = np.frombuffer(k, dtype=np.uint8)
    np.save(os.path.join(d, 'points_key.npy'), key)
    np.save(os.path.join(d, 'points_count.npy'),
            np.array([v for _, v in keyed], dtype=np.float64))
    np.save(os.path.join(d, 'counters.npy'),
            np.array([counters[n] for n in native.COUNTER_FIELDS],
                     dtype=np.float64))


# ---------------------------------------------------------------------------
# CPU reference arm / cpu_baseline: oracle/ only (no product library)
# ---------------------------------------------------------------------------

def oracle_build():
    exe = os.path.join(ROOT, 'oracle', 'dn_oracle_cpp')
    gen = os.path.join(ROOT, 'oracle', 'gen_ndjson')
    if not (os.path.exists(exe) and os.path.exists(gen)):
        subprocess.check_call(['make', '-s', '-C',
                               os.path.join(ROOT, 'oracle')])
    return exe, gen


def run_oracle(plan, path, threads, repeat=1, min_seconds=0.0):
    exe, _ = oracle_build()
    with tempfile.NamedTemporaryFile('w', suffix='.json', delete=False) as f:
        json.dump(plan, f)
        pf = f.name
    try:
        out = subprocess.run([exe, pf, '--threads', str(threads), '--repeat',
                              str(repeat), '--min-seconds', str(min_seconds),
                              path], capture_output=True, check=True).stdout
    finally:
        os.unlink(pf)
    return json.loads(out)


_sample_dir = None


def sample_dir():
    """This run's own directory on tmpfs, removed at exit: samples of another
    run (another build, another user) are never picked up, and none are left
    behind."""
    global _sample_dir
    if _sample_dir is None:
        _sample_dir = tempfile.mkdtemp(
            prefix='dnbench_',
            dir='/dev/shm' if os.path.isdir('/dev/shm') else None)
        atexit.register(shutil.rmtree, _sample_dir, True)
    return _sample_dir


def sample_file(rows, seed, total_rows, first=0):
    """Records [first, first + rows) of the `total_rows`-record workload of
    `seed`, written to tmpfs by oracle/gen_ndjson (byte-identical to the device
    generator: tests/test_gpu_parity.py, tests/test_cabi_cpu.py)."""
    _, gen = oracle_build()
    path = os.path.join(sample_dir(), 'dnbench_sample_%d_%d_%d_%d.ndjson' %
                        (seed, first, rows, total_rows))
    if not os.path.exists(path):
        subprocess.check_call([gen, path + '.tmp', str(seed), str(total_rows),
                               str(first), str(rows),
                               str(min(32, host_cores()[0]))])
        os.rename(path + '.tmp', path)
    return path


def oracle_points(doc):
    import struct
    pts = []
    for p in doc['points']:
        cols = []
        for c in p['cols']:
            if 's' in c:
                cols.append(bytes.fromhex(c['s']))
            else:
                cols.append(struct.unpack('<d', struct.pack(
                    '<Q', int(c['n'], 16)))[0])
        pts.append((cols, p['value']))
    return pts


def cpu_baseline(plan, rows, total_rows, seed, threads, min_seconds):
    """The restated CPU reference on a bounded sample: all threads and one."""
    path = sample_file(rows, seed, total_rows)
    many = run_oracle(plan, path, threads, min_seconds=min_seconds)
    # one thread: a quarter of the sample is plenty (about 0.4 M records/s)
    rows1 = max(1, rows // 8)
    path1 = sample_file(rows1, seed, total_rows)
    one = run_oracle(plan, path1, 1, min_seconds=min(min_seconds, 1.0))
    return {
        'value': rows / many['mean_seconds'], 'unit': 'records/s',
        'cores': threads, 'kind': 'port',
        'best_value': rows / many['seconds'],
        'one_thread_value': rows1 / one['mean_seconds'],
        'sample': 'first %d rows (%.2f GB) of the workload, %d threads, '
                  'file-range sharded, mean of %d scans (>= %.1f s measured); '
                  'one thread: first %d rows; restated CPU oracle '
                  '(oracle/dn_oracle.cpp, -O3): the reference Node path is '
                  'not executable here (no node in the image)' %
                  (rows, os.path.getsize(path) / 1e9, threads, many['reps'],
                   min_seconds, rows1)}, many


def reference_arm(args, rank, world):
    """--impl reference: the restated CPU reference (oracle/dn_oracle.cpp) on
    all host threads; a step = scans of a bounded sample of the workload for
    at least two seconds.  Nothing of the product library is loaded."""
    if rank != 0:
        return
    qconf, ds, desc, _ = QUERIES[args.query]
    plan = make_plan(qconf, ds)
    threads, cores_how = host_cores()
    rows = args.cpu_rows
    path = sample_file(rows, 0xD5A60000, args.rows)
    for _ in range(max(args.warmup, 1)):
        run_oracle(plan, path, threads)
    per, reps = [], 0
    for _ in range(args.steps):
        d = run_oracle(plan, path, threads, min_seconds=2.0)
        per.append(d['mean_seconds'])
        reps += d['reps']
    mean = sum(per) / len(per)
    value = rows / mean
    rows1 = max(1, rows // 8)
    one = run_oracle(plan, sample_file(rows1, 0xD5A60000, args.rows), 1,
                     min_seconds=1.0)
    line = {
        'impl': 'reference', 'metric': 'json_records_per_sec',
        'value': value, 'unit': 'records/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': mean * 1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'u8',
        'data': 'synthetic',
        'config': {'workload': desc, 'rows_per_scan': rows,
                   'scans_per_step': reps / float(args.steps),
                   'query': QUERIES[args.query][3],
                   'note': 'CPU reference arm: C++ restatement of the '
                           'reference Node.js scan path (node and the '
                           "reference's npm dependencies are not in this "
                           'image); bounded sample of the 100M-row workload, '
                           'scanned repeatedly for >= 2 s per step'},
        'cpu_baseline': {'value': value, 'unit': 'records/s',
                         'cores': threads, 'cores_how': cores_how,
                         'kind': 'port',
                         'one_thread_value': rows1 / one['mean_seconds'],
                         'sample': '%d rows (%.2f GB) of the workload, %d '
                                   'threads, file-range sharded, mean over '
                                   '%d scans' %
                                   (rows, os.path.getsize(path) / 1e9,
                                    threads, reps)},
        'e2e': {'value': value, 'unit': 'records/s',
                'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------

def pcie_probe(torch, dev, nbytes=1 << 30, reps=4):
    """Pinned host -> device cudaMemcpyAsync bandwidth (GB/s), best of reps."""
    src = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    dst = torch.empty(nbytes, dtype=torch.uint8, device='cuda:%d' % dev)
    best = 0.0
    for _ in range(reps + 1):
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        dst.copy_(src, non_blocking=True)
        e1.record()
        e1.synchronize()
        best = max(best, nbytes / 1e9 / (e0.elapsed_time(e1) / 1e3))
    del src, dst
    return best


def kernel_name(st):
    if st['kernel'] == 'F path':
        if st['jit']['launches']:
            return ('dng_scan_kernel_j (scan_kernel_f with the run-time '
                    'compiled matcher)')
        return 'dng::scan_kernel_f'
    return 'dng::scan_kernel_w' if st['kernel'] == 'per-warp chunks' \
        else 'dng::scan_kernel'


def gpu_arm(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    os.environ.setdefault('DNG_JIT', 'sync')
    from dragnet_b200 import native

    torch.cuda.set_device(local_rank)
    dev = local_rank
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', dev))
    L = native.lib()
    qconf, ds, desc, _ = QUERIES[args.query]
    plan = make_plan(qconf, ds)
    rows = args.rows
    seed = 0xD5A60000 + rank
    # clocks / throttle reasons of every GPU of the job, sampled by rank 0 from
    # before the warm-up on (see ClockSampler)
    sampler = None
    if rank == 0:
        sampler = ClockSampler(range(world))
        sampler.start()

    # ---- the shard, generated in HBM --------------------------------------
    params = native.gen_params(seed=seed, total_records=rows)
    cap = rows * 226 + (64 << 20)
    buf = torch.empty(cap, dtype=torch.uint8, device='cuda:%d' % dev)
    nbytes = 0
    chunk = 4000000
    ln = ctypes.c_size_t()
    pool_rows = min(args.pool_rows, rows)
    for first in range(0, rows, chunk):
        cnt = min(chunk, rows - first)
        rc = L.dng_gen_device(ctypes.byref(params), dev, first, cnt,
                              buf.data_ptr() + nbytes, cap - nbytes,
                              ctypes.byref(ln))
        if rc != 0:
            raise RuntimeError('dng_gen_device failed: %d' % rc)
        nbytes += ln.value
    torch.cuda.synchronize()

    # ---- NCCL communicator of the library (id exchanged with torch) --------
    comm = None
    if world > 1:
        idbuf = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            raw = ctypes.create_string_buffer(128)
            if L.dng_comm_unique_id(raw) != 0:
                raise RuntimeError('dng_comm_unique_id failed')
            idbuf = torch.frombuffer(bytearray(raw.raw), dtype=torch.uint8)
        idg = idbuf.cuda(dev)
        dist.broadcast(idg, 0)
        ident = bytes(idg.cpu().numpy().tobytes())
        comm = ctypes.c_void_p()
        err = ctypes.create_string_buffer(256)
        rc = L.dng_comm_init(ctypes.byref(comm), world, rank, ident, dev, err,
                             256)
        if rc != 0:
            raise RuntimeError('dng_comm_init: %s' % err.value)

    stream = torch.cuda.current_stream().cuda_stream
    handles = {}

    def plan_handle(q):
        if q not in handles:
            a, d = QUERIES[q][:2]
            handles[q] = native.Plan(json.dumps(make_plan(a, d),
                                                separators=(',', ':')))
        return handles[q]

    def one_scan(feed, merge=True, q=None):
        """-> (points or None, counters, kernel stats, device ms)"""
        s = native.Scan(plan_handle(q or args.query), dev)
        s.set_stream(stream)
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        em = torch.cuda.Event(enable_timing=True)
        e0.record()
        feed(s)
        em.record()
        if comm is not None and merge:
            out = ctypes.c_void_p()
            ctr = native.DngCounters()
            rc = L.dng_merge_nccl(s.handle, comm, 0, ctypes.byref(out),
                                  ctypes.byref(ctr))
            if rc != 0:
                raise RuntimeError('dng_merge_nccl: %d %s' %
                                   (rc, L.dng_scan_error(s.handle)))
            pts = native.Result(out).points() if out.value else None
            counters = ctr.as_dict()
        else:
            res = s.finish()
            pts = res.points()
            counters = s.counters()
        e1.record()
        e1.synchronize()
        st = s.kernel_stats()
        st.update(s.template_stats())
        ms = e0.elapsed_time(e1)
        st['after_feed_ms'] = em.elapsed_time(e1)   # finish / cross-GPU merge
        s.close()
        return pts, counters, st, ms

    def feed_resident(s):
        s.feed_device(buf.data_ptr(), nbytes)

    # ---- pinned host pool for the end-to-end legs -----------------------------
    # the first pool_rows records of the shard, copied out of HBM once; their
    # byte length is what the generator reports for that record range
    tmp = torch.empty(pool_rows * 226 + (1 << 20), dtype=torch.uint8,
                      device='cuda:%d' % dev)
    rc = L.dng_gen_device(ctypes.byref(params), dev, 0, pool_rows,
                          tmp.data_ptr(), tmp.numel(), ctypes.byref(ln))
    assert rc == 0
    pool_len = ln.value
    del tmp
    host_pool = torch.empty(pool_len, dtype=torch.uint8, pin_memory=True)
    host_pool.copy_(buf[:pool_len])
    torch.cuda.synchronize()
    cycles = max(1, rows // pool_rows)
    e2e_rows = cycles * pool_rows

    def feed_host_n(n):
        def feed(s):
            for _ in range(n):
                s.feed_pinned(host_pool.data_ptr(), pool_len)
        return feed

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(feed, steps, warmup, q=None):
        res = None
        for _ in range(warmup):
            res = one_scan(feed, q=q)
        barrier()
        if sampler is not None:
            sampler.mark()
        t0 = time.perf_counter()
        dev_ms, kern_ms, kern_bytes, launches = 0.0, 0.0, 0, 0
        tail_ms = 0.0
        all_launches = 0
        for _ in range(steps):
            res = one_scan(feed, q=q)
            dev_ms += res[3]
            tail_ms += res[2]['after_feed_ms']
            kern_ms += res[2]['kernel_ms']
            kern_bytes += res[2]['kernel_bytes']
            launches += res[2]['launches']
            all_launches += res[2]['all_launches']
        barrier()
        wall = time.perf_counter() - t0
        clocks = sampler.since_mark() if sampler is not None else None
        t = torch.tensor([dev_ms, wall * 1e3, tail_ms], dtype=torch.float64,
                         device='cuda:%d' % dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return {'dev_ms': float(t[0]), 'wall_ms': float(t[1]),
                'tail_ms': float(t[2]),
                'kernel_ms': kern_ms, 'kernel_bytes': kern_bytes,
                'launches': launches, 'all_launches': all_launches,
                'clocks': clocks, 'last': res}

    peak, how = measured_peaks()
    cpu_threads = max(1, host_cores()[0] // world)

    # ---- value: input resident in HBM -------------------------------------------
    R = timed(feed_resident, args.steps, args.warmup)
    ms_per_step = R['dev_ms'] / args.steps
    total_rows = rows * world
    value = total_rows / (ms_per_step / 1e3)

    # ---- e2e: host buffers through the public C ABI ------------------------------
    E = timed(feed_host_n(cycles), max(1, args.e2e_steps), 1)
    e2e_ms = E['dev_ms'] / max(1, args.e2e_steps)
    e2e_value = e2e_rows * world / (e2e_ms / 1e3)
    result_bytes = 0
    if E['last'][0] is not None:
        result_bytes = sum(8 + sum(len(c) if isinstance(c, bytes) else 8
                                   for c in cols)
                           for cols, _ in E['last'][0])
    h2d_peak = pcie_probe(torch, dev)

    # ---- what the oracle says about this rank's pool and about a sample ------
    # (every rank checks its own shard; the oracle's threads are shared out)
    def oracle_tallies(q, path):
        a, d = QUERIES[q][:2]
        doc = run_oracle(make_plan(a, d), path, cpu_threads)
        return {tuple(repr(c) for c in cols): v
                for cols, v in oracle_points(doc)}, doc

    pool_path = sample_file(pool_rows, seed, rows)
    assert os.path.getsize(pool_path) == pool_len
    pool_exp, pool_doc = oracle_tallies(args.query, pool_path)

    def times(tallies, k):
        return {key: v * k for key, v in tallies.items()}

    def as_dict(points):
        return {tuple(repr(c) for c in cols): v for cols, v in points}

    # the e2e leg's own result: at N > 1 the merged tallies are checked below
    e2e_local = one_scan(feed_host_n(cycles), merge=False)
    e2e_parity = 'exact' if as_dict(e2e_local[0]) == times(pool_exp, cycles) \
        and e2e_local[1]['lines'] == pool_doc['counters']['lines'] * cycles \
        else 'MISMATCH'

    # ---- files: the same pool as a tmpfs file through dng_scan_feed_file -------
    file_leg = None
    if world == 1 and args.file_steps > 0:
        if os.environ.get('DNG_BENCH_TRACE'):
            sys.stderr.write('TRACE file leg begins %.3f\n' % time.time())
        Fr = timed(lambda s: s.feed_file(pool_path), args.file_steps, 1)
        if os.environ.get('DNG_BENCH_TRACE'):
            sys.stderr.write('TRACE file leg ends %.3f\n' % time.time())
        fms = Fr['dev_ms'] / args.file_steps
        file_leg = {'value': pool_rows / (fms / 1e3),
                    'unit': 'records/s', 'ms_per_step': fms,
                    'file_bytes': pool_len,
                    'gbs': pool_len / 1e9 / (fms / 1e3),
                    'kernel_ms_per_step': Fr['kernel_ms'] / args.file_steps,
                    'launches_per_step': Fr['launches'] / args.file_steps,
                    'parity': 'exact' if as_dict(Fr['last'][0]) == pool_exp
                    else 'MISMATCH',
                    'note': 'dng_scan_feed_file on a page-cache-resident '
                            'file: reader threads pread into a pinned '
                            'ring, H2D overlapped with the scan'}

    # ---- the other BASELINE configs, resident in HBM ---------------------------
    configs = []
    for q in ('C2', 'C3', 'C4', 'C5'):
        if q != args.query and args.cfg_steps <= 0:
            continue
        C = R if q == args.query else timed(feed_resident, args.cfg_steps, 1,
                                            q=q)
        steps = args.steps if q == args.query else args.cfg_steps
        cms = C['dev_ms'] / steps
        gbs = (C['kernel_bytes'] / 1e9) / (C['kernel_ms'] / 1e3)
        configs.append({
            'config': QUERIES[q][2], 'query': QUERIES[q][3],
            'rows_per_gpu': rows, 'value': total_rows / (cms / 1e3),
            'unit': 'records/s', 'ms_per_step': cms,
            'kernel': kernel_name(C['last'][2]),
            'roofline_frac': gbs / peak, 'kernel_gbs': gbs,
            'points': len(C['last'][0]) if C['last'][0] is not None else None})
    # configs[3] at its stated scale: 1 B rows per GPU do not fit in HBM (224
    # GB), so they are streamed from the pinned pool, cycled; the expected
    # tallies are the oracle's for the pool, times the cycles
    stream_leg = None
    if args.stream_rows > 0:
        scyc = max(1, args.stream_rows // pool_rows)
        c4_exp, c4_doc = oracle_tallies('C4', pool_path)
        barrier()
        S = one_scan(feed_host_n(scyc), merge=False, q='C4')
        t = torch.tensor([S[3]], dtype=torch.float64, device='cuda:%d' % dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sms = float(t[0])
        ok = as_dict(S[0]) == times(c4_exp, scyc) and \
            S[1]['lines'] == c4_doc['counters']['lines'] * scyc
        stream_leg = {
            'config': 'configs[3]: %d rows per GPU streamed from pinned host '
                      'memory (a %d-row pool cycled %dx), '
                      '-b latency[aggr=quantize]' %
                      (scyc * pool_rows, pool_rows, scyc),
            'value': scyc * pool_rows * world / (sms / 1e3),
            'unit': 'records/s', 'ms': sms,
            'h2d_gbs': scyc * pool_len / 1e9 / (sms / 1e3),
            'parity': 'exact' if ok else 'MISMATCH'}

    # ---- parity on a sample of every rank's shard ---------------------------------
    srows = min(args.cpu_rows, rows)
    spath = sample_file(srows, seed, rows)
    s_exp, s_doc = oracle_tallies(args.query, spath)
    sample = open(spath, 'rb').read()
    sbuf = torch.frombuffer(bytearray(sample), dtype=torch.uint8).cuda(dev)
    g = one_scan(lambda s: s.feed_device(sbuf.data_ptr(), len(sample)),
                 merge=False)
    ok = as_dict(g[0]) == s_exp and g[1]['lines'] == s_doc['counters']['lines']
    # the resident buffer starts with exactly these bytes
    ok = ok and bytes(buf[:4096].cpu().numpy().tobytes()) == sample[:4096]
    flags = torch.tensor([1 if ok else 0, 1 if e2e_parity == 'exact' else 0,
                          1 if (stream_leg is None or
                                stream_leg['parity'] == 'exact') else 0],
                         dtype=torch.int32, device='cuda:%d' % dev)
    if world > 1:
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    parity = 'exact' if int(flags[0]) else 'MISMATCH'
    e2e_parity = 'exact' if int(flags[1]) else 'MISMATCH'
    if stream_leg is not None:
        stream_leg['parity'] = 'exact' if int(flags[2]) else 'MISMATCH'

    # ---- N > 1: the merged tallies must equal the sum of the per-rank ones,
    # and (oracle) the merged e2e tallies the sum of the ranks' pool tallies ----
    merge_parity = None
    if world > 1:
        local = one_scan(feed_resident, merge=False)[0]
        gathered = [None] * world if rank == 0 else None
        dist.gather_object((local, times(pool_exp, cycles)), gathered, dst=0)
        if rank == 0:
            acc, exp = {}, {}
            for pts, pe in gathered:
                for cols, v in pts:
                    k = tuple(repr(c) for c in cols)
                    acc[k] = acc.get(k, 0) + v
                for k, v in pe.items():
                    exp[k] = exp.get(k, 0) + v
            merge_parity = 'exact' if as_dict(R['last'][0]) == acc and \
                as_dict(E['last'][0]) == exp else 'MISMATCH'

    if rank != 0:
        if comm is not None:
            L.dng_comm_destroy(comm)
            dist.destroy_process_group()
        return

    # ---- cpu_baseline on a bounded sample (rank 0, N=1 only) ---------------------
    cpu = None
    if world == 1 and args.cpu_rows > 0:
        cpu, _ = cpu_baseline(plan, srows, rows, seed, host_cores()[0],
                              args.cpu_seconds)
        cpu['cores_how'] = host_cores()[1]

    n_launch = max(1, R['launches'])
    st = R['last'][2]
    kname = kernel_name(st)
    # DRAM traffic of the scan kernel: from the `ncu --set full` capture of
    # this very command kept in profiles/ (bench.py cannot run under ncu); only
    # used if it was taken of the kernel this run launched, on this query,
    # built from these very sources (kernel_sources_sha16): null otherwise
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, 'profiles', 'r2_traffic.json')
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            if tj.get('kernel') == kname.split(' ')[0] and \
                    tj.get('query') == args.query and \
                    tj.get('sources_sha16') == kernel_sources_sha16():
                traffic = tj['traffic_over_algorithmic'] * \
                    (R['kernel_bytes'] / n_launch)
                traffic_src = ('dram__bytes_read.sum + dram__bytes_write.sum '
                               'of the ncu capture in profiles/r2_traffic.json'
                               ' (x%.3f algorithmic)' %
                               tj['traffic_over_algorithmic'])
        except Exception:
            pass
    achieved = (R['kernel_bytes'] / 1e9) / (R['kernel_ms'] / 1e3)
    h2d_gbs = cycles * pool_len / 1e9 / (e2e_ms / 1e3)
    line = {
        'metric': 'json_records_per_sec', 'value': value,
        'unit': 'records/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms_per_step,
        'wall_ms_per_step': R['wall_ms'] / args.steps,
        # finish + (N>1) the NCCL merge of the tallies, inside ms_per_step
        'finish_merge_ms_per_step': R['tail_ms'] / args.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'u8', 'data': 'synthetic',
        'config': {
            'workload': desc, 'rows_per_gpu': rows,
            'bytes_per_gpu': nbytes, 'query': QUERIES[args.query][3],
            'parallelism': 'shard-per-gpu x%d, one NCCL reduce of the '
                           'tallies' % world if world > 1 else 'single gpu',
            'l2': 'inputs (%.1f GB) >> L2 (126 MB): no flush needed' %
                  (nbytes / 1e9),
            'points': len(R['last'][0]) if R['last'][0] is not None else None,
            # what the scan specialised itself to from the head of the input
            'kernel': st['kernel'],
            'record_templates': st['templates'],
            'templated_fraction': st['templated_records'] /
            max(1, R['last'][1]['lines'] / world),
            'jit': {'mode': os.environ.get('DNG_JIT'),
                    'state': st['jit']['state'],
                    'compile_ms': st['jit']['compile_ms'],
                    'link_ms': st['jit']['link_ms'],
                    'error': st['jit']['error'],
                    'note': 'matcher compiled at run time for the learned '
                            'templates (NVRTC + nvJitLink), cached per '
                            'process: compiled once, in the warm-up'},
        },
        'roofline': {
            'bound': 'hbm', 'achieved': achieved, 'peak': peak,
            'unit': 'GB/s', 'frac': achieved / peak, 'traffic': traffic,
            'traffic_source': traffic_src,
            'kernel': kname,
            'bytes_per_launch': R['kernel_bytes'] / n_launch,
            'ms_per_launch': R['kernel_ms'] / n_launch,
            'peak_source': '%s HBM copy bandwidth (MEASURED_PEAKS.json)' % how,
        },
        'e2e': {'value': e2e_value, 'unit': 'records/s',
                'h2d_bytes_per_step': cycles * pool_len,
                'd2h_bytes_per_step': result_bytes,
                'ms_per_step': e2e_ms,
                'h2d_gbs': h2d_gbs,
                'parity': e2e_parity,
                'roofline': {'bound': 'pcie', 'achieved': h2d_gbs,
                             'peak': h2d_peak, 'unit': 'GB/s',
                             'frac': h2d_gbs / h2d_peak,
                             'peak_source': 'pinned cudaMemcpyAsync H2D of '
                                            '1 GiB, best of 5, this run'},
                'note': 'pinned host pool of %d rows fed %dx per step via '
                        'dng_scan_feed_pinned (H2D ring overlapped with the '
                        'scan kernel); tallies and line count checked against '
                        'the oracle\'s for the pool x %d' %
                        (pool_rows, cycles, cycles)},
        # every kernel of ours inside the timed steps: the scan kernels (+ the
        # miss kernel of the F path) plus template resolution, newline search
        # and result compaction
        'gpu_launches': R['all_launches'],
        'scan_kernel_launches': R['launches'],
        'clocks': R['clocks'] if rank == 0 else None,
        'parity': parity,
        'merge_parity': merge_parity,
        'e2e_file': file_leg,
        'configs': configs + ([stream_leg] if stream_leg else []),
    }
    if cpu:
        line['cpu_baseline'] = cpu
    if sampler is not None:
        sampler.stop()
    if args.dump_outputs:
        # the last timed step: at N > 1 the merged tallies
        dump_outputs(args.dump_outputs, R['last'][0], R['last'][1])
    print(json.dumps(line), flush=True)
    if comm is not None:
        L.dng_comm_destroy(comm)
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--query', default='C3', choices=sorted(QUERIES))
    ap.add_argument('--rows', type=int,
                    default=int(os.environ.get('DNG_BENCH_ROWS', 100000000)))
    ap.add_argument('--pool-rows', type=int, default=10000000)
    ap.add_argument('--e2e-steps', type=int, default=2)
    ap.add_argument('--cfg-steps', type=int, default=2)
    ap.add_argument('--stream-rows', type=int,
                    default=int(os.environ.get('DNG_BENCH_STREAM_ROWS',
                                               1000000000)))
    ap.add_argument('--cpu-rows', type=int, default=4000000)
    ap.add_argument('--cpu-seconds', type=float, default=4.0)
    ap.add_argument('--file-steps', type=int, default=2)
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the points and counters of the last timed '
                         'step to DIR as .npy files (see dump_outputs)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs: the reference arm scans a different sample')
    rank = int(os.environ.get('RANK', 0))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    if args.impl == 'reference':
        # the oracle only: the product library is not even looked for
        reference_arm(args, rank, world)
        return 0
    import __graft_entry__
    lib_path = os.path.join(ROOT, 'dragnet_b200', 'libdragnet_gpu.so')
    oexe = os.path.join(ROOT, 'oracle', 'dn_oracle_cpp')
    ogen = os.path.join(ROOT, 'oracle', 'gen_ndjson')
    if rank == 0:
        if not (os.path.exists(lib_path) and os.path.exists(oexe) and
                os.path.exists(ogen)):
            __graft_entry__.build()
    else:
        t0 = time.time()
        while not (os.path.exists(lib_path) and os.path.exists(ogen)) and \
                time.time() - t0 < 600:
            time.sleep(1)
    gpu_arm(args, rank, local_rank, world)
    return 0


if __name__ == '__main__':
    sys.exit(main())
