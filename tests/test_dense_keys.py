"""Dense keys: the F kernel counts a record whose breakdown values are all in
a dictionary learned from the head of the input at a per-CTA counter instead
of hashing its key (fast.h FDict, fdict.cpp, jit.cpp dng_jcode,
fast_kernel.cuh).  Results must not depend on it: values outside the
dictionary, values that only look alike, and dictionary values that never
occur again all have to come out as the oracle counts them.

CPU: tests/hostcheck/densecheck.cpp runs the generated lookup on the host and
checks it, and the keys rebuilt from the dictionary, against the F path's own
key code; with `device` the dense source must also build and link for sm_100a.
GPU: parity with the oracle under DNG_DENSE=0 and 1 (and its variants), the
interpreted and the compiled matcher."""

import json
import os
import random
import re
import subprocess
import sys

import pytest

sys.path.insert(0, os.path.dirname(__file__))
import corpus  # noqa: E402
from engines import CSRC, HOSTCHECK_DIR, canon_points, py_engine  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

C2 = corpus.BASELINE_QUERIES['C2'][0]
C3 = corpus.BASELINE_QUERIES['C3'][0]
C5 = corpus.BASELINE_QUERIES['C5'][0]

METHODS = ['"GE"', '"GETX"', '"null"', 'null', '"PATCH"', '"G\\u0045T"',
           '""', '"GET "', 'true']
STATUSES = ['"200"', '200.0', '2e2', 'null', '"null"', '9999', '"20"',
            '2000', 'false', '"abcdefghijklmnopq"']


def _gen(n, seed=0):
    from dragnet_b200 import native
    return native.gen_host(native.gen_params(seed=0xD5A60000 + seed,
                                             total_records=n), 0, n)


def _variant(line, rng):
    """One of the look-alike values in place of a generated one (the record
    keeps its shape, so the templates still take most of them)."""
    r = rng.random()
    if r < 0.45:
        v = ('"method":%s' % rng.choice(METHODS)).encode()
        return re.sub(rb'"method":"[A-Z]+"', lambda _: v, line, count=1)
    if r < 0.9:
        v = ('"statusCode":%s' % rng.choice(STATUSES)).encode()
        return re.sub(rb'"statusCode":\d+', lambda _: v, line, count=1)
    # the field missing altogether
    return line.replace(b'"method":', b'"methox":', 1)


def edge_data(n=6000, head=1500, rate_head=0.004, rate_tail=0.3, seed=1):
    """Generated records; a few look-alikes in the head (so that their shapes
    are templated), many after it (so that most are not in the dictionary)."""
    rng = random.Random(seed)
    lines = _gen(n, seed).split(b'\n')
    out = []
    for i, ln in enumerate(lines):
        if ln and rng.random() < (rate_head if i < head else rate_tail):
            ln = _variant(ln, rng)
        out.append(ln)
    return b'\n'.join(out)


# ---- CPU -------------------------------------------------------------------

@pytest.fixture(scope='session')
def densecheck(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp('densecheck') / 'densecheck')
    subprocess.check_call(['make', '-s', '-C', CSRC, 'build/jit_blob.o'])
    srcs = [os.path.join(HOSTCHECK_DIR, 'densecheck.cpp')] + [
        os.path.join(CSRC, n) for n in ('plan.cpp', 'result.cpp', 'tmpl.cpp',
                                        'fast.cpp', 'fdict.cpp', 'jit.cpp')]
    subprocess.check_call(['g++', '-std=c++17', '-O1', '-w',
                           '-I/usr/local/cuda/include', '-o', exe] + srcs +
                          [os.path.join(CSRC, 'build', 'jit_blob.o'), '-ldl'])
    return exe


def _run_check(exe, tmp_path, argv, learn, data, device=False, env=None):
    pf = tmp_path / 'plan.json'
    pf.write_text(json.dumps(corpus.make_plan(argv)))
    lf = tmp_path / 'learn.log'
    lf.write_bytes(learn)
    df = tmp_path / 'data.log'
    df.write_bytes(data)
    cmd = [exe, str(pf), str(lf), str(df)] + (['device'] if device else [])
    r = subprocess.run(cmd, capture_output=True,
                       env=dict(os.environ, **(env or {})))
    assert r.returncode == 0, r.stderr.decode()
    return json.loads(r.stdout)


@pytest.mark.parametrize('q', ['C2', 'C3', 'C5'])
def test_dense_source_builds_and_links_for_the_device(q, densecheck,
                                                      tmp_path):
    data = _gen(3000)
    argv = corpus.BASELINE_QUERIES[q][0]
    doc = _run_check(densecheck, tmp_path, argv, data, data, device=True)
    # every generated record is counted densely
    assert doc['dict'] > 0 and doc['records'] > 0, doc
    assert doc['dense'] == doc['records'], doc


@pytest.mark.parametrize('argv', [C2, C3, C5], ids=['C2', 'C3', 'C5'])
def test_lookup_and_rebuilt_keys_agree_with_the_key_code(argv, densecheck,
                                                         tmp_path):
    data = edge_data()
    doc = _run_check(densecheck, tmp_path, argv, data, data)
    assert doc['dict'] > 0 and 0 < doc['dense'] < doc['records'], doc


def test_dictionary_learned_from_another_input(densecheck, tmp_path):
    """Most values fall outside a dictionary learned elsewhere."""
    other = b''.join(b'{"req":{"method":"GET"},"res":{"statusCode":%d}}\n' %
                     (500 + i % 2) for i in range(2000))
    data = edge_data()
    doc = _run_check(densecheck, tmp_path, C3, other, data)
    assert doc['dict'] == 2 and 0 < doc['dense'] * 4 < doc['records'], doc
    # (500 is in the generated records' dictionary, 501 is not)
    doc = _run_check(densecheck, tmp_path, C3, data, other)
    assert doc['dict'] > 2 and doc['dense'] * 2 == doc['records'], doc


def test_no_dictionary_for_many_values_or_bucketized_columns(densecheck,
                                                             tmp_path):
    many = b''.join(b'{"req":{"method":"M%d"}}\n' % i for i in range(2000))
    assert _run_check(densecheck, tmp_path, C2, many, many) == {'dict': 0}
    data = _gen(2000)
    c4 = corpus.BASELINE_QUERIES['C4'][0]
    assert _run_check(densecheck, tmp_path, c4, data, data) == {'dict': 0}


def test_dense_off_gives_no_dictionary_source(densecheck, tmp_path):
    data = _gen(2000)
    pf = tmp_path / 'plan.json'
    pf.write_text(json.dumps(corpus.make_plan(C3)))
    (tmp_path / 'd.log').write_bytes(data)
    r = subprocess.run([densecheck, str(pf), str(tmp_path / 'd.log'),
                        str(tmp_path / 'd.log'), 'device'],
                       capture_output=True,
                       env=dict(os.environ, DNG_DENSE='0'))
    assert r.returncode == 3 and b'without dense keys' in r.stderr


# ---- GPU -------------------------------------------------------------------

def _gpu(plan, data, chunk=None):
    from dragnet_b200 import datasource_gpu
    chunk = chunk or len(data)
    chunks = [data[i:i + chunk] for i in range(0, len(data), chunk)]
    r = datasource_gpu.run_plan(plan, chunks=chunks)
    return r.points, r.counters


@pytest.fixture(params=['fast', 'jit'])
def fkernel(request, monkeypatch):
    monkeypatch.setenv('DNG_KERNEL', 'fast')
    monkeypatch.setenv('DNG_JIT', 'sync' if request.param == 'jit' else '0')
    return request.param


def _parity(plan, data, tmp_path, chunk=None):
    p = tmp_path / 'in.log'
    p.write_bytes(data)
    exp_p, exp_c = py_engine(plan, [str(p)])
    act_p, act_c = _gpu(plan, data, chunk)
    assert canon_points(act_p) == canon_points(exp_p)
    assert act_c == exp_c
    # (no point of a zero count, whichever path counted it)
    assert all(v > 0 for _, v in act_p)


@pytest.mark.gpu
@pytest.mark.parametrize('dense', ['0', '1', '3', '5'])
@pytest.mark.parametrize('q', ['C2', 'C3', 'C5'])
def test_look_alike_values_match_the_oracle(q, dense, fkernel, tmp_path,
                                            monkeypatch):
    if fkernel == 'fast' and dense != '1':
        pytest.skip('the interpreted matcher has no dense keys')
    monkeypatch.setenv('DNG_DENSE', dense)
    _parity(corpus.make_plan(corpus.BASELINE_QUERIES[q][0]), edge_data(),
            tmp_path)


@pytest.mark.gpu
@pytest.mark.parametrize('dense', ['0', '1'])
def test_dictionary_values_that_never_occur_again(dense, fkernel, tmp_path,
                                                  monkeypatch):
    """The head has methods the rest of the input never has again (their
    counters stay at zero in every CTA), and the rest has values the head
    never had."""
    monkeypatch.setenv('DNG_DENSE', dense)
    head = b''.join(b'{"req":{"method":"%s"},"res":{"statusCode":%d}}\n' %
                    (m, s) for m in (b'OPTIONS', b'TRACE', b'GET')
                    for s in (200, 404, 500) for _ in range(150))
    rng = random.Random(3)
    tail = b''.join(b'{"req":{"method":"%s"},"res":{"statusCode":%d}}\n' %
                    (rng.choice([b'GET', b'PUT', b'GE']),
                     rng.choice([200, 201, 500])) for _ in range(40000))
    _parity(corpus.make_plan(C3), head + tail, tmp_path)
    _parity(corpus.make_plan(['-b', 'req.method,res.statusCode']),
            head + tail, tmp_path)


@pytest.mark.gpu
@pytest.mark.parametrize('dense', ['0', '1'])
def test_multi_launch_pinned_feeds(dense, fkernel, tmp_path, monkeypatch):
    import torch
    from dragnet_b200 import native
    from engines import py_engine as oracle
    monkeypatch.setenv('DNG_DENSE', dense)
    data = edge_data(n=20000, head=4000)
    p = tmp_path / 'in.log'
    p.write_bytes(data)
    plan = corpus.make_plan(C3)
    exp_p, exp_c = oracle(plan, [str(p)])
    host = torch.frombuffer(bytearray(data), dtype=torch.uint8).pin_memory()
    s = native.Scan(native.Plan(json.dumps(plan)), 0)
    piece = 300007
    for off in range(0, len(data), piece):
        s.feed_pinned(host.data_ptr() + off, min(piece, len(data) - off))
    s.sync()
    res = s.finish()
    sys.path.insert(0, os.path.dirname(__file__))
    from test_gpu_feeds import _decode
    act_p, act_c = _decode(plan, s, res, s.counters())
    assert s.kernel_stats()['launches'] >= 3
    s.close()
    assert canon_points(act_p) == canon_points(exp_p)
    assert act_c == exp_c


@pytest.mark.gpu
@pytest.mark.parametrize('dense', ['0', '1'])
def test_24_warp_launches(dense, fkernel, tmp_path, monkeypatch):
    monkeypatch.setenv('DNG_DENSE', dense)
    monkeypatch.setenv('DNG_F_WARPS', '24')
    _parity(corpus.make_plan(C3), edge_data(n=10000), tmp_path, chunk=700001)
    _parity(corpus.make_plan(C5), edge_data(n=10000, seed=2), tmp_path)
