"""GPU tests of the resource ownership of the host code: the stream-ordered scratch of the device-resident entry points
goes back to the device's default memory pool on success and on failure, and a call traced with GDX_TRACE=1 computes
and reports what the untraced call does, whether it succeeds or fails."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CU_MEMPOOL_ATTR_USED_MEM_CURRENT = 7


@pytest.fixture(scope="module")
def gdx():
    import genedex_b200
    assert genedex_b200._lib.load().gdx_device_count() >= 1
    return genedex_b200


@pytest.fixture(scope="module")
def pool_used(gdx):
    """bytes of the default memory pool of device 0 in use by this process (driver API, read only)"""
    import torch
    torch.cuda.init()
    cu = C.CDLL("libcuda.so.1")
    assert cu.cuInit(0) == 0
    dev, pool = C.c_int(), C.c_void_p()
    assert cu.cuDeviceGet(C.byref(dev), 0) == 0
    assert cu.cuDeviceGetDefaultMemPool(C.byref(pool), dev) == 0

    def used():
        torch.cuda.synchronize()
        v = C.c_uint64()
        assert cu.cuMemPoolGetAttribute(pool, CU_MEMPOOL_ATTR_USED_MEM_CURRENT, C.byref(v)) == 0
        return v.value
    return used


@pytest.fixture(scope="module")
def case(gdx):
    """300 kbp DNA index without lookup levels or seed table, so that a batch of 2^15 queries is sorted, and a batch
    of text windows with its cursors and hit offsets on the device"""
    import torch
    rng = np.random.default_rng(11)
    n, nq, m = 300_000, 1 << 15, 24
    text = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, n)].copy()
    oidx = O.OracleIndex.build([text.tobytes()], O.ALPHABETS["ascii_dna"](), "u32", sampling_rate=4, lookup_depth=0)
    pidx = gdx.FmIndexConfig("u32").lookup_table_depth(0).construct_index([text.tobytes()], gdx.alphabet.ascii_dna())
    pidx.set_seed_table_depth(0)
    starts = rng.integers(0, n - m, nq)
    q = np.ascontiguousarray(text[starts[:, None] + np.arange(m)[None, :]].reshape(-1))
    off = np.arange(nq + 1, dtype=np.uint64) * m
    want_s, want_e = oidx.cursors_many_packed(q, off)
    _, want_hits = oidx.locate_many_packed(q, off)
    d_s = torch.from_numpy(want_s.astype(np.int64)).cuda()
    d_e = torch.from_numpy(want_e.astype(np.int64)).cuda()
    d_off = torch.zeros(nq + 1, dtype=torch.int64, device="cuda")
    d_off[1:] = torch.cumsum(d_e - d_s, 0)
    return dict(pidx=pidx, q=q, nq=nq, m=m, want_counts=want_e - want_s, want_hits=want_hits, d_s=d_s, d_e=d_e,
                d_off=d_off)


def test_failed_locate_intervals_device_returns_its_scratch(gdx, pool_used, case):
    """The second stream-ordered block (the worklist of n + 2 words) cannot be had for n = 2^58: the call fails
    before any kernel runs and must give the first block (the rows) back."""
    import torch
    lib = gdx._lib.load()
    d_hits = torch.zeros((1, 2), dtype=torch.int64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    before = pool_used()
    st = lib.gdx_locate_intervals_device(case["pidx"].handle, case["d_s"].data_ptr(), case["d_e"].data_ptr(), 2 ** 58,
                                         case["d_off"].data_ptr(), 1, d_hits.data_ptr(), stream)
    assert st == gdx._lib.GDX_ERR_OOM, lib.gdx_last_error_message()
    assert pool_used() == before
    # the failure left nothing behind for the next call
    st = lib.gdx_locate_intervals_device(case["pidx"].handle, case["d_s"].data_ptr(), case["d_e"].data_ptr(), 1,
                                         case["d_off"].data_ptr(), 1, d_hits.data_ptr(), stream)
    assert st == gdx._lib.GDX_OK, lib.gdx_last_error_message()


def test_device_entry_points_return_the_pool_to_its_baseline(gdx, pool_used, case):
    import torch
    lib = gdx._lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    nq, m = case["nq"], case["m"]
    dq = torch.from_numpy(case["q"]).cuda()
    qs = gdx._lib.gdx_queries(dq.data_ptr(), None, m, nq)
    d_c = torch.zeros(nq, dtype=torch.int64, device="cuda")
    total = int(case["d_off"][-1].item())
    d_hits = torch.zeros((total, 2), dtype=torch.int64, device="cuda")
    before = pool_used()
    # sorted count: the scratch of the query sort comes from the pool
    assert lib.gdx_count_many_device(case["pidx"].handle, C.byref(qs), d_c.data_ptr(), None, stream) == 0
    assert pool_used() == before
    assert np.array_equal(d_c.cpu().numpy().astype(np.uint64), case["want_counts"])
    assert lib.gdx_locate_intervals_device(case["pidx"].handle, case["d_s"].data_ptr(), case["d_e"].data_ptr(), nq,
                                           case["d_off"].data_ptr(), total, d_hits.data_ptr(), stream) == 0
    assert pool_used() == before
    assert np.array_equal(d_hits.cpu().numpy().astype(np.uint64), case["want_hits"])


TRACE_SCRIPT = r"""
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import genedex_b200 as gdx
from oracle import oracle as O
rng = np.random.default_rng(5)
text = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, 200_000)].tobytes()
pidx = gdx.FmIndexConfig("u32").construct_index([text], gdx.alphabet.ascii_dna())
qs = [text[p:p + 20] for p in rng.integers(0, 190_000, 300_000)]
data, off = O.pack(qs)
counts = pidx.count_many_packed(data, off)
print("counts", int(counts.sum()), int(counts.max()), flush=True)
bad = list(qs[:1000])
bad[700] = b"ACGTNACGT"
data, off = O.pack(bad)
try:
    pidx.count_many_packed(data, off)
    print("no error", flush=True)
except gdx.GenedexError as e:
    print("error", e.status, e.query, pidx._lib.gdx_last_error_query(), str(e), flush=True)
"""


def test_trace_reports_the_untraced_results_and_statuses(gdx):
    """GDX_TRACE=1 prints the chunk timeline of a successful call and releases its events on every path: results,
    statuses and the reported query equal those of the untraced run."""
    runs = {}
    for trace in ("0", "1"):
        env = dict(os.environ, GDX_TRACE=trace)
        p = subprocess.run([sys.executable, "-c", TRACE_SCRIPT, ROOT], env=env, capture_output=True, text=True,
                           timeout=600)
        assert p.returncode == 0, p.stderr
        runs[trace] = p
    assert runs["0"].stdout == runs["1"].stdout
    assert f"error {gdx._lib.GDX_ERR_INVALID_SYMBOL} 700 700 query 700: " in runs["1"].stdout
    assert "[gdx trace] chunk" not in runs["0"].stderr
    assert "[gdx trace] chunk  0 slot 0" in runs["1"].stderr
    assert "[gdx trace] host: all chunks issued" in runs["1"].stderr
