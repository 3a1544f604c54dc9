"""CPU tests of the chunk schedule of the host pipeline (genedex_b200/csrc/chunk_plan.h), built on the host with g++.
The core is a plain transcription of the loop arithmetic search_host used before the schedule moved into the header;
the header must cut the same chunks, chunk for chunk.  No GPU is used here."""
import bisect
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MiB = 1 << 20
U64P = np.ctypeslib.ndpointer(np.uint64, flags="C_CONTIGUOUS")


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    out = tmp_path_factory.mktemp("emul_chunk_plan") / "libchunkplan.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-shared", "-fPIC", "-o", str(out),
                           os.path.join(ROOT, "tests", "host_emul", "chunk_plan_emul.cpp")])
    lib = C.CDLL(str(out))
    lib.emul_chunk_plan.restype = C.c_uint64
    lib.emul_chunk_plan.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_int, U64P,
                                    C.c_double, C.c_double, C.c_int64, C.c_void_p, C.c_void_p, U64P, C.c_uint64,
                                    C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    lib.emul_exception_queries.restype = C.c_uint64
    lib.emul_exception_queries.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, U64P, C.c_uint64,
                                           np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")]
    lib.emul_query_of_symbol.restype = C.c_uint64
    lib.emul_query_of_symbol.argtypes = [U64P, C.c_uint64, C.c_uint64, C.c_uint64]
    return lib


class Batch:
    """A batch shape with the schedule's inputs; `stage_ms` / `backlog` are what a hybrid run observes per chunk."""

    def __init__(self, nq, offsets=None, fixed_len=0, first_symbol=0, prepacked=False, pack=False, hybrid=False,
                 limits=(4 * MiB, 32 * MiB, 4 * MiB, 64 * MiB), pack_rate=4.0e6 * 15, link=50e6, fail_at=-1,
                 stage_ms=None, backlog=None):
        self.nq, self.fixed_len, self.first_symbol = nq, fixed_len, first_symbol
        self.offsets = None if offsets is None else np.ascontiguousarray(offsets, dtype=np.uint64)
        self.prepacked, self.pack, self.hybrid = prepacked, pack, hybrid
        self.limits, self.pack_rate, self.link, self.fail_at = limits, pack_rate, link, fail_at
        self.olist = None if offsets is None else self.offsets.tolist()
        self.cap = cap = min(nq, 1 << 17) + 1  # room for every chunk the tests make
        self.stage_ms = np.zeros(cap) if stage_ms is None else np.resize(np.asarray(stage_ms, dtype=np.float64), cap)
        self.backlog = np.zeros(cap, np.uint64) if backlog is None else np.resize(np.asarray(backlog, dtype=np.uint64), cap)

    def sym(self, i):
        return int(self.offsets[i]) if self.offsets is not None else i * self.fixed_len + self.first_symbol


def run_header(lib, b):
    cap = b.cap
    out = np.zeros(6 * cap, dtype=np.uint64)
    bad, max_sym = C.c_uint64(), C.c_uint64()
    n = lib.emul_chunk_plan(None if b.offsets is None else b.offsets.ctypes.data, b.fixed_len, b.first_symbol, b.nq,
                            int(b.prepacked), int(b.pack), int(b.hybrid), np.array(b.limits, dtype=np.uint64),
                            b.pack_rate, b.link, b.fail_at, b.stage_ms.ctypes.data, b.backlog.ctypes.data, out, cap,
                            C.byref(bad), C.byref(max_sym))
    chunks = [tuple(int(x) for x in out[6 * i: 6 * i + 6]) for i in range(n)]
    assert n < cap or bad.value != 2 ** 64 - 1
    return chunks, (None if bad.value == 2 ** 64 - 1 else bad.value), max_sym.value


def run_model(b):
    """search_host's chunk loop as it was written inline in api.cu, transcribed statement by statement."""
    first, cmax, tail, max_queries = b.limits
    nq, offsets, fixed_len = b.nq, b.offsets, b.fixed_len
    hybrid, prepacked, pack_on = b.hybrid, b.prepacked, b.pack
    sym_end = b.sym(nq)
    pack_rate, raw_next, raw_want, budget = b.pack_rate, hybrid, first, first
    chunks, q0, k = [], 0, 0
    while q0 < nq:
        pack_chunk = pack_on
        if hybrid and pack_on and raw_next:
            pack_chunk = False
        unit = 4 if (pack_chunk or prepacked) else 1
        remaining = sym_end - b.sym(q0)
        want = raw_want if (hybrid and pack_on and not pack_chunk) else budget * unit
        if remaining <= want:
            want = remaining - tail * unit if remaining > 2 * tail * unit else remaining
        if offsets is not None:
            # std::upper_bound(offsets + q0 + 1, offsets + nq + 1, offsets[q0] + want)
            it = bisect.bisect_right(b.olist, b.olist[q0] + want, q0 + 1, nq + 1)
            q1 = q0 + (it - (q0 + 1))
            if q1 == q0:
                q1 = q0 + 1
        else:
            q1 = q0 + (max(1, want // fixed_len) if fixed_len else max_queries)
        q1 = min(q1, min(nq, q0 + max_queries))
        if pack_chunk or not (hybrid and pack_on):
            budget = min(budget * 2, cmax)
        sym0, sym1 = b.sym(q0), b.sym(q1)
        if sym1 < sym0 or sym1 > sym_end:
            return chunks, q0
        nsym = sym1 - sym0
        chunk_packed = False
        if nsym and pack_chunk:
            if k == b.fail_at:
                pack_on = False
            else:
                chunk_packed = True
        chunks.append((q0, q1, sym0, sym1, int(pack_chunk), int(chunk_packed)))
        if hybrid:
            stage_ms = float(b.stage_ms[k])
            if chunk_packed and stage_ms > 0.02:
                pack_rate = 0.5 * pack_rate + 0.5 * nsym / stage_ms
            if chunk_packed:
                t_pack = budget * 4 / pack_rate
                have = float(b.backlog[k])
                need = t_pack * b.link
                raw_next = pack_on and need - have >= float(2 << 20)
                raw_want = min(int(need - have), 4 * cmax) if raw_next else 0
            else:
                raw_next = False
        q0 = q1
        k += 1
    return chunks, None


def random_batch(rng, kind):
    small = rng.random() < 0.5
    limits = (rng.choice([1, 2, 4]) * MiB, rng.choice([1, 2, 4, 8, 32]) * MiB, rng.choice([1, 2, 4]) * MiB,
              rng.choice([1000, 64 * MiB]))
    if small:  # small budgets so that a modest batch makes many chunks
        limits = (rng.choice([1, 3, 64]) * 1024, rng.choice([4, 16, 256]) * 1024, rng.choice([1, 2, 8]) * 1024,
                  rng.choice([300, 5000, 64 * MiB]))
    total = rng.randrange(1, 12 if small else 40) * (64 * 1024 if small else 4 * MiB)
    if kind == "fixed":
        fixed_len = rng.choice([0, 5, 50, 150, 100_000])
        nq = rng.randrange(1, 50_000) if fixed_len == 0 else max(1, total // max(fixed_len, 1))
        args = dict(fixed_len=fixed_len, first_symbol=rng.choice([0, 3, 1001]))
    else:
        nq = rng.randrange(1, 20_000)
        lens = np.array([rng.choice([0, 1, 30, 50, 150, 4000]) for _ in range(min(nq, 64))], dtype=np.uint64)
        lens = np.resize(lens, nq)
        rng_np = np.random.default_rng(rng.randrange(1 << 30))
        rng_np.shuffle(lens)
        offsets = np.concatenate([[rng.choice([0, 7, 12345])], np.cumsum(lens) + 0]).astype(np.uint64)
        offsets[1:] += offsets[0]
        args = dict(offsets=offsets)
    prepacked = rng.random() < 0.25
    pack = not prepacked and rng.random() < 0.7
    hybrid = pack and rng.random() < 0.6
    n = min(nq, 1 << 17) + 1
    stage_ms = [rng.choice([0.0, 0.01, 0.019, 0.021, 0.05, 0.1, 0.5, 3.0, 20.0]) for _ in range(n)] if hybrid else None
    backlog = [rng.choice([0, 1 << 20, 8 << 20, 200 << 20]) for _ in range(n)] if hybrid else None
    fail_at = rng.choice([-1, -1, 0, 1, 2, 5]) if pack else -1
    return Batch(nq, prepacked=prepacked, pack=pack, hybrid=hybrid, limits=limits, fail_at=fail_at, stage_ms=stage_ms,
                 backlog=backlog, pack_rate=rng.choice([4.0e6, 6.0e7]), link=rng.choice([50e6, 5e6]), **args)


def check_properties(b, chunks, bad, max_sym):
    first, cmax, tail, max_queries = b.limits
    assert max_sym == min(b.sym(b.nq) - b.sym(0), 4 * cmax)
    q = 0
    for (q0, q1, sym0, sym1, pack, packed) in chunks:
        assert q0 == q and q1 > q0, "chunks tile the batch in order"
        assert q1 - q0 <= max_queries
        assert (sym0, sym1) == (b.sym(q0), b.sym(q1))
        if q1 - q0 > 1 and first <= cmax:  # (a first budget above the largest one is used as it is)
            assert sym1 - sym0 <= max_sym
        assert not packed or pack
        q = q1
    if bad is None:
        assert q == b.nq, "chunks cover [0, nq)"
        q0, q1, sym0, sym1, pack, _ = chunks[-1]
        unit = 4 if (pack or b.prepacked) else 1
        assert q1 - q0 == 1 or q1 - q0 == max_queries or sym1 - sym0 <= 2 * tail * unit, "the batch ends with a tail chunk"
    else:
        assert bad == q


@pytest.mark.parametrize("kind", ["fixed", "offsets"])
def test_schedule_equals_head_model(lib, kind):
    rng = random.Random(1 if kind == "fixed" else 2)
    seen = set()
    for _ in range(300):
        b = random_batch(rng, kind)
        chunks, bad, max_sym = run_header(lib, b)
        want_chunks, want_bad = run_model(b)
        assert chunks == want_chunks and bad == want_bad, (kind, b.nq, b.limits, b.pack, b.hybrid, b.fail_at)
        check_properties(b, chunks, bad, max_sym)
        seen.add((b.prepacked, b.pack, b.hybrid, b.fail_at >= 0, len(chunks) > 3))
        if b.hybrid:
            seen.add(("raw and packed", any(not c[5] for c in chunks) and any(c[5] for c in chunks)))
    assert (False, True, True, False, True) in seen and (True, False, False, False, True) in seen
    assert ("raw and packed", True) in seen, "no hybrid run alternated raw and packed chunks"


def test_packing_failed_keeps_the_cut_chunk(lib):
    # the chunk whose packing fails was cut with four symbols per link byte; the chunks after it are IO bytes
    b = Batch(100_000, fixed_len=100, pack=True, limits=(64 * 1024, 1 * MiB, 16 * 1024, 64 * MiB), fail_at=2)
    chunks, bad, _ = run_header(lib, b)
    assert bad is None and chunks == run_model(b)[0]
    assert [c[4] for c in chunks[:3]] == [1, 1, 1] and [c[5] for c in chunks[:3]] == [1, 1, 0]
    assert chunks[2][3] - chunks[2][2] == 4 * 256 * 1024 // 100 * 100
    assert all(c[4] == 0 for c in chunks[3:])
    assert chunks[3][3] - chunks[3][2] == 512 * 1024 // 100 * 100


def test_hybrid_raw_chunk_sized_from_pack_time_and_backlog(lib):
    # link at 50 MB/ms, pool at 100 M symbols/ms: the next packed chunk (budget * 4 symbols) takes budget * 4 / 1e8 ms;
    # the link needs that times 50e6 bytes minus what is still queued -- a raw chunk of that size, then a packed one
    kw = dict(fixed_len=1, pack=True, hybrid=True, pack_rate=1e8, limits=(4 * MiB, 32 * MiB, 4 * MiB, 1 << 40))
    b = Batch(1 << 30, stage_ms=[0.0] * 8, backlog=[5 * MiB] * 8, **kw)
    chunks, bad, _ = run_header(lib, b)
    assert bad is None and chunks == run_model(b)[0]
    sizes = [(c[3] - c[2], c[5]) for c in chunks[:4]]
    assert sizes[0] == (4 * MiB, 0), "a hybrid batch opens with a raw chunk"
    assert sizes[1] == (4 * 4 * MiB, 1)  # (the budget doubles on packed chunks only)
    raw = int(8 * MiB * 4 / 1e8 * 50e6 - 5 * MiB)
    assert sizes[2] == (raw, 0) and sizes[3][1] == 1
    # a staging time above 0.02 ms refines the pack rate (an EMA of symbols per ms), one at or below it does not
    for stage_ms in (0.02, 0.05):
        b = Batch(1 << 30, stage_ms=[stage_ms] * 8, backlog=[5 * MiB] * 8, **kw)
        rate = 0.5 * 1e8 + 0.5 * (16 * MiB) / stage_ms if stage_ms > 0.02 else 1e8
        chunks = run_header(lib, b)[0]
        assert chunks[2][3] - chunks[2][2] == min(int(8 * MiB * 4 / rate * 50e6 - 5 * MiB), 4 * 32 * MiB)
    # a backlog that covers the pack time: no raw chunk
    b = Batch(1 << 30, stage_ms=[0.0] * 8, backlog=[1 << 40] * 8, **kw)
    assert [c[5] for c in run_header(lib, b)[0][1:6]] == [1] * 5


def test_bad_offsets_reported_at_first_crossing_boundary(lib):
    rng = random.Random(5)
    for trial in range(200):
        nq = rng.randrange(2, 300)
        offsets = np.concatenate([[0], np.cumsum(np.array([rng.randrange(0, 9) for _ in range(nq)]))]).astype(np.uint64)
        j = rng.randrange(1, nq)
        if trial % 2:
            offsets[j] = int(offsets[nq]) + rng.randrange(1, 100)  # leaves the batch
        else:
            offsets[j] = max(0, int(offsets[j - 1]) - rng.randrange(1, 5)) if offsets[j - 1] else int(offsets[nq]) + 1
        # one query per chunk: every boundary is checked, so the first bad one is found
        b = Batch(nq, offsets=offsets, limits=(64, 64, 16, 1))
        chunks, bad, _ = run_header(lib, b)
        want = next(i for i in range(1, nq + 1)
                    if offsets[i] < offsets[i - 1] or offsets[i] > offsets[nq]) - 1
        assert bad == want and len(chunks) == want
        assert (chunks, bad) == run_model(b)
        # larger chunks: reported at the start of the first chunk whose end crosses them, or by the kernel
        b = Batch(nq, offsets=offsets, limits=(rng.choice([8, 64, 512]), 1024, 8, 1 << 20))
        chunks, bad = run_model(b)
        assert run_header(lib, b)[:2] == (chunks, bad)
        check_properties(b, chunks, bad, run_header(lib, b)[2])
    sorted_offsets = np.arange(0, 1000, 3, dtype=np.uint64)
    assert run_header(lib, Batch(len(sorted_offsets) - 1, offsets=sorted_offsets, limits=(8, 8, 8, 1)))[1] is None


def model_exception_queries(offsets, fixed_len, q0, q1, sym0, exc):
    out = []
    for pos in exc:
        if offsets is not None:
            q = bisect.bisect_right([int(x) for x in offsets], sym0 + pos, q0, q1 + 1) - q0 - 1
            q = min(q % (1 << 64), q1 - q0 - 1)
        else:
            q = pos // fixed_len
        if not out or out[-1] != q:
            out.append(q)
    return out


def test_exception_queries_match_a_scan(lib):
    rng = random.Random(9)
    for trial in range(400):
        nq = rng.randrange(1, 200)
        fixed = trial % 3 == 0
        if fixed:
            fixed_len, offsets = rng.randrange(1, 20), None
            q0 = rng.randrange(0, nq)
            q1 = rng.randrange(q0 + 1, nq + 1)
            sym0, nsym = q0 * fixed_len + 5, (q1 - q0) * fixed_len
        else:
            fixed_len = 0
            offsets = np.concatenate([[rng.randrange(0, 50)], np.array([rng.randrange(0, 6) for _ in range(nq)])]).cumsum()
            offsets = offsets.astype(np.uint64)
            q0 = rng.randrange(0, nq)
            q1 = rng.randrange(q0 + 1, nq + 1)
            unsorted = trial % 3 == 1
            if unsorted and q1 - q0 > 1:  # a decreasing offset inside the chunk (the kernel reports it)
                i = rng.randrange(q0 + 1, q1)
                offsets[i] = rng.randrange(0, int(offsets[q1]) + 3)
            sym0, nsym = int(offsets[q0]), max(int(offsets[q1]) - int(offsets[q0]), 0)
        exc = np.array(sorted(rng.sample(range(nsym), min(nsym, rng.randrange(0, 12)))) if nsym else [], dtype=np.uint64)
        out = np.zeros(max(len(exc), 1), dtype=np.uint32)
        n = lib.emul_exception_queries(None if offsets is None else offsets.ctypes.data, fixed_len, q0, q1, sym0,
                                       np.ascontiguousarray(exc), len(exc), out)
        got = out[:n].tolist()
        assert got == model_exception_queries(offsets, fixed_len, q0, q1, sym0, exc.tolist())
        assert all(0 <= q < q1 - q0 for q in got), "stays inside the chunk"
        if offsets is None or all(offsets[i] <= offsets[i + 1] for i in range(q0, q1)):
            naive = []
            for pos in exc.tolist():
                s = sym0 + pos
                q = (pos // fixed_len if offsets is None
                     else next(i for i in range(q1 - 1, q0 - 1, -1) if offsets[i] <= s) - q0)
                if offsets is not None:
                    assert offsets[q0 + q] <= s < offsets[q0 + q + 1], "the query holds the symbol"
                if not naive or naive[-1] != q:
                    naive.append(q)
            assert got == naive


def test_query_of_symbol(lib):
    offsets = np.array([3, 3, 5, 5, 5, 9, 12], dtype=np.uint64)
    scan = lambda lo, hi, s: max([i for i in range(lo, hi) if offsets[i] <= s], default=lo - 1)
    for lo in range(0, 7):
        for hi in range(lo, 8):
            for s in range(0, 14):
                assert lib.emul_query_of_symbol(offsets, lo, hi, s) == scan(lo, hi, s) % (1 << 64)
