"""GPU tests of the per-call statistics and refusals the locate, count, Hamming and extend paths report through
gdx_stats and their status: walk and verification counters, locate kernel time, the extend error order, and the
refusal of results that cannot fit into device memory on the interval and Hamming locate paths."""
import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gdx():
    import genedex_b200
    assert genedex_b200._lib.load().gdx_device_count() >= 1
    return genedex_b200


@pytest.fixture(scope="module")
def case(gdx):
    """2 Mbp two-text DNA index, suffix array sampled every 4 rows, no dense suffix array (so that the locate walk
    takes steps), and a batch of text windows and random strings."""
    rng = np.random.default_rng(7)
    n = 2_000_000
    text = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, n)].copy()
    texts = [text[:1_300_000].tobytes(), text[1_300_000:].tobytes()]
    oidx = O.OracleIndex.build(texts, O.ALPHABETS["ascii_dna_with_n"](), "u32", sampling_rate=4, lookup_depth=0)
    pidx = gdx.FmIndexConfig("u32").suffix_array_sampling_rate(4).construct_index(texts, gdx.alphabet.ascii_dna_with_n())
    pidx.set_dense_suffix_array(False)
    qs = []
    for i in range(3000):
        m = int(rng.integers(6, 40))
        if i % 3:
            p = int(rng.integers(0, n - 64))
            qs.append(text[p:p + m].tobytes())
        else:
            qs.append(np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, m % 12 + 4)].tobytes())
    data, off = O.pack(qs)
    return dict(oidx=oidx, pidx=pidx, data=data, off=off)


def test_locate_paths_agree_on_walk_counters_without_verification(gdx, case):
    """Without text verification k_search resolves no row to a text position, so locating the batch and locating
    its cursors walk the same rows."""
    pidx, data, off = case["pidx"], case["data"], case["off"]
    pidx.set_text_verification(False)
    try:
        starts, ends = pidx.cursors_many_packed(data, off)
        hoff, hits = pidx.locate_many_packed(data, off)
        s_many = pidx.stats()
        ioff, ihits = pidx.locate_intervals_packed(starts, ends)
        s_iv = pidx.stats()
        counts, chits, release = pidx.locate_many_compact_view(data, off)
        s_compact = pidx.stats()
        release()
    finally:
        pidx.set_text_verification(True)
    assert np.array_equal(hoff, ioff) and np.array_equal(hits, ihits)
    assert np.array_equal(counts, np.diff(hoff).astype(np.uint32))
    assert s_many.hits == s_iv.hits == hits.shape[0] > 0
    assert s_many.locate_walk_steps == s_iv.locate_walk_steps > 0
    assert s_many.walk_steps == s_iv.walk_steps == s_many.locate_walk_steps
    assert s_many.kernel_ms_locate > 0 and s_iv.kernel_ms_locate > 0
    assert s_compact.locate_walk_steps == s_many.locate_walk_steps


def test_dense_suffix_array_needs_no_locate_walk(gdx, case):
    pidx, oidx, data, off = case["pidx"], case["oidx"], case["data"], case["off"]
    pidx.set_dense_suffix_array(True)
    try:
        hoff, hits = pidx.locate_many_packed(data, off)
        s = pidx.stats()
        starts, ends = pidx.cursors_many_packed(data, off)
        pidx.locate_intervals_packed(starts, ends)
        s_iv = pidx.stats()
    finally:
        pidx.set_dense_suffix_array(False)
    ooff, ohits = oidx.locate_many_packed(data, off)
    assert np.array_equal(hoff, ooff) and np.array_equal(hits, ohits)
    assert s.hits > 0 and s.locate_walk_steps == 0
    assert s_iv.hits > 0 and s_iv.locate_walk_steps == 0


def test_count_reports_verification_counters(gdx, case):
    """Without the row context table a verified row walks to its text position."""
    pidx, data, off = case["pidx"], case["data"], case["off"]
    pidx.set_row_context_table(False)
    try:
        with_verify = pidx.count_many_packed(data, off)
        s_on = pidx.stats()
        pidx.set_text_verification(False)
        without = pidx.count_many_packed(data, off)
        s_off = pidx.stats()
    finally:
        pidx.set_text_verification(True)
        pidx.set_row_context_table(True)
    assert np.array_equal(with_verify, without)
    assert s_on.verified_queries > 0 and s_on.walk_steps > 0 and s_on.locate_walk_steps == 0
    assert s_off.verified_queries == 0 and s_off.walk_steps == 0
    assert s_on.lf_steps > 0 and s_off.lf_steps > 0


def test_hamming_locate_and_count_report_the_same_search(gdx, case):
    pidx, data, off = case["pidx"], case["data"], case["off"]
    sub = 500
    sdata, soff = data[: int(off[sub])], off[: sub + 1]
    counts = pidx.count_many_hamming_packed(sdata, soff, 1)
    s_count = pidx.stats()
    hoff, hits = pidx.locate_many_hamming_packed(sdata, soff, 1)
    s_loc = pidx.stats()
    assert s_count.lf_steps == s_loc.lf_steps > 0
    assert s_loc.hits == hits.shape[0] == int(hoff[-1]) == int(counts.sum()) > 0
    assert s_loc.kernel_ms_locate > 0


def test_extend_reports_an_out_of_range_cursor_before_an_invalid_symbol(gdx, case):
    pidx = case["pidx"]
    n = pidx.total_text_len()
    starts = np.zeros(8, dtype=np.uint64)
    ends = np.full(8, n, dtype=np.uint64)
    sym = np.frombuffer(b"ACGTACGT", dtype=np.uint8).copy()
    sym[2] = ord("!")
    ends[5] = n + 1
    with pytest.raises(gdx.GenedexError) as ei:
        pidx.extend_many_packed(starts, ends, sym)
    assert ei.value.status == gdx._lib.GDX_ERR_BAD_ARG
    assert not isinstance(ei.value, gdx.InvalidSymbolError)
    ends[5] = n
    with pytest.raises(gdx.InvalidSymbolError) as ei:
        pidx.extend_many_packed(starts, ends, sym)
    assert ei.value.query == 2


def check_small_locate(case):
    pidx, oidx = case["pidx"], case["oidx"]
    data, off = O.pack([b"ACGTAC", b"TTTTTTTTTTTTTTTTTTTTTTTTTTTTTT", b"GATTACA"])
    ooff, ohits = oidx.locate_many_packed(data, off)
    poff, phits = pidx.locate_many_packed(data, off)
    assert np.array_equal(ooff, poff) and np.array_equal(ohits, phits)


def test_interval_locate_that_cannot_fit_is_refused(gdx, case):
    """30 000 copies of the empty cursor (0, n): 6 * 10^10 hits of 24 device bytes each."""
    pidx = case["pidx"]
    s, e = pidx.cursor_empty().interval
    assert (s, e) == (0, pidx.total_text_len())
    starts = np.full(30_000, s, dtype=np.uint64)
    ends = np.full(30_000, e, dtype=np.uint64)
    with pytest.raises(MemoryError):
        pidx.locate_intervals_packed(starts, ends)
    check_small_locate(case)


def test_hamming_locate_that_cannot_fit_is_refused(gdx, case):
    """30 000 empty queries at k = 0 each match every row."""
    pidx = case["pidx"]
    data, off = O.pack([b""] * 30_000)
    with pytest.raises(MemoryError):
        pidx.locate_many_hamming_packed(data, off, 0)
    check_small_locate(case)
