"""Expected results of the Hamming search (include/genedex_b200.h, "approximate search"), computed without it.  Three
references with one interface, expected(query, k) -> (occ, ivs, rows):
  - Naive: a scan over every window of every text, and the oracle's exact search for the interval of each matching
    window string (small texts);
  - Neighbourhood: every string within k substitutions of the query through the oracle's exact search (short queries
    over few symbols, texts of any size the oracle builds);
  - SeedAndVerify: the oracle's locate of k + 1 exact pieces of the query, each candidate window checked on the dense
    text (long queries, many symbols).
Shared by the host emulation test, the GPU tests and tools/hamming_bench.py (neighbours)."""
import itertools
import math
import random

import numpy as np


def searchable(oa):
    return [c for c in range(256) if 1 <= oa.io_to_dense[c] <= oa.num_searchable]


def hamming_texts(rng: random.Random, oa, ntexts, max_len, p_other=0.1):
    """Texts of mostly searchable symbols (so that windows match), some other valid symbols, and empty texts."""
    ok = bytes(oa.dense_to_io[: oa.num_searchable])
    other = bytes(oa.dense_to_io)
    out = []
    for _ in range(ntexts):
        n = 0 if rng.random() < 0.15 else rng.randrange(max_len + 1)
        out.append(bytes(rng.choice(other) if rng.random() < p_other else rng.choice(ok) for _ in range(n)))
    return out


def hamming_queries(rng: random.Random, oa, texts, n, max_len, k):
    """Windows of searchable symbols sampled from the texts with 0..k substitutions, random queries, and lengths from 0
    up to max_len (so that k >= m occurs).  Any searchable IO byte may stand for its dense symbol (case folding)."""
    syms = searchable(oa)
    sset = set(syms)
    qs = []
    nonempty = [t for t in texts if t]
    while len(qs) < n:
        m = rng.randrange(max_len + 1)
        if nonempty and rng.random() < 0.7:
            t = rng.choice(nonempty)
            p = rng.randrange(len(t))
            w = bytearray(t[p:p + m])
            if any(c not in sset for c in w):
                continue
            for _ in range(rng.randrange(k + 1)):
                if w:
                    w[rng.randrange(len(w))] = rng.choice(syms)
            qs.append(bytes(w))
        else:
            qs.append(bytes(rng.choice(syms) for _ in range(m)))
    return qs


class Naive:
    """Window strings of the texts in the dense representation, with their positions in the concatenated text."""

    def __init__(self, oidx, texts, oa):
        self.oidx, self.oa = oidx, oa
        self.sa = oidx.suffix_array()
        self.n = oidx.text_len
        self.dense = [np.asarray(oa.io_to_dense, dtype=np.uint8)[np.frombuffer(t, dtype=np.uint8)] if t else
                      np.zeros(0, np.uint8) for t in texts]
        self.starts = []
        pos = 0
        for t in texts:
            self.starts.append(pos)
            pos += len(t) + 1
        self._windows = {}

    def windows(self, m):
        """{dense window string: [text positions]} of every window of length m made of searchable symbols."""
        if m not in self._windows:
            w = {}
            ns = self.oa.num_searchable
            for t0, d in zip(self.starts, self.dense):
                if len(d) < m or m == 0:
                    continue
                win = np.lib.stride_tricks.sliding_window_view(d, m)
                ok = np.flatnonzero((win.min(axis=1) >= 1) & (win.max(axis=1) <= ns))
                for p in ok.tolist():
                    w.setdefault(win[p].tobytes(), []).append(t0 + p)
            keys = list(w)
            arr = np.frombuffer(b"".join(keys), dtype=np.uint8).reshape(len(keys), m) if keys else np.zeros((0, m), np.uint8)
            self._windows[m] = (w, keys, arr)
        return self._windows[m][0]

    def expected(self, query, k):
        """-> (occurrences per mismatch count [k + 1], intervals [(start, end, d)] sorted by start, rows per interval)"""
        qd = np.asarray(self.oa.io_to_dense, dtype=np.uint8)[np.frombuffer(query, dtype=np.uint8)]
        m = len(query)
        occ = [0] * (k + 1)
        ivs = []
        if m == 0:
            return [self.n] + [0] * k, [(0, self.n, 0)], [sorted(self.sa.tolist())]
        w = self.windows(m)
        _, keys, arr = self._windows[m]
        dist = np.count_nonzero(arr != qd, axis=1) if len(keys) else np.zeros(0, int)
        for i in np.flatnonzero(dist <= k).tolist():
            win, d = keys[i], int(dist[i])
            pos = w[win]
            occ[d] += len(pos)
            io = bytes(self.oa.dense_to_io[c - 1] for c in win)
            s, e = self.oidx.cursor_for_query(io)
            assert e - s == len(pos), "the oracle's interval of a window string holds its occurrences"
            assert sorted(self.sa[s:e].tolist()) == sorted(pos)
            ivs.append((s, e, d))
        ivs.sort()
        return occ, ivs, [sorted(self.sa[s:e].tolist()) for s, e, _ in ivs]


def neighbourhood_size(m, k, ns):
    """Number of strings within k substitutions of a query of length m over ns symbols."""
    return sum(math.comb(m, d) * (ns - 1) ** d for d in range(min(k, m) + 1))


def neighbours(qd, k, ns):
    """Every string within k substitutions of the dense query qd over the symbols 1..ns, each once: d positions in
    increasing order and, at each, a symbol other than the query's -> (strings [N, m] uint8, distances [N])."""
    qd = np.asarray(qd, dtype=np.uint8)
    m = qd.size
    out, dist = [qd[None, :].copy()], [np.zeros(1, np.int64)]
    for d in range(1, min(k, m) + 1):
        if ns < 2:
            break
        combos = np.array(list(itertools.combinations(range(m), d)), dtype=np.int64)       # (C, d)
        subs = np.array(list(itertools.product(range(1, ns), repeat=d)), dtype=np.int64)  # (S, d)
        cols = np.repeat(combos, len(subs), axis=0)
        offs = np.tile(subs, (len(combos), 1))
        block = np.repeat(qd[None, :], len(cols), axis=0)
        rows = np.arange(len(cols))[:, None]
        block[rows, cols] = ((qd[cols].astype(np.int64) - 1 + offs) % ns + 1).astype(np.uint8)
        out.append(block)
        dist.append(np.full(len(cols), d, np.int64))
    return np.concatenate(out), np.concatenate(dist)


class _OracleRef:
    """What both references share: the oracle, its dense text and where each text starts in it."""

    def __init__(self, oidx, oa):
        self.oidx, self.oa = oidx, oa
        self.n = oidx.text_len
        self.ns = oa.num_searchable
        self.dense_text = oidx.dense_text()
        ends = np.flatnonzero(self.dense_text == 0)  # the sentinel after each text
        self.text_start = np.concatenate([[0], ends[:-1] + 1]).astype(np.int64)
        self.text_len = ends.astype(np.int64) - self.text_start
        self.to_io = np.frombuffer(oa.dense_to_io, dtype=np.uint8)
        self.to_dense = np.asarray(oa.io_to_dense, dtype=np.uint8)

    def _empty(self, k):
        return [self.n] + [0] * k, [(0, self.n, 0)], [list(range(self.n))]

    def _intervals(self, strings, dist, k, positions=None, counts=None):
        """Intervals of the distinct dense strings [N, m] (all occurring) at their distances -> the (occ, ivs, rows)
        of expected().  The width of each interval must equal its number of occurrences: the located rows, and, when
        given, the string's count or its text positions (global, sorted)."""
        m = strings.shape[1]
        occ = [0] * (k + 1)
        if not len(strings):
            return occ, [], []
        data = np.ascontiguousarray(self.to_io[strings.astype(np.int64) - 1].reshape(-1))
        off = np.arange(len(strings) + 1, dtype=np.uint64) * m
        s, e = self.oidx.cursors_many_packed(data, off)
        hoff, hits = self.oidx.locate_many_packed(data, off, nthreads=0)
        assert np.array_equal(np.diff(hoff), e - s), "the oracle locates every row of an interval"
        if counts is not None:
            assert np.array_equal(e - s, counts), "an interval's width is its string's number of occurrences"
        glob = self.text_start[hits[:, 0].astype(np.int64)] + hits[:, 1].astype(np.int64)
        ivs, rows = [], []
        for i in np.argsort(s, kind="stable").tolist():
            pos = sorted(glob[int(hoff[i]):int(hoff[i + 1])].tolist())
            if positions is not None:
                assert pos == positions[i], "the oracle's interval of a window string holds its occurrences"
            assert int(e[i]) > int(s[i])
            occ[int(dist[i])] += int(e[i] - s[i])
            ivs.append((int(s[i]), int(e[i]), int(dist[i])))
            rows.append(pos)
        return occ, ivs, rows


class Neighbourhood(_OracleRef):
    """Enumerates every string within k substitutions of the query and asks the oracle's exact search which occur.
    Cheap while neighbourhood_size(m, k, ns) stays below some 50 000."""

    def expected(self, query, k):
        """-> (occurrences per mismatch count [k + 1], intervals [(start, end, d)] sorted by start, rows per interval)"""
        if not query:
            return self._empty(k)
        strings, dist = neighbours(self.to_dense[np.frombuffer(query, dtype=np.uint8)], k, self.ns)
        data = np.ascontiguousarray(self.to_io[strings.astype(np.int64) - 1].reshape(-1))
        off = np.arange(len(strings) + 1, dtype=np.uint64) * len(query)
        cnt = self.oidx.count_many_packed(data, off, nthreads=0)
        keep = np.flatnonzero(cnt)
        return self._intervals(strings[keep], dist[keep], k, counts=cnt[keep])


class SeedAndVerify(_OracleRef):
    """Pigeonhole: a window within k substitutions of the query matches one of k + 1 pieces of it exactly.  Every
    piece is located with the oracle, each hit gives a candidate window, and the candidates are checked on the dense
    text.  For long queries and many symbols, where enumeration explodes; every piece needs at least 3 symbols."""

    def expected(self, query, k):
        if not query:
            return self._empty(k)
        m = len(query)
        cut = [m * i // (k + 1) for i in range(k + 2)]
        assert min(b - a for a, b in zip(cut, cut[1:])) >= 3, "pieces of fewer than 3 symbols"
        qd = self.to_dense[np.frombuffer(query, dtype=np.uint8)]
        pieces = [query[a:b] for a, b in zip(cut, cut[1:])]
        pdata, poff = np.frombuffer(b"".join(pieces), dtype=np.uint8).copy(), np.array(cut, dtype=np.uint64)
        hoff, hits = self.oidx.locate_many_packed(pdata, poff, nthreads=0)
        cands = []
        for j in range(k + 1):
            h = hits[int(hoff[j]):int(hoff[j + 1])].astype(np.int64)
            t, p = h[:, 0], h[:, 1] - cut[j]
            ok = (p >= 0) & (p + m <= self.text_len[t])
            cands.append(self.text_start[t[ok]] + p[ok])
        cand = np.unique(np.concatenate(cands))
        if not cand.size:
            return [0] * (k + 1), [], []
        win = self.dense_text[cand[:, None] + np.arange(m)]
        dist = np.count_nonzero(win != qd, axis=1)
        good = (win.min(axis=1) >= 1) & (win.max(axis=1) <= self.ns) & (dist <= k)
        strings, inv = np.unique(win[good], axis=0, return_inverse=True)
        inv = inv.reshape(-1)
        positions = [[] for _ in range(len(strings))]
        for i, g in zip(inv.tolist(), cand[good].tolist()):
            positions[i].append(g)
        sdist = np.count_nonzero(strings != qd, axis=1)
        return self._intervals(strings, sdist, k, positions)


class Cheapest:
    """Neighbourhood where the neighbourhood has at most `limit` strings, else SeedAndVerify."""

    def __init__(self, oidx, oa, limit=50_000):
        self.nb, self.sv, self.limit = Neighbourhood(oidx, oa), SeedAndVerify(oidx, oa), limit

    def expected(self, query, k):
        if neighbourhood_size(len(query), k, self.nb.ns) <= self.limit:
            return self.nb.expected(query, k)
        return self.sv.expected(query, k)


SUPERBLOCK = 1 << 16  # rank superblock: positions whose counts come from one sbc row


def multi_superblock_texts(seed, oa, total, ntexts=6, p_other=0.003, run=300):
    """About `total` symbols in ntexts texts (two of them empty) that span several rank superblocks: mostly searchable
    symbols, a few other valid ones, and where the alphabet has them, runs of `run` unsearchable symbols across every
    superblock boundary of the concatenated text."""
    nrng = np.random.default_rng(seed)
    ns = oa.num_searchable
    ok = np.frombuffer(bytes(oa.dense_to_io[:ns]), dtype=np.uint8)
    other = np.frombuffer(bytes(oa.dense_to_io[ns:]), dtype=np.uint8)
    body = nrng.choice(ok, total)
    if other.size:
        sprinkle = np.flatnonzero(nrng.random(total) < p_other)
        body[sprinkle] = nrng.choice(other, sprinkle.size)
        for b in range(SUPERBLOCK, total, SUPERBLOCK):
            lo, hi = b - run // 2, min(b + run // 2, total)
            body[lo:hi] = nrng.choice(other, hi - lo)
    cuts = np.sort(nrng.choice(np.arange(1, total), ntexts - 3, replace=False))
    texts = [t.tobytes() for t in np.split(body, cuts)]
    texts.insert(1, b"")
    texts.append(b"")
    return texts


def window_queries(seed, oa, texts, n, m, k):
    """n queries of length m: windows of the texts (unsearchable symbols replaced) with 0..k substitutions, a quarter
    of them starting next to a superblock boundary of the concatenated text; random strings; windows glued across a
    text border (which match only where the glued string occurs elsewhere)."""
    rng = random.Random(seed)
    syms = bytes(oa.dense_to_io[: oa.num_searchable])
    sset = set(searchable(oa))
    starts, pos = [], 0
    for t in texts:
        starts.append(pos)
        pos += len(t) + 1
    long = [i for i, t in enumerate(texts) if len(t) >= m]

    def clean(w):
        return bytearray(c if c in sset else rng.choice(syms) for c in w)

    qs = []
    while len(qs) < n:
        r = rng.random()
        if r < 0.7 and long:
            i = rng.choice(long)
            t = texts[i]
            if r < 0.2:  # next to a superblock boundary
                b = SUPERBLOCK * rng.randrange(1, max(2, (starts[i] + len(t)) // SUPERBLOCK + 1)) - starts[i]
                p = min(max(b - rng.randrange(m + 1), 0), len(t) - m)
            else:
                p = rng.randrange(len(t) - m + 1)
            w = clean(t[p:p + m])
            for _ in range(rng.randrange(k + 1)):
                w[rng.randrange(m)] = rng.choice(syms)
            qs.append(bytes(w))
        elif r < 0.85 and len(long) > 1 and m > 1:
            a, b = rng.sample(long, 2)
            j = rng.randrange(1, m)
            qs.append(bytes(clean(texts[a][len(texts[a]) - j:] + texts[b][:m - j])))
        else:
            qs.append(bytes(rng.choice(syms) for _ in range(m)))
    return qs
