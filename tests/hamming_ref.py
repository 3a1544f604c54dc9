"""Expected results of the Hamming search (include/genedex_b200.h, "approximate search"), computed without it: a naive
scan over every window of every text, and the oracle's exact search for the interval of each matching window string.
Shared by the host emulation test and the GPU tests."""
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
