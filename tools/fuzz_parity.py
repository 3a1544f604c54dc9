"""Randomised parity fuzzing of the CUDA path against the CPU oracle.

  python tools/fuzz_parity.py --seconds 300 [--seed 1]

Every case draws an alphabet, texts of different shapes (random, long runs, periodic, tiny/empty), a
sampling rate, a lookup depth, storage, construction route and text-section on/off, then compares
cursors / counts / hits (SA-row order) / batched extend / single-query cursors and the invalid-symbol
behaviour with the oracle.  Prints the case seed on the first mismatch.
"""
import argparse
import os
import random
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import gdx_testutil as util  # noqa: E402
import genedex_b200 as gdx  # noqa: E402
from oracle import oracle as O  # noqa: E402

ALPHABETS = ["ascii_dna", "ascii_dna_with_n", "ascii_dna_iupac_as_dna_with_n", "ascii_dna_iupac", "protein20",
             "ascii_amino_acid_iupac", "ascii_printable", "u8_until_0", "u8_until_2", "u8_until_5", "u8_until_40",
             "u8_until_254"]


def make_text(rng, syms, kind, max_len):
    n = rng.randrange(max_len + 1)
    if kind == "random":
        return bytes(rng.choice(syms) for _ in range(n))
    if kind == "runs":
        out = bytearray()
        while len(out) < n:
            out += bytes([rng.choice(syms)]) * rng.randrange(1, 200)
        return bytes(out[:n])
    if kind == "periodic":
        unit = bytes(rng.choice(syms) for _ in range(rng.randrange(1, 7)))
        return (unit * (n // len(unit) + 1))[:n]
    return bytes(rng.choice(syms) for _ in range(rng.randrange(0, 4)))  # tiny


def one_case(seed, alph=None):
    """One random case; `alph` fixes the alphabet (any name gdx_testutil knows), the rest is drawn from the seed as
    it would be otherwise."""
    rng = random.Random(seed)
    drawn = rng.choice(ALPHABETS)
    alph = alph or drawn
    oa = util.oracle_alphabet(alph)
    syms, search = util.all_io_symbols(oa), util.searchable_io_symbols(oa)
    texts = [make_text(rng, syms, rng.choice(["random", "random", "runs", "periodic", "tiny"]),
                       rng.choice([50, 500, 5000, 20000])) for _ in range(rng.randrange(1, 7))]
    s = rng.choice([1, 2, 3, 4, 4, 5, 8, 16, 17, 64])
    depth = rng.randrange(0, 7)
    while oa.num_searchable ** depth > 200_000:
        depth -= 1
    storage = rng.choice(["i32", "u32", "i64"])
    on_device = rng.random() < 0.5
    keep_text = rng.random() < 0.8
    dense = rng.random() < 0.6
    seed_tab = rng.choice([None, None, False, 1, 2, 4, 7])
    row_ctx = rng.random() < 0.7
    desc = f"seed={seed} alph={alph} texts={[len(t) for t in texts]} s={s} D={depth} {storage} dev={on_device} text={keep_text} dense={dense} seed={seed_tab} rowctx={row_ctx}"
    oidx = O.OracleIndex.build(texts, oa, storage, sampling_rate=s, lookup_depth=depth)
    cfg = (gdx.FmIndexConfig(storage).suffix_array_sampling_rate(s).lookup_table_depth(depth)
           .construct_on_device(on_device, verify=on_device).keep_text(keep_text).dense_suffix_array(dense).seed_table(seed_tab is not False).row_context_table(row_ctx))
    pidx = cfg.construct_index(texts, util.product_alphabet(gdx, alph))
    if seed_tab and oa.num_searchable ** seed_tab <= 1 << 22:
        pidx.set_seed_table_depth(seed_tab)

    nonempty = [t for t in texts if t]
    qs = []
    for _ in range(rng.randrange(50, 400)):
        kind = rng.randrange(5)
        if kind <= 2 and nonempty:
            t = rng.choice(nonempty)
            p = rng.randrange(len(t))
            q = bytearray(t[p:p + rng.randrange(0, 120)])
            if kind == 1 and q:  # one substitution
                q[rng.randrange(len(q))] = rng.choice(search)
            if kind == 2 and len(nonempty) > 1:  # glue two text pieces
                t2 = rng.choice(nonempty)
                q = q[: len(q) // 2] + bytearray(t2[: rng.randrange(0, 40)])
            q = bytes(q)
        else:
            q = bytes(rng.choice(search) for _ in range(rng.randrange(0, 40)))
        if depth > 0 and any(oa.io_to_dense[c] > oa.num_searchable for c in q):
            continue  # documented deviation: unsearchable symbols cannot index the lookup table
        qs.append(q)
    try:
        util.assert_same_results(oidx, pidx, qs)
        # batched extend + single-query cursors
        sub = qs[:40]
        if sub:
            cursors = pidx.cursors_for_many_queries(sub)
            symbols = bytes(rng.choice(search) for _ in sub)
            ext = pidx.extend_many(cursors, symbols)
            for c, sym, got, q in zip(cursors, symbols, ext, sub):
                assert got.interval == oidx.extend_query_front(c.interval, sym), ("extend", q)
                assert pidx.cursor_for_query(q).interval == oidx.cursor_for_query(q), ("single", q)
        # invalid symbols: panic <=> exception, per query
        invalid_byte = next((b for b in range(255, -1, -1) if oa.io_to_dense[b] == 0), None)
        if invalid_byte is not None:
            for q in qs[:25]:
                if not q:
                    continue
                qb = bytearray(q)
                qb[rng.randrange(len(qb))] = invalid_byte
                qb = bytes(qb)
                try:
                    want = oidx.count_many([qb]).tolist()
                except O.OraclePanic:
                    for fn in (pidx.count_many, pidx.locate_many, pidx.cursors_for_many_queries):
                        try:
                            fn([qb])
                        except gdx.InvalidSymbolError:
                            continue
                        raise AssertionError(("missing panic", qb))
                    continue
                assert pidx.count_many([qb]) == want, ("count with invalid byte", qb)
    except AssertionError as e:
        print("MISMATCH", desc, e, flush=True)
        raise
    return desc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=120)
    ap.add_argument("--seed", type=int, default=1)
    args = ap.parse_args()
    t0, n, seed = time.time(), 0, args.seed * 1_000_003
    while time.time() - t0 < args.seconds:
        one_case(seed)
        seed += 1
        n += 1
    print(f"fuzz ok: {n} cases in {time.time() - t0:.0f} s (seeds {args.seed * 1_000_003}..{seed - 1})")


if __name__ == "__main__":
    main()
