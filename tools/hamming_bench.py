"""Throughput of the Hamming search on a genome-sized DNA index: gdx_count_many_hamming, gdx_locate_many_hamming and, on
the same queries, the exact gdx_count_many, for k = 0, 1, 2 and query lengths 50 and 100.  The queries are windows of the
text (bench.py's hg38-shaped synthetic genome, ascii_dna_with_n) with 0..2 random substitutions each, seeded.  Prints one
JSON line: queries/s, node expansions (gdx_stats.lf_steps), intervals and hits per query, and the GPU with its power
limit.  Self-checks in the same run: k = 0 counts equal gdx_count_many, and growing k keeps the counts of the smaller
strata and never lowers a total.

  python tools/hamming_bench.py [--text-len 3100000000] [--queries 1000000] [--steps 3] [--warmup 1]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402


def gpu_name_and_power():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power = [x.strip() for x in out[0].split(",")]
        return name, power
    except Exception as e:  # noqa: BLE001 -- reported in the result line
        return f"unknown ({e})", "unknown"


def substitute(q, m, nq, max_subs, seed):
    """0..max_subs substitutions per query (uniform), each to another base."""
    rng = np.random.default_rng(seed)
    qm = q.reshape(nq, m)
    bases = np.frombuffer(b"ACGT", dtype=np.uint8)
    nsub = rng.integers(0, max_subs + 1, nq)
    for r in range(1, max_subs + 1):
        rows = np.flatnonzero(nsub >= r)
        cols = rng.integers(0, m, rows.size)
        cur = qm[rows, cols]
        idx = (np.searchsorted(bases, cur) + rng.integers(1, 4, rows.size)) % 4
        qm[rows, cols] = bases[idx]
    return nsub


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--text-len", type=int, default=3_100_000_000)
    ap.add_argument("--queries", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    import torch

    import bench
    import genedex_b200 as gdx

    dev = torch.device("cuda", 0)
    gpu, power = gpu_name_and_power()
    t0 = time.perf_counter()
    text = bench.make_text_on_device(args.text_len, 0.05, dev)
    nq = args.queries
    batches = {}
    for m in (50, 100):
        q = np.empty(nq * m, dtype=np.uint8)
        bench.fill_query_range(text, q, None, 0, nq, m, dev, seed=bench.QUERY_SEED + 101 + m)
        substitute(q, m, nq, 2, seed=bench.QUERY_SEED + 201 + m)
        batches[m] = q
    host = text.cpu().numpy()
    del text
    torch.cuda.empty_cache()
    idx = (gdx.FmIndexConfig("u32").construct_on_device(True)
           .construct_index_packed(host, np.array([0, host.size], dtype=np.uint64), gdx.alphabet.ascii_dna_with_n()))
    del host
    setup_s = time.perf_counter() - t0

    def timed(fn):
        for _ in range(args.warmup):
            out = fn()
        torch.cuda.synchronize()
        t = time.perf_counter()
        for _ in range(args.steps):
            out = fn()
        torch.cuda.synchronize()  # (every call returns after its results are on the host)
        return (time.perf_counter() - t) / args.steps, out, idx.stats()

    results, checks = {}, {}
    for m, q in batches.items():
        dt, exact, st = timed(lambda: idx.count_many_packed(q, None, m, nq))
        r = {"count_many": {"queries_per_s": nq / dt, "lf_steps_per_query": st.lf_steps / nq,
                            "kernel_ms": st.kernel_ms_search}}
        prev = None
        for k in (0, 1, 2):
            dt, counts, st = timed(lambda: idx.count_many_hamming_packed(q, None, k, m, nq))
            rc = {"queries_per_s": nq / dt, "lf_steps_per_query": st.lf_steps / nq, "kernel_ms": st.kernel_ms_search,
                  "occurrences_per_query": float(counts.sum()) / nq}
            off, _, _, _ = idx.cursors_many_hamming_packed(q, None, k, m, nq)
            rc["intervals_per_query"] = float(off[-1]) / nq
            dt, (hoff, hits), st = timed(lambda: idx.locate_many_hamming_packed(q, None, k, m, nq))
            rl = {"queries_per_s": nq / dt, "hits_per_query": hits.shape[0] / nq, "kernel_ms_search": st.kernel_ms_search,
                  "kernel_ms_locate": st.kernel_ms_locate}
            r[f"k{k}"] = {"count": rc, "locate": rl}
            if k == 0:
                checks[f"m{m}_k0_equals_count_many"] = bool(np.array_equal(counts[:, 0], exact))
            else:
                checks[f"m{m}_k{k}_keeps_smaller_strata"] = bool(np.array_equal(counts[:, :k], prev))
                checks[f"m{m}_k{k}_totals_do_not_decrease"] = bool((counts.sum(axis=1) >= prev.sum(axis=1)).all())
            checks[f"m{m}_k{k}_hits_equal_counts"] = bool(np.array_equal(np.diff(hoff), counts.sum(axis=1)))
            prev = counts
        results[f"m{m}"] = r
    line = {"metric": "Hamming search on a synthetic DNA index", "text_len": args.text_len, "queries": nq,
            "substitutions_per_query": "uniform 0..2", "steps": args.steps, "warmup": args.warmup,
            "gpu": gpu, "power_limit": power, "setup_s": round(setup_s, 1), "results": results,
            "checks": checks, "checks_pass": all(checks.values())}
    print(json.dumps(line))
    return 0 if line["checks_pass"] else 1


if __name__ == "__main__":
    sys.exit(main())
