#!/usr/bin/env python
"""bench.py -- headline benchmark of the batched FM-index search path (BASELINE.json).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...   # CPU reference arm (oracle port)

Workload (every N; BASELINE.json configs[4] = SURVEY 8d "C5", which at N = 8 gives every GPU exactly the
configs[1] = "C2" batch): hg38-shaped synthetic 3.1 Gbp DNA single text (`ascii_dna_with_n`, ~5 % N in
runs <= 10 kbp, u32 storage, sampling rate 4, lookup depth 0 = crate defaults) and ONE batch of 60 M
length-50 queries sampled from the text (3 GB of IO bytes).  The batch is cut into N contiguous ranges by
the library (gdx_shard_range); rank r searches range r on its full index replica through
gdx_count_many_sharded / gdx_locate_many_sharded (n_local = 1, first_shard = r, n_shards = N) -- strong
scaling, no collective on the query path.  The replicas are made by the library's own ncclBroadcast
(gdx_index_broadcast); torch.distributed only carries the 128-byte NCCL id, barriers and the gather that
brings every shard's results to rank 0 for the oracle comparison.  One "step" = one pass over the batch.

`value`    queries/s, the shard's IO bytes already resident in HBM: one k_search launch per rank and step.
`e2e`      the same through the C ABI from ordinary host memory: host 2-bit packing (library thread pool),
           H2D, kernels, D2H of uint32 counts, widening into the caller's uint64 array -- all inside the
           timed region.  `e2e.prepacked`: the caller hands over 2-bit packed reads (pinned), no host packing.
`roofline` the k_search launches of `value`: algorithmic bytes (SURVEY 8d: m + 8 [seed entry] + 2*R*steps + 16
           per query, + R per walk step + 64 per text-verified query; R = 32 B rank record) / CUDA-event time,
           against MEASURED_PEAKS.json; `traffic` = DRAM bytes per launch from the committed ncu capture.
`locate`   the batch through gdx_locate_many_sharded (1 hit per query) and `locate.multi_hit`: 2 M length-14
           queries (~11 hits each) with the dense suffix array and with the configured sampled one (s = 4),
           each with the roofline of the locate kernels (SURVEY 8d: R*walk_steps + 32 + 16 B per hit).
`no_accelerators` the index exactly as BASELINE names it (s = 4, D = 0: no seed table, no dense suffix array,
           no text verification = every LF step of the reference runs), device-resident and end to end.
`single_process` (N > 1) rank 0 alone drives all N GPUs through ONE gdx_count_many_sharded call.
`cpu_baseline` (N = 1) the oracle's port of the reference's 64-query batched search on the host cores.

--dump-outputs DIR  after the run, writes what the timed paths computed in their last step to DIR as float64 .npy files,
           for a fixed, seeded sample of the batch (count_query.npy: the batch positions of the sample): count.npy, the
           counts a caller of gdx_count_many_device receives (`value`), and locate_first_position.npy, the text
           position of each sampled query's first hit from the last `locate` step (not with --no-locate).  The inputs
           are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: the benchmark writes nothing into it
os.environ.setdefault("GDX_ORACLE_NATIVE", "1")  # CPU baseline: oracle rebuilt with -march=native on this box

TEXT_SEED = 0x5EED0001
QUERY_SEED = 0x5EED0002
N_CODE = ord("N")
QCHUNK = 1 << 21  # queries are generated in chunks of this many, each from its own seed
DUMP_SEED = 0x5EED0003
DUMP_SAMPLE = 1 << 21  # --dump-outputs: this many queries (16 MiB of float64 per file, 48 MiB in all)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--text-len", type=int, default=3_100_000_000)
    ap.add_argument("--queries", type=int, default=60_000_000)
    ap.add_argument("--query-len", type=int, default=50)
    ap.add_argument("--lookup-depth", type=int, default=0)
    ap.add_argument("--sampling-rate", type=int, default=4)
    ap.add_argument("--n-fraction", type=float, default=0.05)
    ap.add_argument("--no-locate", action="store_true", help="skip the locate measurements")
    ap.add_argument("--no-extras", action="store_true", help="skip no_accelerators / prepacked / single_process")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip oracle parity + CPU baseline")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU work of the cpu_baseline sample")
    ap.add_argument("--multi-hit-queries", type=int, default=2_000_000)
    ap.add_argument("--multi-hit-len", type=int, default=14)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a seeded sample of the last timed step's counts and hits to DIR as .npy (see the docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the outputs of this repo's CUDA path (--impl ours)")
    return args


# ---- synthetic data (torch on the GPU is plumbing here: RNG + gathers, nothing of the search path) ---
def make_text_on_device(n_symbols, n_fraction, device):
    """hg38-shaped DNA: iid ACGT with ~n_fraction N in runs of 1..10000; returns uint8 IO bytes."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(TEXT_SEED)
    lut = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device=device)
    text = torch.empty(n_symbols, dtype=torch.uint8, device=device)
    step = 1 << 28
    for b in range(0, n_symbols, step):  # chunked to keep the int64 index temporaries small
        e = min(n_symbols, b + step)
        text[b:e] = lut[torch.randint(0, 4, (e - b,), generator=g, device=device, dtype=torch.uint8).long()]
    max_run = min(10_000, max(1, n_symbols // 8))
    n_runs = int(n_fraction * n_symbols / (max_run / 2)) if n_fraction > 0 else 0
    if n_runs:
        cg = torch.Generator()
        cg.manual_seed(TEXT_SEED + 1)
        starts = torch.randint(0, n_symbols - max_run, (n_runs,), generator=cg).tolist()
        lens = torch.randint(1, max_run + 1, (n_runs,), generator=cg).tolist()
        for s, l in zip(starts, lens):
            text[s:s + l] = N_CODE
    return text


def sample_query_chunk(text, chunk, count, m, device, seed=QUERY_SEED):
    """Queries [chunk * QCHUNK, chunk * QCHUNK + count) of the batch: windows of length m sampled uniformly from
    the text, windows containing N rejected.  Every chunk has its own seed, so any rank can make any range."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed * 1_000_003 + chunk)
    n = text.numel()
    ar = torch.arange(m, device=device)
    wins, origins, have = [], [], 0
    while have < count:
        cand = torch.randint(0, n - m, (int((count - have) * 1.3) + 64,), generator=g, device=device)
        win = text[cand[:, None] + ar[None, :]]
        ok = ~(win == N_CODE).any(dim=1)
        win, cand = win[ok][: count - have], cand[ok][: count - have]
        wins.append(win)
        origins.append(cand)
        have += win.shape[0]
    return torch.cat(wins).reshape(-1), torch.cat(origins)


def sample_queries_on_device(text, nq, m, seed, device):
    """nq windows as one device tensor + their origins (tools/: small experiments that keep everything on the GPU)."""
    import torch
    parts = [sample_query_chunk(text, c, min(QCHUNK, nq - c * QCHUNK), m, device, seed) for c in range((nq + QCHUNK - 1) // QCHUNK)]
    return torch.cat([p[0] for p in parts]), torch.cat([p[1] for p in parts])


def fill_query_range(text, q_host, origins_host, b, e, m, device, seed=QUERY_SEED):
    """Writes queries [b, e) of the batch into q_host (uint8, whole-batch sized) and their text positions."""
    import torch
    for chunk in range(b // QCHUNK, (e + QCHUNK - 1) // QCHUNK if e > b else 0):
        c0 = chunk * QCHUNK
        full = min(QCHUNK, origins_host.size - c0) if origins_host is not None else QCHUNK
        win, org = sample_query_chunk(text, chunk, full, m, device, seed)
        lo, hi = max(b, c0), min(e, c0 + full)
        q_host[lo * m:hi * m] = win[(lo - c0) * m:(hi - c0) * m].cpu().numpy()
        if origins_host is not None:
            origins_host[lo:hi] = org[lo - c0:hi - c0].cpu().numpy()
        del win, org
    torch.cuda.empty_cache()


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (NVML every 5 ms in a thread)."""
    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, gpu_index):
        self.samples = []  # (time, sm_mhz, reasons bitmask)
        self.gpu_index = gpu_index
        self.stop_flag = False
        self.thread = None
        self.sm_max = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.gpu_index]) if vis and vis.split(",")[0].isdigit() else self.gpu_index
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))

            def pump():
                while not self.stop_flag:
                    try:
                        mhz = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                        try:
                            reasons = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                        except Exception:
                            reasons = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                        self.samples.append((time.time(), float(mhz), int(reasons)))
                    except Exception:
                        pass
                    time.sleep(0.005)

            self.thread = threading.Thread(target=pump, daemon=True)
            self.thread.start()
        except Exception:
            self.thread = None

    def stop(self, t0, t1):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=1.0)
        sel = [(m, r) for t, m, r in self.samples if t0 <= t <= t1]
        reasons = sorted(name for name, bit in self.BAD.items() if any(r & bit for _, r in sel))
        return {"sm_mhz": statistics.median([m for m, _ in sel]) if sel else None, "sm_max_mhz": self.sm_max,
                "reasons": reasons, "samples": len(sel)}


def ncu_traffic_bytes(name):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch, from a committed ncu --set full summary."""
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    total = 0.0
    try:
        for line in open(os.path.join(ROOT, "profiles", name)):
            f = line.split()
            if len(f) >= 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                total += float(f[1]) * unit[f[2]]
    except Exception:
        return None
    return total or None


def split_host_cores(rank, world, local_rank):
    """Every rank of a multi-process run gets its own share of the host cores (the library sizes its staging
    thread pool from the CPUs the process may run on): the GPU's NUMA node when the box reports one, else a
    contiguous slice.  Returns (number of cores, numa node or None)."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        if world <= 1:
            return len(cores), None
        node = None
        try:
            import torch
            p = torch.cuda.get_device_properties(local_rank)
            bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
            node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        except Exception:
            node = None
        per = max(1, len(cores) // world)
        mine = cores[rank * per:(rank + 1) * per] or cores
        os.sched_setaffinity(0, mine)
        return len(mine), (node if node is not None and node >= 0 else None)
    except Exception:
        return os.cpu_count() or 1, None


def measured_peaks():
    peaks = {"hbm_gbs": 6650.0, "kind": "fallback (B200_PROFILING.md)"}
    try:
        peaks["hbm_gbs"] = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
        peaks["kind"] = "measured (MEASURED_PEAKS.json)"
    except Exception:
        pass
    try:  # random 32 B gather ceiling measured by gdx_measure_random_gather (profiles/r1_gather_ceiling.json)
        rows = json.load(open(os.path.join(ROOT, "profiles", "r1_gather_ceiling.json")))
        peaks["random_lines_per_s"] = max(float(r["gloads_per_s"]) for r in rows if r["record_bytes"] == 32) * 1e9
    except Exception:
        peaks["random_lines_per_s"] = None
    return peaks


def dump_pick(nq):
    """The batch positions --dump-outputs writes: every query up to DUMP_SAMPLE, else a fixed seeded sample (sorted)."""
    if nq <= DUMP_SAMPLE:
        return np.arange(nq)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(nq, DUMP_SAMPLE, replace=False))


def dump_outputs(dirname, arrays):
    """name -> DIR/name.npy as float64 (counts, batch and text positions are integers below 2^53: exact)."""
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), np.asarray(a).astype(np.float64))


def workload_name(args, world):
    return (f"C5: hg38-shaped synthetic {args.text_len / 1e9:.2f} Gbp DNA single text (ascii_dna_with_n, "
            f"{args.n_fraction:.0%} N in runs<=10kbp, u32, s={args.sampling_rate}, D={args.lookup_depth}), ONE batch of "
            f"{args.queries / 1e6:.1f} M len-{args.query_len} queries sampled from the text "
            f"({args.queries * args.query_len / 1e9:.2f} GB), range-sharded by the library over {world} replica(s)")


def download_parts(pidx):
    """BWT, count[], suffix-array samples and border map of a device-built index (host arrays)."""
    rows, pos = pidx.download_text_borders()
    return {"bwt": pidx.download_bwt(), "n": pidx.total_text_len(), "count": pidx.count_array(),
            "samples": pidx.download_samples(), "rows": rows, "pos": pos}


def oracle_from_parts(parts, args, lookup_depth, nthreads, with_locate=True):
    """CPU oracle index (the reference's three-array layout) over those parts."""
    from oracle import oracle as O
    return O.OracleIndex.from_parts(parts["bwt"], O.ALPHABETS["ascii_dna_with_n"](), parts["count"],
                                    np.array([parts["n"] - 1], dtype=np.uint64),
                                    parts["samples"] if with_locate else None, args.sampling_rate,
                                    parts["rows"] if with_locate else None, parts["pos"] if with_locate else None,
                                    lookup_depth=lookup_depth, storage="u32", nthreads=nthreads)


# ---- CPU reference arm -----------------------------------------------------------------------------
def run_reference(args, rank, world):
    if rank != 0:
        return
    import torch

    import genedex_b200 as gdx
    from oracle import oracle as O
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    m, nq = args.query_len, args.queries
    text = make_text_on_device(args.text_len, args.n_fraction, dev)
    # the reference arm times bounded samples: the first 4 M queries of the batch are all it ever touches
    n_have = min(nq, 2 * QCHUNK)
    q = np.empty(n_have * m, dtype=np.uint8)
    fill_query_range(text, q, None, 0, n_have, m, dev)
    text_host = text.cpu().numpy()
    del text
    torch.cuda.empty_cache()
    # The suffix array of 3.1 G symbols is out of reach of the oracle's own simple SACA, so the arm's BWT /
    # samples come from this repo's device construction (setup, untimed) -- and are then checked against the
    # text by the oracle alone (gdxo_verify_against_text: all n rows, BWT symbol + sample + border), so the
    # timed CPU search does not inherit an unnoticed construction bug of the product.
    cfg = (gdx.FmIndexConfig("u32").suffix_array_sampling_rate(args.sampling_rate)
           .lookup_table_depth(0).construct_on_device(True).dense_suffix_array(False).seed_table(False))
    pidx = cfg.construct_index_packed(text_host, np.array([0, text_host.size], dtype=np.uint64),
                                      gdx.alphabet.ascii_dna_with_n())
    cores = O.lib().gdxo_online_cores()
    parts = download_parts(pidx)
    oidx = oracle_from_parts(parts, args, 0, cores)
    del pidx
    torch.cuda.empty_cache()
    tab = np.frombuffer(bytes(O.ALPHABETS["ascii_dna_with_n"]().io_to_dense), dtype=np.uint8)
    dense = np.empty(text_host.size + 1, dtype=np.uint8)
    np.take(tab, text_host, out=dense[:-1])
    dense[-1] = 0
    del text_host
    t0 = time.perf_counter()
    violations, visited = oidx.verify_against_text(dense, nthreads=cores)
    t_verify = time.perf_counter() - t0
    assert violations == 0 and visited == dense.size, f"the CPU arm's index is not the index of the text ({violations})"
    del dense

    def timed(index, label):
        cal = min(n_have, 100_000)
        off = np.arange(cal + 1, dtype=np.uint64) * m
        t0 = time.perf_counter()
        index.count_many_packed(q[: cal * m], off, nthreads=cores)
        rate = cal / (time.perf_counter() - t0)
        # every step a bounded sample; the whole run stays within ~1.5 minutes per index
        per_step = int(min(n_have, max(64 * cores, rate * 90.0 / (args.steps + args.warmup))))
        off = np.arange(per_step + 1, dtype=np.uint64) * m
        times = []
        for it in range(args.warmup + args.steps):
            lo = (it * per_step) % max(1, n_have - per_step + 1)
            t0 = time.perf_counter()
            index.count_many_packed(q[lo * m:(lo + per_step) * m], off, nthreads=cores)
            if it >= args.warmup:
                times.append(time.perf_counter() - t0)
        ms = 1e3 * sum(times) / len(times)
        return per_step / (ms * 1e-3), ms, f"{per_step} of the {nq} queries per step, {cores} threads, contiguous chunk per thread, {label}"

    value, ms, sample = timed(oidx, "lookup depth 0 (crate default)")
    d13 = None
    del oidx
    try:  # the deepest table the crate itself suggests for genomes (config.rs:38-41)
        o13 = oracle_from_parts(parts, args, 13, cores, with_locate=False)
        v13, ms13, s13 = timed(o13, "lookup depth 13")
        d13 = {"value": v13, "unit": "queries/s", "ms_per_step": ms13, "sample": s13}
        del o13
    except Exception as e:  # noqa: BLE001
        d13 = {"unavailable": repr(e)[:200]}
    emit_json({
        "impl": "reference", "metric": "len-50 count queries/s on 3.1 Gbp DNA index", "value": value,
        "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": workload_name(args, args.gpus),
                   "index": "the reference's own three-array condensed Block64 layout, s=4, D=0 (4.65 GB); BWT + samples "
                            "from this repo's device construction (setup, untimed), verified against the text by the "
                            "oracle alone before timing",
                   "index_verified_against_text": {"violations": violations, "rows_visited": visited,
                                                   "seconds": round(t_verify, 1)}},
        "cpu_baseline": {"value": value, "unit": "queries/s", "cores": cores, "kind": "port", "sample": sample},
        "lookup_depth_13": d13,
        "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


# ---- this repo's arm ---------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    host_cores, numa_node = split_host_cores(rank, world, local_rank)  # before the library starts its pool
    import genedex_b200 as gdx
    from genedex_b200.replicate import ReplicaSet, broadcast_index, replicate_transport, shard_range, torch_share_id
    lib = gdx._lib.load()
    pool_threads = int(lib.gdx_host_pool_resize(0))  # the library's default for the CPUs this rank may use
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    m, nq = args.query_len, args.queries
    b, e = shard_range(nq, rank, world)
    snq = e - b
    PACKED = gdx._lib.GDX_QUERIES_PACKED_2BIT

    # a second, CPU-only group: ranks that merely wait (while rank 0 drives every GPU by itself, or builds the
    # oracle) must not sit in an NCCL kernel that spins on their GPU
    cpu_group = dist.new_group(backend="gloo") if world > 1 else None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def cpu_barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(group=cpu_group)

    def reduce(x, op="max"):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
        return float(t.item())

    # ---- data: the whole batch is ONE array; a rank fills (and reads) only the range it owns ------------
    t_setup = time.perf_counter()
    text = make_text_on_device(args.text_len, args.n_fraction, dev)
    q_all = torch.empty(nq * m, dtype=torch.uint8).pin_memory().numpy()   # pinned host memory (the contract's e2e)
    origins = np.zeros(nq, dtype=np.int64)
    need_all = rank == 0 and world > 1 and not args.no_extras   # rank 0 also drives the single-process arm
    fill_query_range(text, q_all, origins, 0 if need_all else b, nq if need_all else e, m, dev)
    multi_q = None
    if not args.no_locate and rank == 0:
        multi_q = np.empty(args.multi_hit_queries * args.multi_hit_len, dtype=np.uint8)
        fill_query_range(text, multi_q, None, 0, args.multi_hit_queries, args.multi_hit_len, dev, seed=QUERY_SEED + 7)
    text_host = text.cpu().numpy() if rank == 0 else None
    del text
    torch.cuda.empty_cache()
    t_data = time.perf_counter() - t_setup

    # ---- index: built on rank 0 (device construction), replicas by the library's own ncclBroadcast -------
    t0 = time.perf_counter()
    alphabet = gdx.alphabet.ascii_dna_with_n()
    pidx = None
    if rank == 0:
        cfg = (gdx.FmIndexConfig("u32").suffix_array_sampling_rate(args.sampling_rate)
               .lookup_table_depth(args.lookup_depth).device(local_rank).construct_on_device(True, verify=True))
        pidx = cfg.construct_index_packed(text_host, np.array([0, text_host.size], dtype=np.uint64), alphabet)
        del text_host
    t_build = time.perf_counter() - t0
    t_bcast, transport = 0.0, None
    if world > 1:
        t0 = time.perf_counter()
        pidx = broadcast_index(pidx, alphabet, rank, world, local_rank, torch_share_id(rank))
        transport = replicate_transport()
        barrier()
        t_bcast = time.perf_counter() - t0
    info = pidx.info()
    rs = ReplicaSet([pidx], first_shard=rank, n_shards=world)
    steps, warm = args.steps, max(args.warmup, 3)

    # ---- value: the shard's IO bytes resident in HBM, one k_search launch per step ---------------------
    stream = torch.cuda.current_stream().cuda_stream
    d_q = torch.from_numpy(q_all[b * m:e * m]).to(dev)
    d_counts = torch.zeros(max(snq, 1), dtype=torch.int64, device=dev)
    d_err = torch.full((1,), -1, dtype=torch.int64, device=dev)

    def device_steps(d_queries, count, fixed_len, n_steps, encoding=0):
        qs = gdx._lib.gdx_queries(d_queries.data_ptr(), None, fixed_len, count, encoding, 0)

        def one():
            rc = lib.gdx_count_many_device(pidx.handle, C.byref(qs), d_counts.data_ptr(), d_err.data_ptr(), stream)
            assert rc == 0, lib.gdx_last_error_message()
        for _ in range(warm):
            one()
        barrier()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_steps + 1)]
        torch.cuda.nvtx.range_push("timed")  # ncu --nvtx --nvtx-include "timed/" lists exactly the timed launches
        evs[0].record()
        for i in range(n_steps):
            one()
            evs[i + 1].record()
        barrier()
        torch.cuda.nvtx.range_pop()
        per = [evs[i].elapsed_time(evs[i + 1]) for i in range(n_steps)]
        assert int(d_err.item()) == -1
        return reduce(evs[0].elapsed_time(evs[-1]) / n_steps), per

    clocks = ClockSampler(local_rank)
    clocks.start()
    t_region0 = time.time()
    kernel_ms, step_ms = device_steps(d_q, snq, m, steps)
    counts_device_path = d_counts[:snq].cpu().numpy().astype(np.uint64)

    # ---- e2e: the whole batch through gdx_count_many_sharded, pinned host buffers in and out ----------------
    counts_all = torch.zeros(nq, dtype=torch.int64).pin_memory().numpy().view(np.uint64)

    def host_steps(fn, n_steps, n_warm=warm):
        for _ in range(n_warm):
            fn()
        barrier()
        torch.cuda.nvtx.range_push("timed")
        t0 = time.perf_counter()
        for _ in range(n_steps):
            fn()  # synchronous: returns with the results on the host
        local = (time.perf_counter() - t0) * 1e3 / n_steps
        torch.cuda.nvtx.range_pop()
        barrier()
        return reduce((time.perf_counter() - t0) * 1e3 / n_steps), local

    e2e_ms, e2e_local = host_steps(lambda: rs.count_many_packed(q_all, None, m, nq, out=counts_all), steps)
    st = rs.stats()
    t_region1 = time.time()
    clock_info = clocks.stop(t_region0, t_region1)
    assert np.array_equal(counts_all[b:e], counts_device_path), "device-resident and host-buffer paths disagree"
    assert snq == 0 or int(counts_all[b:e].min()) >= 1, "a query sampled from the text must occur at least once"
    e2e_by_rank = [(e2e_local, numa_node, host_cores)]
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, e2e_by_rank[0])
        e2e_by_rank = gathered
    h2d = reduce(float(st.h2d_bytes), "sum")
    d2h = reduce(float(st.d2h_bytes), "sum")
    e2e = {"value": nq / (e2e_ms * 1e-3), "unit": "queries/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
           "ms_per_step": e2e_ms, "kernel_ms_inside": st.kernel_ms_search,
           "host_buffers": "pinned IO bytes in, pinned uint64 counts out; inside the call the library's host thread pool "
                           "packs chunks to 2 bits while the PCIe link is busy and sends chunks as they are when it is idle",
           "packed_queries_per_step": int(reduce(float(st.packed_queries), "sum")),
           "host_cores_per_rank": host_cores, "host_pool_threads_per_rank": pool_threads,
           "ms_per_step_by_rank_numa_cores": e2e_by_rank, "gpu_launches_per_step": int(reduce(float(st.kernel_launches), "sum"))}

    extras = not args.no_extras
    # ---- e2e from ordinary (pageable) memory in and out: every byte is packed by the host pool ----------------
    if extras and snq:
        q_page = q_all[b * m:e * m].copy()
        c_page = np.zeros(snq, dtype=np.uint64)
        pg_ms, _ = host_steps(lambda: pidx.count_many_packed(q_page, None, m, snq, out=c_page), max(3, steps // 2), 2)
        gst = pidx.stats()
        assert np.array_equal(c_page, counts_all[b:e])
        e2e["pageable"] = {"value": nq / (pg_ms * 1e-3), "unit": "queries/s", "ms_per_step": pg_ms,
                           "h2d_bytes_per_step": int(reduce(float(gst.h2d_bytes), "sum")),
                           "d2h_bytes_per_step": int(reduce(float(gst.d2h_bytes), "sum")),
                           "packed_queries_per_step": int(reduce(float(gst.packed_queries), "sum")),
                           "host_buffers": "ordinary numpy arrays in and out (a Rust Vec): all bytes packed by the host pool, "
                                           "uint32 counts widened into the caller's array"}
        del q_page, c_page
    # ---- e2e from pre-packed pinned reads (callers that keep their reads 2-bit packed) --------------------
    if extras and (b * m) % 4 == 0 and snq:
        packed_all = torch.empty((nq * m + 3) // 4 + 16, dtype=torch.uint8).pin_memory().numpy()
        sub, first_bad = pidx.pack_queries_2bit(q_all[b * m:e * m], None, m, snq, out=packed_all[b * m // 4:])
        assert first_bad is None
        c32 = torch.empty(nq, dtype=torch.int32).pin_memory().numpy().view(np.uint32)

        def prepacked():
            # the u32 single-replica entry point on the shard's sub-batch (the sharded call widens to u64)
            pidx.count_many_packed(packed_all[b * m // 4:], None, m, snq, out=c32[b:e], encoding=PACKED)
        pp_ms, _ = host_steps(prepacked, steps)
        pst = pidx.stats()
        assert np.array_equal(c32[b:e].astype(np.uint64), counts_all[b:e])
        e2e["prepacked"] = {"value": nq / (pp_ms * 1e-3), "unit": "queries/s", "ms_per_step": pp_ms,
                            "h2d_bytes_per_step": int(reduce(float(pst.h2d_bytes), "sum")),
                            "d2h_bytes_per_step": int(reduce(float(pst.d2h_bytes), "sum")),
                            "host_buffers": "pinned, 2-bit packed by the caller (gdx_pack_queries, untimed), uint32 counts"}
        del packed_all

    # ---- locate: the batch through gdx_locate_many_sharded ------------------------------------------------
    locate = None
    peaks = measured_peaks()
    R = int(info.rank_record_bytes)
    locate_sample, locate_first = None, None
    if not args.no_locate:
        hit_off = torch.zeros(nq + 1, dtype=torch.int64).pin_memory().numpy().view(np.uint64)
        state = {}

        def loc():
            if "release" in state:
                state["release"]()
            state["off"], state["views"], state["first"], state["release"] = rs.locate_many_view(q_all, None, m, nq, hit_offsets=hit_off)
        reps = max(1, min(steps, 5))
        loc_ms, _ = host_steps(loc, reps, 2)
        lst = rs.stats()
        hits = state["views"][0]
        width = (hit_off[b + 1:e + 1] - hit_off[b:e]).astype(np.uint64)
        assert np.array_equal(width, counts_all[b:e]), "locate: hits per query differ from the counts"
        first = hits[(hit_off[b:e] - np.uint64(state["first"][0])).astype(np.int64), 1].astype(np.int64)
        single = width == 1
        assert np.array_equal(first[single], origins[b:e][single]), "locate: a unique hit is not at its origin"
        if args.dump_outputs:  # this shard's part of the sample (every query has a hit: counts >= 1 above)
            pick = dump_pick(nq)
            locate_first = first[pick[(pick >= b) & (pick < e)] - b]
        ns_ = min(snq, 20_000)  # this shard's sample for the oracle comparison on rank 0
        o0 = int(hit_off[b])
        locate_sample = (hit_off[b:b + ns_ + 1] - np.uint64(o0), hits[: int(hit_off[b + ns_]) - o0].copy())
        hits_head = hits[:1000].copy()
        state["release"]()
        # the compact result form: u32 hits per query + (u32 text id, u32 position) hits
        cnt32 = torch.zeros(nq, dtype=torch.int32).pin_memory().numpy().view(np.uint32)
        cstate = {}

        def loc_compact():
            if "release" in cstate:
                cstate["release"]()
            _, cstate["views"], cstate["release"] = rs.locate_many_compact_view(q_all, None, m, nq, hit_counts=cnt32)
        locc_ms, _ = host_steps(loc_compact, reps, 2)
        cst = rs.stats()
        assert np.array_equal(cnt32[b:e].astype(np.uint64), counts_all[b:e])
        assert np.array_equal(cstate["views"][0][:1000].astype(np.uint64), hits_head)
        cstate["release"]()
        compact = {"value": nq / (locc_ms * 1e-3), "unit": "queries/s (e2e, host buffers)", "ms_per_step": locc_ms,
                   "d2h_bytes_per_step": int(reduce(float(cst.d2h_bytes), "sum")),
                   "results": "gdx_locate_many_sharded_compact: u32 hits per query + gdx_hit32 hits (8 B)"}
        del cnt32
        locate = {"value": nq / (loc_ms * 1e-3), "unit": "queries/s (e2e, host buffers)", "ms_per_step": loc_ms, "compact": compact,
                  "hits_per_step": int(reduce(float(lst.hits), "sum")),
                  "locate_walk_steps": int(reduce(float(lst.locate_walk_steps), "sum")),
                  "kernel_ms_locate": reduce(lst.kernel_ms_locate), "kernel_ms_search": reduce(lst.kernel_ms_search),
                  "d2h_bytes_per_step": int(reduce(float(lst.d2h_bytes), "sum"))}
        del hit_off

    # ---- locate with many hits per query (rank 0, one GPU): the locate kernels' own roofline ----------------
    if locate is not None and rank == 0 and extras:
        mq, mm = args.multi_hit_queries, args.multi_hit_len
        multi = {}
        for label, dense in (("dense_suffix_array", True), ("sampled_suffix_array_s%d" % args.sampling_rate, False)):
            if not dense:
                pidx.set_dense_suffix_array(False)
            elif not int(pidx.info().dense_suffix_array_bytes):
                continue
            moff = np.zeros(mq + 1, dtype=np.uint64)
            best = None
            for it in range(4):
                t0 = time.perf_counter()
                _, mh, rel = pidx.locate_many_view(multi_q, None, mm, mq, hit_offsets=moff)
                dt = (time.perf_counter() - t0) * 1e3
                s = pidx.stats()
                rel()
                if it and (best is None or s.kernel_ms_locate < best[1].kernel_ms_locate):
                    best = (dt, s)
            dt, s = best
            alg = int(s.hits) * (32 + 16 + 8) + R * int(s.locate_walk_steps)
            ach = alg / (s.kernel_ms_locate * 1e-3) / 1e9
            multi[label] = {"queries": mq, "query_len": mm, "hits": int(s.hits), "hits_per_query": int(s.hits) / mq,
                            "e2e_ms": dt, "hits_per_s_e2e": int(s.hits) / (dt * 1e-3),
                            "kernel_ms_locate": s.kernel_ms_locate, "kernel_ms_search": s.kernel_ms_search,
                            "hits_per_s_kernel": int(s.hits) / (s.kernel_ms_locate * 1e-3),
                            "locate_walk_steps": int(s.locate_walk_steps),
                            "roofline": {"bound": "hbm", "kernel": "k_expand_rows + k_locate_walk<K32>",
                                         "algorithmic_bytes": alg, "achieved": ach, "peak": peaks["hbm_gbs"],
                                         "unit": "GB/s", "frac": ach / peaks["hbm_gbs"],
                                         "bytes_per_hit": "8 row + 32 SA sector + 16 hit + R per walk step"}}
        pidx.set_dense_suffix_array(True)
        locate["multi_hit"] = multi

    # ---- the index exactly as BASELINE names it: no seed table, no dense suffix array, every LF step --------
    no_accel = None
    if extras:
        seed_depth0 = int(info.seed_table_depth)
        row_ctx0 = int(info.row_context_entry_bytes) != 0
        pidx.set_text_verification(False)
        pidx.set_row_context_table(False)
        pidx.set_dense_suffix_array(False)
        pidx.set_seed_table_depth(0)
        n3 = max(3, steps // 3)
        na_kernel_ms, _ = device_steps(d_q, snq, m, n3)
        assert np.array_equal(d_counts[:snq].cpu().numpy().astype(np.uint64), counts_device_path)
        na_ms, _ = host_steps(lambda: rs.count_many_packed(q_all, None, m, nq, out=counts_all), n3, 1)
        nst = rs.stats()
        na_steps = reduce(float(nst.lf_steps), "sum")
        alg = nq * (m + 16) + 2 * R * na_steps
        no_accel = {"index": "s=%d, D=%d as configured: %.2f GB of reference structures; no seed table, no dense suffix "
                             "array, no text verification (every LF step of batch_computed_cursors.rs:62-70 runs)"
                             % (args.sampling_rate, args.lookup_depth, (int(info.rank_bytes) + int(info.sample_bytes)) / 1e9),
                    "value": nq / (na_kernel_ms * 1e-3), "ms_per_step": na_kernel_ms, "lf_steps_per_step": int(na_steps),
                    "e2e": {"value": nq / (na_ms * 1e-3), "ms_per_step": na_ms},
                    "roofline": {"bound": "hbm", "kernel": "k_query_keys + radix sort + k_search<K32>",
                                 "algorithmic_bytes": alg, "achieved": alg / (na_kernel_ms * 1e-3) / 1e9 / world,
                                 "peak": peaks["hbm_gbs"], "unit": "GB/s per GPU",
                                 "frac": alg / (na_kernel_ms * 1e-3) / 1e9 / world / peaks["hbm_gbs"],
                                 "rank_queries_per_s": 2 * na_steps / (na_kernel_ms * 1e-3)}}
        assert np.array_equal(counts_all[b:e], counts_device_path)
        pidx.set_text_verification(True)
        pidx.set_dense_suffix_array(True)
        if seed_depth0:
            pidx.set_seed_table_depth(seed_depth0)
        if row_ctx0:
            pidx.set_row_context_table(True)
    del d_q

    # ---- every shard's results to rank 0 -----------------------------------------------------------------
    loc_samples = [locate_sample]
    if world > 1:
        pad = max(shard_range(nq, r, world)[1] - shard_range(nq, r, world)[0] for r in range(world))
        mine = torch.zeros(pad, dtype=torch.int64, device=dev)
        mine[:snq] = torch.from_numpy(counts_all[b:e].astype(np.int64)).to(dev)
        parts = [torch.zeros(pad, dtype=torch.int64, device=dev) for _ in range(world)] if rank == 0 else None
        dist.gather(mine, parts, dst=0)
        if rank == 0:
            for r in range(1, world):
                rb, re_ = shard_range(nq, r, world)
                counts_all[rb:re_] = parts[r][: re_ - rb].cpu().numpy().astype(np.uint64)
        del mine, parts
        loc_samples = [None] * world
        dist.all_gather_object(loc_samples, locate_sample)
        if locate_first is not None:  # shards in rank order = the sorted sample in order
            firsts = [None] * world
            dist.all_gather_object(firsts, locate_first)
            locate_first = np.concatenate(firsts)

    # ---- single process, all GPUs: ONE gdx_count_many_sharded call from rank 0 (the other ranks idle) -------
    single = None
    if world > 1 and extras:
        cpu_barrier()
        if rank == 0:
            t0 = time.perf_counter()
            all_rs = ReplicaSet.replicate(pidx, [d for d in range(world) if d != local_rank])
            t_rep = time.perf_counter() - t0
            # this process now stages for every GPU: give it (and a re-created staging pool) all host cores
            os.sched_setaffinity(0, range(os.cpu_count() or 1))
            pool_threads = int(lib.gdx_host_pool_resize(0))
            out = np.zeros(nq, dtype=np.uint64)
            for _ in range(2):
                all_rs.count_many_packed(q_all, None, m, nq, out=out)
            t0 = time.perf_counter()
            reps = max(2, steps // 2)
            for _ in range(reps):
                all_rs.count_many_packed(q_all, None, m, nq, out=out)
            sp_ms = (time.perf_counter() - t0) * 1e3 / reps
            sst = all_rs.stats()
            assert np.array_equal(out, counts_all), "single-process sharded call disagrees with the per-rank shards"
            single = {"value": nq / (sp_ms * 1e-3), "unit": "queries/s", "ms_per_step": sp_ms, "shards": int(sst.shards),
                      "replicate_s": round(t_rep, 2), "transport": replicate_transport(),
                      "host_pool_threads": pool_threads,
                      "note": "one host process, one thread + staging arena per GPU, one shared staging pool; the other "
                              "ranks sit in a barrier meanwhile"}
            del all_rs
        cpu_barrier()

    # ---- oracle: parity on a sample of EVERY shard (+ CPU baseline at N = 1) -------------------------------
    cpu, parity = None, None
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import oracle as O
        cores = O.lib().gdxo_online_cores()
        try:
            os.sched_setaffinity(0, range(os.cpu_count() or 1))
        except Exception:
            pass
        oidx = oracle_from_parts(download_parts(pidx), args, args.lookup_depth, cores)
        checked, loc_checked = 0, 0
        for r in range(world):
            rb, re_ = shard_range(nq, r, world)
            have = (rb, re_) if (need_all or r == 0) else None
            for lo in ([rb, (rb + re_) // 2, max(rb, re_ - 20_000)] if have else []):
                cnt = min(20_000, re_ - lo)
                if cnt <= 0:
                    continue
                off = np.arange(cnt + 1, dtype=np.uint64) * m
                want = oidx.count_many_packed(q_all[lo * m:(lo + cnt) * m], off, nthreads=cores)
                assert np.array_equal(want, counts_all[lo:lo + cnt]), f"shard {r}: GPU counts differ from the oracle"
                checked += cnt
            if loc_samples[r] is not None and have:
                soff, shits = loc_samples[r]
                cnt = soff.size - 1
                off = np.arange(cnt + 1, dtype=np.uint64) * m
                ooff, ohits = oidx.locate_many_packed(q_all[rb * m:(rb + cnt) * m], off, nthreads=cores)
                assert np.array_equal(ooff, soff) and np.array_equal(ohits, shits), f"shard {r}: hits differ from the oracle"
                loc_checked += cnt
        parity = {"count_queries_checked": checked, "locate_queries_checked": loc_checked, "shards_checked": world if need_all or world == 1 else 1,
                  "equal": True}
        if world == 1:
            cal = min(nq, 100_000)
            off = np.arange(cal + 1, dtype=np.uint64) * m
            t0 = time.perf_counter()
            oidx.count_many_packed(q_all[: cal * m], off, nthreads=cores)
            rate = cal / (time.perf_counter() - t0)
            sample_n = int(min(nq, max(cal, rate * args.cpu_seconds)))
            off = np.arange(sample_n + 1, dtype=np.uint64) * m
            best = None
            for _ in range(2):
                t0 = time.perf_counter()
                ocounts = oidx.count_many_packed(q_all[: sample_n * m], off, nthreads=cores)
                dt = time.perf_counter() - t0
                best = dt if best is None else min(best, dt)
            assert np.array_equal(ocounts, counts_all[:sample_n]), "GPU counts differ from the CPU oracle on the baseline sample"
            cpu = {"value": sample_n / best, "unit": "queries/s", "cores": cores, "kind": "port",
                   "sample": f"first {sample_n} of the {nq} queries, best of 2, contiguous chunk per thread",
                   "gpu_counts_equal_oracle_on_sample": True}
        del oidx

    cpu_barrier()  # everyone leaves together (rank 0 was busy with the oracle meanwhile)
    if rank != 0:
        return
    if args.dump_outputs:
        # N > 1: the other shards' counts as gathered above (every rank checked its range of counts_all against its
        # device-path counts)
        pick = dump_pick(nq)
        dumped = {"count": (counts_device_path if world == 1 else counts_all)[pick], "count_query": pick}
        if locate_first is not None:
            dumped["locate_first_position"] = locate_first
        dump_outputs(args.dump_outputs, dumped)
    out = assemble(args, world, info, st, kernel_ms, step_ms, e2e, locate, no_accel, single, cpu, parity, peaks, clock_info,
                   {"data": round(t_data, 2), "index_build": round(t_build, 2), "replicate": round(t_bcast, 2),
                    "replicate_transport": transport}, steps, warm)
    emit_json(out)


def assemble(args, world, info, st, kernel_ms, step_ms, e2e, locate, no_accel, single, cpu, parity, peaks, clock_info, setup_s,
             steps, warm):
    m, nq = args.query_len, args.queries
    R = int(info.rank_record_bytes)
    seed_depth = int(info.seed_table_depth)
    table_depth = max(args.lookup_depth, seed_depth if m >= seed_depth else 0)
    # per-shard statistics of rank 0's last e2e call scaled to the batch (shards are statistically identical)
    scale = nq / max(1, int(st.queries))
    lf_steps = int(st.lf_steps) * scale
    walk = int(st.walk_steps) * scale
    verified = int(st.verified_queries) * scale
    alg_bytes = nq * (m + 16 + (8 if table_depth > 0 else 0)) + 2 * R * lf_steps + R * walk + 64 * verified
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9 / world  # per GPU
    value = nq / (kernel_ms * 1e-3)
    traffic_file = "r2_k_search.txt"
    traffic = ncu_traffic_bytes(traffic_file)  # one launch over a 60 M-query shard (N = 1)
    # (the committed capture is of the default workload with all three accelerators in place)
    default_shape = (args.text_len == 3_100_000_000 and nq == 60_000_000 and m == 50 and args.lookup_depth == 0 and
                     int(info.row_context_entry_bytes) != 0 and seed_depth == 16)
    if traffic and default_shape:
        traffic = traffic / world  # DRAM bytes per launch scale with the queries of the launch
    else:
        traffic = None
    return {
        "metric": "len-50 count queries/s on 3.1 Gbp DNA index (locate: see `locate`)",
        "value": value, "unit": "queries/s", "n_gpus": world, "steps": steps, "warmup": warm,
        "ms_per_step": kernel_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic",
        "config": {"workload": workload_name(args, world), "queries_per_gpu": nq // world,
                   "index": ("replica = the configured index (s=%d, D=%d: rank records %.2f GB + samples %.2f GB) + packed text "
                             "%.2f GB + sampled inverse SA %.2f GB + accelerators derived per replica: dense suffix array %.2f GB, "
                             "seed table depth %d %.2f GB, row context table %.2f GB" % (
                                 args.sampling_rate, args.lookup_depth, int(info.rank_bytes) / 1e9, int(info.sample_bytes) / 1e9,
                                 int(info.text_bytes) / 1e9, int(info.inverse_sample_bytes) / 1e9,
                                 int(info.dense_suffix_array_bytes) / 1e9, seed_depth, int(info.seed_table_bytes) / 1e9,
                                 int(info.row_context_entry_bytes) * int(info.text_len) / 1e9)),
                   "l2": "inputs larger than L2: %.2f GB rank records + %.1f GB seed table + %s accessed at random, %.2f GB of "
                         "queries per GPU" % (
                             int(info.rank_bytes) / 1e9, int(info.seed_table_bytes) / 1e9,
                             ("%.1f GB row context table" % (int(info.row_context_entry_bytes) * int(info.text_len) / 1e9)
                              if int(info.row_context_entry_bytes) else
                              "%.1f GB suffix array + %.2f GB text" % (int(info.dense_suffix_array_bytes) / 1e9, int(info.text_bytes) / 1e9)),
                             nq // world * m / 1e9),
                   "index_image_bytes": int(info.image_bytes), "dense_suffix_array_bytes": int(info.dense_suffix_array_bytes),
                   "seed_table_depth": seed_depth, "seed_table_bytes": int(info.seed_table_bytes),
                   "row_context_table_bytes": int(info.row_context_entry_bytes) * int(info.text_len), "rank_record_bytes": R,
                   "lf_steps_per_step": int(lf_steps), "verified_queries_per_step": int(verified),
                   "verify_walk_steps_per_step": int(walk),
                   "step_ms_min_median_max_rank0": [round(min(step_ms), 3), round(statistics.median(step_ms), 3), round(max(step_ms), 3)],
                   "launches_per_step": "one k_search<K32, VERIFY> per GPU (a lookup level of depth %d replaces the shared steps: no sort)" % table_depth,
                   "setup_s": setup_s},
        "clocks": clock_info,
        "e2e": e2e,
        "gpu_launches": steps * world,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                     "traffic": traffic, "traffic_source": "profiles/%s (ncu --set full of this command at N=1), scaled to the launch's queries" % traffic_file if traffic else None,
                     "peak_kind": peaks["kind"], "kernel": "k_search<K32, VERIFY> (IO-byte queries)",
                     "algorithmic_bytes_per_launch": alg_bytes / world, "per_gpu": True,
                     "dram_achieved_gbs": (traffic / (kernel_ms * 1e-3) / 1e9) if traffic else None,
                     "dram_frac": (traffic / (kernel_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]) if traffic else None,
                     "random_access": ({"dram_lines_per_s": traffic / 128 / (kernel_ms * 1e-3),
                                        "measured_random_line_ceiling_per_s": peaks.get("random_lines_per_s"),
                                        "frac_of_ceiling": (traffic / 128 / (kernel_ms * 1e-3) / peaks["random_lines_per_s"])
                                        if peaks.get("random_lines_per_s") else None} if traffic else None),
                     "queries_per_s_at_survey_ceiling_per_gpu": peaks["hbm_gbs"] * 1e9 / 3266.0,
                     "rank_queries_per_s": 2 * lf_steps / (kernel_ms * 1e-3)},
        "cpu_baseline": cpu,
        "oracle_parity": parity,
        "locate": locate,
        "no_accelerators": no_accel,
        "single_process": single,
    }


_JSON_FD = None


def emit_json(obj):
    """The ONE line of the contract goes to the real stdout; everything else written to fd 1 by libraries
    (NCCL prints its version banner there) was redirected to stderr in main()."""
    line = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, line)


def main():
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
