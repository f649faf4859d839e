#!/usr/bin/env python
"""bench.py — QPS & effective index GB/s of the 4b x 1b BBQ score+top-k path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c3|c3q1|c4|c5] [--impl reference]
                  [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch of synthetic queries: validate + quantise the query batch (K4),
scan + score + top-k over this rank's row shard (K1/K2/K3), and for N > 1 ONE ncclAllGather of the per-shard top-k
lists (64-bit keys, issued inside libbbq_b200.so) + the deterministic merge.  The corpus (BASELINE configs[3] by
default: 100M x 1024, COSINE, k=10, batch of 4096 queries; at N=1 the whole 100M-row index lives on one GPU) is FIXED
and sharded row-wise over the N GPUs => "scaling": "strong".  `--workload c3` / `c2` / `c5` measure the other configs.

value      device-timed whole-job QPS (CUDA events on the launch stream), index resident in HBM, queries on device
e2e        the same through the entry a host binds — bbq_search / bbq_search_sharded with HOST buffers: H2D of the
           queries, search, exchange, D2H of the results all inside the blocking call, timed around it
roofline   the dominant kernel (the scan) against MEASURED_PEAKS.json, plus the tcgen05 int8 rate measured in this run
           by tools/probe/mma_issue_probe
cpu_baseline   the CPU oracle (restatement of the reference's TypeScript path; "port") on a bounded sample,
               same index bytes, 1 thread (the reference is single-threaded Node)
parity     the lists the TIMED configuration returned, checked against the oracle (re-score of the returned rows,
           and no row of a 1M-row sample may beat the k-th returned row)
secondary  (N=1, default run only) the other BASELINE configs, each measured the same way in a few seconds
--dump-outputs DIR   the top-k lists the timed path returned in its last step, as .npy files (inputs are seeded, so
                     two builds run with the same arguments can be compared list for list; bench_outputs/ is ignored by git)
--impl reference   times the CPU path as the main line (the TypeScript reference itself cannot run here:
                   no node / tsc / cargo in the image; see DESIGN.md)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[1..4]
    "c2": dict(n=100_000, dim=768, sim="MAXIMUM_INNER_PRODUCT", k=100, nq=1, qb=4, ib=1,
               name="100k x 768 MAXIMUM_INNER_PRODUCT k=100 single query (BASELINE configs[1])"),
    "c3": dict(n=1_000_000, dim=1024, sim="EUCLIDEAN", k=10, nq=1024, qb=4, ib=1,
               name="1M x 1024 EUCLIDEAN k=10 batch of 1024 queries (BASELINE configs[2])"),
    "c3q1": dict(n=1_000_000, dim=1024, sim="EUCLIDEAN", k=10, nq=1, qb=4, ib=1,
                 name="1M x 1024 EUCLIDEAN k=10 single query (the HBM-bound regime of BASELINE configs[2])"),
    "c4": dict(n=100_000_000, dim=1024, sim="COSINE", k=10, nq=4096, qb=4, ib=1,
               name="100M x 1024 COSINE k=10 batch of 4096 queries, row-sharded (BASELINE configs[3])"),
    "c5": dict(n=10_000_000, dim=1536, sim="COSINE", k=100, nq=1024, qb=8, ib=2, cpu_rows=200_000,
               name="10M x 1536 COSINE k=100 batch of 1024 queries, queryBits=8/indexBits=2 (BASELINE configs[4]; "
                    "EXTENSION: the reference, executed, throws for this config — tests/golden/from_ts/index_bits_2.behaviour.json; "
                    "the index build equals the reference's, the search semantics are this repository's)"),
}
CHUNK = 65536            # corpus generation granularity: chunk c is seeded by (SEED + c) whatever N is
SEED_CORPUS, SEED_QUERY = 20260101, 20260201
METRIC, UNIT = "QPS (4b x 1b BBQ score+top-k)", "queries/s"


# --corpus clustered: a Gaussian mixture (the recall harness's corpus, tools/recall_harness.py --clusters): every row and
# every query is a centre plus noise, so the rankings the parity checks compare are about real neighbours (cluster-mates),
# not about the noise floor of an i.i.d. Gaussian corpus.  The analytic centroid is still 0 (explicit zero centroid).
CORPUS = "gaussian"
N_CENTRES, CLUSTER_NOISE, SEED_CENTRES = 1000, 0.5, 20260301
_centres_cache = {}


def centres_host(dim):
    if dim not in _centres_cache:
        _centres_cache[dim] = np.random.default_rng(SEED_CENTRES).standard_normal((N_CENTRES, dim), dtype=np.float32)
    return _centres_cache[dim]


def gen_chunk_host(c, dim, rows):
    x = np.random.default_rng(SEED_CORPUS + c).standard_normal((rows, dim), dtype=np.float32)
    if CORPUS == "clustered":
        pick = np.random.default_rng(SEED_CORPUS + c + (1 << 20)).integers(0, N_CENTRES, rows)
        x = centres_host(dim)[pick] + np.float32(CLUSTER_NOISE) * x
    return x


def gen_chunk_device(torch, c, dim, rows, device="cuda"):
    """The device-side twin of gen_chunk_host (its own random stream: the two are different corpora of one family)."""
    g = torch.Generator(device=device)
    g.manual_seed(SEED_CORPUS + c)
    x = torch.randn((rows, dim), generator=g, device=device, dtype=torch.float32)
    if CORPUS == "clustered":
        key = ("t", dim, str(device))
        if key not in _centres_cache:
            _centres_cache[key] = torch.from_numpy(centres_host(dim)).to(device)
        pick = torch.randint(0, N_CENTRES, (rows,), generator=g, device=device)
        x = _centres_cache[key][pick] + CLUSTER_NOISE * x
    return x


def gen_queries(nq, dim):
    q = np.random.default_rng(SEED_QUERY).standard_normal((nq, dim), dtype=np.float32)
    if CORPUS == "clustered":
        pick = np.random.default_rng(SEED_QUERY + 1).integers(0, N_CENTRES, nq)
        q = centres_host(dim)[pick] + np.float32(CLUSTER_NOISE) * q
    return q


def load_peaks():
    """-> dict(hbm GB/s, bf16 burst TFLOP/s, bf16 sustained TFLOP/s, source)"""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm": float(d["hbm_gbs"]), "bf16": float(d["bf16_tflops"]),
                "bf16_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                "src": "measured (MEASURED_PEAKS.json)"}
    return {"hbm": 6650.0, "bf16": 1590.0, "bf16_sustained": 1400.0, "src": "fallback (B200_PROFILING.md)"}


def probe_int8_peak():
    """tools/probe/mma_issue_probe peak: cycles per tcgen05.mma.kind::i8 (M128 N208 K32, A in tensor memory) on an idle
    SM, measured on THIS GPU in THIS run (a few microseconds of GPU time, before the timed region)."""
    exe = os.path.join(ROOT, "tools", "probe", "mma_issue_probe")
    try:
        out = subprocess.run([exe, "peak"], capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[-1]
        return json.loads(out)
    except Exception as e:  # the probe is evidence, not the product: report its absence, do not fail the bench
        return {"error": f"{type(e).__name__}: {e}"}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.lines, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True).start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm_sorted = sorted(sm)
        return {"sm_mhz": (sm_sorted[len(sm_sorted) // 2] if sm else None), "sm_max_mhz": (max(mx) if mx else None),
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------------------
# CPU leg: the oracle on host cores (bench.py's cpu_baseline and --impl reference are the only legs that may run it)
# ---------------------------------------------------------------------------------------------------------------
def oracle_index_from_arrays(packed, corr, centroid, dim, sim, index_bits=1):
    from oracle import oracle as O
    return O.OracleIndex(np.ascontiguousarray(centroid, np.float32), np.ascontiguousarray(packed),
                         None, np.ascontiguousarray(corr), dim, sim, index_bits)


def oracle_search(q, oidx, k, qb, mode):
    from oracle import oracle as O
    return O.search_nearest_neighbors(q, oidx, k, query_bits=qb, mode=mode)


def cpu_time_queries(oidx, queries, k, qb, budget_s, max_q):
    """Runs the oracle's searchNearestNeighbors (reference heap selection) query by query, 1 thread."""
    done, t0, res = 0, time.perf_counter(), []
    for q in queries[:max_q]:
        res.append(oracle_search(q, oidx, k, qb, "heap"))
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    return done, time.perf_counter() - t0, res


def build_oracle_index_threaded(w, n_rows):
    """Index build for the reference arm (untimed): the oracle's quantizeVectors over row chunks on all host
    threads (ctypes releases the GIL); explicit zero centroid as in the GPU arm."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle as O
    dim, sim = w["dim"], w["sim"]
    cen = np.zeros(dim, np.float32)
    nchunks = -(-n_rows // CHUNK)

    def one(c):
        rows = min(CHUNK, n_rows - c * CHUNK)
        ix = O.quantize_vectors(gen_chunk_host(c, dim, rows), sim=sim, centroid=cen, want_unpacked=False,
                                index_bits=w["ib"])
        return ix.packed, ix.corr

    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
        parts = list(ex.map(one, range(nchunks)))
    return oracle_index_from_arrays(np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts]),
                                    cen, dim, sim, w["ib"])


def run_reference(args, w, rank):
    """--impl reference: the reference algorithm's CPU path (oracle port) on the box's host cores."""
    if rank != 0:
        return
    n = w["n"]
    sample_rows = min(n, args.ref_rows)
    t0 = time.perf_counter()
    oidx = build_oracle_index_threaded(w, sample_rows)
    build_s = time.perf_counter() - t0
    queries = gen_queries(max(w["nq"], 1), w["dim"])
    from concurrent.futures import ThreadPoolExecutor
    threads = max(1, args.ref_threads or (os.cpu_count() or 1))
    qps_steps = []
    qi = 0
    # one query per host thread at a time — the way a single-threaded Node reference uses a whole box (one worker per
    # core); the oracle's C code runs outside the GIL
    per_step = max(1, args.ref_queries_per_step) * threads
    with ThreadPoolExecutor(max_workers=threads) as ex:
        for step in range(args.warmup + args.steps):
            qs = [queries[(qi + j) % len(queries)] for j in range(per_step)]
            qi += per_step
            t1 = time.perf_counter()
            list(ex.map(lambda q: oracle_search(q, oidx, w["k"], w["qb"], "heap"), qs))
            dt = time.perf_counter() - t1
            if step >= args.warmup:
                qps_steps.append(dt)
    total = sum(qps_steps)
    # per-query cost is linear in the rows scanned: scale the sample to the full corpus (marked as such)
    scale = n / sample_rows
    qps = per_step * args.steps / (total * scale)
    sample = (f"{per_step} queries/step ({threads} threads, one query each at a time) over {sample_rows} of {n} rows"
              + (f", per-query time scaled x{scale:.0f} to the full corpus (extrapolated)" if scale != 1 else "")
              + f"; oracle index build {build_s:.1f}s on {os.cpu_count()} threads (untimed)")
    line = {"impl": "reference", "metric": METRIC, "value": qps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "int32 dot + f64 epilogue", "data": "synthetic",
            "config": {"workload": w["name"], "note": "CPU restatement of the reference TypeScript path (oracle port, C++; pinned bit "
                       "for bit to the reference's own source text by tests/golden/from_ts); the TypeScript reference itself "
                       "cannot be timed here (no node/tsc on the build image or the GPU box: profiles/r02_js_runtime_probe.txt)"},
            "cpu_baseline": {"value": qps, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": qps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ---------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------
def make_format(bbq, w, device):
    return bbq.createBinaryQuantizationFormat(
        {"queryBits": w["qb"], "indexBits": w["ib"],
         "quantizer": {"similarityFunction": w["sim"], "lambda": 0.1, "iters": 5}}, device=device)


def build_shard(torch, fmt, w, r0, r1, device_gen):
    """N(0,1) f32 corpus, generated per 64Ki-row chunk (independent of N), quantised on device (K5), explicit zero
    centroid (the analytic centroid of the synthetic corpus, SURVEY §8d)."""
    n, dim = w["n"], w["dim"]
    cen = np.zeros(dim, np.float32)
    shard = fmt.reserveIndex(max(r1 - r0, 1), dim, cen)
    c, pos = r0 // CHUNK, r0
    while pos < r1:
        c0 = c * CHUNK
        lo, hi = max(pos, c0), min(r1, c0 + CHUNK)
        if device_gen:
            rows = gen_chunk_device(torch, c, dim, min(CHUNK, n - c0))
            part = rows[lo - c0:hi - c0].contiguous()
            fmt.appendRows(shard, d_rows_ptr=part.data_ptr(), n=hi - lo)
            del rows, part
        else:
            rows = gen_chunk_host(c, dim, min(CHUNK, n - c0))
            fmt.appendRows(shard, rows=rows[lo - c0:hi - c0])
        pos = hi
        c += 1
    torch.cuda.synchronize()
    return shard


class Timer:
    def __init__(self, torch, dist, flush, stream):
        self.torch, self.dist, self.flush, self.stream = torch, dist, flush, stream

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def _max_over_ranks(self, tot):
        t = self.torch.tensor([tot], dtype=self.torch.float64, device="cuda")
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def device(self, fn, steps, warmup, cold=True):
        """CUDA events on the launch stream around each step; L2 flushed between steps; max over ranks. -> total ms"""
        torch = self.torch
        for _ in range(warmup):
            fn()
        self.barrier()
        tot = 0.0
        for _ in range(steps):
            if cold:
                self.flush.zero_()             # L2 flush between timed iterations, outside the timed pair
            self.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(self.stream)
            fn()
            e1.record(self.stream)
            e1.synchronize()
            tot += e0.elapsed_time(e1)
        return self._max_over_ranks(tot)

    def host(self, fn, steps, warmup, cold=True):
        """A blocking host call (results are in host memory when it returns): wall clock around it. -> total ms"""
        for _ in range(warmup):
            fn()
        self.barrier()
        tot = 0.0
        for _ in range(steps):
            if cold:
                self.flush.zero_()
            self.barrier()
            t0 = time.perf_counter()
            fn()
            tot += (time.perf_counter() - t0) * 1e3
        return self._max_over_ranks(tot)


def _stage(rank, what):
    if os.environ.get("BBQ_BENCH_WATCHDOG"):
        print(f"[bench r{rank} {time.time() % 1000:.1f}] {what}", file=sys.stderr, flush=True)


DUMP_LIMIT = 64 << 20    # bytes --dump-outputs may write


def dump_outputs(path, idx, sc):
    """--dump-outputs: the top-k lists the timed path returned in its last step, as a caller receives them (global row
    ids as float64, exact below 2**53; f32 scores), one row per query.  Above DUMP_LIMIT a fixed seeded sample of the
    query rows is written; query_rows.npy names the rows either way."""
    os.makedirs(path, exist_ok=True)
    rows = np.arange(idx.shape[0])
    per_row = idx.shape[1] * (8 + 4) + 8
    if rows.size * per_row > DUMP_LIMIT:
        rows = np.sort(np.random.default_rng(0).choice(rows.size, DUMP_LIMIT // per_row, replace=False))
    np.save(os.path.join(path, "query_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(path, "topk_indices.npy"), idx[rows].astype(np.float64))
    np.save(os.path.join(path, "topk_scores.npy"), sc[rows].astype(np.float32))


def measure(args, torch, dist, bbq, w, rank, world, local_rank, steps, warmup, flush, sample_clocks):
    """Builds this rank's shard of workload w and times it.  -> dict of raw measurements (every rank), or None."""
    n, dim, k, nq = w["n"], w["dim"], w["k"], w["nq"]
    r0, r1 = bbq.shard_bounds(n, world, rank)
    fmt = make_format(bbq, w, local_rank)
    t_build = time.perf_counter()
    device_gen = args.datagen == "device" or (args.datagen == "auto" and n > 4_000_000)
    shard = build_shard(torch, fmt, w, r0, r1, device_gen)
    build_s = time.perf_counter() - t_build
    _stage(rank, "shard built")
    searcher = bbq.ShardedSearcher(fmt, shard, r0, rank, world)
    _stage(rank, "communicator up")
    hq = torch.from_numpy(gen_queries(nq, dim)).pin_memory()
    dq = hq.cuda()
    tm = Timer(torch, dist, flush, searcher.stream)

    # --- value: device-resident timing, with the library's per-kernel event taps on --------------------------
    fmt.setProfiling(True)
    for _ in range(warmup):
        searcher.search_device(dq, k)
    torch.cuda.synchronize()
    _stage(rank, "warm-up searches done")
    fmt.resetProfiling()
    l0 = fmt.stats()["kernel_launches"]
    sampler = ClockSampler(local_rank) if (rank == 0 and sample_clocks) else None
    if sampler:
        sampler.start()
    last = []

    def step():
        last[:] = searcher.search_device(dq, k)

    ms_total = tm.device(step, steps, 0)
    outputs = (last[0].cpu().numpy(), last[1].cpu().numpy())     # the last timed step's lists (its stream is synchronised)
    _stage(rank, "device-timed steps done")
    st = fmt.stats()
    launches = st["kernel_launches"] - l0
    fmt.setProfiling(False)
    # --- e2e: HOST buffers through bbq_search / bbq_search_sharded, every step --------------------------------
    e2e_ms = tm.host(lambda: searcher.search(hq, k), steps, warmup)
    _stage(rank, "e2e steps done")
    clocks = sampler.stop() if sampler else None
    # an index smaller than L2 (C2: 11 MB of 126 MB) is L2-resident after the first query: SURVEY §8d asks for the
    # warm figure beside the cold one (`value` / `e2e` are cold: L2 flushed before every step)
    warm = None
    row_bytes = (dim * w["ib"] + 7) // 8
    if (r1 - r0) * (row_bytes + 28) < 100e6:
        warm_ms = tm.device(lambda: searcher.search_device(dq, k), steps, warmup, cold=False)
        warm = {"value": nq / (warm_ms / steps * 1e-3), "unit": UNIT, "ms_per_step": warm_ms / steps,
                "note": "same device-resident search, L2 not flushed between steps (index is L2-resident)"}
    return dict(fmt=fmt, shard=shard, searcher=searcher, hq=hq, st=st, launches=launches, ms_step=ms_total / steps,
                e2e_ms_step=e2e_ms / steps, clocks=clocks, warm=warm, build_s=build_s, device_gen=device_gen,
                rows_local=r1 - r0, r0=r0, outputs=outputs)


def roofline_of(w, m, world, steps, peaks, probe, workload_key):
    st, dim, nq = m["st"], w["dim"], w["nq"]
    rows_local = m["rows_local"]
    bvec = (dim * w["ib"] + 7) // 8 + 16             # algorithmic bytes / scanned vector (SURVEY §8d)
    scan_launch_ms = st["scan_ms"] / max(st["scan_launches"], 1)     # average duration of one scan launch
    scan_ms_step = st["scan_ms"] / steps
    algo_bytes = rows_local * bvec                   # one pass over the shard serves the whole query batch
    index_gbps = algo_bytes / (scan_launch_ms * 1e-3) / 1e9 if scan_launch_ms > 0 else 0.0
    engine = {1: "popcount (LOP3+POPC)", 2: "tcgen05 kind::i8"}.get(st["last_engine"], "popcount (LOP3+POPC)")
    if st["last_engine"] == 2:
        # batched scan = integer contraction [rows x dim*indexBits] . [dim*indexBits x queries(*planes)]: 2*rows*queries*dim*ib
        # ALGORITHMIC ops per launch (an 8-bit query costs two 4-bit B columns per query: machine work, not counted here)
        launches_per_step = max(st["scan_launches"] / steps, 1.0)
        ops = 2.0 * rows_local * (nq / launches_per_step) * dim * w["ib"]
        achieved = ops / (scan_launch_ms * 1e-3) / 1e12
        peak = 2.0 * peaks["bf16"]
        roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TOP/s (int8, = TFLOP/s)",
                    "frac": achieved / peak, "traffic": None,
                    "peak_source": peaks["src"] + ": 2 x bf16_tflops BURST figure (kind::i8 issues at twice the bf16 "
                                   "rate; no int8 number is in MEASURED_PEAKS.json)",
                    "frac_of_2x_bf16_sustained": achieved / (2.0 * peaks["bf16_sustained"]),
                    "kernel": "bbqk::k_scan_mma<SCAN_FILTER>", "algorithmic_ops_per_launch": ops,
                    "queries_resident_per_pass": st["mma_n_tile"], "passes_over_shard": st["mma_passes"],
                    "role_layout": "narrow-batch (4 epilogue warps + 2 expansion groups)" if st.get("mma_layout") else
                                   "wide-batch (8 epilogue warps + 1 expansion group)",
                    "hbm_view": {"algorithmic_bytes_per_launch": algo_bytes, "index_GBps": index_gbps,
                                 "streamed_GBps": index_gbps * st["mma_passes"],
                                 "frac_of_hbm_peak": index_gbps / peaks["hbm"]}}
        if probe and "cycles_per_mma" in probe:
            mhz = (m["clocks"] or {}).get("sm_mhz") or 1965.0
            p8 = probe["int8_ops_per_cycle_per_sm"] * probe["sms"] * mhz * 1e6 / 1e12
            roofline["peak_int8_probe"] = {"value": p8, "unit": "TOP/s", "cycles_per_mma_m128_n208_k32": probe["cycles_per_mma"],
                                           "at_sm_mhz": mhz, "how": "tools/probe/mma_issue_probe peak, run in this process "
                                           "before the timed region: back-to-back tcgen05.mma on idle SMs (no operand feed, no epilogue)"}
            roofline["frac_of_int8_probe"] = achieved / p8
    else:
        roofline = {"bound": "hbm", "achieved": index_gbps, "peak": peaks["hbm"], "unit": "GB/s",
                    "frac": index_gbps / peaks["hbm"], "traffic": None, "peak_source": peaks["src"] + ": hbm_gbs (copy, burst)",
                    "kernel": ("bbqk::k_scan_stream<NB,SCAN_FILTER,W4,CSA>" if nq <= 4 else "bbqk::k_scan<NB,SCAN_FILTER>"),
                    "algorithmic_bytes_per_launch": algo_bytes}
    roofline.update({"avg_scan_launch_ms": scan_launch_ms, "scan_ms_per_step": scan_ms_step,
                     "scan_launches_per_step": st["scan_launches"] / steps,
                     "sample_ms_per_step": st["sample_ms"] / steps,
                     "quantize_ms_per_step": st["quantize_ms"] / steps,
                     "select_ms_per_step": st["select_ms"] / steps,
                     "query_effective_GBps": (nq * algo_bytes / (scan_ms_step * 1e-3) / 1e9) if scan_ms_step > 0 else 0.0,
                     "scan_engine": engine})
    tr, src = load_traffic(workload_key, nq, world, roofline["kernel"])
    roofline["traffic"], roofline["traffic_source"] = tr, src
    roofline["traffic_note"] = ("dram__bytes_read.sum + dram__bytes_write.sum of one launch, copied from the committed "
                                "`ncu --set full` capture of this same command (NOT measured in this run)") if tr else None
    return roofline, index_gbps


def verify_timed_run(w, m, packed, corr, cpu_res, cpu_done, args):
    """Parity of the lists the TIMED configuration returns (same index, same 4096-query batch, same entry point):
    for `parity_queries` queries spread over the batch (a) the k returned rows are exported and re-scored by the
    oracle — f32 scores must be bit-equal and the list must be in canonical order; (b) the oracle's own top-k over
    the exported sample (the first rows of this very index) is computed and no sample row may rank above the k-th
    returned row unless it is in the returned list."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle as O
    dim, sim, k, nq, qb = w["dim"], w["sim"], w["k"], w["nq"], w["qb"]
    shard, searcher, hq = m["shard"], m["searcher"], m["hq"]
    oi, os_ = searcher.search(hq, k)
    oi, os_ = oi.numpy().copy(), os_.numpy().copy()
    qs = hq.numpy()
    cen = shard.getCentroid()
    sample_rows = packed.shape[0]
    oidx = oracle_index_from_arrays(packed, corr, cen, dim, sim, w["ib"])
    want = min(nq, max(args.parity_queries, cpu_done))
    check = sorted(set(range(cpu_done)) | set(int(x) for x in np.linspace(0, nq - 1, want).astype(int)))
    sample_top = {i: cpu_res[i] for i in range(cpu_done)}   # heap lists of the timed cpu leg (same set unless tied)
    rest = [i for i in check if i not in sample_top]
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
        for i, r in zip(rest, ex.map(lambda i: O.search_nearest_neighbors(qs[i], oidx, k, query_bits=qb, mode="canonical"), rest)):
            sample_top[i] = r
    rescored_ok = order_ok = sample_ok = True
    key = lambda s, i: (-(float(s) + 0.0), int(i))
    for i in check:
        rows, scores = oi[i], os_[i]
        keys = [key(s, r) for s, r in zip(scores, rows)]
        order_ok &= keys == sorted(keys) and len(set(rows.tolist())) == len(rows)
        for r, s in zip(rows, scores):
            p, c = shard._export(int(r) - m["r0"], 1)
            one = oracle_index_from_arrays(p, c, cen, dim, sim, w["ib"])
            _, ws = O.search_nearest_neighbors(qs[i], one, 1, query_bits=qb, mode="canonical")
            rescored_ok &= np.float32(ws[0]).view(np.uint32) == np.float32(s).view(np.uint32)
        kth = keys[-1]
        have = set(rows.tolist())
        si, ss = sample_top[i]
        for r, s in zip(si, ss):
            if key(s, r + m["r0"]) < kth and int(r + m["r0"]) not in have:
                sample_ok = False
    return {"timed_configuration_checked": True, "queries_checked": len(check), "of_queries": nq,
            "returned_rows_rescored_bit_equal": bool(rescored_ok), "lists_in_canonical_order": bool(order_ok),
            "sample_rows": sample_rows, "no_sample_row_beats_kth": bool(sample_ok),
            "ok": bool(rescored_ok and order_ok and sample_ok)}


def run_gpu(args, w, rank, world, local_rank):
    import torch
    import bbq_b200

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    bbq_b200.build_library()
    probe = probe_int8_peak() if rank == 0 else None
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    n, dim, sim, k, nq = w["n"], w["dim"], w["sim"], w["k"], w["nq"]
    m = measure(args, torch, dist, bbq_b200, w, rank, world, local_rank, args.steps, args.warmup, flush, True)
    comm = m["fmt"].commInfo()
    if world > 1:
        m["fmt"].commDestroy()       # collective and orderly, on every rank, before the ranks part ways
    qps = nq / (m["ms_step"] * 1e-3)
    e2e_qps = nq / (m["e2e_ms_step"] * 1e-3)
    h2d = nq * dim * 4 * world
    d2h = nq * k * 8 * world

    if rank != 0:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *m["outputs"])
    peaks = load_peaks()
    st = m["st"]
    roofline, index_gbps = roofline_of(w, m, world, args.steps, peaks, probe, args.workload)

    # --- CPU baseline beside it (rank 0): the oracle over THIS index's bytes, bounded sample; then the parity of the
    # timed configuration's own lists -------------------------------------------------------------------------
    cpu = parity = None
    if not args.no_cpu and (world == 1 or args.parity_multi):
        sample_rows = min(m["rows_local"], w.get("cpu_rows", args.cpu_rows))   # bounded sample: the first rows of THIS index
        packed, corr = m["shard"]._export(0, sample_rows)
        oidx = oracle_index_from_arrays(packed, corr, m["shard"].getCentroid(), dim, sim, w["ib"])
        qs = gen_queries(nq, dim)
        done, dt, res = cpu_time_queries(oidx, qs, k, w["qb"], args.cpu_budget, args.cpu_max_queries)
        scale = n / sample_rows                      # per-query cost is linear in the rows scanned
        if world == 1:
            cpu = {"value": done / (dt * scale), "unit": UNIT, "cores": 1, "kind": "port",
                   "sample": f"{done} of {nq} queries over {sample_rows} of the {n} rows of the GPU-built index, 1 thread, "
                             f"{dt:.1f}s" + (f", per-query time scaled x{scale:.0f} to the full corpus (extrapolated)"
                                             if scale != 1 else "")
                             + " (oracle = C++ restatement of the reference TypeScript path, bit-identical to the reference's "
                               "own source on the fixtures of tests/golden/from_ts; not V8)"}
        if world == 1:
            parity = verify_timed_run(w, m, packed, corr, res, done, args)

    line = {"metric": METRIC, "value": qps, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": m["ms_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": ("u8 x u8 -> s32 (tcgen05 kind::i8) + f32 screen + f64 exact replay -> f32 score" if st["last_engine"] == 2
                      else "u32 AND+popcount dot + f64 epilogue -> f32 score"), "data": "synthetic",
            "config": {"workload": w["name"], "rows_total": n, "rows_per_gpu": m["rows_local"], "dim": dim, "k": k,
                       "queries_per_step": nq, "similarity": sim, "query_bits": w["qb"], "index_bits": w["ib"],
                       "sharding": (f"row-wise x{world}; one ncclAllGather of 64-bit top-k keys per step inside "
                                    f"libbbq_b200.so (bbq_search_sharded, NCCL {comm['nccl_version']}, {comm['world']} ranks) + merge"
                                    if world > 1 else "single shard"),
                       "l2": "256 MB flush buffer written between timed iterations",
                       "corpus": ("N(0,1) f32" if CORPUS == "gaussian" else
                                  f"Gaussian mixture f32 ({N_CENTRES} centres ~ N(0,1), noise {CLUSTER_NOISE}; queries drawn the same way)") +
                                 f", {'device' if m['device_gen'] else 'host'}-generated per 65536-row chunk, "
                                 f"explicit zero centroid; index build {m['build_s']:.1f}s (untimed)",
                       "path": {0: "direct", 1: "sampled threshold + filtered scan", 2: "exact chunked"}[st["last_path"]],
                       "remaining_fixed_costs": "per step: one query validation+quantisation, one threshold sample, one "
                                                "selection, one host sync for the overflow flag; with N > 1 every rank "
                                                "quantises the whole batch (redundant), and the all-gather is not "
                                                "overlapped with the next batch's scan"},
            "index_GBps": index_gbps, "index_frac_of_hbm_peak": index_gbps / peaks["hbm"],
            "e2e": {"value": e2e_qps, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": m["e2e_ms_step"],
                    "entry": "bbq_search_sharded" if world > 1 else "bbq_search (via bbq_search_sharded, no communicator)",
                    "timer": "host perf_counter around the blocking C-ABI call (pinned host buffers in, pinned host "
                             "buffers out), max over ranks"},
            "gpu_launches": int(m["launches"]), "roofline": roofline, "clocks": m["clocks"]}
    if m["warm"]:
        line["warm_l2"] = m["warm"]
    if cpu:
        line["cpu_baseline"] = cpu
    if parity:
        line["parity"] = parity
    # free the main index before the secondary workloads
    del m
    torch.cuda.empty_cache()
    if world == 1 and args.workload == "c4" and not args.no_secondary:
        line["secondary"] = secondary_results(args, torch, bbq_b200, local_rank, flush, peaks, probe)
    emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def secondary_results(args, torch, bbq, local_rank, flush, peaks, probe):
    """The other BASELINE configs in the same driver-run line (N=1): each built and timed exactly like the main
    workload, a few seconds apiece, with its top-k lists checked against the oracle on the full (small) index."""
    out = []
    for key in ("c3", "c3q1", "c2"):
        w = dict(WORKLOADS[key])
        try:
            m = measure(args, torch, None, bbq, w, 0, 1, local_rank, args.secondary_steps, 3, flush, True)
            roofline, index_gbps = roofline_of(w, m, 1, args.secondary_steps, peaks, probe, key)
            nq = w["nq"]
            entry = {"workload": w["name"], "value": nq / (m["ms_step"] * 1e-3), "unit": UNIT, "ms_per_step": m["ms_step"],
                     "steps": args.secondary_steps, "warmup": 3,
                     "e2e": {"value": nq / (m["e2e_ms_step"] * 1e-3), "unit": UNIT, "ms_per_step": m["e2e_ms_step"],
                             "h2d_bytes_per_step": nq * w["dim"] * 4, "d2h_bytes_per_step": nq * w["k"] * 8},
                     "gpu_launches": int(m["launches"]), "roofline": roofline, "clocks": m["clocks"],
                     "index_GBps": index_gbps, "index_frac_of_hbm_peak": index_gbps / peaks["hbm"]}
            if m["warm"]:
                entry["warm_l2"] = m["warm"]
            if not args.no_cpu:
                # the whole index is small enough for the oracle: identical lists for a few queries
                packed, corr = m["shard"]._export(0, m["rows_local"])
                oidx = oracle_index_from_arrays(packed, corr, m["shard"].getCentroid(), w["dim"], w["sim"], w["ib"])
                qs = m["hq"].numpy()
                oi, os_ = m["searcher"].search(m["hq"], w["k"])
                oi = oi.numpy()
                nchk = min(nq, 4)
                ok = True
                t0 = time.perf_counter()
                for i in range(nchk):
                    wi, _ = oracle_search(qs[i], oidx, w["k"], w["qb"], "canonical")
                    ok &= oi[i].tolist() == wi.tolist()
                dt = time.perf_counter() - t0
                entry["parity"] = {"queries_checked": nchk, "topk_index_lists_identical": bool(ok)}
                entry["cpu_baseline"] = {"value": nchk / dt, "unit": UNIT, "cores": 1, "kind": "port",
                                         "sample": f"{nchk} queries over the whole index, 1 thread, {dt:.1f}s"}
            out.append(entry)
            del m
        except Exception as e:  # a secondary workload must never take the headline line down with it
            out.append({"workload": w["name"], "error": f"{type(e).__name__}: {e}"})
        torch.cuda.empty_cache()
    out.append(quicksearch_c1(args, bbq))
    return out


def quicksearch_c1(args, bbq):
    """BASELINE configs[0], the reference's own CPU-runnable case: quickSearch(query, vectors, 10, COSINE) on a 1000 x 128
    corpus — the index is REBUILT on every call (src/index.ts:95-111), so this is build + search latency through the
    reference-shaped host API (host rows in, result objects out), beside the oracle's quick_search on one core."""
    try:
        from oracle import oracle as O
        rng = np.random.default_rng(SEED_CORPUS)
        base = rng.standard_normal((1000, 128), dtype=np.float32)
        qs = rng.standard_normal((32, 128), dtype=np.float32)
        for q in qs[:3]:
            bbq.quickSearch(q, base, 10)
        t0 = time.perf_counter()
        got = [bbq.quickSearch(q, base, 10) for q in qs]
        dt = time.perf_counter() - t0
        t1 = time.perf_counter()
        want = [O.quick_search(q, base, 10, "COSINE") for q in qs[:8]]
        dtc = time.perf_counter() - t1
        ok = all([r["index"] for r in got[i]] == want[i][0].tolist() and
                 [np.float32(r["score"]) for r in got[i]] == want[i][1].tolist() for i in range(8))
        return {"workload": "quickSearch on 1000 x 128 f32, k=10, COSINE, index rebuilt per call (BASELINE configs[0])",
                "value": len(qs) / dt, "unit": "quickSearch calls/s", "ms_per_call": 1e3 * dt / len(qs),
                "cpu_baseline": {"value": 8 / dtc, "unit": "quickSearch calls/s", "cores": 1, "kind": "port",
                                 "sample": f"8 calls, {dtc:.2f}s"},
                "parity": {"calls_checked": 8, "lists_and_scores_identical": bool(ok)},
                "note": "host API end to end: H2D of the 512 KB corpus, device index build (K5), query quantisation, "
                        "scan, selection, D2H — per call"}
    except Exception as e:
        return {"workload": "quickSearch (BASELINE configs[0])", "error": f"{type(e).__name__}: {e}"}


_REAL_STDOUT = None


def quiet_stdout():
    """Libraries (NCCL prints its version banner to stdout) must not break the one-JSON-line contract: from here on
    file descriptor 1 goes to stderr and only emit() writes to the real stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def load_traffic(workload, nq, world, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel, from the committed
    `ncu --set full` capture of this same command (profiles/traffic.json names the capture); None when the run is not
    the captured configuration (other query count, sharded corpus)."""
    try:
        table = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except OSError:
        return None, None
    for e in table.get("captures", []):
        if e["workload"] == workload and e["queries_per_step"] == nq and world == 1 and e["kernel"] in kernel:
            return e["dram_bytes_per_launch"], e["source"]
    return None, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--datagen", default="auto", choices=["auto", "host", "device"])
    ap.add_argument("--corpus", default="gaussian", choices=["gaussian", "clustered"],
                    help="clustered: 1000-centre Gaussian mixture (rows and queries), so that the checked rankings are about real neighbours")
    ap.add_argument("--nq", type=int, default=0, help="override the queries per step of the workload (experiments)")
    ap.add_argument("--rows", type=int, default=0, help="override the corpus rows of the workload (experiments)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / parity legs")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary workloads of the default run")
    ap.add_argument("--secondary-steps", type=int, default=0, help="timed steps of each secondary workload (0 = --steps)")
    ap.add_argument("--parity-multi", action="store_true")
    ap.add_argument("--parity-queries", type=int, default=64, help="queries of the timed batch whose lists are verified")
    ap.add_argument("--cpu-budget", type=float, default=15.0, help="seconds of CPU work for cpu_baseline")
    ap.add_argument("--cpu-max-queries", type=int, default=16)
    ap.add_argument("--cpu-rows", type=int, default=1_000_000, help="rows of the index the cpu_baseline leg scans")
    ap.add_argument("--ref-rows", type=int, default=1_000_000, help="--impl reference: rows of the corpus sampled")
    ap.add_argument("--ref-queries-per-step", type=int, default=1, help="--impl reference: queries per thread and step")
    ap.add_argument("--ref-threads", type=int, default=0, help="--impl reference: host threads (0 = all cores)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the top-k lists of the last one as DIR/*.npy (GPU arm)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the GPU arm computed: use it with --impl b200")
    args.secondary_steps = args.secondary_steps or args.steps
    if os.environ.get("BBQ_BENCH_WATCHDOG"):   # diagnostics: dump every Python stack and exit if the run blocks this long
        import faulthandler
        faulthandler.dump_traceback_later(float(os.environ["BBQ_BENCH_WATCHDOG"]), exit=True)
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    w = dict(WORKLOADS[args.workload])
    if args.nq > 0:
        w["nq"] = args.nq
        w["name"] += f" [queries per step overridden: {args.nq}]"
    if args.rows > 0:
        w["n"] = args.rows
        w["name"] += f" [rows overridden: {args.rows}]"
    if args.corpus != "gaussian":
        global CORPUS
        CORPUS = args.corpus
        w["name"] += f" [corpus: {args.corpus}]"
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        quiet_stdout()
        run_reference(args, w, rank)
        return
    if world != args.gpus:
        if args.gpus != 1 and world == 1:
            # launched without torchrun: re-exec under it
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                   "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
            os.execv(sys.executable, cmd)
    quiet_stdout()
    run_gpu(args, w, rank, world, local_rank)


if __name__ == "__main__":
    main()
