#!/usr/bin/env python
"""bench.py — BM25 top-10 queries/sec at 10 M docs on 1/2/4/8 B200 (BASELINE.json metric).

Default workload = configs[1] of BASELINE.json (C2): synthetic 10 M-doc Zipfian corpus (uniform 100..300 tokens per doc,
1 M-term vocabulary, seed 20260101), a batch of 4096 two-to-five-term OR queries (seed 20260102), top-10 (internal
k = 11) WITH BLOCK-MAX PRUNING (`execution = bmw`: exact, byte-identical to the exhaustive result), k1 = 0.9, b = 0.4.
The corpus is generated on the GPU (searchlite_b200.synth) and loaded once into the engine's HBM-resident layout; a
"step" is one pass of the whole 4096-query batch.

  value      queries/sec with the prepared batch already resident in HBM (slg_batch_run), headline execution
  e2e        queries/sec through slg_search_batch with HOST query structs in and HOST hits out
             (H2D of the packed batch + all kernels + D2H of the hits inside the timed region)
  exhaustive the same batch under `execution = bm25` (every posting read and compared): value, e2e, kernel time
  roofline   the exhaustive scoring kernels: algorithmic posting bytes (5 B x sum of df over query terms, SURVEY.md §8d)
             / their CUDA-event time, against the measured HBM copy bandwidth
  pruned     work counters of the pruned run: postings scanned / verified, items dropped, speed-up over exhaustive
  parity     EVERY query of the batch against the oracle's exact top-k (at N > 1: against the oracle's per-segment
             results merged in SortKey order), plus byte-identity of the pruned and exhaustive results
  cpu_baseline  the oracle ("port" of the reference CPU path) timed on the host cores on the same queries

N > 1 (torchrun): the corpus is split into N contiguous doc-range segments, one per rank; every rank scores all
queries on its segment, ONE NCCL all-gather exchanges the packed local top-k blocks and every rank merges (strong
scaling: total corpus fixed).  While the scan runs the shards push their per-query k-th scores into each other's
threshold boards (symmetric memory over NVLink, `--no-threshold-board` switches it off; results are exact either way).

Other configurations (`--config`): c3 (8.84 M short passages, top-1000, bmw), c4 (Bool{must} AND queries behind
And[KeywordEq(lang), I64Range(year)] at 37 / 10 / 1 % selectivity + a 2-term phrase leg, every leg with full-batch oracle
parity), c5 (BM25 top-1000 -> exact 768-d bf16 rerank on the device, 12.5 M docs per GPU, vectors sharded with their docs).
They print the same JSON line shape with their own `config.workload` (tools/bench_configs.py).

`--impl reference` times the reference's own CPU algorithm (oracle restatement, faithful mode: per-query varint
decode + doc-length vector + WAND, the reference's default execution) on the host cores; rank 0 only.

`--dump-outputs DIR` (c2, c3) writes the top-k the last timed step handed its caller to DIR as .npy files, so that two
builds run with the same arguments (hence the same seeded corpus and queries) can be compared output for output:
hits_doc_id, hits_segment_ord (float64, exact) and hits_score (float32, bit for bit) of shape [queries, k], with the
slots past a query's count set to 0; counts (float64, [queries]); query_index (float64): the batch rows written, all
of them unless the dump would pass 64 MB, then a fixed seeded sample.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c4", "c5"])
    ap.add_argument("--docs", type=int, default=0, help="0 = the configuration's size")
    ap.add_argument("--vocab", type=int, default=1_000_000)
    ap.add_argument("--queries", type=int, default=0, help="0 = the configuration's batch")
    ap.add_argument("--limit", type=int, default=0, help="0 = the configuration's limit")
    ap.add_argument("--execution", default="bmw", choices=["bm25", "wand", "bmw"])
    ap.add_argument("--tile-docs", type=int, default=0)
    ap.add_argument("--ctas-per-sm", type=int, default=0)
    ap.add_argument("--sub-docs", type=int, default=0)
    ap.add_argument("--kernel", default="auto", choices=["auto", "cta", "warp", "items", "reg", "warp-inplace", "auto-inplace"])
    ap.add_argument("--option", action="append", default=[], help="engine residency option name=value (slg_set_option)")
    ap.add_argument("--cpu-sample", type=int, default=-1, help="queries checked against / timed on the CPU oracle (-1 = all, 0 = skip)")
    ap.add_argument("--ref-sample", type=int, default=64, help="queries per step of --impl reference")
    ap.add_argument("--candidates", type=int, default=1000, help="c5: BM25 candidates per query handed to the rerank")
    ap.add_argument("--no-phrases", action="store_true", help="c4: skip the phrase leg (positions resident: +21 GB)")
    ap.add_argument("--no-threshold-board", dest="threshold_board", action="store_false",
                    help="N > 1: do not exchange per-query k-th scores between the shards during the scan (NVLink peer pushes, on by default)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-exhaustive", action="store_true", help="skip the exhaustive (bm25) leg and its roofline")
    ap.add_argument("--no-pruned", action="store_true", help=argparse.SUPPRESS)  # (round-1 flag: same as --no-exhaustive)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step to DIR/<name>.npy (c2, c3)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config not in ("c2", "c3")):
        ap.error("--dump-outputs covers --impl ours with --config c2 or c3")
    cfg = {"c2": (10_000_000, 4096, 10), "c3": (8_841_823, 1024, 1000), "c4": (10_000_000, 4096, 10), "c5": (0, 1024, 10)}[args.config]
    args.docs = args.docs or cfg[0]
    args.queries = args.queries or cfg[1]
    args.limit = args.limit or cfg[2]
    args.no_exhaustive = args.no_exhaustive or args.no_pruned
    return args


def read_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


KERNEL_SOURCES = ("slg_scan_kernel.cuh", "slg_stream_kernel.cuh", "slg_items_kernel.cuh", "slg_warp_kernel.cuh", "slg_kernels.cuh",
                  "slg_async.cuh", "slg_launch_items.cu")


def kernel_source_hash() -> str:
    """hash of the sources of the roofline kernels (scan + column pass and what they include): a DRAM-traffic figure taken with
    ncu is only reported next to the kernels it was taken from"""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "searchlite_b200", "csrc")
    for name in KERNEL_SOURCES:
        with open(os.path.join(d, name), "rb") as f:
            h.update(name.encode() + b"\0" + f.read())
    return h.hexdigest()[:16]


def measured_traffic(kernel_key: str):
    """(bytes per launch, source) from profiles/traffic.json when it was captured from THIS build of the kernels, else (None, why)"""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
    except Exception:
        return None, "no ncu capture recorded for this build"
    e = t.get(kernel_key)
    if not e or e.get("source_hash") != kernel_source_hash():
        return None, "the recorded ncu capture belongs to an older build of the kernels"
    return float(e["dram_bytes"]), e.get("file")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                       "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self) -> dict:
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, hits: np.ndarray, counts: np.ndarray) -> None:
    """hits [Q, k] (HIT_DTYPE) and counts [Q] as the .npy files the module docstring lists"""
    n_q, k = hits.shape
    bytes_per_query = k * (8 + 8 + 4) + 8 + 8
    rows = np.arange(n_q)
    if n_q * bytes_per_query > DUMP_LIMIT_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n_q, DUMP_LIMIT_BYTES // bytes_per_query, replace=False))
    hits, counts = hits[rows], counts[rows]
    valid = np.arange(k)[None, :] < counts[:, None]
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"hits_doc_id": np.where(valid, hits["doc_id"], 0).astype(np.float64),
              "hits_segment_ord": np.where(valid, hits["segment_ord"], 0).astype(np.float64),
              "hits_score": np.where(valid, hits["score"], np.float32(0)).astype(np.float32),
              "counts": counts.astype(np.float64), "query_index": rows.astype(np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ---- workloads ---------------------------------------------------------------------------------------------------
def corpus_spec(args, rank: int, world: int):
    from searchlite_b200 import synth
    from searchlite_b200.shard import shard_ranges
    lo, hi = shard_ranges(args.docs, world)[rank]
    if args.config == "c3":  # MS-MARCO-passage-like: short docs (8..104 tokens, mean 56)
        return synth.CorpusSpec(n_docs=hi - lo, vocab=args.vocab, seed=20260103, len_lo=8, len_hi=104, segment_ord=rank, doc_base=lo)
    return synth.CorpusSpec(n_docs=hi - lo, vocab=args.vocab, seed=20260101, segment_ord=rank, doc_base=lo)


def query_batch(args):
    from searchlite_b200 import synth
    return synth.generate_queries(args.queries, args.vocab, seed=20260104 if args.config == "c3" else 20260102)


def workload_name(args, world: int) -> str:
    if args.config == "c3":
        return (f"C3: synthetic {args.docs / 1e6:g}M-passage Zipf(s=1) corpus, uniform 8..104 tokens/doc (mean 56), {args.vocab / 1e6:g}M-term vocab, "
                f"{args.queries} OR queries of 2-5 terms, top-{args.limit} (k={args.limit + 1}), k1=0.9 b=0.4, {world} doc-range segment(s)")
    return (f"C2: synthetic {args.docs / 1e6:g}M-doc Zipf(s=1) corpus, uniform 100..300 tokens/doc, {args.vocab / 1e6:g}M-term vocab, "
            f"{args.queries} OR queries of 2-5 terms, top-{args.limit} (k={args.limit + 1}), k1=0.9 b=0.4, "
            f"{world} doc-range segment(s)")


def run_reference(args, rank: int, world: int):
    """the reference's CPU algorithm on the host cores (oracle port, faithful per-query decode + WAND)"""
    if rank != 0:
        return
    import torch
    from oracle import slo
    slo.build()
    t0 = time.time()
    device = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
    # the reference arm searches the corpus split into `world` segments sequentially, as IndexReader::search does
    # (api/reader.rs:2670), on a bounded sample of the batch per step
    from searchlite_b200 import synth
    oracles = []
    for r in range(world):
        seg = synth.generate_segment(corpus_spec(args, r, world), device).to_host()
        if device.type == "cuda":
            torch.cuda.empty_cache()
        o = slo.OracleIndex(seg)
        o.build_post_image()
        oracles.append(o)
    qb = query_batch(args)
    k = args.limit + 1
    threads = slo.max_threads()
    sample = min(args.ref_sample, args.queries)
    setup_s = time.time() - t0
    times = []
    for step in range(args.warmup + args.steps):
        lo = (step * sample) % max(1, args.queries - sample + 1)
        sub = qb.subset(lo, lo + sample)
        t = time.perf_counter()
        lists = [o.search_batch(sub, k, "wand", faithful=True, threads=threads) for o in oracles]
        if len(oracles) > 1:
            for qi in range(sample):
                slo.merge_hits([h[qi, : c[qi]] for h, c in lists], k)
        dt = time.perf_counter() - t
        if step >= args.warmup:
            times.append(dt)
    ms = 1e3 * float(np.mean(times))
    qps = sample / (ms / 1e3)
    line = {
        "impl": "reference", "metric": "bm25_top10_queries_per_sec", "value": qps, "unit": "queries/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args, world), "execution": "wand (reference default)",
                   "step": f"{sample} queries per step (bounded sample of the {args.queries}-query batch)"},
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} queries/step, faithful mode: per-query varint decode of every term list + per-query "
                                   f"doc-length vector + WAND (oracle restatement; the Rust reference cannot be built here)"},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "setup_s": round(setup_s, 1),
    }
    print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, max(world, args.gpus if world == 1 else world))
        return
    if args.config in ("c4", "c5"):
        from tools import bench_configs
        bench_configs.main(args, rank, local_rank, world)
        return

    import torch
    import torch.distributed as dist
    from searchlite_b200 import GpuIndex, synth
    from searchlite_b200.shard import ShardedSearcher

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    k = args.limit + 1

    t0 = time.time()
    seg = synth.generate_segment(corpus_spec(args, rank, world), device)
    qb = query_batch(args)
    torch.cuda.synchronize()
    gen_s = time.time() - t0
    t0 = time.time()
    options = {kv.split("=")[0]: int(kv.split("=")[1]) for kv in args.option}
    gi = GpuIndex(local_rank, tile_docs=args.tile_docs, ctas_per_sm=args.ctas_per_sm, sub_docs=args.sub_docs, kernel=args.kernel,
                  options=options)
    gi.load_segment(seg)
    load_s = time.time() - t0
    n_postings = gi.segment_stats(rank)["n_postings"]
    del seg
    torch.cuda.empty_cache()

    stream = torch.cuda.ExternalStream(gi.stream_ptr(), device=device)
    searcher = ShardedSearcher(gi, args.queries, k, threshold_board=args.threshold_board) if world > 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        t = torch.tensor([ms], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def time_resident(execution: str):
        """(ms per step, kernel ms, launches per step, results, counters, results of the last timed step) of one execution
        with the batch resident"""
        p = gi.prepare(qb, k, execution)

        def step():
            if world > 1:
                return searcher.run(p)
            p.run(sync=True)
            return None
        for _ in range(args.warmup):
            step()
        barrier()
        c0 = gi.counters()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            ev0.record(stream)
            for _ in range(args.steps):
                last = step()
            ev1.record(stream)
        barrier()
        if world == 1:
            last = p.fetch()  # the one-GPU step leaves its result on the device, where a caller fetches it
        c1 = gi.counters()
        ms = max_over_ranks(ev0.elapsed_time(ev1)) / args.steps
        launches = (c1["kernel_launches"] - c0["kernel_launches"]) / args.steps
        # the scoring kernels' own CUDA-event time (handle's stream): one more, synchronous, pass — the sharded loop above
        # runs asynchronously, so its passes leave no per-kernel time behind; max over ranks like the step time
        c0 = gi.counters()
        if world > 1:
            barrier()
            searcher.attach_board(p)  # (a fresh epoch: the pass must not start from the thresholds its peers left behind)
        p.run(sync=True)
        c1 = gi.counters()
        kernel_ms = max_over_ranks((c1["score_ms_total"] - c0["score_ms_total"]) / max(c1["score_launches"] - c0["score_launches"], 1))
        if world == 1:
            res = p.fetch()
        else:
            res = searcher.exchange_and_merge(p)
            p.fetch()  # (this rank's own work counters)
        ctr = gi.counters()
        p.free()
        return ms, kernel_ms, launches, res, ctr, last

    def time_e2e(execution: str):
        def step():
            if world == 1:
                return gi.search_batch(qb, k, execution)
            p = gi.prepare(qb, k, execution)
            out = searcher.run(p)
            p.free()
            return out
        for _ in range(max(1, args.warmup)):
            step()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.perf_counter()
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(args.steps):
                step()
            e1.record(stream)
        barrier()
        wall_ms = 1e3 * (time.perf_counter() - w0)
        ms = max_over_ranks(max(e0.elapsed_time(e1), wall_ms)) / args.steps
        cc = gi.counters()
        return {"value": args.queries / (ms / 1e3), "unit": "queries/s", "ms_per_step": ms,
                "h2d_bytes_per_step": int(cc["last_h2d_bytes"]), "d2h_bytes_per_step": int(cc["last_d2h_bytes"])}

    # ---- headline execution ----
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ms_step, kernel_ms, launches, (got_h, got_c), ctr, last = time_resident(args.execution)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)
    e2e = None if args.no_e2e else time_e2e(args.execution)

    # ---- exhaustive leg: roofline of the scoring kernels, and the result the pruned run must reproduce byte for byte ----
    exhaustive = None
    ex_h = ex_c = None
    if args.execution != "bm25" and not args.no_exhaustive:
        x_ms, x_kernel_ms, x_launches, (ex_h, ex_c), x_ctr, _ = time_resident("bm25")
        exhaustive = {"execution": "bm25", "value": args.queries / (x_ms / 1e3), "unit": "queries/s", "ms_per_step": x_ms,
                      "kernel_ms": x_kernel_ms, "gpu_launches": x_launches,
                      "postings_scanned": int(x_ctr["last_postings_scattered"]), "postings_verified": int(x_ctr["last_postings_verified"])}
        if not args.no_e2e:
            exhaustive["e2e"] = time_e2e("bm25")
    elif args.execution == "bm25":
        x_kernel_ms, x_ctr = kernel_ms, ctr

    hbm_peak, peak_kind = read_peaks()
    posting_count = ctr["last_posting_count"]
    line = {
        "metric": "bm25_top10_queries_per_sec", "value": args.queries / (ms_step / 1e3), "unit": "queries/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args, world), "execution": args.execution,
                   "l2": "inputs larger than L2 (resident postings >> 126 MB); no explicit flush",
                   "postings_resident_this_rank": int(n_postings), "kernel": args.kernel, "options": options,
                   "threshold_board": bool(searcher is not None and searcher.board is not None)},
        "e2e": e2e,
        "gpu_launches": int(round(launches * args.steps)),
        "clocks": clocks,
        "setup": {"corpus_gen_s": round(gen_s, 1), "load_segment_s": round(load_s, 1), "resident_bytes": int(ctr["resident_bytes"]),
                  "resident": gi.segment_residency(rank)},
    }
    if args.execution != "bm25":
        scanned = int(ctr["last_postings_scattered"])
        line["pruned"] = {
            "execution": args.execution, "kernel_ms": kernel_ms,
            "posting_count": int(posting_count), "postings_scanned": scanned, "postings_scanned_frac": scanned / max(posting_count, 1),
            "postings_verified": int(ctr["last_postings_verified"]), "scan_items": int(ctr["last_items"]),
            "scan_items_dropped": int(ctr["last_items_dropped"]),
            "column_blocks_scored": int(ctr["last_column_blocks_streamed"]), "column_blocks_per_doc": int(ctr["last_subtiles_skipped"]),
            "note": "this rank's segment; posting_count = sum of df over the batch's query terms; a dropped item = 4096 postings of a non-essential term",
        }
        if exhaustive:
            line["pruned"]["speedup_vs_exhaustive"] = exhaustive["ms_per_step"] / ms_step
            line["pruned"]["identical_to_exhaustive"] = bool(ex_h.tobytes() == got_h.tobytes() and ex_c.tobytes() == got_c.tobytes())
    line["exhaustive"] = exhaustive
    if args.execution == "bm25" or exhaustive:
        alg_bytes = 5.0 * posting_count
        achieved = alg_bytes / (x_kernel_ms / 1e3) / 1e9 if x_kernel_ms > 0 else 0.0
        traffic, traffic_src = measured_traffic("scan+columns:bm25:c2" if args.config == "c2" and world == 1 and not options else "none")
        line["roofline"] = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                            "traffic": traffic, "traffic_source": traffic_src, "peak_kind": peak_kind,
                            "kernel": "slg_scan_kernel<false> + slg_score_columns_kernel<false> (execution bm25: every posting read and compared)",
                            "kernel_ms": x_kernel_ms, "algorithmic_bytes_per_launch": alg_bytes,
                            "note": "5 B x sum of df over the batch's query terms (this rank's segment), SURVEY.md §8d; a fraction above 1 means "
                                    "posting bytes are shared between the queries of the batch (one column block read serves every query that names the column)"}

    # ---- CPU baseline + parity on EVERY query (rank 0; at N > 1 against the oracle's merged per-segment results) ----
    n_cpu = args.queries if args.cpu_sample < 0 else min(args.cpu_sample, args.queries)
    line["cpu_baseline"] = None
    if rank == 0 and n_cpu > 0:
        from oracle import slo
        from tests.parity import parity_report
        slo.build()
        threads = slo.max_threads()
        sub = qb.subset(0, n_cpu)
        per_seg = []
        cpu_s = 0.0
        for r in range(world):
            host = synth.generate_segment(corpus_spec(args, r, world), device).to_host()
            torch.cuda.empty_cache()
            ora = slo.OracleIndex(host)
            tcpu = time.perf_counter()
            per_seg.append(ora.search_batch(sub, k, "bm25_dense", threads=threads))
            cpu_s += time.perf_counter() - tcpu
            if world > 1:
                del ora
            del host
        if world == 1:
            ref_h, ref_c = per_seg[0]
        else:
            ref_h = np.zeros_like(per_seg[0][0])
            ref_c = np.zeros_like(per_seg[0][1])
            for qi in range(n_cpu):
                m = slo.merge_hits([h[qi, : c[qi]] for h, c in per_seg], k)
                ref_h[qi, : len(m)] = m
                ref_c[qi] = len(m)
        line["cpu_baseline"] = {"value": n_cpu / cpu_s, "unit": "queries/s", "cores": threads, "kind": "port",
                                "sample": f"{n_cpu} of the {args.queries} queries, oracle bm25_dense (pre-decoded postings, {threads} threads over "
                                          f"queries; the 'fair' port of BASELINE.md §3), {world} segment(s) searched one after the other"}
        rep = parity_report(ref_h, ref_c, got_h[:n_cpu], got_c[:n_cpu])
        rep["note"] = ("every listed query against the oracle's exact result in the reference's (query) summation order: bit_exact = ids, order and "
                       "f32 score bits equal; within_rule = the north-star rule (ids and order equal, scores within 1e-5 relative, id swaps only inside "
                       "1e-5 of the k-th score).  The engine sums a doc's terms without a dense column first, then those with one (declared order)")
        if world == 1:
            from tests.helpers import canonical_batch
            can_h, can_c = ora.search_batch(canonical_batch(gi, sub), k, "bm25_dense", threads=threads)
            rep["bit_exact_declared_order"] = parity_report(can_h, can_c, got_h[:n_cpu], got_c[:n_cpu])["bit_exact"]
        line["parity"] = rep
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
