#!/usr/bin/env python3
"""bench.py -- queries/sec of the Infidex search path on B200 (BASELINE.json metric), one JSON line on rank 0.

  python bench.py --gpus 1 --steps K --warmup W            # our CUDA path; default workload = the metric's own config:
                                                            # BASELINE.json configs[2], 10M multi-field docs, 10k-query batch
  python bench.py --impl reference ...                      # the reference algorithm on the host cores (oracle port; the
                                                            # C# reference itself cannot run here -- no dotnet in the image)
A "step" is one pass of the hot path over one batch of synthetic queries. `value` times the device-resident batch
(ifx_batch_run, CUDA events inside the library); `e2e` times the reference-facing call ifx_search_batch with host buffers
(host->device query upload + device->host result download inside the region). Every run ends with a PARITY assertion: a bounded
sample of a timed batch is answered by the oracle (CPU restatement of the reference) on the host cores -- that run is also the
`cpu_baseline` -- and the GPU's records for those queries must be identical (DocumentId order, Score bits, Tiebreaker bytes);
a mismatch fails the run instead of printing a line.
N > 1: see `run_ours` (one process per GPU under torchrun).
--dump-outputs DIR: the records the `value` path returned for the last timed batch go to DIR/<name>.npy (see dump_outputs); the
corpus and the query batches are seeded, so two builds run with the same arguments can be compared output for output. That path
returns no facet tables (device-resident batches are uploaded without facet capacity), so none are written.
"""
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
    # BASELINE.json configs[1]: 1M synthetic single-field docs, 1k-query batch, top-10
    "c2": dict(n_docs=1_000_000, nq=1000, multi=False, vocab=400_000, filter=False, label="configs[1]: 1M single-field docs, 1k-query batch, top-10, coverage depth 500"),
    # BASELINE.json configs[2] -- the configuration the metric is quoted on
    "c3": dict(n_docs=10_000_000, nq=10_000, multi=True, vocab=400_000, filter=False, label="configs[2]: 10M multi-field docs (title High / description Low), 10k-query batch, top-10, coverage depth 500"),
    # BASELINE.json configs[3]: + Filter.Parse("year >= 2000 AND rating > 7.0") + EnableFacets
    "c4": dict(n_docs=10_000_000, nq=10_000, multi=True, vocab=400_000, filter=True, label="configs[3]: 10M multi-field docs + Filter.Parse('year >= 2000 AND rating > 7.0') + EnableFacets, 10k-query batch, top-10"),
    "small": dict(n_docs=700_000, nq=2000, multi=True, vocab=200_000, filter=False, label="development workload (700k multi-field docs, 2k queries; not a benchmark)"),
    "tiny": dict(n_docs=50_000, nq=200, multi=True, vocab=50_000, filter=False, label="smoke workload (not a benchmark)"),
}
C4_FILTER = "year >= 2000 AND rating > 7.0"


def effective_cpus():
    """CPUs this process may actually use: the affinity mask, capped by the cgroup quota (os.cpu_count() ignores both)."""
    n = len(os.sched_getaffinity(0))
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(p))))
    except Exception:
        pass
    return n


def clocks_sampler(stop, out, gpu_index):
    """ONE long-lived `nvidia-smi -lms 200` process for the timed region (the profiling recipe's clocks line), read line by line: a
    process per sample re-initialises NVML over every GPU of the box each time, which stalls the CUDA calls of all ranks on an 8-GPU node."""
    import shutil
    q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    cmd = ["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "200"]
    if shutil.which("stdbuf"):
        cmd = ["stdbuf", "-oL"] + cmd          # line-buffered stdout into the pipe
    try:
        pr = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, bufsize=1)
    except Exception:
        return
    try:
        while not stop.is_set():
            line = pr.stdout.readline()
            if not line:
                break
            f = [x.strip() for x in line.split(",")]
            try:
                if len(f) >= 6:
                    out.append((float(f[0]), float(f[1]), f[2], f[3], f[4], f[5]))
            except ValueError:
                pass
    finally:
        try:
            pr.terminate(); pr.wait(timeout=5)
        except Exception:
            try:
                pr.kill()
            except Exception:
                pass


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


DUMP_PAD = {"doc_key": -1, "score": 0, "tie": 0}


def dump_outputs(out_dir, arrays):
    """One DIR/<name>.npy per result array (names of ifx_batch_result): float32 as it is, integers as float64 (exact below 2**53).
    Record slots at or beyond a query's n are never written by the library (their memory is undefined): they are saved as DUMP_PAD."""
    n = arrays["n"]
    arrays = dict(arrays)
    for k, fill in DUMP_PAD.items():
        v = arrays[k]; arrays[k] = np.where(np.arange(v.shape[1])[None, :] >= n[:, None], v.dtype.type(fill), v)
    arrays = {k: v if v.dtype == np.float32 else v.astype(np.float64) for k, v in arrays.items()}
    size = sum(v.nbytes for v in arrays.values())
    if size > 64 << 20:                    # 10k queries x top-10: 2.2 MB
        raise ValueError("%d bytes of outputs exceed the 64 MiB dump budget" % size)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def make_corpus(wl):
    from infidex_b200 import synth
    vocab = synth.make_vocab(wl["vocab"])
    docs = synth.gen_docs(wl["n_docs"], vocab, with_description=wl["multi"])
    schema, cols = synth.schema_and_columns(docs, wl["multi"])
    return vocab, docs, schema, cols


def batch_queries(wl, docs, vocab, step, rank=0):
    from infidex_b200 import dist as ifxd
    from infidex_b200 import synth
    return synth.gen_queries(wl["nq"], docs, vocab, seed=ifxd.rank_batch_seed(synth.SEED, step, rank))


def oracle_from_image(eng, schema):
    """The oracle over the same index: its state is taken from the flattened image of the host builder (Index::load_image; checked equal
    to the oracle's own sequential build by tests/test_oracle_image.py and tests/test_host_builder.py -- re-indexing 10M documents with
    the restatement takes ~20 min), every search-time structure and all search code are the oracle's own."""
    from oracle.oracle import Field as OField
    from oracle.oracle import OracleEngine
    orc = OracleEngine([OField(f.Name, f.Weight, f.Indexable, f.Filterable, f.Facetable) for f in schema])
    orc.load_image(eng.image_ptr())
    return orc


def run_reference(args, wl, rank, world):
    """Reference arm: the reference's algorithm (oracle port) on the host cores, all threads, bounded sample of the batch per step."""
    if rank != 0:
        return
    import infidex_b200 as ib
    vocab, docs, schema, cols = make_corpus(wl)
    eng = ib.SearchEngine.__new__(ib.SearchEngine); eng._host = ib.engine._load_host(); eng._builder = None; eng._index = None; eng._gpu = None   # host builder only: no device, no GPU library
    t0 = time.time(); eng.IndexColumns(docs["keys"], schema, cols, upload=False); orc = oracle_from_image(eng, schema); t_index = time.time() - t0
    cores = effective_cpus()
    sample = min(wl["nq"], args.ref_sample)
    fb = ib.Filter.Parse(C4_FILTER).bytecode() if wl["filter"] else None
    times = []
    for s in range(args.warmup + args.steps):
        qs = batch_queries(wl, docs, vocab, s)[:sample]
        t0 = time.perf_counter(); orc.search_batch(qs, 10, 500, True, fb, threads=cores); dt = time.perf_counter() - t0
        if s >= args.warmup:
            times.append(dt)
    total = sum(times); qps = sample * len(times) / total
    line = {"impl": "reference", "metric": "queries/sec", "value": qps, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["label"], "batch": sample, "filter": bool(wl["filter"]), "index_build_s": round(t_index, 1)},
            "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "os_cpu_count": os.cpu_count(), "kind": "port",
                             "sample": "first %d queries of every step's batch, oracle (C++ restatement of the C# reference; dotnet absent), %d host threads" % (sample, cores)},
            "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def parity_and_cpu_baseline(eng, schema, wl, qs, gpu_bufs, flt, args):
    """Answers the first `sample` queries of one timed batch with the oracle on all host cores (timed: the cpu_baseline) and compares the
    GPU's records for the same queries, bit for bit. Returns (cpu_baseline dict, parity dict)."""
    orc = oracle_from_image(eng, schema)
    cores = effective_cpus()
    sample = min(len(qs), args.ref_sample)
    fb = flt.bytecode() if flt else None
    orc.search_batch(qs[: max(8, sample // 16)], 10, 500, True, fb, threads=cores)       # warm-up
    t0 = time.perf_counter(); ok, osc, ot, on, ost = orc.search_batch(qs[:sample], 10, 500, True, fb, threads=cores); dt = time.perf_counter() - t0
    n1 = max(8, sample // 16)
    t1 = time.perf_counter(); orc.search_batch(qs[:n1], 10, 500, True, fb, threads=1); dt1 = time.perf_counter() - t1
    bad = []
    for i in range(sample):
        st = int(gpu_bufs["status"][i]) & ~8
        if ost[i] != 0 or st != 0:
            if (ost[i] != 0) != (st != 0):
                bad.append((qs[i], "status", int(ost[i]), st))
            continue
        n = int(on[i])
        same = n == int(gpu_bufs["n"][i]) and np.array_equal(gpu_bufs["keys"][i, :n], ok[i, :n]) and \
            np.array_equal(gpu_bufs["scores"][i, :n].view(np.uint32), osc[i, :n].view(np.uint32)) and np.array_equal(gpu_bufs["ties"][i, :n], ot[i, :n])
        if not same:
            bad.append((qs[i], gpu_bufs["keys"][i, :3].tolist(), ok[i, :3].tolist()))
    cpu = {"value": sample / dt, "unit": "queries/s", "cores": cores, "os_cpu_count": os.cpu_count(), "kind": "port", "single_thread_value": n1 / dt1,
           "sample": "first %d queries of the first timed batch, oracle (C++ restatement of the C# reference; dotnet absent), %d threads; index state loaded from the builder image" % (sample, cores)}
    return cpu, {"checked": sample, "mismatches": len(bad), "what": "DocumentId order, float32 Score bits, Tiebreaker bytes vs the oracle"}, bad


def run_sharded(args, wl, rank, world, local):
    """N > 1: ONE index, doc-id-range sharded over the N ranks (infidex_b200/dist.py); every batch runs on every shard with NCCL exchanges
    (all-reduce of LD1 union df and of the selector's cardinalities, all-gather of the Stage-1 lists, of the WordMatcher counts and of the
    final records). Strong scaling: the same corpus and the same 10k-query batches as N = 1. Rank 0 also answers a sample of the first
    timed batch with the UNSHARDED oracle; differing queries are counted in `parity` (the MaxScore threshold chain / heap runs per shard:
    documents tied at the Stage-1 cut can differ -- the waiver SURVEY 8e allows, counted here)."""
    import torch
    import torch.distributed as dist
    import infidex_b200 as ib
    from infidex_b200 import dist as ifxd
    from infidex_b200 import synth
    os.environ.setdefault("NCCL_DEBUG", "WARN")          # keep NCCL's version banner off stdout: the JSON line stands alone
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    t_setup = time.time()
    vocab = synth.make_vocab(wl["vocab"]); lo, hi = ifxd.shard_ranges(wl["n_docs"], world)[rank]
    docs = synth.gen_docs(hi - lo, vocab, with_description=wl["multi"], start=lo, threads=max(1, effective_cpus() // world))
    schema, cols = synth.schema_and_columns(docs, wl["multi"])
    eng = ifxd.ShardedSearchEngine(dist, device_index=local)
    t0 = time.time(); eng.IndexShard(docs["keys"], schema, cols, threads=max(1, effective_cpus() // world)); t_index = time.time() - t0
    flt = ib.Filter.Parse(C4_FILTER) if wl["filter"] else None
    n_total = args.warmup + args.steps; corpus = synth.corpus_ref(wl["n_docs"])
    batches, texts = [], []
    for s in range(n_total):          # the SAME batch on every rank
        qs = batch_queries(wl, corpus, vocab, s, 0); qq = []
        for t in qs:
            x = ib.Query(t, 10); x.Filter = flt; x.EnableFacets = bool(flt); qq.append(x)
        batches.append(qq); texts.append(qs)
    t_setup = time.time() - t_setup
    stop = threading.Event(); clk = []
    th = threading.Thread(target=clocks_sampler, args=(stop, clk, local), daemon=True)

    def timed(fn):
        dist.barrier(); torch.cuda.synchronize(); t0 = time.perf_counter(); r = fn(); torch.cuda.synchronize(); dist.barrier(); return r, time.perf_counter() - t0
    # ---- value: batches uploaded beforehand ----------------------------------------------------------------------------------------------
    ups = [eng.UploadBatch(b) for b in batches]
    agg = {k: 0.0 for k in ("ms_prepare", "ms_expand", "ms_stage1", "ms_s1_select", "ms_s1_score_warp", "ms_s1_score_cta", "ms_s1_finish", "ms_wordmatch", "ms_stage2", "ms_final")}
    algo = 0; launches = 0; dev_t = 0.0; first = None
    for s in range(n_total):
        if s == args.warmup:
            if rank == 0:
                th.start()          # one sampler for the job (rank 0's GPU): eight concurrent nvidia-smi loops stall the timed host path
            eng.exchange_ms = {k: 0.0 for k in eng.exchange_ms}; eng.host_ms = {}
        eng.eng.FlushL2(); st = ib.Stats()
        merged, dt = timed(lambda: eng.SearchBatch(None, stats=st, raw=True, uploaded=ups[s]))
        if s >= args.warmup:
            dev_t += dt; algo += st.algo_bytes_stage1; launches += st.kernel_launches
            for k in agg:
                agg[k] += getattr(st, k)
            if first is None:
                first = merged
            last = merged
    exch = dict(eng.exchange_ms); host = dict(eng.host_ms)
    for u in ups:
        eng.FreeBatch(u)
    # ---- e2e: marshalling + upload inside the region ----------------------------------------------------------------------------------------
    e2e_t = 0.0; prepacked = [eng.eng.PackBatch(b) for b in batches]      # marshalled host buffers (as in the N = 1 arm); upload, run, exchanges, download, merge are timed
    for s in range(n_total):
        eng.eng.FlushL2()
        _, dt = timed(lambda: eng.SearchBatch(batches[s], raw=True, packed=prepacked[s]))
        if s >= args.warmup:
            e2e_t += dt
    stop.set(); eng.Close()
    if th.is_alive():
        th.join(timeout=10)
    tt = torch.tensor([dev_t, e2e_t, float(algo)] + [agg[k] for k in agg], dtype=torch.float64, device="cuda")
    mx = tt.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX); sm = tt.clone(); dist.all_reduce(sm)
    if rank != 0:
        dist.barrier(); dist.destroy_process_group(); return 0
    if args.dump_outputs:                  # the merged records every rank holds
        o_key, o_score, o_tie, o_n, total, status, _ = last
        dump_outputs(args.dump_outputs, dict(doc_key=o_key, score=o_score, tie=o_tie, n=o_n, total_candidates=total, status=status))
    dev_t, e2e_t = float(mx[0]), float(mx[1]); algo_all = float(sm[2]); aggm = {k: float(mx[3 + i]) for i, k in enumerate(agg)}
    value = wl["nq"] * args.steps / dev_t; e2e = wl["nq"] * args.steps / e2e_t
    peak, peak_src = measured_peak(); s1_ms = aggm["ms_stage1"] / args.steps
    achieved = (algo_all / args.steps / 1e9) / (s1_ms / 1e3) if s1_ms > 0 else 0.0
    clocks = None
    if clk:
        smc = sorted(c[0] for c in clk); reasons = set()
        for c in clk:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[2:]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        clocks = {"sm_mhz": smc[len(smc) // 2], "sm_max_mhz": max(c[1] for c in clk), "reasons": sorted(reasons), "samples": len(clk)}
    h2d = sum(2 * len(t) for t in texts[0]) + wl["nq"] * 28 + 8
    line = {"metric": "queries/sec", "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dev_t / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["label"], "batch": wl["nq"], "filter": bool(flt), "parallelism": "one index, doc-id-range sharded x%d (65 536-doc boundaries), every batch on every shard" % world,
                       "l2": "256 MiB L2 flush before every timed step", "index_build_s": round(t_index, 1), "setup_s": round(t_setup, 1)},
            "phases_ms_per_step": {k: round(v / args.steps, 3) for k, v in aggm.items()},
            "exchanges_ms_per_step": {k: round(v / args.steps, 3) for k, v in exch.items()},
            "host_wall_ms_per_step_rank0": {k: round(v / args.steps, 3) for k, v in host.items()},
            "roofline": {"bound": "hbm", "kernel": "Stage 1 (k_select_lookup + k_score_cta + k_score_warp + k_s1_finish), all shards", "achieved": achieved, "peak": peak * world, "unit": "GB/s", "frac": achieved / (peak * world),
                         "traffic": None, "algo_bytes_per_launch": algo_all / args.steps, "ms_per_launch": s1_ms, "peak_source": peak_src + " x n_gpus"},
            "e2e": {"value": e2e, "unit": "queries/s", "h2d_bytes_per_step": int(h2d) * world, "d2h_bytes_per_step": int(wl["nq"] * (10 * 13 + 12 + 48)) * world},
            "gpu_launches": int(launches), "clocks": clocks}
    if not args.no_cpu_baseline:
        # the unsharded oracle over the whole corpus (rank 0 builds the full host image for it)
        full = synth.gen_docs(wl["n_docs"], vocab, with_description=wl["multi"]); fs, fc = synth.schema_and_columns(full, wl["multi"])
        he = ib.SearchEngine.__new__(ib.SearchEngine); he._host = ib.engine._load_host(); he._builder = None; he._index = None; he._gpu = None
        he.IndexColumns(full["keys"], fs, fc, upload=False)
        o_key, o_score, o_tie, o_n, total, status, _ = first
        bufs = {"keys": o_key, "scores": o_score, "ties": o_tie, "n": o_n, "status": status}
        cpu, parity, bad = parity_and_cpu_baseline(he, fs, wl, texts[args.warmup], bufs, flt, args)
        parity["what"] += "; UNSHARDED oracle; differences are counted, not fatal, for N > 1 (per-shard MaxScore heaps: ties at the Stage-1 cut)"
        line["cpu_baseline"] = cpu; line["parity"] = parity
    print(json.dumps(line), flush=True)
    dist.barrier(); dist.destroy_process_group()
    return 0


def run_ours(args, wl, rank, world, local):
    import infidex_b200 as ib
    from infidex_b200 import dist as ifxd
    dist = None
    if world > 1:
        return run_sharded(args, wl, rank, world, local)
    t_setup = time.time()
    vocab, docs, schema, cols = make_corpus(wl); t_gen = time.time() - t_setup
    eng = ib.SearchEngine.CreateDefault(device=local)
    t0 = time.time(); eng.IndexColumns(docs["keys"], schema, cols); t_index = time.time() - t0
    text_mb = (docs["title"][1][-1] + (docs["description"][1][-1] if wl["multi"] else 0)) * 2 / 1e6
    flt = ib.Filter.Parse(C4_FILTER) if wl["filter"] else None
    n_total = args.warmup + args.steps
    batches, texts = [], []
    for s in range(n_total):   # a distinct batch per step (and per rank: replicas answer independent batches)
        qs = batch_queries(wl, docs, vocab, s, rank)
        qq = []
        for t in qs:
            x = ib.Query(t, 10); x.Filter = flt; x.EnableFacets = bool(flt); qq.append(x)
        batches.append(qq); texts.append(qs)
    t_setup = time.time() - t_setup

    def barrier():
        if dist is not None:
            dist.barrier()

    # ---- value: device-resident batches, CUDA-event timing inside the library ------------------------------------------------
    handles = [eng.UploadBatch(b) for b in batches]
    stop = threading.Event(); clk = []
    th = threading.Thread(target=clocks_sampler, args=(stop, clk, local), daemon=True)
    agg = {k: 0.0 for k in ("ms_total", "ms_prepare", "ms_expand", "ms_stage1", "ms_s1_select", "ms_s1_score_warp", "ms_s1_score_cta", "ms_s1_finish", "ms_wordmatch", "ms_stage2", "ms_final")}
    algo = 0; launches = 0; q_max = 0.0; q_sum = 0.0; s1_info = {}
    for s in range(n_total):
        if s == args.warmup:
            barrier(); th.start()
        eng.FlushL2()                       # cold L2 before every step (outside the event-timed region)
        st = eng.RunBatch(handles[s])
        if s >= args.warmup:
            for k in agg:
                agg[k] += getattr(st, k)
            algo += st.algo_bytes_stage1; launches += st.kernel_launches; q_max = max(q_max, st.s1_query_ms_max); q_sum += st.s1_query_ms_sum
            s1_info = {"queries_scored_per_warp": st.s1_light + st.s1_mid, "queries_scored_per_cta": st.s1_heavy, "waves": st.s1_waves, "staging_pool_bytes": int(st.s1_pool_bytes)}
    barrier()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, eng.DownloadBatch(handles[-1], wl["nq"], 10))
    for h in handles:
        eng.FreeBatch(h)
    # ---- e2e: host buffers in / out through the C-ABI call ifx_search_batch (query upload + result download inside the region) --
    packed = [eng.PackBatch(b) for b in batches]
    e2e_t = 0.0; h2d = d2h = 0
    for s in range(n_total):
        eng.FlushL2()
        st = ib.Stats(); t0 = time.perf_counter(); eng.SearchPacked(packed[s], st); dt = time.perf_counter() - t0
        if s >= args.warmup:
            e2e_t += dt; h2d, d2h = st.h2d_bytes, st.d2h_bytes
    stop.set()
    if th.is_alive():
        th.join(timeout=10)
    bad_status = int(sum(((p["bufs"]["status"] & ~8) != 0).sum() for p in packed[args.warmup:]))
    dev_ms = agg["ms_total"]
    if dist is not None:
        dev_ms, e2e_t = ifxd.max_over_ranks(dist, [dev_ms, e2e_t], device="cuda")
        ifxd.gather_results(dist, packed[-1]["bufs"]["keys"], device="cuda")      # per-batch result exchange over NCCL
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0
    step_ms = dev_ms / args.steps
    nq_all = wl["nq"] * world
    value = nq_all * args.steps / (dev_ms / 1e3)
    e2e = nq_all * args.steps / e2e_t
    peak, peak_src = measured_peak()
    s1_ms = agg["ms_stage1"] / args.steps; s1_bytes = algo / args.steps
    achieved = (s1_bytes / 1e9) / (s1_ms / 1e3) if s1_ms > 0 else 0.0
    traffic = None
    tp = os.path.join(ROOT, "profiles", "stage1_traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get(args.workload)
    clocks = None
    if clk:
        sm = sorted(c[0] for c in clk); reasons = set()
        for c in clk:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[2:]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        clocks = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(c[1] for c in clk), "reasons": sorted(reasons), "samples": len(clk)}
    line = {"metric": "queries/sec", "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",      # N > 1 splits this same index and batch over N GPUs (run_sharded)
            "config": {"workload": wl["label"], "batch": wl["nq"], "filter": bool(flt), "parallelism": "1 GPU",
                       "l2": "256 MiB L2 flush before every timed step; the index (text alone %.0f MB) also exceeds the 126 MB L2" % text_mb,
                       "corpus_gen_s": round(t_gen, 1), "index_build_s": round(t_index, 1), "setup_s": round(t_setup, 1), "bad_status": bad_status},
            "phases_ms_per_step": {k: round(v / args.steps, 3) for k, v in agg.items()},
            "stage1": s1_info,
            "roofline": {"bound": "hbm", "kernel": "Stage 1 = k_select_lookup (posting streams, selection) + k_score_cta + k_score_warp + k_s1_finish", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "algo_bytes_per_launch": s1_bytes, "ms_per_launch": s1_ms, "peak_source": peak_src,
                         "select_lookup_ms_per_launch": agg["ms_s1_select"] / args.steps,
                         "longest_query_ms": q_max, "sum_query_ms_per_launch": q_sum / args.steps},
            "e2e": {"value": e2e, "unit": "queries/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(launches), "clocks": clocks}
    rc = 0
    if not args.no_cpu_baseline:
        s0 = args.warmup                                                           # the first timed batch
        cpu, parity, bad = parity_and_cpu_baseline(eng, schema, wl, texts[s0], packed[s0]["bufs"], flt, args)
        line["cpu_baseline"] = cpu; line["parity"] = parity
        if bad:
            print("PARITY FAILURE: %d of %d sampled queries differ from the oracle, e.g. %r" % (len(bad), parity["checked"], bad[:3]), file=sys.stderr, flush=True)
            rc = 1
    if rc == 0:
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()
    return rc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=list(WORKLOADS), help="default: c3 = BASELINE.json configs[2], the configuration the metric is quoted on")
    ap.add_argument("--ref-sample", type=int, default=512, help="queries per step of the CPU arms (bounded sample of the batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the oracle leg (cpu_baseline + parity assertion)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the records of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the records of the CUDA path; it does not apply to --impl reference")
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, wl, rank, world)
    sys.exit(run_ours(args, wl, rank, world, local))


if __name__ == "__main__":
    main()
