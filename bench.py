#!/usr/bin/env python
"""bench.py — milli query-time scoring path on B200 (contract: the task's ④; SURVEY.md §8(d)).

Default workload = cfg 3, the configuration BASELINE.json's metric is quoted on:
  synthetic "hackernews" corpus, 10 M docs x 1 searchable field, 1.5 M-word Zipf vocabulary, default criteria, limit 20,
  + one 768-d fp16 embedding per document (cfg 4 generator, 15.4 GB),
  batch = 1024 typo-tolerant 2-4 word queries (cfg 2 generator), each with a query vector, `execute_hybrid(semanticRatio 0.5)`:
  keyword search with ScoringStrategy::Detailed + exact cosine top-20 + the hybrid merge.
One *step* = one such batch through b200_search_batch (mode 2).  `--mode keyword` times Search::execute alone.

  value     queries/sec from the CUDA-event time of the device work of the K steps in a single-lane pass (kernel intervals do not
            overlap there): every host<->device round trip's first..last kernel + the term-derivation sweep + the vector stage
  e2e       queries/sec through the C ABI with HOST buffers: wall clock around the K calls (host-side ranking-rule control flow,
            every H2D/D2H copy, all synchronisation, the hybrid merge)
  roofline  dominant kernel (largest accumulated CUDA-event time): algorithmic bytes (or flops) / its event time vs the measured peak
  cpu_baseline / --impl reference   the CPU oracle ("port": C++ restatement of milli; the Rust reference cannot be built here) on a
            bounded sample of the same queries, fixed thread count, with the latency distribution and a searchCutoffMs-clamped figure
  parity    ALL queries of one timed batch against the oracle: docids, ScoreDetails rank tuples, candidate counts (keyword,
            Detailed) and the merged hybrid hits (docids, scores within 1e-4 relative on the vector similarity)
  --dump-outputs DIR   the search result of the last timed step as DIR/<array>.npy; the same arguments give the same inputs, so two
            builds can be compared output for output

Multi-GPU (torchrun): the path shards by query — every rank holds a replica and serves its own batches; no data-path collective
(DESIGN.md §5); value = all ranks' queries / max-over-ranks time.
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
SEARCH_CUTOFF_S = 1.5  # crates/milli/src/lib.rs:169-173 (searchCutoffMs default)
DIM = 768


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    out = {"hbm": (6650.0, "fallback"), "tensor": (1590.0, "fallback")}
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            out["hbm"] = (float(d["hbm_gbs"]), "measured")
            out["tensor"] = (float(d["bf16_tflops"]), "measured (cuBLAS bf16 burst)")
        except Exception:
            pass
    return out


def ncu_traffic(kernel):
    """dram bytes per launch of `kernel` from the newest committed ncu capture (profiles/*_traffic.json), or None"""
    names = {"eval_paths": "eval_dp_kernel", "scatter": "scatter_kernel", "lev_match": "lev_match_kernel", "act_compact": "act_compact_kernel",
             "pair_probe": "pair_probe_kernel", "emit": "emit_kernel", "vec_gemm_topk": "vec_gemm_topk_kernel", "vec_dist": "vec_dist_kernel"}
    try:
        import glob
        f = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")))[-1]
        return float(json.load(open(f))["kernels"][names[kernel]]["dram_bytes_per_launch"])
    except Exception:
        return None


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self, window=None):
        """summary of the samples that arrived inside `window` = (t0, t1) of time.perf_counter() (nvidia-smi needs about a second
        to start, so the sampler runs from before the warm-up and the timed region is cut out afterwards)"""
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        rows = [r for t, r in self.rows if window is None or window[0] - 0.11 <= t <= window[1] + 0.11]
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
                for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                    if r[col].lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ workload
def build_workload(args, rank, world):
    from corpus.pyindexgen import synthetic_embeddings_f16, synthetic_image
    from meilisearch_b200.tokenizer import TokenBatch

    t = time.time()
    img = synthetic_image(args.docs, args.vocab, seed=0xB200, log=log)
    log(f"[rank {rank}] corpus: {img.n_docs} docs, {img.n_words} words, {type(img).__name__} ready in {time.time() - t:.1f}s")
    batches = [TokenBatch(img.synthetic_queries(args.batch, seed=1000 * rank + i)) for i in range(args.distinct_batches)]
    emb, vecs = None, None
    if args.mode == "hybrid":
        t = time.time()
        emb = synthetic_embeddings_f16(int(img.n_docs), DIM, seed=0xE5BED)
        vecs = [np.random.default_rng(77 + 1000 * rank + i).standard_normal((args.batch, DIM), dtype=np.float32) for i in range(args.distinct_batches)]
        log(f"[rank {rank}] embeddings: {emb.shape[0]} x {DIM} fp16 ({emb.nbytes / 1e9:.1f} GB) generated in {time.time() - t:.1f}s")
    return img, batches, emb, vecs


def metric_name(args):
    if args.mode == "hybrid":
        return "queries/sec (batch=1024, typo-tolerant keyword + 768-d cosine hybrid search, semanticRatio 0.5, top-20)"
    return "queries/sec (batch=1024, typo-tolerant multi-term keyword search, top-20)"


def workload_config(args, img):
    cfg = "cfg3" if img.n_docs >= 5_000_000 else "cfg2"
    txt = (f"{cfg} hackernews-like synthetic: {img.n_docs} docs x 1 field, {img.n_words}-word dictionary, batch={args.batch} queries of 2-4 words "
           "(40% clean / 40% one edit / 20% two edits, last word prefix p=0.3), criteria words,typo,proximity,attributeRank,wordPosition,exactness, "
           "TermsMatchingStrategy::Last, limit 20")
    if args.mode == "hybrid":
        txt += (f"; + {img.n_docs} x {DIM} fp16 L2-normalised N(0,1) embeddings (one per document), one N(0,1) query vector per query, "
                "execute_hybrid(semanticRatio 0.5), keyword side ScoringStrategy::Detailed")
    return {"workload": txt, "mode": args.mode, "batch": args.batch, "docs": int(img.n_docs), "vocab": int(img.n_words),
            "l2": "working set (posting store, per-batch matrices" + (", 15.4 GB embedding matrix" if args.mode == "hybrid" else "") +
                  ") exceeds the 126 MB L2; a different query batch every step"}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_threads():
    return max(1, min(64, (os.cpu_count() or 2) // 2))


def oracle_for(img, emb):
    from oracle.pyoracle import OracleIndex

    o = OracleIndex(img)
    if emb is not None:
        o.set_embeddings(emb)
    return o


def oracle_run(o, args, tokens, vectors, threads, scoring="skip"):
    if args.mode == "hybrid":
        return o.search_batch(tokens, vectors=vectors, hybrid=True, semantic_ratio=0.5, n_threads=threads)
    return o.search_batch(tokens, scoring=scoring, n_threads=threads)


def latency_summary(lat, threads, wall, n):
    lat = np.asarray(lat, np.float64)
    clamped = np.minimum(lat, SEARCH_CUTOFF_S)
    return {"p50_ms": 1e3 * float(np.percentile(lat, 50)), "p95_ms": 1e3 * float(np.percentile(lat, 95)), "mean_ms": 1e3 * float(lat.mean()),
            "max_ms": 1e3 * float(lat.max()), "over_cutoff": int((lat > SEARCH_CUTOFF_S).sum()),
            "qps_if_stopped_at_searchCutoffMs": float(threads / clamped.mean()) if clamped.mean() > 0 else None,
            "qps_measured": n / wall}


def run_reference(args, rank, world):
    """CPU arm: the oracle restatement of milli, one query per thread (the reference's own concurrency model), a bounded sample per step."""
    if rank != 0:
        return
    from meilisearch_b200.tokenizer import TokenBatch

    img, _, emb, _ = build_workload(args, 0, world)
    o = oracle_for(img, emb)
    sample = min(args.batch, args.cpu_sample)
    threads = cpu_threads()
    n_b = args.distinct_batches
    qs = [TokenBatch(img.synthetic_queries(args.batch, seed=i)[:sample]) for i in range(n_b)]
    vs = None
    if args.mode == "hybrid":
        vs = [np.random.default_rng(77 + i).standard_normal((args.batch, DIM), dtype=np.float32)[:sample].copy() for i in range(n_b)]
    for w in range(args.warmup):
        oracle_run(o, args, qs[w % n_b], None if vs is None else vs[w % n_b], threads)
    t0 = time.perf_counter()
    lat = []
    for k in range(args.steps):
        r = oracle_run(o, args, qs[(args.warmup + k) % n_b], None if vs is None else vs[(args.warmup + k) % n_b], threads)
        lat.append(r.seconds.copy())
    dt = time.perf_counter() - t0
    lat = np.concatenate(lat)
    qps = sample * args.steps / dt
    out = {
        "impl": "reference", "metric": metric_name(args), "value": qps, "unit": "queries/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64" if args.mode == "keyword" else "u64+f32", "data": "synthetic",
        "config": workload_config(args, img),
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": threads, "kind": "port",
                         "sample": f"each step = the first {sample} queries of a {args.batch}-query batch of the timed workload, {threads} threads (one query per thread) "
                                   f"of {os.cpu_count()} host threads" + ("; vector stage = one blocked exact scan per step shared by the step's queries" if args.mode == "hybrid" else "") +
                                   "; CPU restatement of milli, not milli itself",
                         "latency": latency_summary(lat, threads, dt, sample * args.steps)},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------ parity
def compare_results(got, want, n, *, sim_rtol=1e-4):
    """docids, score tuples and candidate counts of n queries; returns a dict of mismatch counts"""
    L = min(got.documents_ids.shape[1], want.docids.shape[1])
    nh_g, nh_w = got.n_hits[:n].astype(np.int64), want.n_hits[:n].astype(np.int64)
    pos = np.arange(L)[None, :]
    live = pos < np.minimum(nh_g, nh_w)[:, None]
    ids_eq = (got.documents_ids[:n, :L] == want.docids[:n, :L]) | ~live
    q_ids_ok = ids_eq.all(axis=1) & (nh_g == nh_w)
    ns_eq = (got.n_scores[:n, :L] == want.n_scores[:n, :L]) | ~live
    S = got.score_kind.shape[2]
    spos = np.arange(S)[None, None, :]
    slive = live[:, :, None] & (spos < got.n_scores[:n, :L, None])
    kind_eq = (got.score_kind[:n, :L] == want.score_kind[:n, :L]) | ~slive
    is_vec = (got.score_kind[:n, :L] == 7) & slive
    rank_eq = ((got.score_rank[:n, :L] == want.score_rank[:n, :L]) & (got.score_max[:n, :L] == want.score_max[:n, :L])) | ~slive | is_vec
    gs, ws = got.score_sim[:n, :L].astype(np.float64), want.score_sim[:n, :L].astype(np.float64)
    sim_ok = (np.abs(gs - ws) <= sim_rtol * np.maximum(np.abs(ws), 1e-12) + 2e-6) | ~is_vec
    q_scores_ok = ns_eq.all(axis=1) & kind_eq.all(axis=(1, 2)) & rank_eq.all(axis=(1, 2)) & sim_ok.all(axis=(1, 2))
    cand_ok = got.n_candidates[:n] == want.n_candidates[:n]
    return {"checked": int(n), "docid_mismatches": int((~q_ids_ok).sum()), "score_tuple_mismatches": int((~q_scores_ok & q_ids_ok).sum()),
            "candidate_count_mismatches": int((~cand_ok).sum()), "_bad_ids": np.nonzero(~q_ids_ok)[0]}


def hybrid_tolerated(got, want, q, tol=1e-4):
    """a hybrid docid difference is tolerated when, at every differing position, the two sides' ranking scores agree within tol
    (documents whose weighted scores tie within the float tolerance of the vector similarity may swap)"""
    def gscore(res, i):
        rk, mx, sem = 1, 1, None
        for s in range(int(res.n_scores[q, i])):
            if res.score_kind[q, i, s] == 7:
                sem = max(0.0, float(res.score_sim[q, i, s]))
            else:
                rk = max(rk - 1, 0) * int(res.score_max[q, i, s]) + int(res.score_rank[q, i, s])
                mx *= int(res.score_max[q, i, s])
        return sem if sem is not None else rk / mx
    if got.n_hits[q] != want.n_hits[q]:
        return False
    for i in range(int(got.n_hits[q])):
        if got.documents_ids[q, i] != want.docids[q, i] and abs(gscore(got, i) - gscore(want, i)) > tol:
            return False
    return True


def run_parity(args, ix, img, emb, batches, vecs):
    n = args.batch if args.parity == 0 else min(args.batch, args.parity)
    tb = batches[0].head(n) if n < args.batch else batches[0]
    o = oracle_for(img, emb)
    threads = os.cpu_count() or 1
    t = time.time()
    out = {}
    got = ix.search().query(tb).scoring_strategy("detailed").execute()
    want = o.search_batch(tb, scoring="detailed", n_threads=threads)
    kw = compare_results(got, want, n)
    kw.pop("_bad_ids")
    kw["oracle_seconds"] = round(time.time() - t, 1)
    out["keyword_detailed"] = kw
    if args.mode == "hybrid":
        t = time.time()
        v = np.ascontiguousarray(vecs[0][:n])
        got = ix.search().query(tb).semantic(v).execute_hybrid(0.5)
        want = o.search_batch(tb, vectors=v, hybrid=True, semantic_ratio=0.5, n_threads=threads)
        hy = compare_results(got, want, n)
        bad = hy.pop("_bad_ids")
        hy["docid_mismatches_beyond_1e-4_score_ties"] = int(sum(0 if hybrid_tolerated(got, want, int(q)) else 1 for q in bad))
        hy["semantic_hit_count_mismatches"] = int((got.semantic_hit_count[:n] != want.semantic_hits[:n]).sum())
        hy["oracle_seconds"] = round(time.time() - t, 1)
        out["hybrid"] = hy
    out["checked"] = n
    out["mismatches"] = kw["docid_mismatches"] + kw["score_tuple_mismatches"] + kw["candidate_count_mismatches"] + \
        (out["hybrid"]["docid_mismatches_beyond_1e-4_score_ties"] + out["hybrid"]["score_tuple_mismatches"] if "hybrid" in out else 0)
    return out, o


# ------------------------------------------------------------------------------------------------ cfg 5: corpus-sharded vector stage
def sharded_vector_stage(args, ix, rank, world, local_rank):
    """SURVEY §8(e) / cfg 5, vector side: the embedding matrix is partitioned by contiguous docid range, 12.5 M x 768 fp16 rows per
    GPU (100 M at 8 GPUs).  Every rank scans its shard for the SAME 1024 queries (tcgen05 GEMM + fused top-100), the per-shard
    top-100 lists are exchanged with one ncclAllGather issued by the library on its own stream and merged on the device
    (b200_nns_batch_sharded).  First a 1 M-row subsample is checked against the single-shard CPU oracle."""
    import torch
    import torch.distributed as dist

    from corpus.pyindexgen import synthetic_embeddings_f16

    out = {}
    try:
        dev = torch.device("cuda", local_rank)
        uid = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            uid.copy_(torch.from_numpy(ix.comm_unique_id()).to(dev))
        dist.broadcast(uid, 0)
        ix.comm_init(rank, world, uid.cpu().numpy())
        # (1) correctness on a 1 M-row subsample: merged top-20 == the oracle's scan of all rows
        sub = 1_000_000 // world
        ix.set_embeddings(synthetic_embeddings_f16(sub, DIM, seed=0xE5BED, first_row=rank * sub), np.arange(rank * sub, (rank + 1) * sub, dtype=np.uint32))
        qc = np.random.default_rng(5).standard_normal((32, DIM), dtype=np.float32)
        ids, dst, cnt = ix.nns_by_vector_sharded(qc, 20)
        if rank == 0:
            try:  # rank 0 alone is here: whatever happens, it must reach the collectives below like the other ranks
                o = oracle_small()
                o.set_embeddings(synthetic_embeddings_f16(sub * world, DIM, seed=0xE5BED))
                bad = 0
                for i in range(len(qc)):
                    oid, od = o.nns(qc[i], 20)
                    same = list(ids[i, : cnt[i]]) == list(oid)
                    close = cnt[i] == len(oid) and np.allclose(dst[i, : cnt[i]], od, rtol=1e-4, atol=2e-5)
                    bad += 0 if (same or close) else 1
                out["subsample_check"] = {"rows_total": sub * world, "queries": len(qc), "k": 20, "mismatches": bad}
            except Exception as e:
                out["subsample_check"] = {"error": repr(e)}
        # (2) cfg 5 shape, weak scaling
        n = args.shard_rows
        ix.set_embeddings(synthetic_embeddings_f16(n, DIM, seed=0xE5BED, first_row=rank * n), np.arange(rank * n, (rank + 1) * n, dtype=np.uint32))
        q = np.random.default_rng(7).standard_normal((1024, DIM), dtype=np.float32)
        for _ in range(2):
            ix.nns_by_vector_sharded(q, 100)
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        reps = 5
        for _ in range(reps):
            ids, dst, cnt = ix.nns_by_vector_sharded(q, 100)
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        out.update({"workload": f"corpus-sharded by docid range: {world} x ({n} x {DIM} fp16) rows, the same 1024 queries on every rank, top-100; "
                                f"one ncclAllGather of {world} x 1024 x 100 x (u32 docid, f32 distance) inside the library + device merge",
                    "rows_total": n * world, "ms_per_batch": 1e3 * float(dt[0]) / reps, "queries_per_s": 1024 * reps / float(dt[0]),
                    "all_sorted": bool((np.diff(dst[:, : int(cnt.min())], axis=1) >= 0).all())})
    except Exception as e:  # secondary measurement
        out["error"] = repr(e)
    return out


def oracle_small():
    from corpus.pyindexgen import IndexImage
    from oracle.pyoracle import OracleIndex

    img = IndexImage(1)
    img.add_text(0, 0, "placeholder")
    return OracleIndex(img.build())


# ------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--mode", default="hybrid", choices=["hybrid", "keyword"])
    ap.add_argument("--docs", type=int, default=10_000_000)
    ap.add_argument("--vocab", type=int, default=1_500_000)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--distinct-batches", type=int, default=4)
    ap.add_argument("--cpu-sample", type=int, default=128, help="queries per CPU step (bounded sample of the batch)")
    ap.add_argument("--parity", type=int, default=0, help="queries of the parity check (0 = the whole batch)")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary vector-stage measurements")
    ap.add_argument("--shard-rows", type=int, default=12_500_000, help="embedding rows per GPU of the corpus-sharded stage (N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the search result of the last timed step as DIR/<array>.npy (rank 0)")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    import meilisearch_b200 as mb

    mb.load_library()  # fails loudly if the CUDA extension is missing
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU path; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    # ranks share the host: keep the per-rank worker pools inside the machine's cores
    os.environ.setdefault("B200_HOST_THREADS", str(max(8, min(32, (os.cpu_count() or 64) // max(1, world)))))
    if world >= 4:
        os.environ.setdefault("B200_POOL_SPIN_US", "30")  # idle workers of many ranks must not spin on each other's cores
    img, batches, emb, vecs = build_workload(args, rank, world)
    t = time.time()
    ix = mb.Index(img, device=local_rank)
    if emb is not None:
        ix.set_embeddings(emb)
    log(f"[rank {rank}] staged {ix.stats()['hbm_bytes_staged'] / 1e6:.0f} MB to HBM in {time.time() - t:.1f}s")
    hybrid = args.mode == "hybrid"

    def step(i):
        s = ix.search().query(batches[i % len(batches)])
        if hybrid:
            return s.semantic(vecs[i % len(vecs)]).execute_hybrid(0.5)
        return s.execute()

    sampler = ClockSampler(local_rank)
    sampler.start()
    for w in range(args.warmup):
        res = step(w)
    os.environ["B200_KERNEL_TIMERS"] = "0"  # the e2e region runs as production would: no per-kernel event records
    ix.reset_stats()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    lat = []
    for k in range(args.steps):
        ts = time.perf_counter()
        res = step(args.warmup + k)
        lat.append(time.perf_counter() - ts)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    if world > 1:
        dist.barrier()
    clocks = sampler.stop((t0, t0 + wall))
    st_e2e = ix.stats()
    n_ok = int((res.status == 0).sum())
    # second timed region, software pipeline off (one lane): kernels of different lanes no longer overlap, so the CUDA-event
    # intervals are clean.  `value` and the roofline come from this pass; `e2e` from the pipelined pass above.
    os.environ["B200_SINGLE_LANE"] = "1"
    os.environ["B200_KERNEL_TIMERS"] = "1"
    os.environ["B200_HYBRID_SERIAL"] = "1"  # vector stage after the keyword stage: no overlapping kernel intervals in this pass
    step(args.warmup)
    ix.reset_stats()
    torch.cuda.synchronize()
    for k in range(args.steps):
        step(args.warmup + k)
    torch.cuda.synchronize()
    del os.environ["B200_SINGLE_LANE"]
    del os.environ["B200_HYBRID_SERIAL"]
    st = ix.stats()
    K = st["kernels"]
    dev_s = (st["device_ms"] + K["lev_match"]["ms"] + K["vec_gemm_topk"]["ms"] + K["vec_dist"]["ms"] + K["topk_select"]["ms"]) / 1e3
    if world > 1:
        tt = torch.tensor([wall, dev_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        wall, dev_s = float(tt[0]), float(tt[1])
    total_q = args.batch * args.steps * world
    if rank != 0:
        # the other ranks go straight to the corpus-sharded stage and meet rank 0 there (it first checks parity on its replica)
        if world > 1 and not args.no_extras:
            del emb
            sharded_vector_stage(args, ix, rank, world, local_rank)
        if world > 1:
            dist.destroy_process_group()
        return

    # roofline of the dominant kernel
    peaks = measured_peaks()
    kern = {k: v for k, v in K.items() if v["count"]}
    dom = max(kern, key=lambda k: kern[k]["ms"])
    tot_ms = max(1e-9, sum(x["ms"] for x in kern.values()))

    def roof(name):
        d = kern[name]
        per_launch_ms = d["ms"] / d["count"]
        if name == "vec_gemm_topk":
            flops = 2.0 * args.batch * float(img.n_docs) * DIM
            ach = flops / (per_launch_ms * 1e-3) / 1e12 if per_launch_ms > 0 else 0.0
            return {"bound": "tensor", "kernel": name, "achieved": ach, "peak": peaks["tensor"][0], "peak_source": peaks["tensor"][1], "unit": "TFLOP/s",
                    "frac": ach / peaks["tensor"][0], "traffic": ncu_traffic(name), "launches": int(d["count"]), "avg_launch_ms": per_launch_ms,
                    "algorithmic_flops_per_launch": flops, "algorithmic_bytes_per_launch": d["bytes"] / d["count"]}
        ach = (d["bytes"] / d["count"]) / (per_launch_ms * 1e-3) / 1e9 if per_launch_ms > 0 else 0.0
        return {"bound": "hbm", "kernel": name, "achieved": ach, "peak": peaks["hbm"][0], "peak_source": peaks["hbm"][1], "unit": "GB/s",
                "frac": ach / peaks["hbm"][0], "traffic": ncu_traffic(name), "launches": int(d["count"]), "avg_launch_ms": per_launch_ms,
                "algorithmic_bytes_per_launch": d["bytes"] / d["count"]}

    roofline = roof(dom)
    # a "launch" of the keyword kinds is the group of kernels of that kind in one device step, timed by one pair of CUDA events on the
    # lane's stream (eval_paths = eval_dp_kernel of every shared-memory class + walk_kernel); `traffic` is ncu's DRAM bytes per such group
    roofline["launch_unit"] = "one device step's kernels of this kind (eval_paths: eval_dp_kernel x classes + walk_kernel)"
    roofline["kernel_time_share"] = {k: round(v["ms"] / tot_ms, 4) for k, v in kern.items()}
    roofline["all_kernels"] = {k: {"frac": round(roof(k)["frac"], 4), "unit": roof(k)["unit"], "achieved": round(roof(k)["achieved"], 1),
                                   "ms_per_step": round(kern[k]["ms"] / args.steps, 3)} for k in kern}

    # parity on the whole first batch (checker only; not in any timed region); the multi-GPU runs check a sample (the full batch is
    # checked by the N = 1 run of the same code on the same corpus)
    if world > 1 and args.parity == 0:
        args.parity = 64
    t = time.time()
    parity, o = run_parity(args, ix, img, emb, batches, vecs)
    log(f"parity ({time.time() - t:.1f}s): {parity}")

    # CPU baseline: oracle on a bounded sample of a timed batch, fixed thread count
    sample = min(args.batch, args.cpu_sample)
    threads = cpu_threads()
    bi = args.warmup % len(batches)
    sq = batches[bi].head(sample)
    sv = None if vecs is None else np.ascontiguousarray(vecs[bi][:sample])
    tc = time.perf_counter()
    r = oracle_run(o, args, sq, sv, threads)
    dtc = time.perf_counter() - tc
    cpu = {"value": sample / dtc, "unit": "queries/s", "cores": threads, "kind": "port",
           "sample": f"the first {sample} queries of a timed {args.batch}-query batch, {threads} threads (one query per thread) of {os.cpu_count()} host threads"
                     + ("; vector stage = one blocked exact scan shared by the sample's queries" if hybrid else "") + "; CPU restatement of milli, not milli itself",
           "latency": latency_summary(r.seconds, threads, dtc, sample)}
    del o

    out = {
        "metric": metric_name(args), "value": total_q / dev_s, "unit": "queries/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dev_s / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64" if not hybrid else "u64+f16/f32", "data": "synthetic",
        "config": workload_config(args, img),
        "e2e": {"value": total_q / wall, "unit": "queries/s", "ms_per_step": 1e3 * wall / args.steps, "p50_batch_ms": 1e3 * float(np.median(lat)),
                "h2d_bytes_per_step": int(st_e2e["h2d_bytes"] / args.steps), "d2h_bytes_per_step": int(st_e2e["d2h_bytes"] / args.steps),
                "device_steps_per_batch": st_e2e["device_steps"] / args.steps, "lanes": os.environ.get("B200_DRIVERS", "4") + "x" + os.environ.get("B200_LANES_PER_DRIVER", "1")},
        "gpu_launches": int(st_e2e["kernel_launches"]),
        "clocks": clocks,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "parity": parity,
        "queries_ok": n_ok,
        "host_ms_per_step": {k: v / args.steps for k, v in st_e2e["host_ms"].items()},
        "engine": {"deferred_activations_per_step": st_e2e["deferred"] / args.steps, "arena_peak_bytes": int(st_e2e["arena_peak_bytes"]),
                   "eval_class_tiles": st["eval_class_tiles"], "eval_class_launches": st["eval_class_launches"]},
        "algorithmic_bytes_per_step": {"posting": int(st["posting_bytes"] / args.steps), "matrix": int(st["matrix_bytes"] / args.steps),
                                       "dictionary": int(st["dictionary_bytes"] / args.steps), "vector": int(st["vector_bytes"] / args.steps)},
    }

    if world > 1 and not args.no_extras:
        del emb
        emb = None
        out["vector_stage_sharded"] = sharded_vector_stage(args, ix, rank, world, local_rank)
    if not args.no_extras and world == 1:
        extras(args, ix, img, emb, batches, out, peaks)
    if args.dump_outputs:  # res: the last step of the e2e pass, which runs as production does
        dump_outputs(res, args.dump_outputs)
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


RESULT_ARRAYS = ("documents_ids", "n_hits", "n_scores", "score_kind", "score_rank", "score_max", "score_sim", "n_candidates",
                 "semantic_hit_count", "status", "degraded", "used_negative_operator")
DUMP_LIMIT_BYTES = 60 << 20  # array data; with the .npy headers and query_index.npy the files stay below 64 MB


def dump_outputs(res, out_dir):
    """The arrays of a SearchResult as out_dir/<name>.npy, so that two builds can be compared output for output: score_sim stays
    float32, the integer arrays become float64 (exact: every value is below 2**53).  A batch whose arrays exceed 64 MB is cut to a
    seeded sample of its queries, whose row numbers go to query_index.npy."""
    n = len(res.n_hits)
    per_query = sum((4 if name == "score_sim" else 8) * getattr(res, name)[:1].size for name in RESULT_ARRAYS)
    keep = min(n, DUMP_LIMIT_BYTES // per_query)
    rows = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name in RESULT_ARRAYS:
        a = getattr(res, name)[rows]
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))
    if keep < n:
        np.save(os.path.join(out_dir, "query_index.npy"), rows.astype(np.float64))


def extras(args, ix, img, emb, batches, out, peaks):
    """secondary lines: keyword-only throughput of the same corpus, and the vector stage alone (cfg 4 shapes on the staged matrix)"""
    try:
        os.environ["B200_KERNEL_TIMERS"] = "0"
        if args.mode == "hybrid":
            for w in range(2):
                ix.search().query(batches[w % len(batches)]).execute()
            t0 = time.perf_counter()
            reps, lat = 4, []
            for i in range(reps):
                t1 = time.perf_counter()
                ix.search().query(batches[i % len(batches)]).execute()
                lat.append(time.perf_counter() - t1)
            wall = time.perf_counter() - t0
            out["keyword_only"] = {"workload": "the same batches through Search::execute (ScoringStrategy::Skip), end to end from host buffers",
                                   "e2e_queries_per_s": args.batch * reps / wall, "p50_batch_ms": 1e3 * float(np.median(lat))}
        os.environ["B200_KERNEL_TIMERS"] = "1"
        if emb is None:
            return
        n = int(emb.shape[0])
        rng = np.random.default_rng(0xE5BED)
        q = rng.standard_normal((8, DIM), dtype=np.float32)
        for _ in range(3):
            ix.nns_by_vector(q[:1], 100)
        ix.reset_stats()
        tv = time.perf_counter()
        reps = 10
        for i in range(reps):
            ix.nns_by_vector(q[i % 8: i % 8 + 1], 100)
        wall_v = time.perf_counter() - tv
        sv = ix.stats()["kernels"]["vec_dist"]
        gbs = sv["bytes"] / (sv["ms"] * 1e-3) / 1e9
        out["vector_stage"] = {"workload": f"cfg4: {n} x {DIM} fp16 rows, B=1 cosine top-100", "kernel": "vec_dist",
                               "avg_launch_ms": sv["ms"] / sv["count"], "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peaks["hbm"][0],
                               "e2e_queries_per_s": reps / wall_v, "e2e_ms_per_query": 1e3 * wall_v / reps}
        qb = rng.standard_normal((1024, DIM), dtype=np.float32)
        for _ in range(2):
            ix.nns_by_vector(qb, 100)
        ix.reset_stats()
        tv = time.perf_counter()
        reps = 4
        for i in range(reps):
            ix.nns_by_vector(qb, 100)
        wall_b = time.perf_counter() - tv
        sg = ix.stats()["kernels"]["vec_gemm_topk"]
        if sg["count"]:
            ms = sg["ms"] / sg["count"]
            tflops = 2.0 * 1024 * n * DIM / (ms * 1e-3) / 1e12
            out["vector_stage_batched"] = {"workload": f"cfg4 batched: 1024 queries x ({n} x {DIM} fp16), cosine top-100, fp16 operands / fp32 accumulate",
                                           "kernel": "vec_gemm_topk (+vec_merge)", "avg_launch_ms": ms,
                                           "roofline": {"bound": "tensor", "achieved": tflops, "peak": peaks["tensor"][0], "peak_source": peaks["tensor"][1],
                                                        "unit": "TFLOP/s", "frac": tflops / peaks["tensor"][0]},
                                           "kernel_queries_per_s": 1024 / (ms * 1e-3), "e2e_queries_per_s": 1024 * reps / wall_b}
    except Exception as e:  # the headline number must not die with a secondary one
        out["extras_error"] = str(e)


if __name__ == "__main__":
    main()
