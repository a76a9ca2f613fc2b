#!/usr/bin/env python
"""bench.py — the BASELINE.json metric: queries/sec (+ decoded-postings/sec) on the synthetic Zipfian index.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload and2|or10|tree8|and2l] [--sub or10,tree8,and2l|none]

One "step" = one pass of the hot path over one batch of synthetic queries.  Default workload (BASELINE.json configs[1]): a batch of
1000 2-term AND queries on the 100M-doc Zipfian synthetic index, GOOGLE codec, DocumentsOnly.  The same run also measures configs[2]
(10-term OR, BM25 top-100, LUCENE) and configs[3] (8-term AND/OR/NOT trees) at a reduced step count and reports them under
`workloads` (value, e2e, roofline, parity), so every driver record carries all three at every N.

  value      whole-job queries/s with the index resident in HBM and results left in HBM (kernels only), CUDA events, max over ranks
  e2e        the same through the public C-ABI call (trn_exec_batch) with HOST buffers: plans H2D + every matched docID (or top-k) D2H
             — the number to quote as throughput
  roofline   of the fused exec kernel: SURVEY 8(d) algorithmic bytes (sum of the queries' term chunks + emitted bytes) / event time
  cpu_baseline / parity   the reference's own exec_query (oracle/_ref) on the host cores over a bounded sample of the same batch; its
             results double as the full-size checker of the GPU batch (N = 1: this rank's results; N > 1: per-query match counts and
             docID checksums all-gathered from every rank / the merged top-k, checked on rank 0 against the UNSHARDED reference)

N > 1: the docID space is partitioned across ranks (strong scaling: the same 100M-doc index, each rank holds the postings of its docID
range, SURVEY.md 8e).  Docs-only results need no exchange (shard order == docID order); the top-k workload merges per-shard top-k with
ONE all-gather (NCCL) + a merge kernel.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

WORKLOADS = {
    "and2": dict(codec=0, mode=0, desc="1000 x 2-term AND, DocumentsOnly, GOOGLE codec"),
    "or10": dict(codec=1, mode=2, desc="10-term OR, BM25 top-100, LUCENE codec"),
    "tree8": dict(codec=0, mode=0, desc="8-term mixed AND/OR/NOT trees, DocumentsOnly, GOOGLE codec"),
    "and2l": dict(codec=1, mode=0, desc="1000 x 2-term AND, DocumentsOnly, LUCENE codec (the headline batch on the other postings format)"),
}
BYTES_PER_POSTING = {0: 4.54, 1: 1.95}  # measured on the synthetic index (with positions): GOOGLE inline hits / LUCENE index file only


def gen_queries(workload: str, nq: int, nterms: int, seed: int = 0xC0FFEE):
    """term ranks drawn ~ 1/r (query-log-like), BASELINE.md section 3"""
    rng = np.random.default_rng(seed)
    w = 1.0 / np.arange(1, nterms + 1)
    w /= w.sum()
    names = [f"t{r:04d}" for r in range(1, nterms + 1)]
    out, ranks = [], []
    for _ in range(nq):
        if workload in ("and2", "and2l"):
            t = rng.choice(nterms, size=2, replace=False, p=w)
            out.append(f"{names[t[0]]} AND {names[t[1]]}")
        elif workload == "or10":
            t = rng.choice(nterms, size=10, replace=False, p=w)
            out.append(" OR ".join(names[i] for i in t))
        else:
            t = rng.choice(nterms, size=8, replace=False, p=w)
            n = [names[i] for i in t]
            k = int(rng.integers(0, 4))
            out.append([
                f"({n[0]} OR {n[1]}) AND ({n[2]} OR {n[3]}) AND {n[4]} NOT ({n[5]} OR {n[6]} OR {n[7]})",
                f"{n[0]} AND {n[1]} AND {n[2]} NOT {n[3]} NOT {n[4]}",
                f"({n[0]} AND {n[1]}) OR ({n[2]} AND {n[3]}) OR ({n[4]} AND {n[5]}) NOT {n[6]} NOT {n[7]}",
                f"{n[0]} AND ({n[1]} OR {n[2]} OR {n[3]}) NOT ({n[4]} AND {n[5]}) AND ({n[6]} OR {n[7]})",
            ][k])
        ranks.append(t)
    return out, ranks


def synth_dfs(ndocs: int, nterms: int, min_df: int = 1000) -> np.ndarray:
    """document frequencies of the UNSHARDED synthetic index (closed form of the generator)"""
    return np.array([min(ndocs, max(min_df, ndocs // (2 * r))) for r in range(1, nterms + 1)], dtype=np.int64)


def config_of(args, wl, world: int) -> dict:
    """what the job measures — identical in the product arm and the reference arm (no measured quantities in here)"""
    est = float(synth_dfs(args.ndocs, args.nterms).sum()) * BYTES_PER_POSTING[wl["codec"]] / max(1, world)
    l2 = (f"inputs larger than L2: ~{est / 1e6:.0f} MB of index per GPU vs 126 MB L2, no flush between steps" if est > 126e6
          else f"TEST SIZE: ~{est / 1e6:.0f} MB of index per GPU fits the 126 MB L2")
    return {"workload": f"{wl['desc']}; {args.ndocs} docs, {args.nterms} terms, Zipf(1) df, batch {args.nq}, seed 0xC0FFEE",
            "codec": "GOOGLE" if wl["codec"] == 0 else "LUCENE",
            "docid_sharding": f"{world} x contiguous docID range" if world > 1 else "none", "l2": l2}


def metric_name(workload: str) -> str:
    return "queries/sec (batched 2-term AND, 100M-doc Zipfian synthetic index)" if workload == "and2" else f"queries/sec ({workload})"


def host_info() -> dict:
    model = ""
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    try:
        usable = len(os.sched_getaffinity(0))
    except AttributeError:
        usable = os.cpu_count() or 1
    return {"nproc": os.cpu_count() or 1, "usable_cores": usable, "cpu_model": model}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md clocks line)"""

    def __init__(self, device: int):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 7:
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel per 1000-query batch, from the committed ncu --set full capture
    of this same command (profiles/traffic.json, values copied from the ncu summaries it names); None if not captured"""
    p = ROOT / "profiles" / "traffic.json"
    if p.exists():
        try:
            return json.loads(p.read_text()).get(kernel)
        except Exception:
            return None
    return None


def numa_bind(local_rank: int, world: int) -> dict:
    """pin this rank's threads (and with them its first-touch pinned allocations) to the NUMA node its GPU hangs off; the node's cores
    are split between the ranks that share it.  Eight unbound ranks on a two-socket host had their result copies cross the socket link
    (SCALE_r01: e2e at 8 GPUs below 4 GPUs)."""
    out = {"bound": False}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True, timeout=20).stdout.split()
        node_of = []
        for bus in q:
            p = Path("/sys/bus/pci/devices") / bus.lower()[-12:] / "numa_node"
            node_of.append(int(p.read_text()) if p.exists() else -1)
        node = node_of[local_rank]
        if node < 0:
            return out
        cpus = []
        for part in (Path("/sys/devices/system/node") / f"node{node}" / "cpulist").read_text().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        peers = [r for r in range(min(world, len(node_of))) if node_of[r] == node]
        share = cpus[peers.index(local_rank)::len(peers)] if local_rank in peers and len(peers) > 1 else cpus
        os.sched_setaffinity(0, set(share))
        out = {"bound": True, "numa_node": node, "cores": len(share)}
    except Exception as e:  # binding is an optimisation, never a reason to fail the bench
        out["error"] = repr(e)[:120]
    return out


def full_size_parity(res, mode, k, counts, sums, tid, tsc, n):
    """the reference run of the cpu_baseline leg doubles as the full-size checker of the GPU batch `res` (same index bytes, same
    queries): per-query match counts and docID checksums (DocumentsOnly) / counts and top-k scores (top-k mode, 1e-5 relative)"""
    import trinity_b200 as tb
    out = {"queries_checked": int(n), "match_counts_equal": bool(np.array_equal(np.asarray(res.match_counts[:n], np.uint64), counts[:n]))}
    if mode == tb.MODE_DOCS_ONLY:
        got = res.checksums()[:n]  # exact in uint64; a compact result is replayed through trn_result_decode first
        out["docid_checksums_equal"] = bool(np.array_equal(got, sums[:n]))
    elif mode == tb.MODE_SCORED_TOPK:
        worst = 0.0
        for q in range(n):
            d, s = res.query(q)
            want = tsc[q][: len(s)]
            if len(s) != int(min(k, counts[q])):
                worst = float("inf")
                break
            if len(s):
                worst = max(worst, float(np.max(np.abs(np.asarray(s, np.float64) - want) / np.maximum(np.abs(want), 1e-30))))
        out["topk_scores_max_rel_err"] = worst
        out["topk_scores_within_1e-5"] = bool(worst <= 1e-5)
    return out


def sharded_parity(mode, k, n, counts, sums, tsc, g_counts, g_sums, merged_scores):
    """N > 1: `g_counts` / `g_sums` = per-query match counts and docID checksums summed over all ranks (uint64, wrap-around), `merged_scores`
    = the merged [nq, k] top-k scores (padding < 0) — against the UNSHARDED reference run on rank 0"""
    out = {"queries_checked": int(n), "match_counts_equal": bool(np.array_equal(g_counts[:n], counts[:n]))}
    if mode == 0:
        out["docid_checksums_equal"] = bool(np.array_equal(g_sums[:n], sums[:n]))
    else:
        worst = 0.0
        for q in range(n):
            s = merged_scores[q]
            s = s[s >= 0]
            want = tsc[q][: len(s)]
            if len(s) != int(min(k, counts[q])):
                worst = float("inf")
                break
            if len(s):
                worst = max(worst, float(np.max(np.abs(np.asarray(s, np.float64) - want) / np.maximum(np.abs(want), 1e-30))))
        out["topk_scores_max_rel_err"] = worst
        out["topk_scores_within_1e-5"] = bool(worst <= 1e-5)
    return out


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, res, mode: int):
    """what a caller of the timed path receives from its last step, as float64 .npy files (exact for docIDs, counts and 32-bit halves of
    the checksums): per-query match counts and docID checksums, and the matched docIDs themselves, or a fixed seeded sample of their
    positions in the concatenated result when they exceed DUMP_BYTES; top-k mode: the [nq, k] docIDs and scores (-1 = no entry)"""
    import trinity_b200 as tb
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    counts = np.asarray(res.match_counts[: res.nq], np.uint64)
    np.save(d / "match_counts.npy", counts.astype(np.float64))
    if mode == tb.MODE_SCORED_TOPK:
        ids, sc = np.full((res.nq, res.k), -1.0), np.full((res.nq, res.k), -1.0)
        for q in range(res.nq):
            qd, qs = res.query(q)
            ids[q, : len(qd)], sc[q, : len(qs)] = qd, qs
        np.save(d / "topk_docids.npy", ids)
        np.save(d / "topk_scores.npy", sc)
        return
    sums = res.checksums()
    np.save(d / "docid_checksums_hi.npy", (sums >> np.uint64(32)).astype(np.float64))
    np.save(d / "docid_checksums_lo.npy", (sums & np.uint64(0xFFFFFFFF)).astype(np.float64))
    total = int(counts.sum())
    cap = (DUMP_BYTES - 64 * res.nq) // 16   # sampled docIDs and their positions, 8 bytes each
    pos = np.arange(total, dtype=np.int64) if total <= cap else np.sort(np.random.default_rng(0x5EED).choice(total, cap, replace=False))
    out = np.empty(len(pos), np.float64)
    ends = np.cumsum(counts.astype(np.int64))
    buf = np.empty(max(1, int(counts.max()) if res.nq else 1), np.uint32)
    lo = 0
    for q in range(res.nq):
        hi = int(np.searchsorted(pos, ends[q]))
        if hi > lo:
            qd = res.query(q)[0] if res.docids is not None else res.decode_query(q, buf)
            out[lo:hi] = qd[pos[lo:hi] - (ends[q] - int(counts[q]))]
        lo = hi
    np.save(d / "docids.npy", out)
    np.save(d / "docids_position.npy", pos.astype(np.float64))


def reference_sample(r, texts, scored, k, cores, budget_s):
    """run the reference's exec_query over a prefix of the batch sized by a probe for ~budget_s of host time"""
    probe = min(len(texts), 64)
    el, *_ = r.exec_batch(texts[:probe], scored, k, cores)
    n = max(min(32, len(texts)), min(len(texts), int(budget_s * probe / max(el, 1e-9))))
    el, counts, sums, tid, tsc = r.exec_batch(texts[:n], scored, k, cores)
    return n, el, counts, sums, tid, tsc


# ======================================================================================================================= product arm
class Job:
    def __init__(self, args):
        import torch
        import torch.distributed as dist

        self.args, self.torch, self.dist = args, torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device — trinity_b200 has no CPU path (use --impl reference for the CPU arm)")
        self.numa = numa_bind(self.local_rank, self.world) if not args.no_numa_bind else {"bound": False}
        torch.cuda.set_device(self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        self.stream = torch.cuda.current_stream()
        self.indexes = {}  # codec -> (synth shard, GpuIndexSource, build_s, upload_s)
        self.refs = {}     # codec -> reference index over the UNSHARDED bytes (rank 0 only)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def index(self, codec):
        import trinity_b200 as tb
        from trinity_b200.sharded import shard_range
        if codec not in self.indexes:
            a = self.args
            t0 = time.time()
            lo, hi = shard_range(a.ndocs, self.rank, self.world)
            threads = max(1, len(os.sched_getaffinity(0)))
            synth = tb.SynthIndex(codec, a.ndocs, a.nterms, threads=threads, doc_range=(lo, hi))
            build_s = time.time() - t0
            g = tb.GpuIndexSource(self.local_rank)
            g.set_stream(self.stream.cuda_stream)
            t0 = time.time()
            g.upload(codec, np.asarray(synth.index), np.asarray(synth.terms), a.ndocs)
            self.indexes[codec] = (synth, g, build_s, time.time() - t0)
        return self.indexes[codec]

    def drop_index(self, codec):
        if codec in self.indexes:
            self.indexes.pop(codec)[1].close()
        self.refs.pop(codec, None)

    def reference(self, codec):
        """rank 0: the reference's IndexSource over the unsharded index bytes (the shard itself at N = 1)"""
        import trinity_b200 as tb
        sys.path.insert(0, str(ROOT / "tests"))
        from refharness import RefIndex, load_ref
        if codec not in self.refs:
            a = self.args
            synth = self.index(codec)[0] if self.world == 1 else tb.SynthIndex(codec, a.ndocs, a.nterms, threads=max(1, len(os.sched_getaffinity(0))))
            self.refs[codec] = (RefIndex.from_bytes(load_ref(), codec, np.asarray(synth.index), np.asarray(synth.hits), synth.names, np.asarray(synth.terms),
                                                    a.ndocs, synth.sum_hits), synth)
        return self.refs[codec][0]

    def run(self, workload: str, K: int, W: int, cpu_budget_s: float, with_clocks: bool, dump_dir: str | None = None) -> dict:
        import trinity_b200 as tb
        from trinity_b200.sharded import device_view
        torch, dist, args, world, rank = self.torch, self.dist, self.args, self.world, self.rank
        wl = WORKLOADS[workload]
        codec, mode = wl["codec"], wl["mode"]
        synth, g, build_s, upload_s = self.index(codec)
        info = g.info()
        stream = self.stream

        texts, _ = gen_queries(workload, args.nq, args.nterms)
        tdict = tb.TermDictionary(synth.names)
        plans = [tb.parse_query(q, tdict) for q in texts]
        full_df = synth_dfs(args.ndocs, args.nterms)
        # the mode the product calls run in: DocumentsOnly workloads return their matches in the compact encoding unless told otherwise
        emode = tb.MODE_DOCS_COMPACT if (mode == tb.MODE_DOCS_ONLY and args.result_encoding == "compact") else mode
        if mode != tb.MODE_DOCS_ONLY:  # global BM25 weights: df summed over shards == the unsharded df (similarity.h:209-217)
            for p in plans:
                for x in p:
                    if x["kind"] == tb.NODE_TERM and x["term"] != tb.EMPTY_TERM:
                        x["weight"] = tb.bm25_idf(int(full_df[x["term"]]), args.ndocs)
        # full-scan accounting numerator (same for CPU and GPU): sum of term.documents over the UNSHARDED index
        postings_per_batch = int(sum(int(full_df[x["term"]]) for p in plans for x in p if x["kind"] == tb.NODE_TERM and x["term"] != tb.EMPTY_TERM))

        gathered = merged_d = merged_s = None
        if world > 1 and mode == tb.MODE_SCORED_TOPK:
            gathered = (torch.empty((world, args.nq, args.k), dtype=torch.int32, device="cuda"),
                        torch.empty((world, args.nq, args.k), dtype=torch.float32, device="cuda"))
            merged_d = torch.empty((args.nq, args.k), dtype=torch.int32, device="cuda")
            merged_s = torch.empty((args.nq, args.k), dtype=torch.float32, device="cuda")

        def exchange():
            """the ONE exchange step of the sharded path: all-gather of per-shard top-k + merge kernel"""
            if gathered is None:
                return
            dptr, sptr, _ = g.last_topk_device()
            dist.all_gather_into_tensor(gathered[0].view(-1), device_view(dptr, args.nq * args.k, torch.int32))
            dist.all_gather_into_tensor(gathered[1].view(-1), device_view(sptr, args.nq * args.k, torch.float32))
            g.merge_topk(gathered[0].data_ptr(), gathered[1].data_ptr(), world, args.nq, args.k, merged_d.data_ptr(), merged_s.data_ptr())

        # ---------------- warm-up (also sizes every grow-only buffer) ----------------
        packed = g.pack(plans)
        for _ in range(W):
            res = g.exec_batch(plans, emode, args.k, copy=False, packed=packed)
            exchange()
        for _ in range(W):  # the device-resident form has its own (whole-batch) buffers: warm those too
            g.exec_batch_device(plans, emode, args.k, packed=packed)
            exchange()
        matches_per_batch = int(res.match_counts.sum())
        # bytes of one batch's result as it leaves the device: matched docIDs (plain: 4 B each; compact: the encoded segments + their
        # descriptors) or the top-k lists
        out_bytes_per_batch = res.result_bytes() if mode == tb.MODE_DOCS_ONLY else args.nq * args.k * 8

        # ---------------- timed: device-resident ----------------
        sampler = ClockSampler(self.local_rank) if with_clocks else None
        if sampler:
            sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        kern_ms, launches, tms = [], 0, []
        self.barrier()
        ev0.record(stream)
        for _ in range(K):
            g.exec_batch_device(plans, emode, args.k, packed=packed)
            exchange()
        ev1.record(stream)
        self.barrier()
        dev_ms_total = ev0.elapsed_time(ev1)

        # ---------------- timed: end to end through the C ABI with host buffers ----------------
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(K):
            res = g.exec_batch(plans, emode, args.k, copy=False, packed=packed)
            exchange()
            kern_ms.append(res.exec_kernel_ms)
            launches += res.kernel_launches + (1 if gathered is not None else 0)
            tms.append(g.last_timings())
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        clocks = sampler.stop() if sampler else None
        if dump_dir and rank == 0:
            dump_outputs(dump_dir, res, emode)
        # the same end-to-end step with plain 32-bit docIDs out (TRN_MODE_DOCS_ONLY), for comparison with the compact encoding
        plain = None
        if emode != mode:
            for _ in range(2):
                rp = g.exec_batch(plans, mode, args.k, copy=False, packed=packed)
            self.barrier()
            t0 = time.perf_counter()
            for _ in range(K):
                rp = g.exec_batch(plans, mode, args.k, copy=False, packed=packed)
            torch.cuda.synchronize()
            tp = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(tp, op=dist.ReduceOp.MAX)
            plain = {"value": args.nq * K / float(tp[0]), "unit": "queries/s", "d2h_bytes_per_step": int(rp.result_bytes()) + (args.nq + 1) * 8 + args.nq * 8}
            res = g.exec_batch(plans, emode, args.k, copy=False, packed=packed)  # the parity check below reads the compact result

        times = torch.tensor([dev_ms_total / 1e3, e2e_s], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(times, op=dist.ReduceOp.MAX)
        dev_s, e2e_s = float(times[0]), float(times[1])

        # per-rank breakdown of one e2e step (mean over the K steps): where a rank's host-buffer call spends its wall time
        mine = {k2: float(np.mean([t[k2] for t in tms])) for k2 in tms[0]} if tms else {}
        mine["bytes_d2h"] = int(out_bytes_per_batch)
        per_rank = [mine]
        if world > 1:
            box = [None] * world
            dist.all_gather_object(box, mine)
            per_rank = box

        plan_bytes = int(sum(p.nbytes for p in plans))
        d2h = out_bytes_per_batch + (args.nq + 1) * 8 + args.nq * 8
        peak, peak_src = measured_peak()
        kernel_name = "k_exec_docs" if mode == tb.MODE_DOCS_ONLY else ("k_score_flat" if codec == 1 else "k_exec_tiles")
        # the host-buffer path pipelines a set-query batch in chunks (TRN_PIPELINE_CHUNKS, default 4): one fused-kernel launch per chunk
        # (as many as the referenced postings pay for, at most TRN_PIPELINE_CHUNKS = 8: the engine reports what it used)
        nlaunch = max(1, int(round(float(np.mean([t.get("chunks", 1.0) for t in tms]))))) if tms else 1
        k_ms_step = float(np.mean(kern_ms)) if kern_ms else None          # all fused-kernel launches of one step
        k_ms = k_ms_step / nlaunch if k_ms_step else None                 # average duration of ONE launch
        traffic = ncu_traffic(f"{kernel_name}:{workload}") if (world == 1 and args.ndocs == 100_000_000 and args.nq == 1000) else None
        if traffic is not None:
            traffic = int(traffic) // nlaunch  # the capture is per 1000-query batch; the line reports per launch, like `achieved`
        algo_bytes = (int(res.index_bytes_touched) + out_bytes_per_batch) // nlaunch   # algorithmic bytes of ONE launch
        achieved = algo_bytes / (k_ms * 1e-3) / 1e9 if k_ms else None

        line = {
            "metric": metric_name(workload),
            "value": args.nq * K / dev_s,
            "unit": "queries/s",
            "n_gpus": world,
            "steps": K,
            "warmup": W,
            "ms_per_step": dev_s * 1e3 / K,
            "higher_is_better": True,
            "scaling": "strong",
            "vs_baseline": None,
            "dtype": "u32",
            "data": "synthetic",
            "impl": "ours",
            "config": config_of(args, wl, world),
            "index": {"index_bytes_rank0": int(info["index_bytes"]), "directory_bytes_rank0": int(info["directory_bytes"]),
                      "index_build_s": round(build_s, 1), "upload_s": round(upload_s, 1)},
            "decoded_postings_per_s": postings_per_batch * K / dev_s,
            "matches_per_batch_rank0": matches_per_batch,
            "e2e": {"value": args.nq * K / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": plan_bytes, "d2h_bytes_per_step": d2h,
                    "decoded_postings_per_s": postings_per_batch * K / e2e_s, "per_rank_ms": per_rank,
                    "result_encoding": ("compact (TRN_MODE_DOCS_COMPACT: per docID tile a bitmap / bucketed 8-bit offsets / 16-bit offsets / docIDs, whichever is smallest; replayed on the host by trn_result_for_each)"
                                        if emode != mode else ("u32 docIDs" if mode == tb.MODE_DOCS_ONLY else "top-k (docID, score)")),
                    "matched_docids_per_step": matches_per_batch, "plain_u32": plain},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": kernel_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": algo_bytes, "kernel_ms": k_ms, "launches_per_step": nlaunch,
                         "note": "achieved = SURVEY 8(d) algorithmic bytes (every referenced list once per query, skipped blocks included) / kernel time: an EFFECTIVE rate, not HBM utilisation (the kernels skip blocks and are instruction-issue bound); see DESIGN.md section 4"},
        }
        if clocks is not None:
            line["clocks"] = clocks

        # ---------------- reference leg: CPU baseline + full-size parity (rank 0 runs the reference; every rank contributes its results)
        if not args.no_cpu_baseline and not (ROOT / "oracle" / "_ref" / "libtrinity_ref.so").exists():
            line["cpu_baseline"] = line["parity"] = {"skipped": "oracle/_ref (the reference's own code) is not built"}
        elif not args.no_cpu_baseline:
            g_counts = g_sums = m_scores = None
            if world > 1:
                # per-query match counts + docID checksums of THIS rank's shard, summed over ranks (uint64 arithmetic, wrap-around is fine)
                cnt = torch.from_numpy(np.asarray(res.match_counts, np.uint64).astype(np.int64)).cuda()
                if mode == tb.MODE_DOCS_ONLY:
                    sm = torch.from_numpy(res.checksums().view(np.int64).copy()).cuda()
                else:
                    sm = torch.zeros(args.nq, dtype=torch.int64, device="cuda")
                dist.all_reduce(cnt)
                dist.all_reduce(sm)
                g_counts, g_sums = cnt.cpu().numpy().view(np.uint64), sm.cpu().numpy().view(np.uint64)
                if merged_s is not None:
                    m_scores = merged_s.cpu().numpy()
            if rank == 0:
                mine_aff = os.sched_getaffinity(0)
                try:
                    os.sched_setaffinity(0, range(os.cpu_count() or 1))  # the checker may use the whole host: the other ranks idle at the barrier
                except OSError:
                    pass
                cores = len(os.sched_getaffinity(0))
                r = self.reference(codec)
                n, el, counts, sums, tid, tsc = reference_sample(r, texts, mode != 0, args.k, cores, cpu_budget_s)
                os.sched_setaffinity(0, mine_aff)
                cb = {"value": n / el, "unit": "queries/s", "cores": cores, "kind": "reference",
                      "sample": f"first {n} queries of the same batch, one query per host thread ({cores} threads), {el:.2f} s wall",
                      "seconds": el, "host": host_info()}
                try:
                    if world == 1:
                        cb["parity"] = full_size_parity(res, mode, args.k, counts, sums, tid, tsc, n)
                    else:
                        cb["parity"] = sharded_parity(mode, args.k, n, counts, sums, tsc, g_counts, g_sums, m_scores)
                        cb["parity"]["checked"] = f"results of all {world} ranks combined vs the UNSHARDED reference index on rank 0"
                except Exception as e:  # the checker must never take the bench line down
                    cb["parity"] = {"error": repr(e)}
                line["cpu_baseline"] = cb
                line["parity"] = cb["parity"]
            if world > 1:
                self.barrier()
        return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="and2", choices=list(WORKLOADS))
    ap.add_argument("--sub", default="auto", help="workloads measured besides the primary one at a reduced step count: 'or10,tree8,and2l', 'none', 'auto' (= all three for the default primary)")
    ap.add_argument("--ndocs", type=int, default=100_000_000)
    ap.add_argument("--nterms", type=int, default=4096)
    ap.add_argument("--nq", type=int, default=1000)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--cpu-sample", type=int, default=0, help="(reference arm) queries per step (0 = auto)")
    ap.add_argument("--result-encoding", default="compact", choices=["compact", "u32"],
                    help="DocumentsOnly workloads: how the matched docIDs leave the device — TRN_MODE_DOCS_COMPACT (per tile: bitmap / bucketed 8-bit offsets / 16-bit offsets / docIDs, "
                         "replayed by trn_result_decode) or plain 32-bit docIDs (TRN_MODE_DOCS_ONLY)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the primary workload's results of the last timed step to DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    W = max(3, args.warmup) if args.impl == "ours" else args.warmup
    K = max(1, args.steps)
    if args.impl == "reference":
        return reference_arm(args, rank, world, K, W)

    job = Job(args)
    line = job.run(args.workload, K, W, cpu_budget_s=30.0, with_clocks=True, dump_dir=args.dump_outputs)
    line["numa"] = job.numa
    subs = []
    if args.sub == "auto":
        subs = [w for w in ("or10", "tree8", "and2l") if w != args.workload] if args.workload == "and2" else []
    elif args.sub != "none":
        subs = [w for w in args.sub.split(",") if w in WORKLOADS and w != args.workload]
    if subs:
        line["workloads"] = {}
        # tree8 shares the GOOGLE index of and2: run it first, then release that index before the LUCENE one is built
        for w in sorted(subs, key=lambda x: WORKLOADS[x]["codec"] != WORKLOADS[args.workload]["codec"]):
            for c in list(job.indexes):
                if c != WORKLOADS[w]["codec"]:
                    job.drop_index(c)
            sub = job.run(w, min(K, 3), 3, cpu_budget_s=12.0, with_clocks=False)
            keep = ("value", "unit", "ms_per_step", "steps", "warmup", "config", "e2e", "roofline", "decoded_postings_per_s", "gpu_launches", "parity", "cpu_baseline")
            line["workloads"][w] = {k2: sub[k2] for k2 in keep if k2 in sub}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        job.dist.destroy_process_group()


# ===================================================================================================================== reference arm
def reference_arm(args, rank, world, K, W):
    """--impl reference: the reference's own CPU exec_query on the box's host cores (oracle/_ref), same config/metric.  Nothing of the
    product is loaded here: the index is authored by the reference's own Encoders (tref_synth_build, the same workload generator;
    byte-equal to the product builder's GOOGLE index, decode-equal for LUCENE — tests/test_codecs_cpu.py)."""
    if rank != 0:
        return
    sys.path.insert(0, str(ROOT / "tests"))
    from refharness import RefIndex, load_ref

    wl = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    t0 = time.time()
    r = RefIndex.synth_build(load_ref(), wl["codec"], args.ndocs, args.nterms, threads=cores)
    build_s = time.time() - t0
    texts, _ = gen_queries(args.workload, args.nq, args.nterms)
    # each step = the whole batch when W + K passes fit ~300 s of host time, else the longest prefix that does (the batch is in random order)
    n = args.cpu_sample
    if not n:
        probe = min(len(texts), 128)
        el, *_ = r.exec_batch(texts[:probe], wl["mode"] != 0, args.k, cores)
        n = max(min(32, len(texts)), min(len(texts), int(300.0 * (probe / max(el, 1e-9)) / max(1, K + W))))
    qs = texts[:n]
    for _ in range(W):
        r.exec_batch(qs, wl["mode"] != 0, args.k, cores)
    tot, best = 0.0, None
    for _ in range(K):
        el, *_ = r.exec_batch(qs, wl["mode"] != 0, args.k, cores)
        tot += el
        best = el if best is None else min(best, el)
    v = n * K / tot
    print(json.dumps({
        "metric": metric_name(args.workload),
        "value": v, "unit": "queries/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": tot * 1e3 / K, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u32", "data": "synthetic", "impl": "reference",
        "config": config_of(args, wl, world),
        "index": {"index_build_s": round(build_s, 1), "built_by": "reference Encoders (oracle/_ref), one IndexSession per term"},
        "cpu_baseline": {"value": v, "unit": "queries/s", "cores": cores, "kind": "reference", "best_step_value": n / best, "host": host_info(),
                         "sample": (f"each step = the whole {n}-query batch" if n == len(texts) else f"each step = first {n} queries of the batch")
                         + f", one query per host thread ({cores} threads)"},
        "e2e": {"value": v, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


if __name__ == "__main__":
    main()
