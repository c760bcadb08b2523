#!/usr/bin/env python3
"""bench.py — ops merged/sec of the Peritext op-log apply + flatten hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c4|c2|c3|c5] [--docs D] [--impl engine|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" is one pass of the hot path (pt_batch_merge: apply every op of every log + flatten to spans + digest) over one
batch of synthetic logs.  Default workload = BASELINE.json configs[3] ("c4": 100K docs x 1K ops fuzz-generated, 3
concurrent replicas => 300K logs, 3x10^8 op records, 7.15 GB of packed input — the configuration the north star quotes its
roofline target on; it fits one GPU).  `value` counts op records applied per second summed over docs AND replicas (each
replica really applies every op in the reference, src/micromerge.ts:513), inputs resident in HBM; `e2e` is the same metric
through the public C-ABI path with pinned-host inputs (pt_batch_upload, uncompressed) and packed results read back inside
the timed region.  `extra_configs` (N = 1 only) carries the device-timed numbers of configs[1] and configs[2] (c2, c3).

N > 1: the SAME 100K documents are sharded by doc id across the ranks (peritext_b200.sharding.shard_range — "strong", what
configs[3] names: "doc-sharded 8xB200"); the path's only exchange is one all-gather of the 32-byte per-log result headers
(digests) per step for the convergence check, issued on a side stream so that it overlaps the next step's merge.  `weak`
carries the same measurement with the per-GPU document count held fixed (every rank merges its own 100K documents).

--impl reference: the reference's sequential algorithm (C++ restatement in oracle/, Node.js is unavailable in this
image) on all host cores, on a bounded sample of the same workload.  It never loads the engine library.
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

METRIC = "ops merged/sec across batch"
UNIT = "ops/s"


def sample_clocks(stop_evt, out, device_index):
    """Polls the B200_PROFILING.md clocks line (one nvidia-smi query per sample, back to back) while the bench runs."""
    q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    while not stop_evt.is_set():
        try:
            r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(device_index)],
                               capture_output=True, text=True, timeout=5)
            if r.returncode == 0 and r.stdout.strip():
                parts = [x.strip() for x in r.stdout.strip().split(",")]
                if len(parts) >= 9:
                    out.append(parts)
        except Exception:
            pass
        stop_evt.wait(0.02)


def clocks_summary(samples):
    if not samples:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
    sm = sorted(float(s[1]) for s in samples if s[1].replace(".", "").isdigit())
    mx = max((float(s[2]) for s in samples if s[2].replace(".", "").isdigit()), default=None)
    reasons = set()
    for s in samples:
        for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], s[5:9]):
            if v.lower().startswith("active"):
                reasons.add(name)
    return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(samples)}


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(config, n_docs):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture (profiles/ncu_traffic.json),
    valid for the same config and docs-per-GPU; None otherwise."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        e = json.load(open(p)).get(config)
        if e and int(e.get("docs_per_gpu", -1)) == int(n_docs):
            return float(e["dram_bytes_per_launch"]), e.get("source")
    except Exception:
        pass
    return None, None


def build_checker_only():
    """The reference arm and the cpu_baseline leg need the oracle and the workload generator, NOT the engine."""
    import __graft_entry__ as g
    g.build(load_engine=False)


def cpu_replay_rate(batch, threads, repeats=3):
    """Median-of-`repeats` ops/s of the oracle replay (sequential reference algorithm, one log per thread)."""
    from oracle.packed import replay_packed
    rates, secs = [], []
    for _ in range(repeats):
        _, dt = replay_packed(batch, threads=threads, flatten=True)
        rates.append(batch.n_ops / dt); secs.append(dt)
    k = sorted(range(repeats), key=lambda i: rates[i])[repeats // 2]
    return rates[k], secs[k], rates


def cpu_sample_docs(config, n_docs, cores):
    # bounded sample: the reference is O(N^2) per document, so a step replays a slice of the workload sized for ~5-10 s
    if config in ("c2", "c3"):
        return min(n_docs, max(cores, 16))
    if config == "c4":
        return min(n_docs, max(cores * 32, 1024))
    return 1


def cpu_baseline(config, n_docs_total, ops_per_doc):
    from peritext_b200 import workload
    cores = os.cpu_count() or 1
    sample_docs = cpu_sample_docs(config, n_docs_total, cores)
    batch = workload.generate(config, n_docs=sample_docs, ops_per_doc=ops_per_doc)
    rate, dt, rates = cpu_replay_rate(batch, cores)
    info = (f"first {sample_docs} of {n_docs_total} docs x {batch.meta['replicas']} replicas ({batch.n_ops} op records), median of 3 replays "
            f"({dt:.2f} s), apply+flatten, one log per thread; C++ restatement of the reference algorithm (Node.js unavailable in image)")
    return {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": info, "per_thread": rate / cores,
            "runs": [round(r) for r in rates]}


def ingest_throughput(config, logs=240):
    """Native wire-format ingest (pt_ingest_parse: JSON Change[] -> packed records + change table), all host threads, on a
    bounded sample of the workload re-expressed as JSON; checked by merging the ingested batch (same visible text)."""
    from peritext_b200 import workload
    from peritext_b200.engine import BatchEngine, pack_logs_native
    cores = os.cpu_count() or 1
    R = workload.CONFIGS[config]["replicas"]
    sample = workload.generate(config, n_docs=max(1, logs // R), ops_per_doc=1000 if config != "c4" else None)
    texts = [workload.to_change_json(sample, i) for i in range(sample.n_logs)]
    nbytes = sum(len(t) for t in texts)
    pack_logs_native(texts[:8])
    best = None
    for _ in range(3):
        t0 = time.perf_counter()
        got = pack_logs_native(texts, threads=cores)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    eng = BatchEngine(0)
    a, b = eng.run(sample), eng.run(got)
    eng.close()
    same = bool((a.results["n_visible"] == b.results["n_visible"]).all() and (a.results["n_spans"] == b.results["n_spans"]).all()
                and a.text.tobytes() == b.text.tobytes() and (b.results["status"] == 0).all())
    return {"api": "pt_ingest_parse (C-ABI) via engine.pack_logs_native, includes copying the packed arrays to numpy", "threads": cores,
            "logs": sample.n_logs, "op_records": sample.n_ops, "json_bytes": nbytes, "seconds": best, "mb_per_s": nbytes / best / 1e6,
            "ops_per_s": sample.n_ops / best, "merge_of_ingested_batch_matches": same}


def run_reference(args, rank, world):
    """--impl reference arm: rank 0 only; never loads the engine library."""
    if rank != 0:
        return 0
    build_checker_only()
    from peritext_b200 import workload
    cfg = workload.CONFIGS[args.config]
    n_docs = args.docs or cfg["n_docs"]
    cores = os.cpu_count() or 1
    sample_docs = cpu_sample_docs(args.config, n_docs, cores)
    batch = workload.generate(args.config, n_docs=sample_docs, ops_per_doc=args.ops_per_doc)
    from oracle.packed import replay_packed
    for _ in range(max(0, min(args.warmup, 1))):
        replay_packed(batch, threads=cores)
    per_step = []
    for _ in range(args.steps):
        merged, dt = replay_packed(batch, threads=cores)
        per_step.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, merged, DUMP_BYTES)
    ms = 1e3 * sum(per_step) / max(1, args.steps)
    value = batch.n_ops / (ms / 1e3)
    med = sorted(per_step)[len(per_step) // 2]
    sample = (f"{sample_docs} of {n_docs} docs x {batch.meta['replicas']} replicas per step ({batch.n_ops} op records); C++ restatement "
              f"of the reference algorithm (Node.js unavailable in image), one log per thread")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": f"{args.config}: {cfg['label']}", "sample": sample},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "per_thread": value / cores,
                             "median_step_value": batch.n_ops / med},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


def bind_to_gpu_numa_node(torch, local_rank):
    """N > 1: pin this rank (and so its pinned staging buffers) to the CPU cores of its GPU's NUMA node; on an 8-GPU box
    ranks that float across sockets contend for one socket's memory bandwidth on the host <-> device legs."""
    try:
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id if hasattr(torch.cuda.get_device_properties(local_rank), "pci_bus_id") else None
        if bus is None:
            out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local_rank)], capture_output=True, text=True, timeout=10).stdout.strip()
            bus = out.lower().replace("00000000:", "0000:")
        else:
            bus = "0000:%02x:00.0" % bus
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus)}
    except Exception as e:      # topology files missing: run unbound
        return {"error": str(e)[:80]}


class DeviceRun:
    """One engine handle with a batch resident in HBM; `timed(steps)` = K merges (+ the digest all-gather on a side stream)."""

    def __init__(self, torch, dist, dev, local_rank, world, batch, counts):
        from peritext_b200.engine import BatchEngine
        self.torch, self.dist, self.dev, self.world, self.batch = torch, dist, dev, world, batch
        self.counts, self.max_logs = counts, max(counts)
        self.stream = torch.cuda.Stream(device=dev)
        self.side = torch.cuda.Stream(device=dev)
        self.eng = BatchEngine(local_rank, stream=self.stream.cuda_stream)
        self.eng.upload(batch)
        self.n_logs = batch.n_logs

        class _DevView:   # zero-copy torch view of the engine-owned per-log result headers
            def __init__(s, ptr, nbytes):
                s.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}
        n = self.n_logs
        self.res_dev = torch.as_tensor(_DevView(self.eng.device_results_ptr(), n * 32), device=dev) if n else torch.zeros(0, dtype=torch.uint8, device=dev)
        if world > 1:
            self.stage = torch.zeros(self.max_logs * 32, dtype=torch.uint8, device=dev)
            self.gathered = torch.empty(world * self.max_logs * 32, dtype=torch.uint8, device=dev)
            self.ev_staged = torch.cuda.Event()
            self.ev_gathered = torch.cuda.Event()
            self.ev_gathered.record(self.side)

    def step(self):
        torch = self.torch
        with torch.cuda.stream(self.stream):
            self.eng.merge()
            if self.world > 1:
                # the path's only exchange: result headers (digests) for the convergence check; staged so that the all-gather
                # of step k runs on the side stream while step k+1 merges
                self.stream.wait_event(self.ev_gathered)
                self.stage[: self.n_logs * 32].copy_(self.res_dev, non_blocking=True)
                self.ev_staged.record(self.stream)
        if self.world > 1:
            from peritext_b200 import sharding
            with torch.cuda.stream(self.side):
                self.side.wait_event(self.ev_staged)
                sharding.all_gather_results(self.stage, self.world, out=self.gathered)
                self.ev_gathered.record(self.side)

    def timed(self, steps, warmup):
        torch, dist = self.torch, self.dist
        for _ in range(warmup):
            self.step()
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        l0 = self.eng.launch_count
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        evs[0].record(self.stream)
        for k in range(steps):
            self.step()
            evs[k + 1].record(self.stream)
        end = torch.cuda.Event(enable_timing=True)
        if self.world > 1:
            self.stream.wait_event(self.ev_gathered)      # the last step's exchange is inside the timed region
        end.record(self.stream)
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        total = evs[0].elapsed_time(end)
        per = sorted(evs[k].elapsed_time(evs[k + 1]) for k in range(steps))
        return total, per, self.eng.launch_count - l0

    def lone_merge_ms(self, reps=5):
        v = []
        for _ in range(reps):
            self.eng.merge(); self.eng.sync(); v.append(self.eng.last_merge_ms)
        return sorted(v)[len(v) // 2]

    def check(self):
        """(result headers, all statuses ok, replicas converged) over this rank's logs and — after an exchange — every rank's."""
        from peritext_b200 import sharding
        R = self.batch.meta["replicas"]
        results = self.eng.results()
        rep = sharding.convergence_report(results, R)
        ok, conv = rep["all_status_ok"], rep["replicas_converged"]
        if self.world > 1:
            self.torch.cuda.synchronize()
            allres = sharding.headers_from_bytes(self.gathered.cpu().numpy()).reshape(self.world, self.max_logs)
            for r in range(self.world):
                rr = sharding.convergence_report(allres[r, : self.counts[r]], R)
                ok = ok and rr["all_status_ok"]; conv = conv and rr["replicas_converged"]
        return results, ok, conv

    def close(self):
        self.eng.close()


DUMP_BYTES = 64_000_000   # --dump-outputs writes at most this much (split evenly over the ranks)
DUMP_SEED = 0x5EED


def _ranges(starts, counts):
    """Concatenation of range(s, s + c) over the pairs: the element indices of variable-length records."""
    starts, counts = np.asarray(starts, np.int64), np.asarray(counts, np.int64)
    first = np.concatenate([[0], np.cumsum(counts)[:-1]])
    return np.arange(int(counts.sum()), dtype=np.int64) + np.repeat(starts - first, counts)


def dump_outputs(out_dir, merged, budget, prefix=""):
    """Writes a MergedBatch (what pt_batch_download hands the caller) as float64 .npy files, at most `budget` bytes, so
    that two builds can be compared array for array.  Every field is a u32, exact in float64; each 64-bit digest word is
    stored as its low and high halves.  Logs are chosen in one fixed seeded order, so equal outputs give equal files.
      results.npy          [n, 9] log, status, n_elems, n_visible, n_spans, digest[0] lo, hi, digest[1] lo, hi
                           (every log if that takes at most half the budget, else a sample)
      sample_logs.npy      [k, 4] log, n_visible, n_spans, comments: the logs whose full output follows, as many as fit
      sample_tokens.npy    their visible tokens, log after log
      sample_spans.npy     [m, 3] start, flags, link_attr of their spans (flags >> 8 = the span's comment count)
      sample_comments.npy  the comment ranks of those spans, span after span (offset-free, unlike comment_off)"""
    res = merged.results
    n = len(res)
    order = np.random.default_rng(DUMP_SEED).permutation(n)
    rows = np.sort(order[: min(n, budget // 2 // (9 * 8))])
    dg = res["digest"][rows]
    results = np.stack([np.asarray(c, np.float64) for c in (rows, res["status"][rows], res["n_elems"][rows], res["n_visible"][rows],
                        res["n_spans"][rows], dg[:, 0] & 0xFFFFFFFF, dg[:, 0] >> 32, dg[:, 1] & 0xFFFFFFFF, dg[:, 1] >> 32)], axis=1)
    span_off, n_spans = merged.span_off[:n].astype(np.int64), res["n_spans"].astype(np.int64)
    per_span = np.concatenate([[0], np.cumsum(merged.spans["flags"] >> 8, dtype=np.int64)])
    n_comments = per_span[span_off + n_spans] - per_span[span_off]
    cost = 8 * (4 + res["n_visible"].astype(np.int64) + 3 * n_spans + n_comments)
    room = budget - results.nbytes - 5 * 256             # the .npy header of each file
    sel = np.sort(order[: int(np.searchsorted(np.cumsum(cost[order]), room, side="right"))])
    spans = merged.spans[_ranges(span_off[sel], n_spans[sel])]
    arrays = {"results": results,
              "sample_logs": np.stack([sel, res["n_visible"][sel], n_spans[sel], n_comments[sel]], axis=1),
              "sample_tokens": merged.text[_ranges(merged.text_off[sel], res["n_visible"][sel])],
              "sample_spans": np.stack([spans["start"], spans["flags"], spans["link_attr"]], axis=1),
              "sample_comments": merged.comment_pool[_ranges(spans["comment_off"], spans["flags"] >> 8)]}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), np.asarray(a, np.float64))
    return {name: a.shape[0] for name, a in arrays.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--config", default="c4", choices=["c2", "c3", "c4", "c5"])
    ap.add_argument("--docs", type=int, default=0, help="documents in the whole job (default: the config's; c5: 16 per GPU)")
    ap.add_argument("--ops-per-doc", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra configs (c2, c3) reported beside the headline")
    ap.add_argument("--no-weak", action="store_true", help="N > 1: skip the weak-scaling measurement")
    ap.add_argument("--e2e-compact", action="store_true", help="also time the e2e leg on the compact wire format (host conversion inside the timed region)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's outputs to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "engine" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device; this engine has no CPU fallback"}))
        return 2
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        numa = bind_to_gpu_numa_node(torch, local_rank)
        dist.init_process_group("nccl", device_id=dev)

    import __graft_entry__ as g
    g.build()
    from peritext_b200 import sharding, workload
    from peritext_b200.packing import INSDEL_DT, MARK_DT, PackedBatch

    cfg = workload.CONFIGS[args.config]
    n_docs_total = args.docs or (cfg["n_docs"] if args.config != "c5" else 16 * world)
    gen_threads = max(1, len(os.sched_getaffinity(0)) if world > 1 else (os.cpu_count() or 8))

    # ---- strong: the job's documents sharded by doc id over the ranks --------------------------------------------------
    first, count = sharding.shard_range(n_docs_total, rank, world)
    R = cfg["replicas"]
    counts = [sharding.shard_range(n_docs_total, r, world)[1] * R for r in range(world)]      # logs per rank
    t0 = time.time()
    batch = workload.generate(args.config, n_docs=count, ops_per_doc=args.ops_per_doc, doc_first=first, threads=gen_threads)
    gen_s = time.time() - t0
    in_bytes = batch.insdel.nbytes + batch.marks.nbytes + batch.desc.nbytes

    stop_evt, samples = threading.Event(), []
    th = threading.Thread(target=sample_clocks, args=(stop_evt, samples, local_rank), daemon=True)
    th.start()

    run = DeviceRun(torch, dist, dev, local_rank, world, batch, counts)
    total_ms, per_step, launches = run.timed(args.steps, args.warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, run.eng.download(), DUMP_BYTES // world, f"rank{rank}_" if world > 1 else "")
    lone_ms = run.lone_merge_ms(min(5, args.steps))
    results, ok, converged = run.check()
    stats = run.eng.stats()
    ops_local = batch.n_ops
    alg_bytes = batch.algorithmic_bytes(results)

    # ---- e2e through the public API: pinned host -> device (pt_batch_upload), merge, packed results back to host ----------
    e2e = None
    if not args.no_e2e:
        from peritext_b200.engine import PipelinedEngine

        def pinned(a):
            return torch.from_numpy(a.view(np.uint8).reshape(-1)).pin_memory() if a.nbytes else torch.zeros(16, dtype=torch.uint8).pin_memory()
        p_ins, p_mk = pinned(batch.insdel), pinned(batch.marks)
        pbatch = PackedBatch(batch.desc, p_ins.numpy()[: batch.insdel.nbytes].view(INSDEL_DT), p_mk.numpy()[: batch.marks.nbytes].view(MARK_DT),
                             batch.values, batch.link_attrs, batch.comment_ids, batch.other_attrs, batch.meta)
        # the public batch API: PipelinedEngine cuts the batch into 4 runs of logs (own handle + stream each) so that the
        # upload of one overlaps the merge and the download of the others
        pipe = PipelinedEngine(local_rank, chunks=4)

        def timed_e2e(compact):
            outs = None
            for _ in range(2):
                outs = pipe.run(pbatch, compact=compact, threads=gen_threads)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            e_steps = max(3, min(args.steps, 8))
            t0 = time.perf_counter()
            for _ in range(e_steps):
                outs = pipe.run(pbatch, compact=compact, threads=gen_threads)
            torch.cuda.synchronize()
            ms = 1e3 * (time.perf_counter() - t0) / e_steps
            d2h = sum(o.results.nbytes + o.text.nbytes + o.spans.nbytes + o.comment_pool.nbytes + o.text_off.nbytes + o.span_off.nbytes for o in outs)
            e_res = np.concatenate([o.results for o in outs])
            good = bool((e_res["status"] == 0).all()) and e_res["digest"].tobytes() == results["digest"].tobytes()
            return ms, int(d2h), good

        # (1) the packed records as they are (pt_batch_upload); (2) the compact wire format: every chunk is converted on the
        # host (pt_compact_ops, all threads of this rank) INSIDE the timed region and uploaded as half the bytes
        u_ms, u_d2h, u_ok = timed_e2e(False)
        ok = ok and u_ok
        e2e = {"ms": u_ms, "h2d": int(in_bytes), "d2h": u_d2h, "form": "uncompressed", "plain_ms": u_ms}
        try:
            if not args.e2e_compact:     # measured on B200 boxes: the host-side conversion costs more than the PCIe bytes it saves
                raise RuntimeError("not measured (pass --e2e-compact)")
            c_ms, c_d2h, c_ok = timed_e2e(True)
            ok = ok and c_ok
            e2e["compact_ms"] = c_ms
            if c_ms < u_ms:
                e2e = {"ms": c_ms, "h2d": int(batch.insdel.nbytes // 2 + batch.marks.nbytes // 2 + batch.desc.nbytes), "d2h": c_d2h, "form": "compact", "plain_ms": u_ms, "compact_ms": c_ms}
        except Exception as ex:      # a log that the compact form cannot represent, or not requested: the plain form stands
            if args.e2e_compact:
                e2e["compact_error"] = str(ex)[:120]
        pipe.close()
        del pbatch, p_ins, p_mk

    # reduce over ranks: time = max, work = sum
    def reduce_max(*vals):
        if world == 1:
            return list(vals)
        t = torch.tensor(list(vals), device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def reduce_sum(v):
        if world == 1:
            return v
        t = torch.tensor([float(v)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t[0])

    t_ms, e2e_ms, e2e_plain_ms = reduce_max(total_ms, e2e["ms"] if e2e else 0.0, e2e["plain_ms"] if e2e else 0.0)
    total_ops = reduce_sum(ops_local)
    total_logs = reduce_sum(batch.n_logs)
    ms_per_step = t_ms / args.steps
    value = total_ops / (ms_per_step / 1e3)
    n_logs_local = batch.n_logs
    unique_local = batch.meta["unique_ops"]
    run.close()
    del run, batch

    # ---- weak: every rank merges its own full-size batch (N > 1 only) ----------------------------------------------------
    weak = None
    if world > 1 and not args.no_weak:
        per_gpu = n_docs_total
        wb = workload.generate(args.config, n_docs=per_gpu, ops_per_doc=args.ops_per_doc, doc_first=sharding.weak_doc_first(per_gpu, rank), threads=gen_threads)
        wrun = DeviceRun(torch, dist, dev, local_rank, world, wb, [wb.n_logs] * world)
        w_total, w_per, _ = wrun.timed(args.steps, args.warmup)
        _, w_ok, w_conv = wrun.check()
        (w_ms,) = reduce_max(w_total)
        w_ops = reduce_sum(wb.n_ops)
        weak = {"value": w_ops / (w_ms / args.steps / 1e3), "unit": UNIT, "ms_per_step": w_ms / args.steps, "docs_per_gpu": per_gpu,
                "all_status_ok": w_ok, "replicas_converged": w_conv}
        ok = ok and w_ok; converged = converged and w_conv
        wrun.close()
        del wrun, wb

    # ---- the other single-GPU configs, device-timed (N = 1 only) ------------------------------------------------------------
    extras = None
    if world == 1 and not args.no_extras and args.config == "c4":
        extras = {}
        peak, _ = hbm_peak()
        for name in ("c3", "c2"):
            xb = workload.generate(name, threads=gen_threads)
            xr = DeviceRun(torch, dist, dev, local_rank, 1, xb, [xb.n_logs])
            x_total, x_per, _ = xr.timed(args.steps, args.warmup)
            x_res, x_ok, x_conv = xr.check()
            x_ms = x_total / args.steps
            x_alg = xb.algorithmic_bytes(x_res)
            extras[name] = {"workload": workload.CONFIGS[name]["label"], "value": xb.n_ops / (x_ms / 1e3), "unit": UNIT, "ms_per_step": x_ms,
                            "ms_per_step_min": x_per[0], "roofline_frac": x_alg / (x_ms / 1e3) / 1e9 / peak,
                            "algorithmic_bytes_per_launch": int(x_alg), "all_status_ok": x_ok, "replicas_converged": x_conv,
                            "kernel_paths": xr.eng.stats()}
            ok = ok and x_ok; converged = converged and x_conv
            xr.close()
            del xr, xb

    stop_evt.set(); th.join(timeout=2)

    if rank == 0:
        peak, peak_src = hbm_peak()
        achieved = alg_bytes / (lone_ms / 1e3) / 1e9
        traffic, traffic_src = ncu_traffic(args.config, count)
        warp_share = stats.get("logs_deferred_to_big_bin", 0) == 0 and args.config == "c4"
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32",
            "data": "synthetic",
            "config": {"workload": f"{args.config}: {cfg['label']}", "docs_total": n_docs_total, "docs_per_gpu": count, "replicas": R,
                       "logs_per_gpu": n_logs_local, "op_records_per_step": int(total_ops), "op_records_per_step_per_gpu": ops_local,
                       "unique_ops_per_gpu": unique_local, "input_bytes_per_gpu": in_bytes,
                       "parallelism": f"doc-sharded x{world} (strong: shard_range over {n_docs_total} docs)",
                       "l2": "input (%.0f MB per GPU) larger than the 126 MB L2; no flush needed" % (in_bytes / 1e6)
                       if in_bytes > 130e6 else "input smaller than L2 (steps may hit L2)",
                       "generator_s": round(gen_s, 2), "all_status_ok": ok, "replicas_converged": converged,
                       "docs_per_sec": total_logs / (ms_per_step / 1e3), "kernel_paths": stats,
                       "ms_per_step_min": per_step[0], "ms_per_step_median": per_step[len(per_step) // 2], "ms_per_step_max": per_step[-1],
                       "exchange": "none (1 rank)" if world == 1 else "all-gather of 32-byte result headers per step, side stream, inside the timed region",
                       "rank0_cpu_binding": numa},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "ptk::merge_logs_warp_kernel" if warp_share else "ptk::merge_logs_team_kernel" if args.config == "c2" else "ptk::merge_logs_kernel",
                         "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": int(alg_bytes), "launch_ms": lone_ms},
            "clocks": clocks_summary(samples),
        }
        if e2e:
            api = ("peritext_b200.engine.PipelinedEngine.run over the C-ABI, 4 chunks: "
                   + ("pt_compact_ops [host conversion of the packed records to the compact wire format, inside the timed region] / pt_batch_upload_compact"
                      if e2e["form"] == "compact" else "pt_batch_upload")
                   + " / pt_batch_merge / pt_batch_download_begin [device-side packing of the outputs] / pt_batch_download per chunk")
            line["e2e"] = {"value": total_ops / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(e2e["h2d"]),
                           "d2h_bytes_per_step": int(e2e["d2h"]), "ms_per_step": e2e_ms, "wire_form": e2e["form"], "api": api,
                           "uncompressed": {"value": total_ops / (e2e_plain_ms / 1e3), "ms_per_step": e2e_plain_ms, "h2d_bytes_per_step": int(in_bytes),
                                            "api": "same pipeline with pt_batch_upload (16 / 32 byte records as packed)"}}
            if "compact_ms" in e2e:      # rank 0's own time; the compact wire form halves the PCIe bytes but its host-side conversion
                line["e2e"]["compact_wire_form"] = {"ms_per_step_rank0": e2e["compact_ms"], "includes_host_conversion": True}     # (pt_compact_ops) is inside the timed region
            if "compact_error" in e2e:
                line["e2e"]["compact_error"] = e2e["compact_error"]
        if weak:
            line["weak"] = weak
        if extras:
            line["extra_configs"] = extras
        if world == 1 and not args.no_extras:
            line["ingest"] = ingest_throughput(args.config)
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(args.config, n_docs_total, args.ops_per_doc)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0 if (ok and converged) else 3


if __name__ == "__main__":
    sys.exit(main())
