#!/usr/bin/env python3
"""Benchmark of the BPE merge-loop hot path (BASELINE.json metric: BPE train merges/sec + encode GB/s at
1/2/4/8 B200 vs the reference's CPU path, with the HBM roofline fraction of the dominant kernel).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl engine|reference] [--workload c1|c2|c3|c4|c5]
                  [--dump-outputs DIR]

One "step" = one complete run of the workload from the byte corpus (widen, count, all merges).
  value : merges/s with the corpus already resident in HBM (CUDA events on the engine's stream, max over ranks)
  e2e   : the same through the C-ABI context calls with HOST buffers: pinned corpus -> H2D, train, merges + ids ->
          D2H, all inside the timed region.  N = 1 also reports the one-call entry point bpe_cuda_train() (pageable
          buffers, context creation inside) and the drop-in compress() on a file (e2e_paths).
Workloads (SURVEY.md §8d, BASELINE.json configs):
  c3 : synthetic 1 GB byte-level Zipf corpus, 32,000 merges, sharded over N GPUs; the deltas of every pass
       travel between the GPUs' pair tables over NVLink peer memory       (DEFAULT at every N: the configuration
       the 1/2/4/8 scaling curve is asked for; it also fits one GPU)
  c2 : synthetic 100 MB Zipf-word ASCII corpus, 4,096 merges                (also measured inside the N = 1 line: "c2")
  c1 : the reference's random_text.txt to exhaustion (parity configuration; L2-resident)
  c4 : encode a 10 GB corpus with the 32,000-merge table learned from c3's corpus (8 GPUs)     [value: GB/s of input]
  c5 : synthetic 8 GB byte-level corpus, 50,000 merges (8 GPUs)
N > 1 is launched by torch.distributed.run (one rank per GPU); torch.distributed (gloo) is only the bootstrap
(NCCL id broadcast, barriers, max-over-ranks), the data path is the engine's own exchange.

--impl reference times the UNMODIFIED reference (oracle/_ref/ref_harness, compiled from the reference sources) on
the host cores, each step a bounded sample of the same workload (first merges of a prefix, scaled; stated in the line).

--dump-outputs DIR writes what the engine's last timed step returned (merge list, ids) as DIR/<name>.npy (see
dump_outputs()): the corpora are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes as C
import gzip
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MB = 1_000_000
# ref_bytes / ref_merges: the bounded sample the reference's CPU path is timed on (its per-merge cost is linear in
# the token count: full recount + table fold + rewrite every iteration, bpe.c:669-783)
WORKLOADS = {
    "c1": dict(desc="random_text.txt (1,048,576 B, bundled with the reference), merges to exhaustion", kind=None, mode="train",
               size=1048576, seed=0, merges=0, ref_bytes=1048576, ref_merges=100),
    "c2": dict(desc="synthetic 100 MB Zipf-word ASCII corpus (zipf_ascii seed 1234), 4,096 merges", kind=0, mode="train",
               size=100 * MB, seed=1234, merges=4096, ref_bytes=100 * MB, ref_merges=16),
    "c3": dict(desc="synthetic 1 GB byte-level Zipf corpus (zipf_bytes seed 4321), 32,000 merges", kind=1, mode="train",
               size=1000 * MB, seed=4321, merges=32000, ref_bytes=64 * MB, ref_merges=2),
    "c4": dict(desc="encode a synthetic 10 GB byte-level Zipf corpus (80 chunks of 125 MB, zipf_bytes seeds 777+k, c3's word "
                    "list) with the 32,000-merge table learned from c3's corpus", kind=1, mode="encode", size=10000 * MB,
               seed=777, chunk=125 * MB, merges=32000, table="c3", ref_bytes=128 * MB, ref_merges=32),
    "c5": dict(desc="synthetic 8 GB byte-level Zipf corpus (64 chunks of 125 MB, zipf_bytes seeds 8888+k), 50,000 merges", kind=1,
               mode="train", size=8000 * MB, seed=8888, chunk=125 * MB, merges=50000, ref_bytes=64 * MB, ref_merges=2),
}
REF_BIN = os.path.join(ROOT, "oracle/_ref/ref_harness")
ORACLE_CLI = os.path.join(ROOT, "oracle/_build/bpe_oracle_cli")
TRAFFIC = os.path.join(ROOT, "profiles", "r2_traffic.json")   # measured dram bytes of the dominant kernel (ncu --set full)
DUMP_IDS = 1 << 21   # --dump-outputs keeps a fixed sample of this many ids of a longer stream (32 MB with its positions)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def fill_corpus(w, arr, lo, hi):
    """arr[:] = bytes [lo, hi) of workload w's corpus."""
    from llmtokenizer_b200 import _lib
    lib = _lib.load_corpus()
    words = 50000 if w["kind"] == 0 else 65536
    if w["kind"] is None:
        with gzip.open(os.path.join(ROOT, "tests/golden/random_text.txt.gz"), "rb") as f:
            arr[:] = np.frombuffer(f.read(), dtype=np.uint8)[lo:hi]
    elif "chunk" not in w:
        if lo == 0 and hi == w["size"]:
            assert lib.gen_corpus_fill(w["kind"], arr.ctypes.data, hi, w["seed"], words) == 0
        else:
            # one sequential stream: a prefix is generated directly, anything else is cut out of the whole
            tmp = np.empty(hi, dtype=np.uint8)
            assert lib.gen_corpus_fill(w["kind"], tmp.ctypes.data, hi, w["seed"], words) == 0
            arr[:] = tmp[lo:hi]
    else:
        ch = w["chunk"]
        jobs = []
        for k in range(lo // ch, (hi + ch - 1) // ch):
            c0, c1 = max(lo, k * ch), min(hi, (k + 1) * ch)

            def one(k=k, c0=c0, c1=c1):
                if c0 == k * ch:
                    assert lib.gen_corpus_fill(w["kind"], arr[c0 - lo:].ctypes.data, c1 - c0, w["seed"] + k, words) == 0
                else:
                    tmp = np.empty(c1 - k * ch, dtype=np.uint8)
                    assert lib.gen_corpus_fill(w["kind"], tmp.ctypes.data, tmp.size, w["seed"] + k, words) == 0
                    arr[c0 - lo:c1 - lo] = tmp[c0 - k * ch:]
            jobs.append(threading.Thread(target=one))
        for j in jobs:   # (ctypes releases the GIL: the chunks are generated in parallel)
            j.start()
        for j in jobs:
            j.join()


def make_shard(w, rank, world, pinned=True):
    """This rank's contiguous shard of the corpus in (pinned) host memory."""
    import torch
    n = w["size"]
    lo, hi = n * rank // world, n * (rank + 1) // world
    t = torch.empty(hi - lo, dtype=torch.uint8, pin_memory=pinned and torch.cuda.is_available())
    arr = t.numpy()
    fill_corpus(w, arr, lo, hi)
    return t, arr


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True).start()
        except OSError:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---- the reference's CPU path (bounded samples) ----------------------------------------------------
def run_reference_sample(corpus_path, merges):
    """The first `merges` merges of the file's corpus through the unmodified reference (or the oracle port)."""
    out = f"/tmp/bench_ref_{os.getpid()}"
    if os.path.exists(REF_BIN):
        cmd, kind = [REF_BIN, corpus_path, str(merges), out], "reference"
    else:
        cmd, kind = [ORACLE_CLI, "train", corpus_path, str(merges), "1", out], "port"
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"{cmd}: rc={r.returncode} {r.stderr[-300:]}")
    f = r.stdout.split()
    done, secs = int(f[0]), float(f[2])
    for ext in (".merges", ".ids"):
        try:
            os.remove(out + ext)
        except OSError:
            pass
    return done, secs, kind


def reference_train_sample(w, name):
    """(merges/s scaled to the full corpus, raw merges/s on the sample, description, kind)"""
    nb = min(w["ref_bytes"], w["size"])
    arr = np.empty(nb, dtype=np.uint8)
    fill_corpus(w, arr, 0, nb)
    path = f"/tmp/bench_corpus_{name}_{os.getpid()}.bin"
    arr.tofile(path)
    try:
        done, secs, kind = run_reference_sample(path, int(os.environ.get("BPE_BENCH_REF_MERGES") or w["ref_merges"]))
    finally:
        os.remove(path)
    raw = done / secs
    scale = nb / w["size"]
    what = (f"first {done} merges of the first {nb / MB:.0f} MB of the same corpus ({secs:.1f} s: compress() incl. file read + "
            f"widen, 16 worker threads + main as hard-coded in bpe.c:409)")
    if scale < 1:
        what += (f"; value = {raw:.3f} merges/s on the sample x {scale:.4f} (the reference recounts and rewrites the whole "
                 f"stream every merge, bpe.c:669-783: time per merge is linear in the corpus size)")
    return raw * scale, raw, what, kind


def reference_encode_sample(w, merges_np):
    """The reference has no encoder; its rewrite loop (bpe.c:760-772) applied rank by rank is what oracle/bo_encode
    restates: time the first ref_merges ranks on a slice -> GB/s of input for the WHOLE table, extrapolated."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_api
    nb = min(w["ref_bytes"], w["size"])
    arr = np.empty(nb, dtype=np.uint8)
    fill_corpus(w, arr, 0, nb)
    r = min(w["ref_merges"], len(merges_np))
    o = oracle_api.load()
    t0 = time.perf_counter()
    o.encode(arr, merges_np[:r])
    secs = time.perf_counter() - t0
    full = secs * len(merges_np) / max(1, r)          # upper bound: later ranks see a shorter stream
    return (nb / 1e9) / full, f"oracle bo_encode (bpe.c:760-772 per rank, 1 thread): first {r} of {len(merges_np)} ranks on a " \
                              f"{nb / MB:.0f} MB slice took {secs:.1f} s; extrapolated linearly to the whole table"


# ---- distributed bootstrap -------------------------------------------------------------------------
def dist_setup(n_gpus):
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group(backend="gloo")
    assert world == n_gpus or world == 1, f"--gpus {n_gpus} but WORLD_SIZE={world}"
    return rank, world, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()


def max_over_ranks(x, world):
    if world == 1:
        return x
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0])


def sum_over_ranks(x, world):
    if world == 1:
        return x
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t[0])


def sha_over_ranks(ids, rank, world):
    """SHA-256 of the ranks' id arrays concatenated in rank order (rank 0 returns it)."""
    h = hashlib.sha256()
    if world == 1:
        h.update(np.ascontiguousarray(ids, dtype="<u4").tobytes())
        return h.hexdigest()
    import torch
    import torch.distributed as dist
    if rank == 0:
        h.update(np.ascontiguousarray(ids, dtype="<u4").tobytes())
        for r in range(1, world):
            n = torch.zeros(1, dtype=torch.int64)
            dist.recv(n, src=r)
            buf = torch.empty(int(n[0]), dtype=torch.int32)
            if int(n[0]):
                dist.recv(buf, src=r)
            h.update(buf.numpy().tobytes())
        return h.hexdigest()
    dist.send(torch.tensor([ids.size], dtype=torch.int64), dst=0)
    if ids.size:
        dist.send(torch.from_numpy(np.ascontiguousarray(ids).view(np.int32)), dst=0)
    return None


def bench_reference(args, w, rank, world):
    if rank != 0:
        return
    name = args.workload
    if w["mode"] == "encode":
        # the table comes from the oracle port on a small prefix of the table corpus: only its shape matters for timing
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_api
        tw = WORKLOADS[w["table"]]
        small = np.empty(4 * MB, dtype=np.uint8)
        fill_corpus(tw, small, 0, small.size)
        _, merges_np, _, _ = oracle_api.load().train(small, 256, oracle_api.FAST_CF)
        vals = []
        for i in range(args.warmup + args.steps):
            v, what = reference_encode_sample(dict(w, ref_merges=min(w["ref_merges"], 256)), merges_np)
            if i >= args.warmup:
                vals.append(v)
        val, raw, kind, unit, metric = float(np.mean(vals)), float(np.mean(vals)), "port", "GB/s", "bpe_encode_gb_per_sec"
        ms = 0.0
    else:
        vals, raws, secs_tot = [], [], 0.0
        what, kind = "", "reference"
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            v, r, what, kind = reference_train_sample(w, name)
            if i >= args.warmup:
                vals.append(v)
                raws.append(r)
                secs_tot += time.perf_counter() - t0
        val, raw, unit, metric = float(np.mean(vals)), float(np.mean(raws)), "merges/s", "bpe_train_merges_per_sec"
        ms = 1e3 * secs_tot / max(1, args.steps)
    line = {
        "impl": "reference", "metric": metric, "value": val, "unit": unit, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": f"{name}: {w['desc']}", "merges": w["merges"], "corpus_bytes": w["size"]},
        "cpu_baseline": {"value": val, "unit": unit, "cores": os.cpu_count(), "kind": kind, "raw_sample_value": raw, "sample": what},
        "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---- the engine ------------------------------------------------------------------------------------
def load_traffic():
    if os.path.exists(TRAFFIC):
        return json.load(open(TRAFFIC))
    return None


def time_training(ctx, M, steps, warmup, world, local, sample_clocks=True):
    import torch
    for _ in range(warmup):
        st = ctx.train(M)
    sampler = ClockSampler(local)
    barrier(world)
    torch.cuda.synchronize()
    if sample_clocks:
        sampler.start()
    dev_ms, merges_done, launches = 0.0, 0, 0
    t0 = time.perf_counter()
    for _ in range(steps):
        st = ctx.train(M)
        dev_ms += st["ms_device"]
        merges_done += st["n_merges"]
        launches += st["kernel_launches"]
    torch.cuda.synchronize()
    barrier(world)
    wall_ms = max_over_ranks((time.perf_counter() - t0) * 1e3, world)
    clocks = sampler.stop() if sample_clocks else None
    dev_ms = max_over_ranks(dev_ms, world)
    return dict(value=merges_done / (dev_ms * 1e-3), dev_ms=dev_ms, wall_ms=wall_ms, clocks=clocks, launches=launches, stats=st)


def dump_outputs(out_dir, merges, ids):
    """Write what a step returned as float64 arrays (exact: ids and positions are below 2^53): merges.npy [k, 2] (training
    only) and ids.npy.  A stream longer than DUMP_IDS is sampled at fixed positions (seed 0, ascending), which go to
    ids_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    if merges is not None:
        np.save(os.path.join(out_dir, "merges.npy"), merges.astype(np.float64))
    if ids.size > DUMP_IDS:
        idx = np.sort(np.random.default_rng(0).choice(ids.size, DUMP_IDS, replace=False))
        np.save(os.path.join(out_dir, "ids_index.npy"), idx.astype(np.float64))
        ids = ids[idx]
    np.save(os.path.join(out_dir, "ids.npy"), ids.astype(np.float64))


def profiled_roofline(ctx, run, world, shard_bytes, kernel_desc):
    """One extra step with CUDA events around every pass of the dominant kernel."""
    ctx.set_option("profile_replace", 1)
    sp = run()
    ctx.set_option("profile_replace", 0)
    peak, peak_src = peaks()
    k_ms = max_over_ranks(sp["replace_ms"], world)
    k_bytes = sp["replace_bytes"] / world  # algorithmic bytes on one rank ~ global / N
    achieved = k_bytes / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0
    step_ms = max_over_ranks(sp["ms_device"], world)
    r = {
        "bound": "hbm", "kernel": kernel_desc, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "peak_source": peak_src, "traffic": None, "launches": sp["replace_passes"],
        "avg_launch_us": 1e3 * k_ms / max(1, sp["replace_passes"]),
        "merges_per_pass": sp["n_merges"] / max(1, sp["replace_passes"]),
        "algorithmic_bytes_per_step": sp["replace_bytes"], "algorithmic_bytes_per_launch_per_gpu": k_bytes / max(1, sp["replace_passes"]),
        "kernel_share_of_step": k_ms / step_ms if step_ms else None,
        "other_kernels_ms": {"apply_select_incl_exchange": sp["apply_ms"] + sp["select_ms"], "host_gaps": sp["gap_ms"]},
        "how": "CUDA events on the engine's stream around every pass (replace_stream_kernel / replace_kernel launch) in one "
               "extra step of the same workload (events off in the timed steps), max over ranks; bytes = sum over PASSES "
               "of 4*(tokens in + tokens out) - a pass that carries several provably-next merges is counted once",
    }
    whole = (sp["replace_bytes"] / world + 9 * shard_bytes) / (step_ms * 1e-3) / 1e9
    r["whole_step_gbs"] = whole
    r["whole_step_frac"] = whole / peak
    return r, sp


def bench_engine(args, w, rank, world, local):
    import torch
    import llmtokenizer_b200 as L
    from llmtokenizer_b200 import _lib
    lib = _lib.load()
    assert lib.bpe_cuda_device_count() > local, "no CUDA device: the engine has no CPU fallback"
    torch.cuda.set_device(local)
    name = args.workload
    encode_mode = w["mode"] == "encode"
    ctx = L.Context(local)
    if world > 1:
        import torch.distributed as dist
        idt = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            idt[:] = torch.frombuffer(bytearray(L.nccl_unique_id()), dtype=torch.uint8)
        dist.broadcast(idt, 0)
        ctx.set_comm(rank, world, bytes(idt.numpy().tobytes()))
    M = w["merges"]
    peak, peak_src = peaks()
    traffic = load_traffic()

    # ---- c4: learn the table first (c3's corpus, all ranks), then the workload is the encode of the big corpus ------
    table = None
    if encode_mode:
        tw = WORKLOADS[w["table"]]
        _, tshard = make_shard(tw, rank, world)
        ctx.upload_ptr(tshard.ctypes.data, tshard.size)
        barrier(world)
        ctx.train(tw["merges"])
        table, _ = ctx.download(tokens=False)
        del tshard

    pin_t, shard = make_shard(w, rank, world)
    n = w["size"]
    ctx.upload_ptr(shard.ctypes.data, shard.size)
    barrier(world)   # (the ranks generate their shards at different speeds)

    if encode_mode:
        run = lambda: ctx.encode(table)
        for _ in range(args.warmup):
            st = run()
        sampler = ClockSampler(local)
        barrier(world)
        torch.cuda.synchronize()
        sampler.start()
        dev_ms, launches = 0.0, 0
        for _ in range(args.steps):
            st = run()
            dev_ms += st["ms_device"]
            launches += st["kernel_launches"]
        torch.cuda.synchronize()
        barrier(world)
        clocks = sampler.stop()
        dev_ms = max_over_ranks(dev_ms, world)
        value = n * args.steps / (dev_ms * 1e-3) / 1e9
        metric, unit = "bpe_encode_gb_per_sec", "GB/s"
        final_tokens = st["n_tokens"]
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, None, ctx.download(merges=False)[1])
    else:
        run = lambda: ctx.train(M)
        tt = time_training(ctx, M, args.steps, args.warmup, world, local)
        value, dev_ms, clocks, launches, st = tt["value"], tt["dev_ms"], tt["clocks"], tt["launches"], tt["stats"]
        metric, unit = "bpe_train_merges_per_sec", "merges/s"
        final_tokens = st["n_tokens"]
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, *ctx.download())

    # ---- end to end through host buffers (context API, pinned) ---------------------------------------
    nm, nt = ctx.result_sizes()
    out_m = torch.empty((max(nm, 1), 2), dtype=torch.int32, pin_memory=True)
    out_t = torch.empty(max(nt + 1024, 1), dtype=torch.int32, pin_memory=True)

    def e2e_step():
        ctx.upload_ptr(shard.ctypes.data, shard.size)          # H2D of this step's input
        s = run()
        ctx.download_into(out_m.data_ptr(), out_t.data_ptr())  # D2H of merges + ids
        return s

    e2e_step()
    barrier(world)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e2e_units = 0
    for _ in range(args.steps):
        s = e2e_step()
        e2e_units += n / 1e9 if encode_mode else s["n_merges"]
        launches += s["kernel_launches"]
    torch.cuda.synchronize()
    barrier(world)
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3, world)
    e2e_value = e2e_units / (e2e_ms * 1e-3)
    h2d = int(shard.size)
    d2h = int((0 if encode_mode else nm * 8) + nt * 4)

    # ---- roofline of the dominant kernel (replace+scan+delta), one extra profiled step ----------------------
    kdesc = ("replace_stream_kernel (fused replace + prefix-scan compaction + pair-count deltas; a == b passes: replace_kernel)")
    roofline, sp = profiled_roofline(ctx, run, world, shard.size, kdesc)
    if traffic and name in traffic:
        roofline["traffic"] = traffic[name].get("dram_bytes_per_launch")
        roofline["traffic_detail"] = traffic[name]

    # ---- the other half of the metric: encode GB/s with the learned table, at every N, with its own roofline -------
    encode = None
    if not encode_mode and name in ("c2", "c3", "c5"):
        merges_np, _ = ctx.download(tokens=False)
        ctx.encode(merges_np)
        se = ctx.encode(merges_np)
        enc_ms = max_over_ranks(se["ms_device"], world)
        enc_roof, sep = profiled_roofline(ctx, lambda: ctx.encode(merges_np), world, shard.size, kdesc + " driven by the given merge list")
        encode = {"value": n / (enc_ms * 1e-3) / 1e9, "unit": "GB/s of input", "ranks": int(len(merges_np)), "ms": enc_ms,
                  "passes": se["replace_passes"], "n_gpus": world,
                  "roofline": {k: enc_roof[k] for k in ("bound", "achieved", "peak", "unit", "frac", "launches", "avg_launch_us",
                                                        "kernel_share_of_step", "algorithmic_bytes_per_step")}}

    # ---- parity at full size, outside every timed region --------------------------------------------------
    checks = {}
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()
    if not encode_mode:
        run()
        m_b, t_b = ctx.download()
        ids_sha = sha_over_ranks(t_b, rank, world)
        total_ids = int(sum_over_ranks(t_b.size, world))
        gold = {"c2": "c2_full.json", "c3": "c3_full.json", "c1": "c1_exhaustion.json"}.get(name)
        gpath = os.path.join(ROOT, "tests", "golden", gold) if gold else None
        if gpath and os.path.exists(gpath):
            g = json.load(open(gpath))   # digests of the CPU oracle's result for this very corpus (tools/make_*_golden.py)
            checks["equals_oracle_digest"] = bool(sha(m_b) == g["merges_sha256"] and (rank != 0 or ids_sha == g["ids_sha256"])
                                                  and total_ids == g["n_ids"])
            checks["oracle_digest"] = gold
        elif name == "c3":
            # the full 32,000-merge oracle run takes hours; its first 4,000 merges are committed
            g = json.load(open(os.path.join(ROOT, "tests", "golden", "c3_first4000.json")))
            checks["first_4000_merges_equal_oracle_digest"] = bool(sha(m_b[:4000]) == g["merges_sha256"])
        checks["merges_sha256"] = sha(m_b)[:16]
        checks["ids_sha256"] = (ids_sha or "")[:16]
        if world == 1:
            nbytes = ctx.decode(m_b, download=False)       # ids -> bytes on the device, compared with the shard there
            checks["decode_round_trip_mismatching_bytes"] = int(ctx.decode_mismatches() if nbytes == shard.size else -1)
            ctx.encode(m_b)
            _, t_e = ctx.download(merges=False)
            checks["encode_with_learned_merges_reproduces_training_ids"] = bool(sha(t_e) == sha(t_b))
            if n <= 200 * MB:
                ctx.set_option("batch_max", 1)             # one merge per pass: the sequential order by construction
                ctx.train(M)
                m_1, t_1 = ctx.download()
                ctx.set_option("batch_max", 15)             # (clamped to the build's BATCH_MAX)
                checks["batched_passes_equal_one_merge_per_pass"] = bool(sha(m_b) == sha(m_1) and sha(t_b) == sha(t_1))
    else:
        run()
        _, t_b = ctx.download(merges=False)
        checks["ids_sha256"] = (sha_over_ranks(t_b, rank, world) or "")[:16]
        checks["total_ids"] = int(sum_over_ranks(t_b.size, world))

    # ---- N = 1 extras: config 2 in the same line, the one-call and drop-in e2e paths, the CPU reference ---------
    c2 = None
    e2e_paths = None
    cpu = None
    if world == 1 and not args.quick:
        if name == "c3":
            w2 = WORKLOADS["c2"]
            ctx2 = L.Context(local)
            _, s2 = make_shard(w2, 0, 1)
            ctx2.upload_ptr(s2.ctypes.data, s2.size)
            t2 = time_training(ctx2, w2["merges"], args.steps, args.warmup, 1, local, sample_clocks=False)
            r2, sp2 = profiled_roofline(ctx2, lambda: ctx2.train(w2["merges"]), 1, s2.size, kdesc)
            if traffic and "c2" in traffic:
                r2["traffic"] = traffic["c2"].get("dram_bytes_per_launch")
                r2["traffic_detail"] = traffic["c2"]
            m2, t2ids = ctx2.download()
            g2 = json.load(open(os.path.join(ROOT, "tests", "golden", "c2_full.json")))
            c2 = {"workload": f"c2: {w2['desc']}", "value": t2["value"], "unit": "merges/s", "ms_per_step": t2["dev_ms"] / args.steps,
                  "roofline": r2, "equals_oracle_digest": bool(sha(m2) == g2["merges_sha256"] and sha(t2ids) == g2["ids_sha256"])}
            ctx2.close()
            del s2
        if not encode_mode:
            # (1) the one-call C-ABI entry point a reference-side caller binds: pageable buffers, contexts created inside
            t0 = time.perf_counter()
            m1, t1, s1 = L.train(shard, max_merges=M, n_gpus=1)
            one_call = (time.perf_counter() - t0)
            # (2) the drop-in compress() on a file (get_file + strlen cut + engine + dyn_arr result), bpe.c:541-811
            dropin = None
            so = os.path.join(ROOT, "llmtokenizer_b200", "dropin", "libbpe.so")
            if os.path.exists(so):
                path = f"/tmp/bench_dropin_{os.getpid()}.bin"
                shard.tofile(path)
                dl = C.CDLL(so)
                dl.compress_n.restype = C.c_void_p
                dl.compress_n.argtypes = [C.c_char_p, C.POINTER(C.POINTER(C.c_uint32)), C.POINTER(C.c_size_t), C.c_size_t, C.c_int]
                dl.dyn_arr_free.argtypes = [C.c_void_p]
                enc, ln = C.POINTER(C.c_uint32)(), C.c_size_t()
                t0 = time.perf_counter()
                arr = dl.compress_n(path.encode(), C.byref(enc), C.byref(ln), M, 1)
                dropin = time.perf_counter() - t0
                ok = bool(arr) and ln.value == len(t1)
                if arr:
                    dl.dyn_arr_free(arr)
                    C.CDLL(None).free(enc)
                os.remove(path)
                dropin = {"value": len(m1) / dropin, "unit": "merges/s", "seconds": dropin, "ids_match_one_call": ok,
                          "what": "compress_n(path, &ids, &len, merges, 1) of the drop-in libbpe.so on a file: file read, "
                                  "NUL cut, H2D, training, D2H, dyn_arr vocabulary (bpe.c:541-811)"}
            e2e_paths = {"bpe_cuda_train": {"value": len(m1) / one_call, "unit": "merges/s", "seconds": one_call,
                                            "inside_ms": {k: round(s1[k], 1) for k in ("ms_h2d", "ms_device", "ms_d2h", "ms_total")},
                                            "what": "one call from pageable host memory: context + table creation, H2D, training, "
                                                    "D2H into malloc'd buffers"},
                         "dropin_compress": dropin}
        if not args.no_cpu_baseline:
            if encode_mode:
                v, what = reference_encode_sample(w, table)
                cpu = {"value": v, "unit": "GB/s", "cores": 1, "kind": "port", "sample": what}
            else:
                v, raw, what, kind = reference_train_sample(w, name)
                cpu = {"value": v, "unit": "merges/s", "cores": os.cpu_count(), "kind": kind, "raw_sample_value": raw, "sample": what}
                if encode is not None:
                    merges_np, _ = ctx.download(tokens=False)
                    ev, ewhat = reference_encode_sample(dict(w, ref_bytes=min(128 * MB, w["size"]), ref_merges=32), merges_np)
                    encode["cpu_baseline"] = {"value": ev, "unit": "GB/s", "cores": 1, "kind": "port", "sample": ewhat}

    if rank == 0:
        line = {
            "metric": metric, "value": value, "unit": unit, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": f"{name}: {w['desc']}", "merges": M, "corpus_bytes": n,
                       "shards": world, "final_tokens": int(final_tokens),
                       "l2": "every step starts from the resident byte corpus and re-widens it into a 4 B/token stream (4 GB for "
                             "c3, 400 MB for c2: larger than the 126 MB L2); no flush between steps" if n >= 50 * MB
                       else "stream fits in L2 (parity configuration, not a bandwidth one)"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / args.steps, "steps": args.steps,
                    "path": "bpe_cuda_ctx_upload (pinned host shard) + ctx_train/ctx_encode + ctx_download, per rank"},
            "e2e_paths": e2e_paths,
            "gpu_launches": int(launches),
            "roofline": roofline,
            "cpu_baseline": cpu,
            "encode": encode,
            "c2": c2,
            "checks": checks,
            "engine_stats": {k: sp[k] for k in ("same_bucket_ties", "threshold_edges", "resolver_runs", "census_runs",
                                                 "table_rehashes", "table_capacity", "final_distinct", "replace_passes",
                                                 "batch_merges", "batch_passes")},
        }
        print(json.dumps(line), flush=True)
    ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--workload", default=None, choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="skip the N = 1 extras (c2 block, one-call / drop-in e2e, CPU legs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's merge list and ids to DIR/*.npy "
                                                          "(--impl engine, --gpus 1)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.impl != "engine" or args.gpus != 1):
        ap.error("--dump-outputs writes the engine's result on one GPU: it needs --impl engine and --gpus 1")
    if args.workload is None:
        # The 1/2/4/8 curve is asked for on the 1 GB corpus (BASELINE.json configs[2]); it fits one GPU, so every N runs
        # it and the per-N values are comparable.  Config 2 (100 MB, 1 GPU) is measured inside the N = 1 line ("c2").
        args.workload = os.environ.get("BPE_BENCH_WORKLOAD") or "c3"
    w = dict(WORKLOADS[args.workload])
    if os.environ.get("BPE_BENCH_SCALE"):
        # plumbing test only (tests / dry runs): a smaller corpus of the same kind; the line says so in config.workload
        f = float(os.environ["BPE_BENCH_SCALE"])
        w["size"] = int(w["size"] * f)
        w["desc"] += f" [SCALED x{f}: NOT the named configuration]"
    rank, world, local = dist_setup(args.gpus)
    if args.impl == "reference":
        bench_reference(args, w, rank, world)
    else:
        bench_engine(args, w, rank, world, local)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
