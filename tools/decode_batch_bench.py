#!/usr/bin/env python3
"""decode_batch on one GPU: the document mixes of tools/encode_batch_bench.py, encoded with config 3's 32,000-merge
table by encode_batch, then decoded per document.

  (a) docs   the first 256 MB of config 4's corpus cut into log-normal documents (median 1,500 B, sigma 1.0, clipped to
             [1, 65,536])
  (b) tiny   64 MB of the same corpus as documents of 32-256 B, where the per-document work weighs most

Per mix:
  - Context.decode_batch: warm-up calls, then --steps timed calls with the vocabulary kept on the context; documents/s
    and output GB/s from the CUDA-event time of the kernels (median over the steps).  Its output is checked once
    against the documents (cut at their first NUL) and their lengths.
  - the floor: plain decode() of the same concatenated ids, whose kernels are those of Context.decode (D1-D3; the
    context form decodes only a context's resident stream, so it cannot take these ids); its CUDA-event kernel time,
    median over --steps calls after the same warm-up.  decode() sets up a fresh context per call, so the one-call
    decode_batch() of the same batch is timed the same way, and ratio = one-call batch / floor compares like with like.
  - a small batch (64 sequences of 256 ids): per-call wall time of Context.decode_batch with the vocabulary cached
    (median of 50 calls) against the one-call decode_batch() (median of 10 calls: context set-up, vocabulary flatten and
    upload, copies and all).
  - with --kernels, after the timed calls: per-kernel device time of decode() and of Context.decode_batch on the same
    batch, from torch.profiler (3 calls each, kept out of the timed windows because tracing slows the host).
Every timed call reads the ids (about 300 MB for (a)) and writes the bytes (256 MB) afresh; (b)'s 75 MB of ids and
64 MB of output partly stay in the 126 MB L2 from one call to the next.  The card's name and power limit are read in
the same run.

  python tools/decode_batch_bench.py --steps 5 --warmup 2 --kernels --out profiles/decode_batch_b200.json
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import batch_cases as bc  # noqa: E402
import llmtokenizer_b200 as L  # noqa: E402
from encode_batch_bench import gpu_card, uniform_docs  # noqa: E402
from parity_cases import corpus  # noqa: E402


def workloads(which):
    out = {}
    if "docs" in which:
        out["docs"] = bc.c4_docs(256_000_000)
    if "tiny" in which:
        out["tiny"] = (corpus(1, 64_000_000, 778), uniform_docs(64_000_000, 32, 256, 5))
    return out


def check(data, off, out, boff):
    docs = [bc.nul_cut(data[int(off[i]):int(off[i + 1])]) for i in range(len(off) - 1)]
    lens_ok = np.array_equal(boff, np.concatenate([[0], np.cumsum([len(d) for d in docs])]).astype(np.uint64))
    return bool(lens_ok and out == b"".join(docs))


def kernel_us(f, calls=3):
    """microseconds of device time per call of each kernel f launches (torch.profiler, CUDA activity)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        for _ in range(calls):
            f()
    return {e.key.split("(")[0]: round(e.device_time_total / calls, 1) for e in p.key_averages()
            if e.device_time_total > 0 and "kernel" in e.key}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--workloads", default="docs,tiny")
    ap.add_argument("--kernels", action="store_true", help="also profile the kernels (a separate pass)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from llmtokenizer_b200 import _lib
    if _lib.load().bpe_cuda_device_count() < 1:
        sys.exit("decode_batch_bench needs a GPU")
    merges = np.load(os.path.join(ROOT, "tests", "golden", "full", "c3_full_merges.npz"))["merges"]
    res = {"gpu": gpu_card(), "table": "config 3's 32,000 merges", "steps": args.steps, "warmup": args.warmup,
           "workloads": {}}
    ctx = L.Context(0)
    for name, (data, off) in workloads(args.workloads.split(",")).items():
        ids, toff, _ = ctx.encode_batch((data, off), merges)
        batch = (ids, toff)
        n_docs = len(toff) - 1
        out, boff, _ = ctx.decode_batch(batch, merges)
        ok = check(data, off, out, boff)
        del out
        for _ in range(args.warmup):
            ctx.decode_batch(batch, merges, download=False)
            L.decode(ids, merges)
            L.decode_batch(batch, merges)
        dev, tot, floor, one = [], [], [], []
        for _ in range(args.steps):
            nb, _, st = ctx.decode_batch(batch, merges, download=False)
            dev.append(st["ms_device"])
            tot.append(st["ms_total"])
            floor.append(L.decode(ids, merges)[1]["ms_device"])
            one.append(L.decode_batch(batch, merges)[2]["ms_device"])
        ms, ms_floor, ms_one = float(np.median(dev)), float(np.median(floor)), float(np.median(one))
        # a small batch with the vocabulary cached, against the one-call form
        small = (ids[:64 * 256], np.arange(0, 64 * 256 + 1, 256, dtype=np.uint64))
        ctx.decode_batch(small, merges)
        ctx_ms, one_ms = [], []
        for _ in range(50):
            t0 = time.perf_counter()
            s_out, _, _ = ctx.decode_batch(small, merges)
            ctx_ms.append((time.perf_counter() - t0) * 1e3)
        for _ in range(10):
            t0 = time.perf_counter()
            o_out, _, _ = L.decode_batch(small, merges)
            one_ms.append((time.perf_counter() - t0) * 1e3)
        res["workloads"][name] = {
            "bytes": int(nb), "n_docs": n_docs, "n_ids": int(len(ids)), "kernel_launches": st["kernel_launches"],
            "ms_device_median": round(ms, 4), "ms_device_all": [round(x, 4) for x in dev],
            "docs_per_s": round(n_docs / (ms / 1e3), 1), "output_GB_per_s": round(nb / (ms / 1e3) / 1e9, 3),
            "ctx_call_ms_median": round(float(np.median(tot)), 3),
            "floor_plain_decode_ms_device_median": round(ms_floor, 4), "floor_ms_device_all": [round(x, 4) for x in floor],
            "one_call_batch_ms_device_median": round(ms_one, 4), "one_call_batch_ms_device_all": [round(x, 4) for x in one],
            "ratio_one_call_batch_over_plain": round(ms_one / ms_floor, 3), "ratio_ctx_batch_over_plain": round(ms / ms_floor, 3),
            "small_batch": {"sequences": 64, "ids_each": 256, "ctx_call_ms_median": round(float(np.median(ctx_ms)), 4),
                            "one_call_ms_median": round(float(np.median(one_ms)), 4), "same_bytes": s_out == o_out},
            "check_against_documents": ok}
        if args.kernels:
            res["workloads"][name]["kernel_us_per_call"] = {
                "decode": kernel_us(lambda: L.decode(ids, merges)),
                "ctx_decode_batch": kernel_us(lambda: ctx.decode_batch(batch, merges, download=False))}
        print(name, json.dumps(res["workloads"][name]), flush=True)
    ctx.close()
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
