#!/usr/bin/env python3
"""encode_batch on one GPU: three seeded document mixes encoded with config 3's 32,000-merge table.

  (a) docs   the first 256 MB of config 4's corpus cut into log-normal documents (median 1,500 B, sigma 1.0, clipped to
             [1, 65,536]): the 256 MB version of tests/golden/c4_docs_encode_batch.json
  (b) tiny   64 MB of the same corpus as documents of 32-256 B, where the fixed cost of a document dominates
  (c) long   256 MB as documents of 256 KB - 4 MB, all in the global-memory tier (about 30 s per call on a B200: no
             separate one-call run)
  docs8k     (a) with the lengths clipped to 8,192 (every document in shared memory): how much of (a)'s time is the
             global-memory tier's tail

Per mix: warm-up calls, then --steps timed calls of Context.encode_batch (the rank table is built once and kept);
documents/s and input GB/s from the CUDA-event time of the kernels (median over steps), and one one-call
encode_batch() end to end (context set-up, copies and all).  A seeded sample of each mix is checked: 200 documents
against the CPU oracle for (a) and (b); for (c), whose documents take the oracle minutes each, 8 documents against
encode() of the document alone (encode() is pinned to the oracle by the test suite).

Baselines for scale: the per-document path (Context.upload + encode + download) on the first 100 documents of (a), and
the whole-stream encode() of (a)'s concatenation (different semantics: merges cross document boundaries).

  python tools/encode_batch_bench.py --workloads docs,tiny,long,docs8k --steps 3 --warmup 1 \
      --out profiles/encode_batch_b200.json          (the committed run; about 4 minutes of one GPU)
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import batch_cases as bc  # noqa: E402
import llmtokenizer_b200 as L  # noqa: E402
from parity_cases import corpus  # noqa: E402


def uniform_docs(total, lo, hi, seed):
    rng = np.random.default_rng(seed)
    lens = rng.integers(lo, hi + 1, total // lo + 1)
    off = np.concatenate([[0], np.cumsum(lens)])
    k = int(np.searchsorted(off, total))
    off = off[:k + 1].copy()
    off[k] = total
    return off.astype(np.uint64)


def workloads(which):
    out = {}
    if "docs" in which:
        out["docs"] = bc.c4_docs(256_000_000)
    if "tiny" in which:
        out["tiny"] = (corpus(1, 64_000_000, 778), uniform_docs(64_000_000, 32, 256, 5))
    if "docs8k" in which:
        out["docs8k"] = (corpus(1, 256_000_000, 777), bc.lognormal_docs(256_000_000, 777, hi=8192))
    if "long" in which:
        out["long"] = (corpus(1, 256_000_000, 779), uniform_docs(256_000_000, 256 << 10, 4 << 20, 6))
    return out


def gpu_card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def check_sample(name, data, off, ids, toff, merges, oracle):
    n = len(off) - 1
    rng = np.random.default_rng(2024)
    k = 8 if name == "long" else 200
    pick = np.sort(rng.choice(n, min(k, n), replace=False))
    for i in pick:
        doc = data[int(off[i]):int(off[i + 1])]
        want = L.encode(doc, merges)[0] if name == "long" else oracle.encode(doc, merges)
        if not np.array_equal(ids[int(toff[i]):int(toff[i + 1])], want):
            return False, int(i)
    return True, len(pick)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--workloads", default="docs,tiny,long")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from llmtokenizer_b200 import _lib
    if _lib.load().bpe_cuda_device_count() < 1:
        sys.exit("encode_batch_bench needs a GPU")
    import oracle_api
    oracle = oracle_api.load()
    merges = np.load(os.path.join(ROOT, "tests", "golden", "full", "c3_full_merges.npz"))["merges"]
    res = {"gpu": gpu_card(), "table": "config 3's 32,000 merges", "steps": args.steps, "warmup": args.warmup,
           "workloads": {}}
    mixes = workloads(args.workloads.split(","))
    ctx = L.Context(0)
    for name, (data, off) in mixes.items():
        n_docs = len(off) - 1
        for _ in range(args.warmup):
            ctx.encode_batch((data, off), merges)
        dev, tot = [], []
        for _ in range(args.steps):
            ids, toff, st = ctx.encode_batch((data, off), merges)
            dev.append(st["ms_device"])
            tot.append(st["ms_total"])
        ms = float(np.median(dev))
        one_call, st1, same = None, None, None
        if name != "long":
            t0 = time.perf_counter()
            ids1, toff1, st1 = L.encode_batch((data, off), merges)
            one_call = round((time.perf_counter() - t0) * 1e3, 2)
            st1 = {k: round(st1[k], 2) for k in ("ms_h2d", "ms_device", "ms_d2h", "ms_total")}
            same = bool(np.array_equal(ids1, ids) and np.array_equal(toff1, toff))
        ok, info = check_sample(name, data, off, ids, toff, merges, oracle)
        lens = np.diff(off.astype(np.int64))
        res["workloads"][name] = {
            "bytes": int(off[-1]), "n_docs": n_docs, "doc_len_median": float(np.median(lens)), "doc_len_max": int(lens.max()),
            "n_ids": int(len(ids)), "kernel_launches": st["kernel_launches"],
            "ms_device_median": round(ms, 3), "ms_device_all": [round(x, 3) for x in dev],
            "docs_per_s": round(n_docs / (ms / 1e3), 1), "input_GB_per_s": round(st["n_input"] / (ms / 1e3) / 1e9, 4),
            "ctx_call_ms_median": round(float(np.median(tot)), 2),
            "one_call_ms": one_call, "one_call_stats_ms": st1,
            "one_call_equals_ctx": same,
            "sample_check": {"ok": ok, ("checked" if ok else "first_mismatch"): info,
                             "against": "encode() per document" if name == "long" else "oracle per document"}}
        print(name, json.dumps(res["workloads"][name]), flush=True)
    if "docs" in mixes:
        data, off = mixes["docs"]
        t0 = time.perf_counter()
        for i in range(100):
            ctx.upload(data[int(off[i]):int(off[i + 1])])
            ctx.encode(merges)
            ctx.download(merges=False)
        dt = time.perf_counter() - t0
        ids, st = L.encode(data, merges)
        res["baselines"] = {
            "per_document_upload_encode_download": {"n_docs": 100, "bytes": int(off[100]), "seconds": round(dt, 3),
                                                    "docs_per_s": round(100 / dt, 1)},
            "whole_stream_encode_of_docs_concat": {"bytes": int(off[-1]), "ms_device": round(st["ms_device"], 2),
                                                   "input_GB_per_s": round(st["n_input"] / (st["ms_device"] / 1e3) / 1e9, 4),
                                                   "note": "merges cross document boundaries: for scale only"}}
        print("baselines", json.dumps(res["baselines"]), flush=True)
    ctx.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
