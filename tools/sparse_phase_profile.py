#!/usr/bin/env python3
"""Where a config-3 training step spends its device time, pass kind by pass kind.

Trains bench.py's config 3 (1 GB byte-level Zipf corpus, 32,000 merges) on one GPU: a warm-up run, then one run with
the engine's per-launch CUDA events on (`profile_replace`).  Prints, per phase, the total and the mean per pass, plus
the steps that were enqueued speculatively and fell through, and writes the same as one JSON object together with the
card's name, power limit and SM clocks read in the same call.

  python tools/sparse_phase_profile.py [--workload c3] [--warmup 1] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PHASES = ("dense_pass_ms", "sparse_scan_ms", "apply_ms", "select_ms", "gap_ms", "convert_ms")


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        return {"query": q, "value": None}
    return {"query": q, "value": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c3")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None, help="write the JSON object here as well")
    args = ap.parse_args()

    import bench
    import llmtokenizer_b200 as L
    from llmtokenizer_b200 import _lib
    assert _lib.load().bpe_cuda_device_count() > 0, "no CUDA device: the engine has no CPU fallback"
    w = bench.WORKLOADS[args.workload]
    _, shard = bench.make_shard(w, 0, 1)
    ctx = L.Context(0)
    ctx.upload_ptr(shard.ctypes.data, shard.size)
    for _ in range(args.warmup):
        ctx.train(w["merges"])
    ctx.set_option("profile_replace", 1)
    st = ctx.train(w["merges"])
    ctx.set_option("profile_replace", 0)
    merges, _ = ctx.download(tokens=False)
    ctx.close()

    passes, sparse = st["replace_passes"], st["sparse_passes"]
    dense = passes - sparse
    per_pass = {"dense_pass_ms": dense, "sparse_scan_ms": sparse}
    phases = {}
    for k in PHASES:
        n = per_pass.get(k, passes)
        phases[k] = {"ms": st[k], "per_pass_us": 1e3 * st[k] / n if n else None, "passes": n}
    res = {
        "workload": w["desc"],
        "card": card(),
        "ms_device": st["ms_device"],
        "n_merges": st["n_merges"],
        "passes": passes, "dense_passes": dense, "sparse_passes": sparse,
        "steps_enqueued": st["replace_launches"],
        "steps_fell_through": st["replace_launches"] - passes,
        "kernel_launches": st["kernel_launches"],
        "replace_ms": st["replace_ms"],
        "phases": phases,
        "sparse_entries": st["sparse_entries"],
        "sparse_replacements": st["sparse_replacements"],
        "merges_digest": bench.hashlib.sha256(merges.tobytes()).hexdigest()[:16],
        "how": "one profiled run after warm-up; CUDA events on the engine's stream after every launch of a step (host "
               "gaps are the intervals that end at the start of a step or of a conversion); per-pass means divide by "
               "the passes of that kind (all passes for apply / select / gap / convert)",
    }
    for k in PHASES:
        p = phases[k]
        print(f"{k:16s} {p['ms']:9.1f} ms  {p['per_pass_us'] or 0:8.1f} us/pass over {p['passes']} passes", file=sys.stderr)
    print(f"steps enqueued {res['steps_enqueued']}, fell through {res['steps_fell_through']}, sparse entries checked "
          f"{res['sparse_entries']} for {res['sparse_replacements']} replacements, kernel launches {res['kernel_launches']}", file=sys.stderr)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
