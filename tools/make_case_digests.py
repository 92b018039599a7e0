#!/usr/bin/env python3
"""Compute the CPU oracle's results for the heavier parity cases (tests/parity_cases.py) and commit them under
tests/golden/cases/: the -m gpu suite then compares the engine with these instead of running the oracle inline
on the GPU box (fixed time budget there).

  python tools/make_case_digests.py [-j 4] [--force] [KEY ...]
"""
import os
import sys
import time
from concurrent.futures import ProcessPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def one(key):
    import oracle_api
    import parity_cases as pc
    t0 = time.time()
    o = oracle_api.load()
    if key in pc.TRAIN_CASES:
        d = pc.compute_train(o, key)
        info = f"{len(d['merges'])} merges, {d['n_ids']} ids, ties {d['same_bucket_ties']}, edges {d['threshold_edges']}"
    else:
        d = pc.compute_encode(o, key)
        info = f"{d['n_ids']} ids"
    d["made_by"] = f"tools/make_case_digests.py {key} (oracle FAST_CF mode, 1 thread)"
    d["oracle_seconds"] = round(time.time() - t0, 1)
    pc.save(key, d)
    return key, time.time() - t0, info


def main():
    import parity_cases as pc
    args = sys.argv[1:]
    force = "--force" in args
    jobs = 4
    if "-j" in args:
        jobs = int(args[args.index("-j") + 1])
        del args[args.index("-j"):args.index("-j") + 2]
    keys = [a for a in args if not a.startswith("-")]
    train = [k for k in pc.TRAIN_CASES if (not keys or k in keys) and (force or not os.path.exists(pc._path(k)))]
    enc = [k for k in pc.ENCODE_CASES if (not keys or k in keys) and (force or not os.path.exists(pc._path(k)))]
    for group in (train, enc):   # encode cases need their train case's merges
        with ProcessPoolExecutor(jobs) as ex:
            for key, dt, info in ex.map(one, group):
                print(f"{key:24s} {dt:8.1f} s  {info}", flush=True)


if __name__ == "__main__":
    main()
