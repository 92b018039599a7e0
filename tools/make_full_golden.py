#!/usr/bin/env python3
"""Full-length parity fixtures that keep the MERGE LIST itself (so a test can compare any prefix of it) plus the
SHA-256 of the final ids.  Runs the CPU oracle (oracle/, pinned against the compiled reference) offline; hours for
the 1 GB corpus.

  python tools/make_full_golden.py c1_exhaustion                       # random_text.txt to exhaustion (config 1)
  python tools/make_full_golden.py c3_full 1000000000 4321 32000 1     # name, bytes, seed, merges, kind (1 = zipf_bytes)
  python tools/make_full_golden.py c5_chunk0_70k 125000000 8888 70000 1   # ids past 65,535 (22 minutes, 8 threads)

BO_WORKERS=n (default: all cores) splits the oracle's two whole-array loops over helper threads (same results,
tests/test_oracle.py); the 1 GB corpus then takes about an hour instead of most of a day.
"""
import ctypes
import gzip
import hashlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracle_api  # noqa: E402
from llmtokenizer_b200 import _lib  # noqa: E402


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype="<u4").tobytes()).hexdigest()


def main():
    name = sys.argv[1]
    if len(sys.argv) >= 6:
        size, seed, merges, kind = (int(x) for x in sys.argv[2:6])
        words = 50000 if kind == 0 else 65536
        buf = np.zeros(size, dtype=np.uint8)
        assert _lib.load_corpus().gen_corpus_fill(kind, buf.ctypes.data, size, seed, words) == 0
        corpus = {"kind": "zipf_ascii" if kind == 0 else "zipf_bytes", "bytes": size, "seed": seed, "words": words}
    else:
        with gzip.open(os.path.join(ROOT, "tests", "golden", "random_text.txt.gz"), "rb") as f:
            buf = np.frombuffer(f.read(), dtype=np.uint8)
        merges = int(sys.argv[2]) if len(sys.argv) > 2 else 0
        corpus = {"kind": "file", "file": "tests/golden/random_text.txt.gz", "bytes": int(buf.size)}
    t0 = time.time()
    orc = oracle_api.load()
    workers = int(os.environ.get("BO_WORKERS", os.cpu_count() or 1))
    orc.lib.bo_set_workers.argtypes = [ctypes.c_int, ctypes.c_size_t]
    orc.lib.bo_set_workers(workers, 1 << 22)
    rc, m, ids, st = orc.train(buf, merges, oracle_api.FAST_CF)
    assert rc == 0
    out = {"corpus": corpus, "cap": merges, "merges": int(len(m)), "n_ids": int(len(ids)), "merges_sha256": sha(m),
           "ids_sha256": sha(ids), "same_bucket_ties": int(st["same_bucket_ties"]),
           "threshold_edges": int(st["threshold_edges"]), "final_distinct": int(st["final_distinct"]),
           "thread_buckets": [int(x) for x in st["thread_buckets"]],
           "made_by": f"tools/make_full_golden.py {' '.join(sys.argv[1:])} (oracle FAST_CF mode, {workers} helper threads)",
           "oracle_seconds": round(time.time() - t0, 1)}
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "full", name + "_merges.npz"), merges=m.astype(np.uint32))
    with open(os.path.join(ROOT, "tests", "golden", name + ".json"), "w") as f:
        json.dump(out, f, indent=1)
    print(out)


if __name__ == "__main__":
    main()
