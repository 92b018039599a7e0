#!/usr/bin/env python3
"""Batch-encode fixture: the first 32 MB of config 4's corpus (zipf_bytes, sampling seed 777, config 3's word list) cut
into documents of seeded log-normal lengths (median 1,500 B, sigma 1.0, clipped to [1, 65,536]; tests/batch_cases.py),
each document encoded on its own by the CPU oracle (bo_encode, rank by rank) with config 3's committed 32,000-merge
table.  Writes tests/golden/<name>.json: number of documents and ids, SHA-256 of the ids and of the offsets.

  python tools/make_encode_batch_golden.py c4_docs_encode_batch 32000000 [workers]
"""
import hashlib
import json
import os
import sys
import time
from multiprocessing import Pool

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import batch_cases  # noqa: E402
import oracle_api  # noqa: E402

TABLE = "tests/golden/full/c3_full_merges.npz"
_job = {}


def _init(size):
    _job["data"], _job["off"] = batch_cases.c4_docs(size)
    _job["merges"] = np.load(os.path.join(ROOT, TABLE))["merges"]
    _job["oracle"] = oracle_api.load()


def _encode_range(rng):
    data, off, m, o = _job["data"], _job["off"], _job["merges"], _job["oracle"]
    return [o.encode(data[int(off[i]):int(off[i + 1])], m) for i in range(*rng)]


def main():
    name, size = sys.argv[1], int(sys.argv[2])
    workers = int(sys.argv[3]) if len(sys.argv) > 3 else os.cpu_count()
    _, off = batch_cases.c4_docs(size)
    n = len(off) - 1
    step = 256
    t0 = time.time()
    with Pool(workers, initializer=_init, initargs=(size,)) as pool:
        parts = pool.map(_encode_range, [(i, min(n, i + step)) for i in range(0, n, step)])
    ids = [x for part in parts for x in part]
    tok_off = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum([len(x) for x in ids], out=tok_off[1:])
    flat = np.concatenate(ids).astype("<u4") if ids else np.zeros(0, "<u4")
    out = {"corpus": {"kind": "zipf_bytes", "bytes": size, "seed": 777, "words": 65536},
           "documents": {"lengths": "log-normal, median 1500, sigma 1.0, clipped to [1, 65536], numpy default_rng(777)",
                         "n_docs": n},
           "table": TABLE + " (config 3's 32,000 merges)", "n_ids": int(flat.size),
           "ids_sha256": hashlib.sha256(flat.tobytes()).hexdigest(),
           "offsets_sha256": hashlib.sha256(tok_off.astype("<u8").tobytes()).hexdigest(),
           "made_by": f"tools/make_encode_batch_golden.py (oracle bo_encode per document, {workers} processes)",
           "oracle_seconds": round(time.time() - t0, 1)}
    with open(os.path.join(ROOT, "tests", "golden", name + ".json"), "w") as f:
        json.dump(out, f, indent=1)
    print(out)


if __name__ == "__main__":
    main()
