#!/usr/bin/env python3
"""Encode fixtures: a chunk of a zipf_bytes corpus (config 3's word list, sampling seed as given) encoded with a committed
merge table by the CPU oracle (bo_encode: bpe.c:760-772 rank by rank, one thread).  Writes tests/golden/<name>.json (digest
of the ids).  The table is a tests/golden/full/<table>_merges.npz, config 3's 32,000 merges by default.

  python tools/make_encode_golden.py c4_chunk0_encode 125000000 777                     # about half an hour
  python tools/make_encode_golden.py c4_2m_encode_c5_70k 2000000 777 c5_chunk0_70k      # config 5's chunk, 70,000 merges
"""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracle_api  # noqa: E402
from parity_cases import corpus, sha  # noqa: E402


def main():
    name, size, seed = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])
    tname = sys.argv[4] if len(sys.argv) > 4 else "c3_full"
    table = f"tests/golden/full/{tname}_merges.npz"
    merges = np.load(os.path.join(ROOT, table))["merges"]
    data = corpus(1, size, seed)
    t0 = time.time()
    ids = oracle_api.load().encode(data, merges)
    what = " (config 3's 32,000 merges)" if tname == "c3_full" else f" ({len(merges):,} merges)"
    out = {"corpus": {"kind": "zipf_bytes", "bytes": size, "seed": seed, "words": 65536},
           "table": table + what, "ranks": int(len(merges)), "n_ids": int(len(ids)),
           "ids_sha256": sha(ids), "made_by": f"tools/make_encode_golden.py {' '.join(sys.argv[1:])} (oracle bo_encode, 1 thread)",
           "oracle_seconds": round(time.time() - t0, 1)}
    with open(os.path.join(ROOT, "tests", "golden", name + ".json"), "w") as f:
        json.dump(out, f, indent=1)
    print(out)


if __name__ == "__main__":
    main()
