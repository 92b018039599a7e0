"""TEST INFRASTRUCTURE: the seeded inputs of the heavier parity cases and their committed oracle results.

The CPU oracle (oracle/, pinned against the compiled reference) needs seconds to minutes for these inputs; the
`-m gpu` suite has a fixed time budget on the GPU box, so the oracle's answers are computed offline by
tools/make_case_digests.py and committed under tests/golden/cases/KEY.npz (merge list, SHA-256 of the ids, the
oracle's tie / threshold counters and its 16 worker-table bucket counts).  A case without a committed file is
computed inline (slow path, same check)."""
import hashlib
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASE_DIR = os.path.join(ROOT, "tests", "golden", "cases")


def corpus(kind, size, seed):
    from llmtokenizer_b200 import _lib
    lib = _lib.load_corpus()
    buf = np.zeros(size, dtype=np.uint8)
    assert lib.gen_corpus_fill(kind, buf.ctypes.data, size, seed, 50000 if kind == 0 else 65536) == 0
    return buf


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype="<u4").tobytes()).hexdigest()


def _random_text():
    import gzip
    with gzip.open(os.path.join(ROOT, "tests", "golden", "random_text.txt.gz"), "rb") as f:
        return np.frombuffer(f.read(), dtype=np.uint8)


def _rt_big():
    rt = _random_text()
    return np.concatenate([rt, rt[::-1], rt[:300000]])  # 2.4 M tokens, dynamic regime throughout


def _ranged(ranges, i):
    rng = np.random.default_rng(1000 + ranges)
    cases = [rng.integers(97, 100, 1_300_000, dtype=np.uint8),
             np.repeat(rng.integers(97, 101, 500_000, dtype=np.uint8), rng.integers(1, 5, 500_000))[:1_200_000]]
    return cases[i] if i < 2 else corpus(0, 1_500_000, 31 + ranges)


def _runs(P):
    rng = np.random.default_rng(P)
    return np.repeat(rng.integers(97, 100, 400_000, dtype=np.uint8), rng.integers(1, 30, 400_000))[:4_000_001]


def _tie_heavy(copies=60):
    # the 20 KB random-text prefix (9 same-bucket ties when trained alone) repeated past 1,048,576 tokens with a
    # different separator byte between the copies: trained to exhaustion the late merges tie all the time
    rt = _random_text()[:20000]
    parts = []
    for k in range(copies):
        parts.append(rt[(k * 37) % 500:])
        parts.append(np.array([1 + k % 31], dtype=np.uint8))
    return np.concatenate(parts)


def _wide_ties(n=88_000):
    # n random bytes from 1..255, twice: nearly every pair count is 2, so every iteration is a hash-table tie-break.
    # Trained to exhaustion each copy collapses to one token after about 70,300 merges, so ids past 65,535 are born
    # in the static regime (the stream never holds more than 2 n tokens)
    r = np.random.default_rng(65536).integers(1, 256, n, dtype=np.uint8)
    return np.concatenate([r, r])


# key -> (input factory, merge cap [0 = to exhaustion])
TRAIN_CASES = {
    "zipfa6m_300": (lambda: corpus(0, 6_000_000, 99), 300),
    "zipfb5m_150": (lambda: corpus(1, 5_000_000, 98), 150),
    "rt2p4m_120": (_rt_big, 120),
    "zipfa12m_2500": (lambda: corpus(0, 12_000_000, 71), 2500),
    "zipfb8m_2200": (lambda: corpus(1, 8_000_000, 72), 2200),
    "zipfa9m_2000": (lambda: corpus(0, 9_000_000, 73), 2000),
    "zipfa12m_10000": (lambda: corpus(0, 12_000_000, 11), 10000),
    "uniform14m_2600": (lambda: np.random.default_rng(4).integers(33, 127, 14_000_000, dtype=np.uint8), 2600),
    "zipfa8m_200": (lambda: corpus(0, 8_000_000, 7), 200),
    "zipfb6m_100": (lambda: corpus(1, 6_000_000, 8), 100),
    "zipfa12m_1300": (lambda: corpus(0, 12_000_000, 71), 1300),
    "same3m_1": (lambda: np.full(3_000_003, 120, dtype=np.uint8), 1),
    "zipfa3m_300": (lambda: corpus(0, 3_000_000, 9), 300),
    # steep counts (byte-level Zipf): a handful of pairs above half the maximum, candidate lists that run empty
    "zipfb3m_1500": (lambda: corpus(1, 3_000_000, 55), 1500),
    # stream that falls below 1,048,576 tokens (the reference's static slicing, bpe.c:449) while merges share passes
    "cross1m_400": (lambda: corpus(0, 1_400_000, 21), 400),
    # tie-heavy, to exhaustion, above and below the static limit
    "ties1m2_exh": (_tie_heavy, 0),
    # 4.3 M tokens that stay above the static limit for all 1,000 merges, 4 of them same-bucket ties
    "ties4m_1000": (lambda: _tie_heavy(220), 1000),
    # ids past 65,535 (70,306 merges, 3,599 same-bucket ties), all born in the static regime
    "wideties88k_exh": (_wide_ties, 0),
}
for _r in (1, 5, 64, 0):
    for _i in range(3):
        TRAIN_CASES[f"ranged{_r}_{_i}"] = ((lambda r=_r, i=_i: _ranged(r, i)), 60)
for _P in (2, 4, 8):
    TRAIN_CASES[f"runs4m_12_P{_P}"] = ((lambda P=_P: _runs(P)), 12)

# key -> (train case whose merges are applied, input factory): what oracle.encode(other, merges) returns
ENCODE_CASES = {
    "enc_zipfa12m_2500": ("zipfa12m_2500", lambda: corpus(0, 3_000_000, 171)),
    "enc_zipfb8m_2200": ("zipfb8m_2200", lambda: corpus(1, 3_000_000, 172)),
    "enc_zipfa9m_2000": ("zipfa9m_2000", lambda: corpus(0, 3_000_000, 173)),
    "enc_zipfa12m_10000": ("zipfa12m_10000", lambda: corpus(0, 400_000, 12)),
    "enc_zipfa3m_300": ("zipfa3m_300", lambda: corpus(0, 2_000_001, 10)),
}


def train_input(key):
    return TRAIN_CASES[key][0](), TRAIN_CASES[key][1]


def _path(key):
    return os.path.join(CASE_DIR, key + ".npz")


def compute_train(oracle, key):
    import oracle_api
    data, cap = train_input(key)
    rc, m, t, st = oracle.train(data, cap, oracle_api.FAST_CF)
    assert rc == 0, (key, rc)
    return {"merges": m.astype(np.uint32), "n_ids": len(t), "ids_sha256": sha(t), "same_bucket_ties": int(st["same_bucket_ties"]),
            "threshold_edges": int(st["threshold_edges"]), "thread_buckets": np.asarray(st["thread_buckets"], dtype=np.uint64),
            "cap": cap, "n_input": int(data.size)}


def compute_encode(oracle, key):
    tkey, make = ENCODE_CASES[key]
    m = expected_train(tkey, oracle)["merges"]
    data = make()
    t = oracle.encode(data, m)
    return {"n_ids": len(t), "ids_sha256": sha(t), "n_input": int(data.size), "train_case": tkey}


def save(key, d):
    os.makedirs(CASE_DIR, exist_ok=True)
    np.savez_compressed(_path(key), **{k: np.asarray(v) for k, v in d.items()})


def _load(key):
    z = np.load(_path(key))
    d = {}
    for k in z.files:
        v = z[k]
        d[k] = v if v.ndim else v.item()
    return d


def expected_train(key, oracle=None):
    """The oracle's result for TRAIN_CASES[key]: committed file, else computed now."""
    if os.path.exists(_path(key)):
        d = _load(key)
        d["thread_buckets"] = [int(x) for x in d["thread_buckets"]]
        return d
    assert oracle is not None, f"no committed oracle result for {key}"
    d = compute_train(oracle, key)
    d["thread_buckets"] = [int(x) for x in d["thread_buckets"]]
    return d


def expected_encode(key, oracle=None):
    if os.path.exists(_path(key)):
        return _load(key)
    assert oracle is not None, f"no committed oracle result for {key}"
    return compute_encode(oracle, key)
