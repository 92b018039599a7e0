"""encode_batch: every document encoded on its own, in one call.  The CPU part pins the algorithm the batch kernel
implements (min-rank-first, and its select-and-compact scan) against the oracle and the C ABI's argument checks; the
GPU part compares the kernel with the oracle per document."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import batch_cases as bc

HERE = os.path.dirname(os.path.abspath(__file__))
WARP_CAP, BLOCK_CAP, TILE = 512, 8192, 4096   # tier limits of bpe_encode_batch.cuh


def _c3_merges():
    return np.load(os.path.join(HERE, "golden", "full", "c3_full_merges.npz"))["merges"]


def _random_case(rng, max_len=60, max_k=30):
    alphabet = rng.choice(256, int(rng.integers(1, 5)), replace=False)
    n = int(rng.integers(0, max_len + 1))
    doc = bytearray(rng.choice(alphabet, n).astype(np.uint8).tobytes())
    if n and rng.random() < 0.2:
        doc[int(rng.integers(n))] = 0
    return bytes(doc), bc.random_table(rng, alphabet, int(rng.integers(0, max_k + 1)))


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_min_rank_first_equals_rank_by_rank(oracle):
    """The restatement the kernel implements equals the oracle's rank-by-rank encode: tiny alphabets, a == b pairs,
    repeated pairs, NULs, empty and 1-byte documents."""
    rng = np.random.default_rng(20261020)
    for _ in range(4000):
        doc, m = _random_case(rng)
        assert bc.min_rank_first(doc, m) == oracle.encode(doc, m).tolist(), (doc, m.tolist())


def test_min_rank_first_on_a_real_vocabulary(oracle):
    data, off = bc.c4_docs(200_000)
    m = _c3_merges()
    for i in range(6):
        doc = data[int(off[i]):int(off[i + 1])]
        assert bc.min_rank_first(doc, m) == oracle.encode(doc, m).tolist()


def test_scan_select_and_compact_equals_greedy_pass():
    """The kernel's step 2 (segment summaries, one scan per tile, a carry between tiles, in-place writes) restated:
    the same output as the reference's greedy pass, runs of a == b included, at many tile shapes."""
    rng = np.random.default_rng(7)
    for _ in range(3000):
        al = int(rng.integers(1, 4))
        toks = rng.integers(0, al, int(rng.integers(0, 90))).tolist()
        a = int(rng.integers(0, al))
        b = a if rng.random() < 0.4 else int(rng.integers(0, al))
        items, threads = int(rng.integers(1, 5)), int(rng.integers(1, 5))
        assert bc.scan_replace(toks, a, b, 99, items, threads) == bc.greedy_replace(toks, a, b, 99)


def test_segmented_cascade_equals_rank_by_rank(oracle):
    """The global-memory tier's segment-local form (compaction inside segments, per-segment minimum ranks, a selected
    last pair reaching into the next non-empty segment) restated at tiny segment sizes, where segments empty out."""
    rng = np.random.default_rng(11)
    for _ in range(2000):
        alphabet = rng.choice(np.arange(1, 256), int(rng.integers(1, 4)), replace=False)
        doc = rng.choice(alphabet, int(rng.integers(0, 120))).astype(np.uint8).tobytes()
        m = bc.random_table(rng, alphabet, int(rng.integers(0, 40)))
        assert bc.segmented_cascade(doc, m, int(rng.integers(1, 9))) == oracle.encode(doc, m).tolist()


def _abi_call(lib, data, off, merges, tokens=True):
    """bpe_cuda_encode_batch on numpy arrays (None: a NULL pointer)"""
    ptr = lambda a: None if a is None else a.ctypes.data
    toks, toff, nt = C.POINTER(C.c_uint32)(), C.POINTER(C.c_uint64)(), C.c_size_t()
    rc = lib.bpe_cuda_encode_batch(ptr(data), ptr(off), 0 if off is None else len(off) - 1, ptr(merges),
                                   0 if merges is None else len(merges), C.byref(toks) if tokens else None,
                                   C.byref(toff), C.byref(nt), None)
    if rc == 0:
        lib.bpe_cuda_free(toks)
        lib.bpe_cuda_free(toff)
    return rc


def test_argument_errors_through_the_c_abi():
    from llmtokenizer_b200 import _lib
    lib = _lib.load()
    data = np.frombuffer(b"abcabcab", dtype=np.uint8)
    good = np.array([[97, 98], [256, 99]], dtype=np.uint32)
    off = np.array([0, 3, 8], dtype=np.uint64)
    assert _abi_call(lib, data, np.array([0, 5, 3], dtype=np.uint64), good) == -1
    assert b"must not decrease" in lib.bpe_cuda_last_error()
    assert _abi_call(lib, data, None, good) == -1                        # NULL offsets
    assert _abi_call(lib, None, off, good) == -1                         # NULL bytes, non-empty batch
    assert _abi_call(lib, data, off, good, tokens=False) == -1           # NULL output
    rc = lib.bpe_cuda_encode_batch(data.ctypes.data, off.ctypes.data, 2, None, 2, C.byref(C.POINTER(C.c_uint32)()),
                                   C.byref(C.POINTER(C.c_uint64)()), C.byref(C.c_size_t()), None)
    assert rc == -1                                                       # NULL merges, n_merges > 0
    bad = np.array([[97, 98], [257, 99]], dtype=np.uint32)                # rank 1 names id 257
    assert _abi_call(lib, data, off, bad) == -1
    assert lib.bpe_cuda_last_error() == b"merge 1 refers to an id that does not exist yet"   # as bpe_cuda_ctx_encode
    assert lib.bpe_cuda_ctx_encode_batch(None, data.ctypes.data, off.ctypes.data, 2, good.ctypes.data, 2, None, None,
                                         None) == -1
    if lib.bpe_cuda_device_count() == 0:
        assert _abi_call(lib, data, off, good) == -4                     # no CPU fallback
        assert _abi_call(lib, data, np.array([0], dtype=np.uint64), None) == -4   # an empty batch too


def test_python_batch_forms_agree_on_the_cpu_side():
    """A list of bytes-like objects and an (array, offsets) tuple describe the same batch."""
    from llmtokenizer_b200.bpe import _as_batch
    docs = [b"ab", b"", bytearray(b"c\x00d"), np.frombuffer(b"xyz", dtype=np.uint8)]
    data, off = _as_batch(docs)
    assert data.tobytes() == b"abc\x00dxyz" and off.tolist() == [0, 2, 2, 5, 8]
    d2, o2 = _as_batch((data, off))
    assert d2.tobytes() == data.tobytes() and o2.tolist() == off.tolist()
    with pytest.raises(ValueError):
        _as_batch((data, np.array([0, 99], dtype=np.uint64)))
    two = (np.frombuffer(b"ab", dtype=np.uint8), np.frombuffer(b"cde", dtype=np.uint8))   # two documents, not offsets
    d3, o3 = _as_batch(two)
    assert d3.tobytes() == b"abcde" and o3.tolist() == [0, 2, 5]


# ---- GPU ---------------------------------------------------------------------------------------------------------
def _check_batch(engine, oracle, docs, merges, expected=None):
    ids, off, st = engine.encode_batch(docs, merges)
    assert off.shape == (len(docs) + 1,) and off[0] == 0 and off[-1] == len(ids)
    for i, d in enumerate(docs):
        want = oracle.encode(d, merges) if expected is None else expected[i]
        assert np.array_equal(ids[off[i]:off[i + 1]], want), f"document {i} (length {len(d)})"
    assert st["n_tokens"] == len(ids) and st["n_merges"] == len(merges)
    assert st["n_input"] == sum(len(bc.nul_cut(d)) for d in docs)
    return ids, off, st


@pytest.mark.gpu
def test_edge_cases(engine, oracle):
    m = np.array([[97, 98], [97, 97], [256, 99], [258, 258], [97, 98], [120, 97]], dtype=np.uint32)
    ids, off, st = engine.encode_batch([], m)
    assert len(ids) == 0 and off.tolist() == [0] and st["n_tokens"] == 0
    docs = [b"", b"\x00", b"\x00abab", b"a", b"z", b"ab", b"abc\x00abc", b"a" * 1001, b"a" * 4096, b"a" * 9000 + b"bc",
            b"abcabc" * 300, b"xa", b"by", b""]
    _check_batch(engine, oracle, docs, m)
    _check_batch(engine, oracle, docs, np.zeros((0, 2), dtype=np.uint32))          # no merges: the bytes themselves
    # concatenation merges across the boundary of "xa" | "by", the batch does not
    m2 = np.array([[97, 98]], dtype=np.uint32)
    ids, off, _ = engine.encode_batch([b"xa", b"by"], m2)
    assert ids.tolist() == [120, 97, 98, 121] and off.tolist() == [0, 2, 4]
    cat, _ = engine.encode(b"xaby", m2)
    assert cat.tolist() == [120, 256, 121]


def _tier_lengths():
    out = []
    for lim in (WARP_CAP, BLOCK_CAP, TILE, 2 * TILE + TILE // 2):
        out += [lim - 1, lim, lim + 1]
    return out + [0, 1, 2, 31, 32, 33, 200, 3000, 20000]


@pytest.mark.gpu
def test_random_batches_against_the_oracle(engine, oracle):
    rng = np.random.default_rng(31337)
    for trial in range(6):
        alphabet = rng.choice(np.arange(1, 256), int(rng.integers(2, 6)), replace=False)
        lens = _tier_lengths() + rng.integers(0, 3000, 40).tolist()
        rng.shuffle(lens)
        docs = []
        for n in lens:
            d = bytearray(rng.choice(alphabet, n).astype(np.uint8).tobytes())
            if n > 2 and rng.random() < 0.1:
                d[int(rng.integers(n))] = 0
            docs.append(bytes(d))
        k = int(rng.integers(50, 400))
        if trial % 2:
            m = bc.random_table(rng, alphabet, k)
        else:   # a learned table (no occurrences missing) over a sample of the same alphabet
            _, m, _, _ = oracle.train(rng.choice(alphabet, 20000).astype(np.uint8), k)
        _check_batch(engine, oracle, docs, m)


@pytest.mark.gpu
def test_real_vocabulary_against_the_oracle(engine, oracle):
    """1 MB of config 4's corpus cut into about 2,000 documents (log-normal, median 300 B) with config 3's 32,000-merge
    table, every document against the oracle."""
    from parity_cases import corpus
    data = corpus(1, 1_000_000, 777)
    off = bc.lognormal_docs(len(data), 11, median=300)
    docs = [data[int(off[i]):int(off[i + 1])] for i in range(len(off) - 1)]
    assert len(docs) >= 1500
    _check_batch(engine, oracle, docs, _c3_merges())


@pytest.mark.gpu
def test_global_memory_tier(engine, oracle):
    """Documents far beyond shared memory (segment-local cascade) with config 3's whole 32,000-rank table: 1 MB and
    4 MB equal to encode() of each document alone, which is pinned to the oracle with this table on 125 MB of the
    same corpus; 100 KB, 1 MB (first 1,500 ranks) and long a == b runs against the oracle inline."""
    from parity_cases import corpus
    m = _c3_merges()
    docs = [corpus(1, 1_000_000, 4001), corpus(1, 4_000_000, 4002), b"ab" * 5000 + b"b" * 3001]
    ids, off, st = engine.encode_batch(docs, m)
    for i, d in enumerate(docs):
        want, _ = engine.encode(d, m)
        assert np.array_equal(ids[off[i]:off[i + 1]], want), f"document {i}"
    _check_batch(engine, oracle, [corpus(1, 100_000, 4003), docs[2], b"a" * 50_001], m)
    _check_batch(engine, oracle, docs[:1], m[:1500])


@pytest.mark.gpu
def test_config4_documents_match_the_committed_digest(engine):
    """32 MB of config 4's corpus as 12,807 documents of log-normal lengths, encoded with config 3's table: the digest
    of the oracle's per-document ids (tests/golden/c4_docs_encode_batch.json, tools/make_encode_batch_golden.py)."""
    g = json.load(open(os.path.join(HERE, "golden", "c4_docs_encode_batch.json")))
    data, off = bc.c4_docs(g["corpus"]["bytes"])
    assert len(off) - 1 == g["documents"]["n_docs"]
    ids, toff, st = engine.encode_batch((data, off), _c3_merges())
    assert len(ids) == g["n_ids"]
    assert hashlib.sha256(ids.astype("<u4").tobytes()).hexdigest() == g["ids_sha256"]
    assert hashlib.sha256(toff.astype("<u8").tobytes()).hexdigest() == g["offsets_sha256"]


@pytest.mark.gpu
def test_context_batches_keep_the_resident_state(engine, oracle):
    rng = np.random.default_rng(99)
    alphabet = np.frombuffer(b"abcd", dtype=np.uint8)
    docs = [rng.choice(alphabet, int(n)).astype(np.uint8).tobytes() for n in rng.integers(0, 3000, 300)]
    m1 = bc.random_table(rng, alphabet, 300)
    m2 = bc.random_table(rng, alphabet, 300)
    shard = rng.choice(alphabet, 200_000).astype(np.uint8)
    ctx = engine.Context(0)
    try:
        ctx.upload(shard)
        ctx.train(64)
        trained = ctx.download()
        exp1 = [oracle.encode(d, m1) for d in docs]
        exp2 = [oracle.encode(d, m2) for d in docs]
        launches = []
        for m, exp in ((m1, exp1), (m1, exp1), (m2, exp2), (m1, exp1)):   # same table, then another, then back
            ids, off, st = ctx.encode_batch(docs, m)
            launches.append(st["kernel_launches"])
            for i in range(len(docs)):
                assert np.array_equal(ids[off[i]:off[i + 1]], exp[i])
            got = ctx.download()
            assert np.array_equal(got[0], trained[0]) and np.array_equal(got[1], trained[1])
        assert launches[1] == launches[0] - 1 and launches[2] == launches[0] and launches[3] == launches[0]
        ctx.encode(m1)                                     # a stream encode in between
        enc = ctx.download()[1]
        ids, off, _ = ctx.encode_batch(docs[:20], m1)
        for i in range(20):
            assert np.array_equal(ids[off[i]:off[i + 1]], exp1[i])
        assert np.array_equal(ctx.download()[1], enc)
        assert np.array_equal(enc, oracle.encode(shard, m1))
        ctx.train(64)
        assert np.array_equal(ctx.download()[0], trained[0])
    finally:
        ctx.close()


@pytest.mark.gpu
def test_launch_count_does_not_depend_on_the_batch(engine):
    rng = np.random.default_rng(5)
    m = bc.random_table(rng, np.frombuffer(b"ab", dtype=np.uint8), 100)
    small = [rng.integers(97, 99, 50).astype(np.uint8).tobytes() for _ in range(10)]
    big = [rng.integers(97, 99, int(n)).astype(np.uint8).tobytes() for n in rng.integers(0, 2000, 10_000)]
    _, _, s1 = engine.encode_batch(small, m)
    _, _, s2 = engine.encode_batch(big, _c3_merges())
    assert s1["kernel_launches"] == s2["kernel_launches"] > 0


@pytest.mark.gpu
def test_round_trip(engine):
    data, off = bc.c4_docs(2_000_000, len_seed=3)
    data = data.copy()
    data[::9973] = 0                                          # some documents end early
    m = _c3_merges()
    ids, toff, _ = engine.encode_batch((data, off), m)
    back, _ = engine.decode(ids, m)
    assert back == b"".join(bc.nul_cut(data[int(off[i]):int(off[i + 1])]) for i in range(len(off) - 1))
