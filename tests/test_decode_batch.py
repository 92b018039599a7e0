"""decode_batch: every id sequence of a batch decoded on its own, with per-document byte offsets, in one call.  The CPU
part pins the C ABI's argument checks, the Python batch forms, and a restatement of how the kernels compute the byte
offsets; the GPU part compares every document with the oracle's (or the engine's) decode of its ids alone."""
import bisect
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import batch_cases as bc

HERE = os.path.dirname(os.path.abspath(__file__))
TILE = 2048   # DEC_TILE of bpe_decode.cuh: ids per block


def _c3_merges():
    return np.load(os.path.join(HERE, "golden", "full", "c3_full_merges.npz"))["merges"]


# ---- CPU ---------------------------------------------------------------------------------------------------------
def _one_call(lib, ids, off, merges, n_docs=None, outs=(True, True, True)):
    """bpe_cuda_decode_batch on numpy arrays (None: a NULL pointer)"""
    ptr = lambda a: None if a is None else a.ctypes.data
    out, boff, nb = C.POINTER(C.c_uint8)(), C.POINTER(C.c_uint64)(), C.c_size_t()
    if n_docs is None:
        n_docs = 0 if off is None else len(off) - 1
    rc = lib.bpe_cuda_decode_batch(ptr(ids), ptr(off), n_docs, ptr(merges), 0 if merges is None else len(merges),
                                   C.byref(out) if outs[0] else None, C.byref(boff) if outs[1] else None,
                                   C.byref(nb) if outs[2] else None, None)
    if rc == 0:
        lib.bpe_cuda_free(out)
        lib.bpe_cuda_free(boff)
    return rc


def _ctx_call(lib, ids, off, merges, n_docs=None, outs=(True, True)):
    """bpe_cuda_ctx_decode_batch with a NULL context: every argument is checked before the context"""
    ptr = lambda a: None if a is None else a.ctypes.data
    if n_docs is None:
        n_docs = 0 if off is None else len(off) - 1
    boff = np.zeros(max(1, n_docs + 1 if n_docs < 1000 else 1), dtype=np.uint64)
    return lib.bpe_cuda_ctx_decode_batch(None, ptr(ids), ptr(off), n_docs, ptr(merges), 0 if merges is None else len(merges),
                                         boff.ctypes.data if outs[0] else None, C.byref(C.c_size_t()) if outs[1] else None,
                                         None)


def test_argument_errors_through_the_c_abi():
    from llmtokenizer_b200 import _lib
    lib = _lib.load()
    ids = np.array([97, 256, 98, 257, 99], dtype=np.uint32)
    off = np.array([0, 2, 5], dtype=np.uint64)
    good = np.array([[97, 98], [256, 99]], dtype=np.uint32)
    bad = np.array([[97, 98], [257, 99]], dtype=np.uint32)                # rank 1 names id 257
    for call in (_one_call, _ctx_call):
        assert call(lib, ids, None, good) == -1
        assert lib.bpe_cuda_last_error() == b"invalid argument: NULL tok_offsets or merges"
        assert call(lib, None, off, good) == -1
        assert lib.bpe_cuda_last_error() == b"invalid argument: NULL tokens"
        assert call(lib, ids, np.array([0, 4, 3], dtype=np.uint64), good) == -1
        assert lib.bpe_cuda_last_error() == b"invalid argument: tok_offsets[2] < tok_offsets[1] (offsets must not decrease)"
        assert call(lib, ids, off, bad) == -1
        assert lib.bpe_cuda_last_error() == b"merge 1 refers to an id that does not exist yet"   # as decode()
        assert call(lib, ids, off, good, n_docs=2 ** 32 - 1) == -1
        assert b"at most 4,294,967,294" in lib.bpe_cuda_last_error()
    # NULL merges with n_merges > 0
    nb = C.c_size_t()
    assert lib.bpe_cuda_decode_batch(ids.ctypes.data, off.ctypes.data, 2, None, 2, C.byref(C.POINTER(C.c_uint8)()),
                                     C.byref(C.POINTER(C.c_uint64)()), C.byref(nb), None) == -1
    assert lib.bpe_cuda_last_error() == b"invalid argument: NULL tok_offsets or merges"
    boff = np.zeros(3, dtype=np.uint64)
    assert lib.bpe_cuda_ctx_decode_batch(None, ids.ctypes.data, off.ctypes.data, 2, None, 2, boff.ctypes.data, C.byref(nb),
                                         None) == -1
    assert lib.bpe_cuda_last_error() == b"invalid argument: NULL tok_offsets or merges"
    # NULL outputs
    for outs in ((False, True, True), (True, False, True), (True, True, False)):
        assert _one_call(lib, ids, off, good, outs=outs) == -1
        assert lib.bpe_cuda_last_error() == b"invalid argument: NULL output pointer"
    for outs in ((False, True), (True, False)):
        assert _ctx_call(lib, ids, off, good, outs=outs) == -1
        assert lib.bpe_cuda_last_error() == b"invalid argument: NULL output buffer"
    # a valid call: the context is checked last; the one-call form needs a device (no CPU fallback)
    assert _ctx_call(lib, ids, off, good) == -1
    assert lib.bpe_cuda_last_error() == b"invalid argument: NULL context"
    assert _one_call(lib, None, np.array([3, 3], dtype=np.uint64), good) in (0, -4)   # NULL tokens, empty batch: valid
    if lib.bpe_cuda_device_count() == 0:
        assert _one_call(lib, ids, off, good) == -4
        assert _one_call(lib, None, np.array([0], dtype=np.uint64), None) == -4      # an empty batch too


def test_python_batch_forms_agree_on_the_cpu_side():
    """A list of id arrays and an (ids, uint64 offsets) tuple describe the same batch."""
    from llmtokenizer_b200.bpe import _as_id_batch
    docs = [[97, 256], [], np.array([0, 1], dtype=np.uint32), (300,), np.array([5], dtype=np.int64)]
    ids, off = _as_id_batch(docs)
    assert ids.dtype == np.uint32 and ids.tolist() == [97, 256, 0, 1, 300, 5] and off.tolist() == [0, 2, 2, 4, 5, 6]
    assert off.dtype == np.uint64
    i2, o2 = _as_id_batch((ids, off))
    assert i2.tolist() == ids.tolist() and o2.tolist() == off.tolist()
    i3, o3 = _as_id_batch((np.arange(10, dtype=np.uint32), np.array([3, 5, 9], dtype=np.uint64)))   # offsets need not start at 0
    assert i3.size == 10 and o3.tolist() == [3, 5, 9]
    with pytest.raises(ValueError):
        _as_id_batch((ids, np.array([0, 99], dtype=np.uint64)))
    two = (np.array([1, 2], dtype=np.uint32), np.array([3, 4, 5], dtype=np.uint32))   # two documents, not offsets
    i4, o4 = _as_id_batch(two)
    assert i4.tolist() == [1, 2, 3, 4, 5] and o4.tolist() == [0, 2, 5]
    i5, o5 = _as_id_batch([])
    assert i5.size == 0 and o5.tolist() == [0]


def restated_byte_offsets(lens, tok_off, threads, per_thread):
    """The byte offsets as the kernels compute them (bpe_decode.cuh, D4): tile sums and their exclusive scan (D1, D2);
    one binary search per tile for the first entry of tok_off that starts in it (decode_batch_tiles_kernel); per tile, each
    thread's exclusive byte position (s_pos), and per document that thread's position plus at most per_thread - 1
    lengths; documents that start at the end of the batch take the last tile's end.  lens: expansion length of every id
    of the batch.  Returns the offsets and the most lengths read for one document."""
    base, tile = int(tok_off[0]), threads * per_thread
    n = int(tok_off[-1]) - base
    n_ends = len(tok_off)
    if n == 0:
        return [0] * n_ends, 0
    nt = (n + tile - 1) // tile
    sums = [sum(lens[t * tile:(t + 1) * tile]) for t in range(nt)]
    tile_off = [0]
    for s in sums:
        tile_off.append(tile_off[-1] + s)
    tile_doc = [bisect.bisect_left(tok_off, base + t * tile) for t in range(nt)] + [n_ends]
    out, most = [None] * n_ends, 0
    for t in range(nt):
        lo = t * tile
        tile_ids = min(tile, n - lo)
        mine = [sum(lens[lo + k * per_thread:min(lo + tile_ids, lo + (k + 1) * per_thread)]) for k in range(threads)]
        s_pos = np.concatenate([[0], np.cumsum(mine)[:-1]]).astype(np.int64).tolist()
        for i in range(tile_doc[t], tile_doc[t + 1]):
            j = int(tok_off[i]) - base - lo
            assert 0 <= j <= tile_ids and (j < tile_ids or t == nt - 1)
            b = tile_off[t + 1] - tile_off[t]
            if j < tile_ids:
                th = j // per_thread
                b = s_pos[th] + sum(lens[lo + th * per_thread:lo + j])
                most = max(most, j - th * per_thread)
            assert out[i] is None
            out[i] = tile_off[t] + b
    assert None not in out
    return out, most


def test_restated_offsets_equal_the_cumulative_lengths():
    """At small tile and thread sizes: documents starting exactly on tile and thread boundaries, runs of empty
    documents, trailing empties, tok_offsets[0] > 0."""
    rng = np.random.default_rng(4242)
    for trial in range(1500):
        threads, per_thread = int(rng.integers(1, 5)), int(rng.integers(1, 5))
        tile = threads * per_thread
        base = int(rng.integers(0, 3)) * int(rng.integers(0, 7))
        n = int(rng.integers(0, 12 * tile))
        cuts = set(rng.integers(0, n + 1, int(rng.integers(0, 12))).tolist())
        cuts |= {k * tile + d for k in range(n // tile + 1) for d in (-1, 0, 1) if rng.random() < 0.3}
        cuts |= {k * per_thread for k in range(n // per_thread + 1) if rng.random() < 0.2}
        starts = sorted(c for c in cuts if 0 <= c <= n)
        ends = []
        for c in starts:                           # runs of empty documents
            ends += [c] * int(rng.choice([1, 1, 1, 2, 3]))
        if rng.random() < 0.3:
            ends += [n] * int(rng.integers(1, 4))  # trailing empties
        tok_off = [base] + [base + c for c in ends] + [base + n]
        lens = rng.integers(0 if trial % 5 == 0 else 1, 40, n).tolist()
        got, most = restated_byte_offsets(lens, tok_off, threads, per_thread)
        cum = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        assert got == [int(cum[o - base]) for o in tok_off], (threads, per_thread, tok_off)
        assert most <= per_thread - 1


# ---- GPU ---------------------------------------------------------------------------------------------------------
def _docs_of(ids, off):
    return [ids[int(off[i]):int(off[i + 1])] for i in range(len(off) - 1)]


def _check(engine, oracle, docs, merges, expected=None):
    """decode_batch against the oracle's decode of every document alone; the concatenation against decode()."""
    out, boff, st = engine.decode_batch(docs, merges)
    ids, off = engine.bpe._as_id_batch(docs)
    parts = _docs_of(ids, off)
    assert boff.dtype == np.uint64 and boff.shape == (len(parts) + 1,) and boff[0] == 0 and boff[-1] == len(out)
    for i, d in enumerate(parts):
        want = oracle.decode(d, merges) if expected is None else expected[i]
        assert out[int(boff[i]):int(boff[i + 1])] == want, f"document {i} ({len(d)} ids)"
    cat = ids[int(off[0]):int(off[-1])]
    assert out == engine.decode(cat, merges)[0]
    assert st["n_input"] == len(cat) and st["n_tokens"] == len(out) and st["n_merges"] == len(merges)
    return out, boff, st


@pytest.mark.gpu
def test_edge_cases(engine, oracle):
    m = np.array([[0, 0], [97, 98], [256, 256], [257, 0], [99, 99]], dtype=np.uint32)
    out, boff, st = engine.decode_batch([], m)
    assert out == b"" and boff.tolist() == [0] and st["kernel_launches"] == 0
    out, boff, st = engine.decode_batch([[], [], []], m)                        # all documents empty
    assert out == b"" and boff.tolist() == [0, 0, 0, 0] and st["kernel_launches"] == 0
    docs = [[], [], [97, 257], [0, 256, 0], [], [258, 259, 260], [], [98], [259], [], []]
    _check(engine, oracle, docs, m)                                              # empties first, middle, last; 0x00 bytes
    out, _, _ = _check(engine, oracle, [[256], [0, 0]], m)
    assert out == b"\0" * 4
    _check(engine, oracle, [[97, 0, 255], [1, 2]], np.zeros((0, 2), dtype=np.uint32))   # no merges
    # tok_offsets[0] > 0: ids before and after the batch are not read (they are outside the vocabulary here)
    ids = np.array([9999, 9999, 97, 256, 258, 0, 98, 9999], dtype=np.uint32)
    off = np.array([2, 4, 4, 7], dtype=np.uint64)
    out, boff, _ = _check(engine, oracle, (ids, off), m)
    assert boff.tolist() == [0, 3, 3, len(out)]


def _random_table_and_ids(rng, k, n):
    alphabet = rng.choice(256, int(rng.integers(1, 6)), replace=False)
    m = bc.random_table(rng, alphabet, k)
    ids = rng.integers(0, 256 + k, n).astype(np.uint32)
    return m, ids


@pytest.mark.gpu
def test_documents_at_tile_boundaries(engine, oracle):
    """Document starts at 2,048-id tile boundaries +-1, runs of empty documents there, and one document spanning many
    tiles."""
    rng = np.random.default_rng(2048)
    m, ids = _random_table_and_ids(rng, 300, 40 * TILE + 77)
    cuts = []
    for t in (1, 2, 3, 5, 8):
        cuts += [t * TILE - 1, t * TILE, t * TILE, t * TILE + 1]
    cuts += [9 * TILE + 5, 30 * TILE + 3, 40 * TILE, 40 * TILE + 77, 40 * TILE + 77]   # 9..30: one long document
    off = np.array([0] + sorted(cuts), dtype=np.uint64)
    _check(engine, oracle, (ids, off), m)


@pytest.mark.gpu
def test_long_expansions_carry_document_starts(engine, oracle):
    """A vocabulary of doubling runs (a, aa, aaaa, ...): tiles whose output exceeds the 32 KB that are staged in shared
    memory, so the straight-to-global branch of the expand kernel writes the document offsets."""
    k = 12
    m = np.array([[97, 97]] + [[256 + r, 256 + r] for r in range(k - 1)] + [[98, 256 + k - 1]], dtype=np.uint32)
    lens = np.array([1] * 256 + [2 ** (r + 1) for r in range(k)] + [1 + 2 ** k], dtype=np.int64)
    rng = np.random.default_rng(7)
    ids = rng.integers(0, 256 + k + 1, 5 * TILE + 100).astype(np.uint32)
    tile_bytes = [int(lens[ids[t * TILE:(t + 1) * TILE]].sum()) for t in range(5)]   # the five full tiles
    assert min(tile_bytes) > 32 * 1024
    cuts = sorted(rng.integers(0, len(ids), 60).tolist() + [TILE, TILE, 3 * TILE - 1, 4 * TILE + 1, len(ids)])
    off = np.array([0] + cuts, dtype=np.uint64)
    _check(engine, oracle, (ids, off), m)


@pytest.mark.gpu
def test_random_batches_against_the_oracle(engine, oracle):
    rng = np.random.default_rng(31337)
    for trial in range(6):
        k = int(rng.integers(0, 500))
        n_docs = int(rng.integers(1, 400))
        lens = rng.integers(0, 3 * TILE if trial % 2 else 60, n_docs)
        lens[rng.random(n_docs) < 0.15] = 0
        m, ids = _random_table_and_ids(rng, k, int(lens.sum()))
        docs = _docs_of(ids, np.concatenate([[0], np.cumsum(lens)]))
        _check(engine, oracle, docs, m)


@pytest.mark.gpu
def test_round_trip_of_config4_documents(engine):
    """About 2 MB of config 4's corpus as log-normal documents, config 3's 32,000-merge table: decode_batch of
    encode_batch gives back every document up to its first NUL, and the offsets are their lengths."""
    data, off = bc.c4_docs(2_000_000, len_seed=3)
    data = data.copy()
    data[::9973] = 0                                          # some documents end early
    m = _c3_merges()
    ids, toff, _ = engine.encode_batch((data, off), m)
    out, boff, st = engine.decode_batch((ids, toff), m)
    docs = [bc.nul_cut(data[int(off[i]):int(off[i + 1])]) for i in range(len(off) - 1)]
    assert boff.tolist() == np.concatenate([[0], np.cumsum([len(d) for d in docs])]).tolist()
    assert out == b"".join(docs)
    assert st["table_rehashes"] == 1


@pytest.mark.gpu
def test_round_trip_of_the_committed_document_set(engine):
    """The 12,807 documents of tests/golden/c4_docs_encode_batch.json (32 MB): the ids are the committed ones, and
    decoding them per document gives back the documents."""
    g = json.load(open(os.path.join(HERE, "golden", "c4_docs_encode_batch.json")))
    data, off = bc.c4_docs(g["corpus"]["bytes"])
    m = _c3_merges()
    ids, toff, _ = engine.encode_batch((data, off), m)
    assert hashlib.sha256(ids.astype("<u4").tobytes()).hexdigest() == g["ids_sha256"]
    out, boff, _ = engine.decode_batch((ids, toff), m)
    docs = [bc.nul_cut(data[int(off[i]):int(off[i + 1])]) for i in range(len(off) - 1)]
    assert len(docs) == g["documents"]["n_docs"]
    assert boff.tolist() == np.concatenate([[0], np.cumsum([len(d) for d in docs])]).tolist()
    assert out == b"".join(docs)


@pytest.mark.gpu
def test_out_of_vocabulary_id(engine, oracle):
    m = np.array([[97, 98], [256, 99]], dtype=np.uint32)
    docs = [[97], [], [256, 257], [98, 258, 97], [], [300]]                     # 258 is the first id outside (258 entries)
    with pytest.raises(engine.BpeCudaError) as e:
        engine.decode_batch(docs, m)
    assert e.value.rc == -1 and "document 3 holds id 258" in str(e.value)
    ctx = engine.Context(0)
    try:
        with pytest.raises(engine.BpeCudaError) as e:
            ctx.decode_batch(docs, m)
        assert e.value.rc == -1 and "document 3 holds id 258" in str(e.value)
        good = [[97], [], [256, 257], [98, 97]]
        out, boff, _ = ctx.decode_batch(good, m)                                  # the context is still usable
        assert out == b"a" + b"ab" + b"abc" + b"ba" and boff.tolist() == [0, 1, 1, 6, 8]
    finally:
        ctx.close()


@pytest.mark.gpu
def test_launch_count_does_not_depend_on_the_batch(engine):
    rng = np.random.default_rng(5)
    m, ids = _random_table_and_ids(rng, 100, 4_000_000)
    small = _docs_of(ids[:2560], np.arange(0, 2561, 256))
    lens = rng.integers(0, 40, 100_000)
    big = (ids, np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64))
    _, _, s1 = engine.decode_batch(small, m)
    _, boff, s2 = engine.decode_batch(big, m)
    assert len(boff) == 100_001
    assert s1["kernel_launches"] == s2["kernel_launches"] == 4


@pytest.mark.gpu
def test_context_keeps_the_vocabulary_and_the_resident_state(engine, oracle):
    rng = np.random.default_rng(99)
    alphabet = np.frombuffer(b"abcd", dtype=np.uint8)
    shard = rng.choice(alphabet, 200_000).astype(np.uint8)
    m1 = bc.random_table(rng, alphabet, 300)
    m2 = bc.random_table(rng, alphabet, 300)
    lens = rng.integers(0, 500, 300)
    ids = rng.integers(0, 556, int(lens.sum())).astype(np.uint32)
    docs = (ids, np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64))
    parts = _docs_of(*docs)
    exp = {id(m): [oracle.decode(d, m) for d in parts] for m in (m1, m2)}
    ctx = engine.Context(0)
    try:
        ctx.upload(shard)
        ctx.train(64)
        trained = ctx.download()
        assert ctx.decode(trained[0]) == shard.tobytes() and ctx.decode_mismatches() == 0
        rebuilt = []
        for m in (m1, m1, m2, m1, m1):                    # alternating lists, and a repeated one
            out, boff, st = ctx.decode_batch(docs, m)
            rebuilt.append(st["table_rehashes"])
            assert [out[int(boff[i]):int(boff[i + 1])] for i in range(len(parts))] == exp[id(m)]
            got = ctx.download()
            assert np.array_equal(got[0], trained[0]) and np.array_equal(got[1], trained[1])
        assert rebuilt == [1, 0, 1, 1, 0]
        assert ctx.decode(trained[0]) == shard.tobytes() and ctx.decode_mismatches() == 0   # between batch decodes
        nb, boff, st = ctx.decode_batch(docs, m2, download=False)                          # bytes stay on the device
        assert st["table_rehashes"] == 1 and nb == boff[-1] == sum(len(x) for x in exp[id(m2)])
        buf = np.zeros(nb, dtype=np.uint8)
        assert ctx.lib.bpe_cuda_ctx_decode_download(ctx.h, buf.ctypes.data) == 0
        assert buf.tobytes() == b"".join(exp[id(m2)])
        assert ctx.decode_batch(docs, m2)[2]["table_rehashes"] == 0
        assert ctx.decode(trained[0], download=False) == len(shard) and ctx.decode_mismatches() == 0
        ctx.train(64)                                      # the resident shard is still the one uploaded
        assert np.array_equal(ctx.download()[0], trained[0])
    finally:
        ctx.close()
