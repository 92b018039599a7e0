"""Vocabularies past 65,536 ids: training, encode, encode_batch, decode and decode_batch where ids no longer fit 16 bits.

Three oracle results cross the boundary:
  (A) parity_cases "wideties88k_exh": 88,000 random bytes twice, to exhaustion in the static regime (70,306 merges, ids up
      to 70,560, 3,599 same-bucket ties);
  (B) config 5's first 125 MB chunk to 70,000 merges (tests/golden/c5_chunk0_70k.json + full/): id 65,536 is born inside
      batched passes on a stream of tens of millions of tokens;
  (C) a foreign table made here from a seed, whose ids past 65,535 alias a byte or an early id in their low 16 bits.
The CPU part checks that the fixtures cross the boundary and that a kernel which looked pairs up by the low 16 bits of the
ids would fail the GPU part (a model of such a kernel differs from the oracle on the very inputs used there), plus the
vocabulary checks of the C ABI at the boundary.  Every GPU test asserts that what it compared holds ids >= 65,536."""
import ctypes as C
import heapq
import json
import os

import numpy as np
import pytest

import batch_cases as bc
import parity_cases as pc
from parity_cases import corpus, sha
from test_gpu_parity import _full_golden, assert_case, check_result

HERE = os.path.dirname(os.path.abspath(__file__))
WIDE = 1 << 16                 # the first id that does not fit 16 bits
WIDE_RANK = WIDE - 256         # its rank (65,280)
TIER_LENGTHS = (511, 512, 513, 8191, 8192, 8193)   # WARP_CAP and BLOCK_CAP of bpe_encode_batch.cuh, +-1
C4_TEXT = (2_000_000, 777)     # config 4's corpus: the first 2 MB, encoded with (B)'s table


def _c5_70k():
    return _full_golden("c5_chunk0_70k")


# ---- (C): a foreign table whose wide ids alias bytes and early ids ------------------------------------------------
def _t(p, q):
    """id of the byte pair (p, q), p and q in 1..255, in the table below"""
    return 256 + (p - 1) * 255 + (q - 1)


def foreign_wide_table(n_wide=2000, seed=65536):
    """(merges, named ids) of a valid table of 65,280 + n_wide + 5 ranks:
      ranks 0 .. 65,024       every ordered pair of bytes 1..255, (p, q) at rank (p-1)*255 + q-1.  A pair (low, high)
                              (p <= 127 < q) ranks below every pair that starts with a high byte, so a text of such pairs
                              collapses to their ids first
      ranks 65,025 .. 65,279  255 distinct pairs of those (low, high) ids: ids 65,281 .. 65,535
      rank 65,280             (65,535, T): id 65,536; rank 65,281: (65,536, 65,536): id 65,537
      ranks up to n_wide      distinct pairs of (low, high) ids: id 65,536 + k for k < n_wide, which a 16-bit lookup takes
                              for byte k (k < 256) or for the early id k
      5 more                  pairs that a 16-bit lookup sees as an earlier pair: (65,536 + 97, 98) ('a' 'b' is rank 24,577),
                              (x, x) for x = 65,536 + 200 and 65,537, and (65,536 + (1, 130), T') where ((1, 130), T') is
                              rank 65,025
    Expansions stay at most 16 bytes, so decode's flattened vocabulary is about 1 MB."""
    rng = np.random.default_rng(seed)
    m = [(a, b) for a in range(1, 256) for b in range(1, 256)]
    used = set()

    def fresh_pair(first=None):
        while True:
            a = first if first is not None else _t(int(rng.integers(1, 128)), int(rng.integers(128, 256)))
            b = _t(int(rng.integers(1, 128)), int(rng.integers(128, 256)))
            if (a, b) not in used:
                used.add((a, b))
                return a, b

    ta, tb, tc = _t(3, 200), _t(5, 140), _t(9, 255)
    used |= {(tb, tc), (tc, ta), (tc, tc)}     # 65,536 and 65,537 must spell as intended
    level2 = [fresh_pair(_t(1, 130))] + [fresh_pair() for _ in range(253)]
    used.add((ta, tb))
    level2.append((ta, tb))                   # id 65,535
    m += level2
    assert len(m) == WIDE_RANK
    m += [(WIDE - 1, tc), (WIDE, WIDE)]       # ids 65,536 and 65,537
    m += [fresh_pair() for _ in range(n_wide - 2)]
    ids = {"last_narrow": WIDE - 1, "first_wide": WIDE, "second_wide": WIDE + 1, "alias_a": WIDE + 97,
           "alias_200": WIDE + 200, "alias_tok": WIDE + _t(1, 130)}
    specials = {"a_then_b": (WIDE + 97, 98), "xx_200": (WIDE + 200, WIDE + 200), "xx_65537": (WIDE + 1, WIDE + 1),
                "alias_tok_pair": (WIDE + _t(1, 130), level2[0][1])}
    for name, pair in specials.items():
        ids[name] = 256 + len(m)
        m.append(pair)
    return np.array(m, dtype=np.uint32), ids


def _vocab(merges):
    v = [bytes([i]) for i in range(256)]
    for a, b in np.asarray(merges).tolist():
        v.append(v[a] + v[b])
    return v


def foreign_wide_phrases(merges, ids):
    """Byte strings whose encoding with the table is the named wide id, or a wide id next to a token that a 16-bit lookup
    would merge with it.  A phrase that ends in 'b' (a low byte) must end its document: 'b' would pair with the first
    byte of a following phrase."""
    v = _vocab(merges)
    inner = [v[ids[k]] for k in ("last_narrow", "first_wide", "second_wide", "alias_tok")]
    inner += [v[WIDE + 200] + bytes([201]),                      # (65,736, 201): no rank; (200, 201) has one
              v[WIDE + 200] * 2, v[WIDE + 1] * 3,              # (x, x) pairs, an odd run
              v[ids["alias_tok"]] + v[merges[WIDE_RANK - 255][1]]]
    return inner, v[WIDE + 97] + b"b"


def foreign_wide_text(merges, ids, n, seed):
    """n bytes of phrases, random wide ids (their 4-byte spellings), narrow ids and loose high bytes"""
    rng = np.random.default_rng(seed)
    v = _vocab(merges)
    inner, _ = foreign_wide_phrases(merges, ids)
    parts, size = [], 0
    while size < n:
        u = rng.random()
        if u < 0.15:
            p = inner[int(rng.integers(len(inner)))]
        elif u < 0.65:
            p = v[WIDE + int(rng.integers(2, len(merges) - WIDE_RANK - 5))]
        elif u < 0.85:
            p = v[_t(int(rng.integers(1, 128)), int(rng.integers(128, 256)))]
        else:
            p = bytes([int(rng.integers(128, 256))])
        parts.append(p)
        size += len(p)
    return b"".join(parts)[:n]


def foreign_wide_docs(merges, ids):
    """the (C) documents: every phrase alone, texts at every tier length, one for the global-memory tier"""
    inner, tail = foreign_wide_phrases(merges, ids)
    docs = inner + [tail, inner[0] + inner[4] + tail]
    docs += [foreign_wide_text(merges, ids, n - len(tail), n) + tail if n % 2 else foreign_wide_text(merges, ids, n, n)
             for n in TIER_LENGTHS]
    docs.append(foreign_wide_text(merges, ids, 60_000, 60_000))
    return docs


# ---- a model of a kernel that looks pairs up by the low 16 bits of the ids ------------------------------------------
def truncating_encode(doc, merges, mask=0xFFFF):
    """min-rank-first (batch_cases.min_rank_first, which equals rank-by-rank encoding) with the pair -> rank lookup keyed
    by (a & mask, b & mask): what a kernel gives that keeps 16-bit ids in its pair table.  mask=None: the exact lookup,
    i.e. the oracle.  The ids it writes are not truncated.  One step takes every pair of the smallest rank present (from a
    heap of (rank, position) entries, checked against the tokens when taken) and merges them left to right, a pair
    whose first token was consumed by its left neighbour being skipped: the greedy rule of a run of equal tokens."""
    key = (lambda a, b: (a & mask, b & mask)) if mask is not None else (lambda a, b: (a, b))
    table = {}
    for r, (a, b) in enumerate(np.asarray(merges, dtype=np.int64).reshape(-1, 2).tolist()):
        table.setdefault(key(a, b), r)
    tok = list(bc.nul_cut(doc))
    n = len(tok)
    nxt, prv, alive = list(range(1, n + 1)), list(range(-1, n - 1)), [True] * n
    heap = []

    def push(p):
        q = nxt[p]
        r = table.get(key(tok[p], tok[q])) if q < n else None
        if r is not None:
            heapq.heappush(heap, (r, p, tok[p], tok[q]))

    for p in range(n - 1):
        push(p)
    while heap:
        r = heap[0][0]
        done = []
        while heap and heap[0][0] == r:            # popped in position order
            _, p, a, b = heapq.heappop(heap)
            q = nxt[p]
            if not alive[p] or q >= n or tok[p] != a or tok[q] != b or (done and done[-1] == p):
                continue
            tok[p] = 256 + r
            alive[q] = False
            nxt[p] = nxt[q]
            if nxt[q] < n:
                prv[nxt[q]] = p
            done.append(p)
        for p in done:                             # the pairs the step made
            push(p)
            if prv[p] >= 0:
                push(prv[p])
    return np.array([tok[p] for p in range(n) if alive[p]], dtype=np.uint32)


def c5_alias_phrases(oracle, merges):
    """(phrase, z): byte strings that encode to [..., z, b] with the table, a wide id z = 65,536 + k (k < 256) left next
    to its last byte b although (k, b) is a merge of the table, which a 16-bit lookup would apply"""
    v = _vocab(merges)
    ranked = set(map(tuple, np.asarray(merges[:WIDE_RANK]).tolist()))
    out = []
    for k in range(256):
        for b in range(1, 256):
            if (k, b) in ranked:
                ph = v[WIDE + k] + bytes([b])
                if oracle.encode(ph, merges)[-2:].tolist() == [WIDE + k, b]:
                    out.append((ph, WIDE + k))
                    break
    return out


def c5_docs(oracle, merges):
    """config 5's corpus cut at every tier length, each document ending in one of the phrases above (the first one that
    keeps its z next to b after the text in front of it), and one document for the global-memory tier with 64 phrases
    inside"""
    ph = c5_alias_phrases(oracle, merges)
    data = corpus(1, 200_000, 8888).tobytes()
    docs, pos, j = [], 0, 0
    for n in TIER_LENGTHS:
        while True:
            p, z = ph[j]
            j += 1
            d = data[pos:pos + n - len(p)] + p
            if oracle.encode(d, merges)[-2:].tolist() == [z, p[-1]]:
                break
        docs.append(d)
        pos += n
    docs.append(b"".join(data[pos + 1000 * i:pos + 1000 * (i + 1)] + ph[i][0] for i in range(64)))
    return docs


# ---- CPU -----------------------------------------------------------------------------------------------------------
def test_fixtures_cross_the_boundary():
    exp = pc.expected_train("wideties88k_exh")
    assert len(exp["merges"]) == 70_306 > WIDE_RANK and int(exp["merges"].max()) >= WIDE
    assert exp["n_ids"] == 2 and exp["same_bucket_ties"] == 3599
    g = _c5_70k()
    m = g["merge_list"]
    assert len(m) == g["merges"] == g["cap"] > WIDE_RANK and int(m.max()) >= WIDE and sha(m) == g["merges_sha256"]
    m50 = _full_golden("c5_chunk0_50k")["merge_list"]
    assert np.array_equal(m[:50_000], m50)
    mc, _ = foreign_wide_table()
    assert len(mc) > WIDE_RANK and int(mc.max()) >= WIDE


def test_foreign_wide_table_spells_what_it_says(oracle):
    """The (C) phrases encode to the ids they are built for, and 65,535 .. 65,537 occur."""
    m, ids = foreign_wide_table()
    assert all(a < 256 + r and b < 256 + r for r, (a, b) in enumerate(m.tolist()))
    v = _vocab(m)
    for name, x in ids.items():
        assert oracle.encode(v[x], m).tolist() == [x], name
    seen = set()
    for d in foreign_wide_docs(m, ids):
        seen |= set(oracle.encode(d, m).tolist())
    assert {WIDE - 1, WIDE, WIDE + 1} <= seen and max(seen) >= WIDE + 2000


def test_truncating_lookup_would_fail_the_gpu_inputs(oracle):
    """The model with the exact lookup is the oracle; with 16-bit keys it differs from the oracle on the (C) documents and
    on config 5's documents with (B)'s table, so a kernel that truncates cannot pass the GPU tests below."""
    m, ids = foreign_wide_table()
    docs = foreign_wide_docs(m, ids)
    for i, d in enumerate(docs):
        want = oracle.encode(d, m)
        assert np.array_equal(truncating_encode(d, m, mask=None), want), i
        # the first four phrases spell 65,535, 65,536, 65,537 and 65,921 without a wide id in a lookup; every other
        # document holds a pair that the 16-bit lookup takes for an earlier one
        assert np.array_equal(truncating_encode(d, m), want) == (i < 4), i
    mb = _c5_70k()["merge_list"]
    assert len(c5_alias_phrases(oracle, mb)) >= 64
    for i, d in enumerate(c5_docs(oracle, mb)):
        want = oracle.encode(d, mb)
        assert np.array_equal(truncating_encode(d, mb, mask=None), want), i
        assert not np.array_equal(truncating_encode(d, mb), want), i


def _decode_batch_call(lib, ids, off, merges):
    out, boff, nb = C.POINTER(C.c_uint8)(), C.POINTER(C.c_uint64)(), C.c_size_t()
    rc = lib.bpe_cuda_decode_batch(ids.ctypes.data, off.ctypes.data, len(off) - 1, merges.ctypes.data, len(merges),
                                   C.byref(out), C.byref(boff), C.byref(nb), None)
    if rc == 0:
        lib.bpe_cuda_free(out)
        lib.bpe_cuda_free(boff)
    return rc


def _decode_call(lib, ids, merges):
    out, nb = C.POINTER(C.c_uint8)(), C.c_size_t()
    rc = lib.bpe_cuda_decode(ids.ctypes.data, len(ids), merges.ctypes.data, len(merges), C.byref(out), C.byref(nb), None)
    if rc == 0:
        lib.bpe_cuda_free(out)
    return rc


def _encode_batch_call(lib, data, off, merges):
    toks, toff, nt = C.POINTER(C.c_uint32)(), C.POINTER(C.c_uint64)(), C.c_size_t()
    rc = lib.bpe_cuda_encode_batch(data.ctypes.data, off.ctypes.data, len(off) - 1, merges.ctypes.data, len(merges),
                                   C.byref(toks), C.byref(toff), C.byref(nt), None)
    if rc == 0:
        lib.bpe_cuda_free(toks)
        lib.bpe_cuda_free(toff)
    return rc


def test_vocabulary_checks_of_the_abi_at_the_boundary():
    """A merge list of n ranks is a vocabulary of 256 + n ids.  Rank r may name ids up to 256 + r - 1: 65,535 at rank
    65,280 and 65,536 at rank 65,281 are accepted, the id being defined (256 + r) is not.  Ids of a decoded stream are
    checked on the device: the last id, 256 + n - 1 >= 65,536, decodes; 256 + n is rejected with -1.  Without a device
    every call that passes the argument checks returns -4."""
    from llmtokenizer_b200 import _lib
    lib = _lib.load()
    has_gpu = lib.bpe_cuda_device_count() > 0
    m, _ = foreign_wide_table()
    n = len(m)
    last = np.array([WIDE - 1, 256 + n - 1], dtype=np.uint32)
    off = np.array([0, 1, 2], dtype=np.uint64)
    data = np.frombuffer(b"abc", dtype=np.uint8)
    doff = np.array([0, 3], dtype=np.uint64)
    assert m[WIDE_RANK].tolist() == [WIDE - 1, m[WIDE_RANK][1]] and m[WIDE_RANK + 1].tolist() == [WIDE, WIDE]
    for r, pair in ((WIDE_RANK, (WIDE, 97)), (WIDE_RANK + 1, (97, WIDE + 1)), (n - 1, (256 + n - 1, 98))):
        bad = m[:r + 1].copy()
        bad[r] = pair                                  # names the id rank r defines
        for call in (lambda: _decode_batch_call(lib, last[:1], off[:2], bad),
                     lambda: _encode_batch_call(lib, data, doff, bad)):
            assert call() == -1
            assert lib.bpe_cuda_last_error() == f"merge {r} refers to an id that does not exist yet".encode()
        boff = np.zeros(2, dtype=np.uint64)
        assert lib.bpe_cuda_ctx_decode_batch(None, last.ctypes.data, off.ctypes.data, 1, bad.ctypes.data, len(bad),
                                             boff.ctypes.data, C.byref(C.c_size_t()), None) == -1
        assert b"refers to an id that does not exist yet" in lib.bpe_cuda_last_error()
    # the argument checks pass: the context is checked last
    boff = np.zeros(3, dtype=np.uint64)
    assert lib.bpe_cuda_ctx_decode_batch(None, last.ctypes.data, off.ctypes.data, 2, m.ctypes.data, n, boff.ctypes.data,
                                         C.byref(C.c_size_t()), None) == -1
    assert lib.bpe_cuda_last_error() == b"invalid argument: NULL context"
    over = np.array([WIDE - 1, 256 + n], dtype=np.uint32)
    if has_gpu:
        assert _decode_batch_call(lib, last, off, m) == 0 and _decode_call(lib, last, m) == 0
        assert _decode_batch_call(lib, over, off, m) == -1
        assert lib.bpe_cuda_last_error() == f"decode_batch: document 1 holds id {256 + n}, outside the vocabulary ({256 + n} entries)".encode()
        assert _decode_call(lib, over, m) == -1
        assert _encode_batch_call(lib, data, doff, m) == 0
    else:
        assert _decode_batch_call(lib, last, off, m) == -4
        assert _decode_call(lib, last, m) == -4
        assert _encode_batch_call(lib, data, doff, m) == -4


# ---- GPU -----------------------------------------------------------------------------------------------------------
def _device_count():
    from llmtokenizer_b200 import _lib
    return _lib.load().bpe_cuda_device_count()


def _wide(ids):
    """ids >= 65,536 among what is compared: a test that stops reaching them must fail, not pass quietly"""
    k = int(np.count_nonzero(np.asarray(ids, dtype=np.uint32) >= WIDE))
    assert k > 0
    return k


def _c5_expected(g):
    return {"merges": g["merge_list"], "n_ids": g["n_ids"], "ids_sha256": g["ids_sha256"],
            "same_bucket_ties": g["same_bucket_ties"], "threshold_edges": g["threshold_edges"],
            "thread_buckets": g["thread_buckets"]}


@pytest.mark.gpu
@pytest.mark.parametrize("P", [1, 2, 8])
def test_train_static_tie_heavy_past_65536(engine, oracle, P):
    """(A): 176,000 tokens to exhaustion, every iteration a tie-break, 3,599 of them inside one bucket; about 5,000 ids past
    65,535 are born in the static regime.  Merges, ids, tie counters and worker-table bucket counts as the oracle's."""
    if _device_count() < P:
        pytest.skip(f"needs {P} GPUs")
    _, m, t, st = assert_case(engine, oracle, "wideties88k_exh", n_gpus=P)
    assert len(m) == 70_306 and _wide(m) > 0 and _wide(t) == 2
    assert st["same_bucket_ties"] == 3599


@pytest.mark.gpu
def test_train_streaming_past_65536(engine):
    """(B): config 5's first chunk to 70,000 merges.  Id 65,536 is born inside batched passes on a stream of about 30 M
    tokens; the stream is decoded on the device and compared with the chunk, and encoding the chunk with the learned
    table gives the training ids again.  Without batching every merge past 65,280 is a pass of its own: same result."""
    g = _c5_70k()
    data = corpus(1, g["corpus"]["bytes"], g["corpus"]["seed"])
    stats = []
    for bm in (None, 1):
        ctx = engine.Context(0)
        try:
            if bm:
                ctx.set_option("batch_max", bm)
            ctx.upload(data)
            st = ctx.train(g["cap"])
            m, t = ctx.download()
            assert ctx.decode(m, download=False) == data.size and ctx.decode_mismatches() == 0
        finally:
            ctx.close()
        check_result(_c5_expected(g), m, t, st, 1, f"config 5, first chunk, 70,000 merges, batch_max {bm}")
        assert st["final_distinct"] == g["final_distinct"]
        _wide(m)
        _wide(t)
        stats.append(st)
    assert stats[0]["batch_merges"] > 0 and stats[1]["batch_merges"] == 0 and stats[1]["replace_passes"] == g["cap"]
    enc, se = engine.encode(data, m)
    assert len(enc) == g["n_ids"] and sha(enc) == g["ids_sha256"], se


@pytest.mark.gpu
@pytest.mark.parametrize("P", [1, 2])
def test_stream_encode_with_wide_tables(engine, oracle, P):
    """encode() with (B)'s table on 2 MB of config 4's corpus (the oracle's digest is committed) and on config 5's
    documents with their aliasing phrases, and with (C)'s table on 250 KB of its phrases (the oracle inline)."""
    if _device_count() < P:
        pytest.skip(f"needs {P} GPUs")
    g = json.load(open(os.path.join(HERE, "golden", "c4_2m_encode_c5_70k.json")))
    m = _c5_70k()["merge_list"]
    assert g["ranks"] == len(m) and (g["corpus"]["bytes"], g["corpus"]["seed"]) == C4_TEXT
    ids, st = engine.encode(corpus(1, *C4_TEXT), m, n_gpus=P)
    assert len(ids) == g["n_ids"] and sha(ids) == g["ids_sha256"], st
    _wide(ids)
    text = b"".join(c5_docs(oracle, m))
    ids, st = engine.encode(text, m, n_gpus=P)
    assert np.array_equal(ids, oracle.encode(text, m)), st
    _wide(ids)
    mc, names = foreign_wide_table()
    text = foreign_wide_text(mc, names, 250_000, 1)
    ids, st = engine.encode(text, mc, n_gpus=P)
    want = oracle.encode(text, mc)
    assert np.array_equal(ids, want), st
    assert _wide(ids) > 25_000 and {WIDE - 1, WIDE, WIDE + 1} <= set(ids.tolist())


def _batch_cases(oracle):
    """(table, documents, the oracle's encoding of each document alone) for (B)'s table and (C)'s"""
    mb = _c5_70k()["merge_list"]
    mc, names = foreign_wide_table()
    out = []
    for m, docs in ((mb, c5_docs(oracle, mb)), (mc, foreign_wide_docs(mc, names))):
        out.append((m, docs, [oracle.encode(d, m) for d in docs]))
    return out


def _check_batch(ids, off, docs, want, what):
    assert off.shape == (len(docs) + 1,) and off[0] == 0 and off[-1] == len(ids)
    for i, w in enumerate(want):
        assert np.array_equal(ids[int(off[i]):int(off[i + 1])], w), f"{what}: document {i} ({len(docs[i])} bytes)"


@pytest.mark.gpu
def test_encode_batch_with_wide_tables(engine, oracle):
    """Documents at every tier edge and one for the global-memory tier, each against the oracle's encoding of it alone.  On
    one context: the whole table, its prefix below 65,536 ids, the whole table again - the cached pair -> rank table is
    rebuilt when only the number of merges changes."""
    cases = _batch_cases(oracle)
    for m, docs, want in cases:
        ids, off, st = engine.encode_batch(docs, m)
        _check_batch(ids, off, docs, want, f"{len(m)} merges")
        assert all(_wide(w) for w in want[-7:])        # every tier document holds wide ids
        assert _wide(ids) == sum(int(np.count_nonzero(w >= WIDE)) for w in want)
    m, docs, want = cases[0]
    short = m[:50_000]
    want_short = [oracle.encode(d, short) for d in docs]
    ctx = engine.Context(0)
    try:
        launches = []
        for mm, w in ((m, want), (short, want_short), (m, want), (m, want)):
            ids, off, st = ctx.encode_batch(docs, mm)
            _check_batch(ids, off, docs, w, f"context, {len(mm)} merges")
            launches.append(st["kernel_launches"])
        assert launches[0] == launches[1] == launches[2] == launches[3] + 1   # the table is built for each new list
        assert int(max(w.max() for w in want_short)) < 50_256
    finally:
        ctx.close()


@pytest.mark.gpu
def test_decode_with_wide_tables(engine, oracle):
    """decode and decode_batch of the encodings above (against the oracle and the input bytes), of documents made only of
    wide ids, and the out-of-vocabulary error at 256 + n_merges, which names its document and leaves the context usable.
    On one context: the whole table, its prefix, the whole table again."""
    cases = _batch_cases(oracle)
    rng = np.random.default_rng(65536)
    for m, docs, want in cases:
        V = 256 + len(m)
        cut = [bc.nul_cut(d) for d in docs]
        out, boff, st = engine.decode_batch(want, m)
        assert [out[int(boff[i]):int(boff[i + 1])] for i in range(len(docs))] == cut
        cat = np.concatenate(want)
        _wide(cat)
        assert engine.decode(cat, m)[0] == b"".join(cut) == oracle.decode(cat, m)
        only = [rng.integers(WIDE, V, int(n)).astype(np.uint32) for n in (1, 2047, 2048, 2049, 9000)]
        only.append(np.array([V - 1, WIDE, V - 1], dtype=np.uint32))
        out, boff, _ = engine.decode_batch(only, m)
        assert [out[int(boff[i]):int(boff[i + 1])] for i in range(len(only))] == [oracle.decode(d, m) for d in only]
        bad = [want[0], only[1], np.concatenate([only[2], [V]]).astype(np.uint32), [V - 1]]
        with pytest.raises(engine.BpeCudaError) as e:
            engine.decode_batch(bad, m)
        assert e.value.rc == -1 and f"document 2 holds id {V}, outside the vocabulary ({V} entries)" in str(e.value)
        with pytest.raises(engine.BpeCudaError) as e:
            engine.decode(np.array([V - 1, V], dtype=np.uint32), m)
        assert e.value.rc == -1
        assert engine.decode(np.array([V - 1], dtype=np.uint32), m)[0] == oracle.decode([V - 1], m)
    m, docs, want = cases[0]
    short = m[:50_000]
    narrow = [oracle.encode(d, short) for d in docs]
    ctx = engine.Context(0)
    try:
        with pytest.raises(engine.BpeCudaError) as e:
            ctx.decode_batch([want[0], [256 + len(m)]], m)
        assert e.value.rc == -1 and "document 1 holds id" in str(e.value)
        rebuilt = []
        for mm, dd in ((m, want), (short, narrow), (m, want), (m, want)):
            out, boff, st = ctx.decode_batch(dd, mm)
            rebuilt.append(st["table_rehashes"])
            assert [out[int(boff[i]):int(boff[i + 1])] for i in range(len(dd))] == [oracle.decode(d, mm) for d in dd]
        assert rebuilt == [0, 1, 1, 0]          # the first list was flattened by the failed call
        with pytest.raises(engine.BpeCudaError) as e:   # a wide id past the prefix's vocabulary
            ctx.decode_batch([narrow[0], want[-1]], short)
        assert e.value.rc == -1 and "document 1 holds id" in str(e.value)
        out, boff, _ = ctx.decode_batch(want, m)
        assert out == b"".join(bc.nul_cut(d) for d in docs)
    finally:
        ctx.close()
