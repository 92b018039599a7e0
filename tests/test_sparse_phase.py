"""The sparse late phase (LAYOUT_SPARSE, llmtokenizer_b200/csrc/bpe_sparse.cuh).

Without a GPU: a Python restatement of the layout (tokens at their byte offsets, start_of at token ends), the frozen
pair index, the creation lists, the run pairing of a == a merges and the pair-count deltas of a pass, checked against
the oracle's streams and a full recount on small inputs.  On the GPU: runs whose oracle results are committed or
computed inline, with sparse passes asserted to have run, across pauses, the static limit and a == a merges."""
import numpy as np
import pytest

import oracle_api
import parity_cases as pc
from parity_cases import corpus, sha

SENT = 0xFFFFFFFF


class SparseModel:
    """tok[p] = id starting at byte p (SENT elsewhere), so[e] = start of the token ending at byte e."""

    def __init__(self, dense, merges_so_far):
        self.len = {t: 1 for t in range(256)}
        for k, (a, b) in enumerate(merges_so_far):
            self.len[256 + k] = self.len[int(a)] + self.len[int(b)]
        lens = np.array([self.len[int(t)] for t in dense], dtype=np.int64)
        pos = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64)
        self.n0 = int(lens.sum())
        self.tok = np.full(self.n0 + 8, SENT, dtype=np.int64)
        self.so = np.zeros(self.n0 + 8, dtype=np.int64)
        self.tok[pos] = dense
        self.so[pos + lens - 1] = pos
        self.zsw = 256 + len(merges_so_far)
        # frozen index: every pair instance, bucketed by pair
        self.frozen = {}
        for i in range(len(dense) - 1):
            self.frozen.setdefault((int(dense[i]), int(dense[i + 1])), []).append(int(pos[i]))
        self.created = {}
        self.scanned = 0

    def prev_tok(self, p):
        return SENT if p == 0 else int(self.tok[self.so[p - 1]])

    def occurrences(self, a, b):
        if a < self.zsw and b < self.zsw:
            return 0, self.frozen.get((a, b), [])
        la = self.created.get(a, []) if a >= self.zsw else None
        lb = self.created.get(b, []) if b >= self.zsw else None
        if lb is None or (la is not None and len(la) <= len(lb)):
            return 1, la
        return 2, lb

    def apply_pass(self, batch, z0):
        """One pass of merges batch[i] -> z0 + i.  Returns the deltas {(i, t, k): v} as the scan kernel emits them."""
        lens = self.len
        for i, (a, b) in enumerate(batch):
            lens[z0 + i] = lens[a] + lens[b]
        reps, deltas = [], {}

        def add(i, t, k):
            deltas[(i, t, k)] = deltas.get((i, t, k), 0) + 1

        for i, (a, b) in enumerate(batch):
            kind, lst = self.occurrences(a, b)
            self.scanned += len(lst)
            for e in lst:
                if kind == 2:
                    q = e
                    if self.tok[q] != b or q == 0:
                        continue
                    p = int(self.so[q - 1])
                    if self.tok[p] != a:
                        continue
                else:
                    p = e
                    if self.tok[p] != a:
                        continue
                    q = p + lens[a]
                    if self.tok[q] != b:
                        continue
                if a == b:
                    x = self.prev_tok(p)
                    if x == a:
                        continue  # not the start of its run
                    cur, first = p, True
                    while True:
                        q2 = cur + lens[a]
                        if self.tok[q2] != a:
                            break
                        yp = q2 + lens[a]
                        y = int(self.tok[yp])
                        nm = y == a and self.tok[yp + lens[a]] == a
                        xx = x if first else a
                        if xx != SENT:
                            if xx != a:
                                add(i, xx, 0)
                            add(i, xx if first else z0, 2)
                        if y != SENT and not nm:
                            if y != a:
                                add(i, y, 1)
                            add(i, y, 3)
                        reps.append((cur, i))
                        first = False
                        if not nm:
                            break
                        cur = yp
                    continue
                xp = int(self.so[p - 1]) if p else 0
                x = int(self.tok[xp]) if p else SENT
                xn = x
                for j, (aj, bj) in enumerate(batch):
                    if x == bj and xp > 0 and self.tok[self.so[xp - 1]] == aj:
                        xn = z0 + j
                yp = q + lens[b]
                y = int(self.tok[yp])
                nm = any(y == aj and self.tok[yp + lens[aj]] == bj for aj, bj in batch)
                if x != SENT:
                    add(i, x, 0)
                    add(i, xn, 2)
                if y != SENT and not nm:
                    add(i, y, 1)
                    add(i, y, 3)
                reps.append((p, i))
        # the write phase
        for p, i in reps:
            a, b = batch[i]
            q = p + lens[a]
            self.tok[p] = z0 + i
            self.tok[q] = SENT
            self.so[q + lens[b] - 1] = p
            self.created.setdefault(z0 + i, []).append(p)
        return deltas

    def dense(self):
        t = self.tok[:self.n0]
        return t[t != SENT].astype(np.uint32)


def _batches(merges, start):
    """consecutive merges grouped the way a batched pass may carry them: pairwise different ids, none made in the
    group, no a == a pair (those take a pass of their own)"""
    out, k = [], start
    while k < len(merges):
        g = [tuple(int(v) for v in merges[k])]
        used = set(g[0])
        k += 1
        if g[0][0] != g[0][1]:
            while k < len(merges) and len(g) < 12:
                a, b = (int(v) for v in merges[k])
                made = {256 + start2 for start2 in range(k - len(g), k)}
                if a == b or a in used or b in used or a in made or b in made:
                    break
                g.append((a, b))
                used |= {a, b}
                k += 1
        out.append(g)
    return out


def _check(data, merges, switch, oracle):
    toks = data.astype(np.uint32)
    for k in range(switch):
        toks = oracle.rewrite(toks, int(merges[k][0]), int(merges[k][1]), 256 + k)
    model = SparseModel(toks, merges[:switch])
    k = switch
    for batch in _batches(merges, switch):
        before = oracle_api.pair_counts(toks)
        deltas = model.apply_pass(batch, 256 + k)
        for i, (a, b) in enumerate(batch):
            toks = oracle.rewrite(toks, a, b, 256 + k + i)
        assert np.array_equal(model.dense(), toks), f"stream differs after the pass of merge {k}"
        # the deltas say how every pair's count changes, except the merged pairs' own
        want = {}
        for (i, t, kk), v in deltas.items():
            a, b = batch[i]
            z = 256 + k + i
            key = [(t, a), (b, t), (t, z), (z, t)][kk]
            want[key] = want.get(key, 0) + (v if kk >= 2 else -v)
        after = oracle_api.pair_counts(toks)
        merged = {a | (b << 32) for a, b in batch}
        for key in set(before) | set(after) | {x | (y << 32) for x, y in want}:
            if key in merged:
                continue
            x, y = key & 0xFFFFFFFF, key >> 32
            assert after.get(key, 0) - before.get(key, 0) == want.get((x, y), 0), (k, batch, (x, y))
        k += len(batch)
    return model


@pytest.mark.parametrize("kind,size,cap,switch", [(0, 60_000, 400, 40), (1, 40_000, 300, 10), (2, 30_000, 200, 0)])
def test_sparse_restatement_matches_the_oracle(oracle, kind, size, cap, switch):
    data = corpus(kind, size, 77 + kind)
    rc, m, t, _ = oracle.train(data, cap)
    assert rc == 0
    model = _check(data, m, switch, oracle)
    assert np.array_equal(model.dense(), t)


def test_sparse_restatement_runs_of_equal_tokens(oracle):
    """a == a merges whose runs cross one another's creations: odd and even runs, runs at both ends"""
    rng = np.random.default_rng(5)
    data = np.repeat(rng.integers(97, 100, 3000, dtype=np.uint8), rng.integers(1, 12, 3000))
    data = np.concatenate([[97] * 7, data, [98] * 5]).astype(np.uint8)
    rc, m, t, _ = oracle.train(data, 120)
    assert rc == 0 and any(a == b for a, b in m[20:])
    model = _check(data, m, 3, oracle)
    assert np.array_equal(model.dense(), t)


# ---------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


def _train_case(engine, oracle, key, options=None):
    data, cap = pc.train_input(key)
    exp = pc.expected_train(key, oracle)
    ctx = engine.Context(0)
    try:
        for k, v in (options or {}).items():
            ctx.set_option(k, v)
        ctx.upload(data)
        st = ctx.train(cap)
        m, t = ctx.download()
    finally:
        ctx.close()
    from test_gpu_parity import check_result
    check_result(exp, m, t, st, 1, key)
    return data, m, t, st


@gpu
@pytest.mark.parametrize("key", ["zipfa12m_10000", "zipfb8m_2200", "uniform14m_2600"])
def test_sparse_passes_run_and_match_the_oracle(engine, oracle, key):
    _, m, t, st = _train_case(engine, oracle, key)
    assert st["sparse_passes"] > 0, st


@gpu
def test_sparse_phase_pauses_for_ties(engine, oracle):
    """Ties above the static limit: every one of them pauses the sparse phase for the resolver (dense layout) and
    the run goes back to sparse passes after it."""
    _, m, t, st = _train_case(engine, oracle, "ties4m_1000")
    assert st["sparse_passes"] > 0 and st["same_bucket_ties"] > 0 and st["resolver_runs"] > 0, st


@gpu
def test_sparse_phase_then_the_static_limit(engine, oracle):
    """1.2 M tokens trained to exhaustion: sparse passes, then the stream falls below 1,048,576 tokens and the run
    continues on the dense layout (static slicing, census, 419 same-bucket ties)."""
    _, m, t, st = _train_case(engine, oracle, "ties1m2_exh")
    assert st["sparse_passes"] > 0 and st["census_runs"] > 0, st


@gpu
def test_sparse_phase_with_runs_of_equal_tokens(engine, oracle):
    """a == a merges on the sparse layout: runs of a rare byte (lengths 1-9, at both ends of the stream too) are
    merged pairwise from their left ends, twice over, after a rare pair."""
    rng = np.random.default_rng(11)
    data = rng.integers(97, 123, 2_400_000, dtype=np.uint8)
    for p in rng.choice(np.arange(20, data.size - 20), 400, replace=False):
        data[p:p + 2] = (2, 3)
    for p in rng.choice(np.arange(20, data.size - 20), 300, replace=False):
        data[p:p + int(rng.integers(1, 10))] = 1
    data[:9] = 1
    data[-7:] = 1
    # 200 ranks whose pairs never occur come first, so that the loop has switched layouts before the real ones
    F = 200
    z = 256 + F + 1  # the id (1, 1) makes
    merges = np.array([(200 + i % 50, 250 + i // 50) for i in range(F)] +
                      [(2, 3), (1, 1), (z, z), (z, 1), (z + 1, 1), (1, z), (97, 98), (z + 1, z + 1)], dtype=np.uint32)
    ids, st = engine.encode(data, merges)
    assert np.array_equal(ids, oracle.encode(data, merges))
    assert st["sparse_passes"] > 0, st


@gpu
def test_encode_on_the_sparse_layout_reproduces_training(engine, oracle):
    data, m, t, st = _train_case(engine, oracle, "zipfa12m_10000")
    ids, est = engine.encode(data, m)
    assert len(ids) == len(t) and sha(ids) == sha(t)
    assert est["sparse_passes"] > 0, est
