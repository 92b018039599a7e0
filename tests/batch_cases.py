"""TEST INFRASTRUCTURE for encode_batch: the min-rank-first restatement that the batch kernel implements, a
restatement of the kernel's select-and-compact scan, seeded random merge tables, and the document mix of config 4's
corpus (tests/test_encode_batch.py, tools/make_encode_batch_golden.py, tools/encode_batch_bench.py)."""
import numpy as np


def nul_cut(doc):
    doc = bytes(doc)
    k = doc.find(b"\0")
    return doc if k < 0 else doc[:k]


def rank_table(merges):
    """pair -> smallest rank (a pair listed twice acts at its first rank only)"""
    t = {}
    for r, (a, b) in enumerate(np.asarray(merges, dtype=np.int64).reshape(-1, 2).tolist()):
        t.setdefault((a, b), r)
    return t


def greedy_replace(toks, a, b, z):
    """one rank pass of the reference (bpe.c:760-772): left to right, an occurrence consumes both tokens"""
    out, i = [], 0
    while i < len(toks):
        if i + 1 < len(toks) and toks[i] == a and toks[i + 1] == b:
            out.append(z)
            i += 2
        else:
            out.append(toks[i])
            i += 1
    return out


def min_rank_first(doc, merges, replace=greedy_replace):
    """Repeat { r* = smallest rank among the adjacent pairs; replace every occurrence of merges[r*] greedily } until no
    adjacent pair has a rank.  Equal to the rank-by-rank passes of encode() for a valid merge list."""
    toks = list(nul_cut(doc))
    table = rank_table(merges)
    mg = np.asarray(merges, dtype=np.int64).reshape(-1, 2).tolist()
    while True:
        ranks = [table.get((toks[i], toks[i + 1])) for i in range(len(toks) - 1)]
        present = [r for r in ranks if r is not None]
        if not present:
            return toks
        r = min(present)
        toks = replace(toks, mg[r][0], mg[r][1], 256 + r)


# ---- the kernel's step 2 (bpe_encode_batch.cuh), restated ----------------------------------------------------------
# A segment of positions is summarised as (f0, f1, c0, c1): the selection bit after the segment and the number of kept
# positions, for a selection bit of 0 / 1 before it.  Segments combine associatively, so one scan over the threads of
# a tile gives every thread its incoming bit and its first write index.
IDENTITY = (0, 1, 0, 0)


def seg_summary(match):
    s = [0, 1]
    c = [0, 0]
    for m in match:
        for h in (0, 1):
            c[h] += not s[h]
            s[h] = int(m and not s[h])
    return (s[0], s[1], c[0], c[1])


def seg_combine(l, r):
    return (r[l[0]], r[l[1]], l[2] + r[2 + l[0]], l[3] + r[2 + l[1]])


def scan_replace(toks, a, b, z, items=4, threads=8):
    """greedy_replace() computed the way the kernel does: tiles of threads * items positions, one exclusive scan of
    segment summaries per tile, a carry (bit, count) from tile to tile, writes in place at the scanned index."""
    toks = list(toks)
    n = len(toks)
    match = [int(i + 1 < n and toks[i] == a and toks[i + 1] == b) for i in range(n)]
    out = list(toks)
    s_carry, base = 0, 0
    for lo0 in range(0, n, threads * items):
        segs = [list(range(lo0 + t * items, min(n, lo0 + (t + 1) * items))) for t in range(threads)]
        summ = [seg_summary([match[i] for i in seg]) for seg in segs]
        pref = IDENTITY
        writes = []
        for t, seg in enumerate(segs):
            sel, o = pref[s_carry], base + pref[2 + s_carry]
            for i in seg:
                if not sel:
                    assert o <= i   # in place: never ahead of the position being read
                    writes.append((o, z if match[i] else toks[i]))
                    o += 1
                    sel = match[i]
                else:
                    sel = 0
            pref = seg_combine(pref, summ[t])
        for o, v in writes:
            out[o] = v
        base += pref[2 + s_carry]
        s_carry = pref[s_carry]
    return out[:base]


def random_table(rng, alphabet, k, same_frac=0.3, dup_frac=0.1):
    """A valid foreign merge list of k ranks over the given byte alphabet: merges[r] uses ids < 256 + r, about
    same_frac of them a == b, about dup_frac of them a repeat of an earlier pair."""
    ids = [int(x) for x in alphabet]
    m = []
    for r in range(k):
        if m and rng.random() < dup_frac:
            m.append(m[int(rng.integers(len(m)))])
        else:
            a = ids[int(rng.integers(len(ids)))]
            b = a if rng.random() < same_frac else ids[int(rng.integers(len(ids)))]
            m.append((a, b))
        ids.append(256 + r)
    return np.array(m, dtype=np.uint32).reshape(-1, 2)


def lognormal_docs(total, seed, median=1500, sigma=1.0, lo=1, hi=65536):
    """Offsets (uint64, n_docs + 1) that cut `total` bytes into documents of seeded log-normal lengths, clipped to
    [lo, hi]; the last document takes what is left."""
    rng = np.random.default_rng(seed)
    lens = []
    acc = 0
    while acc < total:
        ls = np.clip(np.rint(rng.lognormal(np.log(median), sigma, 65536)), lo, hi).astype(np.int64)
        lens.append(ls)
        acc += int(ls.sum())
    lens = np.concatenate(lens)
    off = np.concatenate([[0], np.cumsum(lens)])
    k = int(np.searchsorted(off, total))
    off = off[:k + 1].copy()
    off[k] = total
    return off.astype(np.uint64)


def c4_docs(total, seed=777, len_seed=777):
    """config 4's corpus (zipf_bytes, sampling seed 777, config 3's word list), first `total` bytes, cut into documents
    of log-normal lengths (median 1,500 B, sigma 1.0, clipped to [1, 65,536])"""
    from parity_cases import corpus
    return corpus(1, total, seed), lognormal_docs(total, len_seed)


def segmented_cascade(doc, merges, seg=8):
    """The global-memory tier of the kernel (cascade_segmented) restated: segments of `seg` positions compact only
    inside themselves; segmin[s] covers the pairs that start in s (the last one reaches into the next non-empty
    segment); an iteration refreshes the segments marked in the last one, takes the minimum over segmin, and selects
    in the segments that hold it, in order, a selected last pair removing the first token of the next non-empty
    segment.  Returns the ids (gaps closed)."""
    toks = list(nul_cut(doc))
    table = rank_table(merges)
    S = (len(toks) + seg - 1) // seg
    segs = [toks[s * seg:(s + 1) * seg] for s in range(S)]
    rk = [[None] * len(x) for x in segs]
    dirty = set(range(S))
    NO = float("inf")
    segmin = [NO] * S
    zprev = None

    def nxt_first(s):
        for q in range(s + 1, S):
            if segs[q]:
                return segs[q][0]
        return None

    def prev_nonempty(s):
        for q in range(s - 1, -1, -1):
            if segs[q]:
                return q
        return None

    while True:
        for s in dirty:
            nf = nxt_first(s)
            for p, x in enumerate(segs[s]):
                y = segs[s][p + 1] if p + 1 < len(segs[s]) else nf
                if zprev is None or x == zprev or y == zprev:
                    r = table.get((x, y)) if y is not None else None
                    rk[s][p] = NO if r is None else r
            segmin[s] = min(rk[s], default=NO)
        dirty = set()
        best = min(segmin, default=NO)
        if best == NO:
            return [t for x in segs for t in x]
        z = 256 + best

        def select(s, s_in):
            sel, out_t, out_r = s_in, [], []
            for t, r in zip(segs[s], rk[s]):
                if not sel:
                    m = r == best
                    out_t.append(z if m else t)
                    out_r.append(r)
                    sel = m
                else:
                    sel = False
            segs[s], rk[s] = out_t, out_r
            dirty.add(s)
            q = prev_nonempty(s)
            if q is not None:
                dirty.add(q)
            return sel

        listed = [s for s in range(S) if segmin[s] == best]
        carry = None
        for s in listed:
            if carry is not None and carry < s:
                select(carry, True)
            out = select(s, carry == s)
            carry = None
            if out:
                q = s + 1
                while q < S and not segs[q]:
                    q += 1
                carry = q if q < S else None
        if carry is not None:
            select(carry, True)
        zprev = z
