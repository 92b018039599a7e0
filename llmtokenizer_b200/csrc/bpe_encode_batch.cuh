// bpe_encode_batch.cuh — one-pass encoder for a batch of independent documents (bpe_cuda_encode_batch).
//
// Per document the merges are applied MIN-RANK-FIRST: repeat { r* = smallest rank among the adjacent pairs; replace
// every occurrence of merges[r*] greedily left to right (a run of L equal tokens under an a == b pair becomes L/2
// merged ids, paired from the start of the run) } until no adjacent pair has a rank.  This equals the rank-by-rank
// passes of bpe_cuda_encode (DESIGN.md §4): a rewrite only creates pairs that contain z = 256 + r*, which a valid
// list merges only at ranks above r*, so no smaller rank can appear again; a pair listed twice acts at its first rank
// only, so the pair -> rank table keeps the minimum.
//
// Launches of one batch (independent of the number of documents and of the table size):
//   E1 batch_rank_table_kernel  pair -> min rank, open addressing (only when the merge list changed)
//   E2 batch_cascade_kernel     persistent CTAs take work items from an atomic counter, longest documents first
//   E3 decode_scan_kernel       exclusive scan of the per-document id counts -> tok_offsets (shared with decode)
//   E4 batch_gather_kernel      the ids of document i, left at its byte offset by E2, compacted to tok_offsets[i]
//
// E2 keeps, per document, tok[] and rk[] (rank of the pair (tok[p], tok[p+1]), or NO_RANK) and runs the cascade in
// place.  One iteration is three barriers for a document that fits one tile:
//   1. min pass (striped): refresh rk[p] where tok[p] or tok[p+1] is the id made by the previous iteration, reduce min
//   2. per tile of CAS_THREADS * CAS_ITEMS positions: each thread loads its CAS_ITEMS consecutive positions into
//      registers, one scan over the group decides the greedy selection and every kept position's new index
//      (state: the selection bit after the segment and the kept count, each for both values of the bit before it),
//      then the kept tokens are written back compacted (write index <= read index, so in place is safe)
//   3. barrier, next iteration
// Tiers, by the document's length after its NUL cut (chosen automatically):
//   warp   len <= WARP_CAP      one warp per document, 8 documents per CTA, shared memory, __syncwarp only
//   block  len <= BLOCK_CAP     one CTA, shared memory
//   global len >  BLOCK_CAP     one CTA, tok[] and rk[] in the batch's global buffers, compacted inside segments of
//                               4,096 positions with a per-segment minimum rank (cascade_segmented).  Correct at any
//                               length below 4 GiB; documents beyond a few hundred KB are encode()'s job (DESIGN §4)
#pragma once
#include "bpe_kernels.cuh"

namespace bpe
{

constexpr int CAS_THREADS = 256;
constexpr int CAS_WARPS = CAS_THREADS / 32;
constexpr int CAS_ITEMS = 16;                                  // consecutive positions per thread in the scatter step
constexpr u32 CAS_TILE = CAS_THREADS * CAS_ITEMS;              // 4096
constexpr u32 WARP_CAP = 32 * CAS_ITEMS;                       // 512
constexpr u32 BLOCK_CAP = 2 * CAS_TILE;                        // 8192
constexpr u32 NO_RANK = 0xFFFFFFFFu;
constexpr u64 RT_EMPTY = ~0ull;                                // (no valid pair has a == b == 0xFFFFFFFF)

// shared-memory words of one tok[] or rk[] array: one pad word every 32 keeps the blocked accesses of step 2
// (thread t reads positions 16t .. 16t+15) free of bank conflicts
__host__ __device__ constexpr u32 cas_pidx(u32 p) { return p + (p >> 5); }
constexpr u32 CAS_SMEM_WORDS = cas_pidx(BLOCK_CAP) + 1;
constexpr size_t CAS_SMEM_BYTES = 2 * CAS_SMEM_WORDS * sizeof(u32);
static_assert(CAS_WARPS * 2 * (cas_pidx(WARP_CAP) + 1) <= 2 * CAS_SMEM_WORDS, "warp tier fits the block tier's memory");

struct RankTable
{
    const u64 *__restrict__ key;  // a | b << 32, RT_EMPTY where free
    const u32 *__restrict__ rank; // smallest rank of that pair
    u32 mask;                     // capacity - 1 (a power of two)
};

__device__ __forceinline__ u32 rt_hash(u64 k) { return (u32)((k * 0x9E3779B97F4A7C15ull) >> 32); }

__device__ __forceinline__ u32 rank_of(const RankTable &t, u32 a, u32 b)
{
    const u64 k = (u64)a | ((u64)b << 32);
    for (u32 h = rt_hash(k) & t.mask;; h = (h + 1) & t.mask)
    {
        const u64 s = __ldg(t.key + h);
        if (s == k)
            return __ldg(t.rank + h);
        if (s == RT_EMPTY)
            return NO_RANK;
    }
}

// E1: key[] = RT_EMPTY and rank[] = NO_RANK beforehand (memset); capacity >= 2 * n_merges
__global__ void __launch_bounds__(256) batch_rank_table_kernel(const uint2 *__restrict__ merges, u32 n_merges, u64 *key,
                                                               u32 *rank, u32 mask)
{
    for (u32 r = blockIdx.x * blockDim.x + threadIdx.x; r < n_merges; r += gridDim.x * blockDim.x)
    {
        const uint2 m = merges[r];
        const u64 k = (u64)m.x | ((u64)m.y << 32);
        for (u32 h = rt_hash(k) & mask;; h = (h + 1) & mask)
        {
            const u64 prev = atomicCAS(&key[h], RT_EMPTY, k);
            if (prev == RT_EMPTY || prev == k)
            {
                atomicMin(&rank[h], r);
                break;
            }
        }
    }
}

// ---- scan state of step 2 ----------------------------------------------------------------------------------
// bits 0-13: positions kept if the bit before the segment is 0, bits 14-27: if it is 1 (a tile has <= 4096),
// bit 28: selection bit after the segment if the bit before is 0, bit 29: if it is 1
constexpr u32 SEL_IDENTITY = 1u << 29;
__device__ __forceinline__ u32 sel_cnt(u32 x, u32 s) { return (x >> (14 * s)) & 0x3FFFu; }
__device__ __forceinline__ u32 sel_out(u32 x, u32 s) { return (x >> (28 + s)) & 1u; }
// the segment l followed by the segment r
__device__ __forceinline__ u32 sel_combine(u32 l, u32 r)
{
    const u32 l0 = sel_out(l, 0), l1 = sel_out(l, 1);
    return (sel_cnt(l, 0) + sel_cnt(r, l0)) | ((sel_cnt(l, 1) + sel_cnt(r, l1)) << 14) | (sel_out(r, l0) << 28) |
           (sel_out(r, l1) << 29);
}

struct CasScratch
{
    u32 red[CAS_WARPS];
    u32 scan[2][CAS_WARPS]; // alternate by tile: a fast thread may publish the next tile's while a slow one still reads
};

// Step 2 on one tile: positions [lo0, lo0 + NT * CAS_ITEMS) of tok[0..n) are selected (rk == best, greedy) and
// written back compacted from index base_carry on; s_carry is the selection bit of the position before the tile.  Both
// carries are updated for the next tile.  The group must be converged (a barrier inside for NT > 32).
template <int NT, bool PAD>
__device__ __forceinline__ void select_tile(u32 *tok, u32 *rk, u32 n, u32 lo0, u32 best, u32 &s_carry, u32 &base_carry,
                                            u32 &parity, CasScratch *sc)
{
    auto P = [](u32 p) { return PAD ? cas_pidx(p) : p; };
    const u32 t = NT == 32 ? (threadIdx.x & 31) : threadIdx.x;
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const u32 z = 256 + best; // positions with rk == best hold exactly the pair merges[best]
    const u32 lo = lo0 + t * CAS_ITEMS;
    u32 tv[CAS_ITEMS], rv[CAS_ITEMS];
    u32 s0 = 0, s1 = 1, c0 = 0, c1 = 0;
#pragma unroll
    for (int k = 0; k < CAS_ITEMS; k++)
    {
        const u32 i = lo + k;
        tv[k] = i < n ? tok[P(i)] : 0;
        rv[k] = i < n ? rk[P(i)] : NO_RANK;
        if (i < n) // positions past n leave the bit as it is: it is the carry into the next tile or segment
        {
            c0 += !s0;
            c1 += !s1;
            const u32 m = rv[k] == best;
            s0 = m & !s0;
            s1 = m & !s1;
        }
    }
    const u32 mine = c0 | (c1 << 14) | (s0 << 28) | (s1 << 29);
    u32 incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const u32 y = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= (u32)o)
            incl = sel_combine(y, incl);
    }
    u32 ex = __shfl_up_sync(0xFFFFFFFFu, incl, 1);
    if (lane == 0)
        ex = SEL_IDENTITY;
    u32 total;
    if (NT > 32)
    {
        u32 *s = sc->scan[parity];
        parity ^= 1;
        if (lane == 31)
            s[warp] = incl;
        __syncthreads();
        u32 before = SEL_IDENTITY;
        total = SEL_IDENTITY;
#pragma unroll
        for (int w = 0; w < NT / 32; w++)
        {
            if ((u32)w < warp)
                before = sel_combine(before, s[w]);
            total = sel_combine(total, s[w]);
        }
        ex = sel_combine(before, ex);
    }
    else
    {
        total = __shfl_sync(0xFFFFFFFFu, incl, 31);
    }
    u32 sel = sel_out(ex, s_carry);
    u32 o = base_carry + sel_cnt(ex, s_carry);
    // every thread of the group has read its positions (the scan above is a barrier for the CTA; a warp's shuffles
    // converge it), so the compacted writes cannot clobber an unread position
#pragma unroll
    for (int k = 0; k < CAS_ITEMS; k++)
    {
        const u32 i = lo + k;
        if (i < n)
        {
            const u32 m = rv[k] == best;
            if (!sel)
            {
                tok[P(o)] = m ? z : tv[k];
                rk[P(o)] = rv[k];
                o++;
                sel = m;
            }
            else
                sel = 0;
        }
    }
    base_carry += sel_cnt(total, s_carry);
    s_carry = sel_out(total, s_carry);
}

// The cascade of one document of n tokens (tok[] already holds them), in shared memory.  NT = 32: one warp, else the
// whole CTA.  PAD: cas_pidx() layout.  Returns the final number of tokens (tok[0..n)).
template <int NT, bool PAD>
__device__ u32 cascade(u32 *tok, u32 *rk, u32 n, const RankTable &rt, CasScratch *sc)
{
    auto P = [](u32 p) { return PAD ? cas_pidx(p) : p; };
    const u32 t = NT == 32 ? (threadIdx.x & 31) : threadIdx.x;
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u32 zprev = NO_RANK; // NO_RANK: every rk[] is still to be computed
    u32 parity = 0;
    for (;;)
    {
        // 1. refresh and reduce
        u32 best = NO_RANK;
        for (u32 p = t; p < n; p += NT)
        {
            u32 r = rk[P(p)];
            const u32 x = tok[P(p)];
            const u32 y = p + 1 < n ? tok[P(p + 1)] : NO_RANK;
            if (zprev == NO_RANK || x == zprev || y == zprev)
            {
                r = p + 1 < n ? rank_of(rt, x, y) : NO_RANK;
                rk[P(p)] = r;
            }
            best = min(best, r);
        }
        best = __reduce_min_sync(0xFFFFFFFFu, best);
        if (NT > 32)
        {
            if (lane == 0)
                sc->red[warp] = best;
            __syncthreads();
#pragma unroll
            for (int w = 0; w < NT / 32; w++)
                best = min(best, sc->red[w]);
        }
        else
            __syncwarp();
        if (best == NO_RANK)
            return n;
        // 2. select and compact, tile by tile
        u32 s_carry = 0, base_carry = 0;
        for (u32 lo0 = 0; lo0 < n; lo0 += NT * CAS_ITEMS)
            select_tile<NT, PAD>(tok, rk, n, lo0, best, s_carry, base_carry, parity, sc);
        n = base_carry;
        zprev = 256 + best;
        if (NT == 32)
            __syncwarp();
        else
            __syncthreads();
    }
}

// ---- global-memory tier: segment-local compaction ------------------------------------------------------------------
// The document is cut into segments of SEG positions.  Segment s keeps its live tokens at tok[s*SEG .. s*SEG + cnt[s])
// (compaction never crosses a segment) and segmin[s] = the smallest rank among its pairs, the pair of its last token
// with the first token of the next non-empty segment included.  An iteration therefore costs O(segments) for the
// minimum plus the work in the segments that hold r* (and in the neighbours whose pairs changed), not O(length).
constexpr u32 SEG = CAS_TILE;
constexpr u32 SEG_DIRTY = 0xFFFFFFFEu; // segmin[s]: rk[] of the segment must be refreshed first (no rank is this large)
constexpr u32 SEG_NONE = 0xFFFFFFFFu;

struct SegScratch
{
    u32 list[CAS_THREADS];
    u32 wsum[CAS_WARPS];
    u32 red[2][CAS_WARPS]; // alternate from refresh to refresh
    u32 bcast[2];
};

// ordered list of the indices whose flag is set, one per thread of the CTA -> list[0..return)
__device__ __forceinline__ u32 block_list(bool f, u32 idx, SegScratch *ss)
{
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const u32 b = __ballot_sync(0xFFFFFFFFu, f);
    if (lane == 0)
        ss->wsum[warp] = __popc(b);
    __syncthreads();
    u32 before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < CAS_WARPS; w++)
    {
        before += (u32)w < warp ? ss->wsum[w] : 0;
        total += ss->wsum[w];
    }
    if (f)
        ss->list[before + __popc(b & ((1u << lane) - 1))] = idx;
    __syncthreads();
    return total;
}

// the whole CTA: recompute rk[] of segment s where a token of the pair is zprev (all of it when zprev == NO_RANK),
// then segmin[s].  All loads of a thread are issued before any store (they do not depend on each other).
__device__ void seg_refresh(u32 *tok, u32 *rk, const u32 *cnt, u32 *segmin, u32 s, u32 S, u32 zprev, const RankTable &rt,
                            u32 &parity, SegScratch *ss)
{
    const u32 t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const u32 n = cnt[s];
    u32 *tk = tok + (u64)s * SEG, *rr = rk + (u64)s * SEG;
    u32 x[CAS_ITEMS], y[CAS_ITEMS], r[CAS_ITEMS];
#pragma unroll
    for (int k = 0; k < CAS_ITEMS; k++)
    {
        const u32 p = t + k * CAS_THREADS;
        x[k] = p < n ? tk[p] : 0;
        y[k] = p + 1 < n ? tk[p + 1] : NO_RANK;
        r[k] = p < n ? rr[p] : NO_RANK;
        if (p + 1 == n) // the last pair reaches into the next non-empty segment
            for (u32 q = s + 1; q < S; q++)
                if (cnt[q])
                {
                    y[k] = tok[(u64)q * SEG];
                    break;
                }
    }
    u32 best = NO_RANK;
#pragma unroll
    for (int k = 0; k < CAS_ITEMS; k++)
    {
        const u32 p = t + k * CAS_THREADS;
        if (p < n && (zprev == NO_RANK || x[k] == zprev || y[k] == zprev))
        {
            r[k] = y[k] != NO_RANK ? rank_of(rt, x[k], y[k]) : NO_RANK;
            rr[p] = r[k];
        }
        best = min(best, r[k]);
    }
    best = __reduce_min_sync(0xFFFFFFFFu, best);
    u32 *red = ss->red[parity];
    parity ^= 1;
    if (lane == 0)
        red[warp] = best;
    __syncthreads();
    if (t == 0)
    {
#pragma unroll
        for (int w = 0; w < CAS_WARPS; w++)
            best = min(best, red[w]);
        segmin[s] = best;
    }
}

// select and compact segment s (one tile) with selection bit s_in before it; marks it and the non-empty segment before
// it for refresh.  Returns the selection bit of its last position.
__device__ u32 seg_select(u32 *tok, u32 *rk, u32 *cnt, u32 *segmin, u32 s, u32 s_in, u32 best, u32 &parity,
                          CasScratch *sc)
{
    u32 s_carry = s_in, base = 0;
    select_tile<CAS_THREADS, false>(tok + (u64)s * SEG, rk + (u64)s * SEG, cnt[s], 0, best, s_carry, base, parity, sc);
    __syncthreads(); // every thread has read cnt[s]
    if (threadIdx.x == 0)
    {
        cnt[s] = base;
        segmin[s] = SEG_DIRTY;
        for (u32 q = s; q-- > 0;)
            if (cnt[q])
            {
                segmin[q] = SEG_DIRTY;
                break;
            }
    }
    return s_carry;
}

// the non-empty segment after s (SEG_NONE if there is none); read by thread 0, broadcast
__device__ u32 seg_next(const u32 *cnt, u32 s, u32 S, SegScratch *ss)
{
    __syncthreads();
    if (threadIdx.x == 0)
    {
        u32 q = s + 1;
        while (q < S && !cnt[q])
            q++;
        ss->bcast[0] = q < S ? q : SEG_NONE;
    }
    __syncthreads();
    return ss->bcast[0];
}

// The cascade of one document in global memory, segment-local.  Returns the final number of tokens, compacted to
// tok[0..m).
__device__ u32 cascade_segmented(u32 *tok, u32 *rk, u32 n, u32 *cnt, u32 *segmin, const RankTable &rt, CasScratch *sc,
                                 SegScratch *ss)
{
    const u32 t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const u32 S = (n + SEG - 1) / SEG;
    for (u32 s = t; s < S; s += CAS_THREADS)
    {
        cnt[s] = min(SEG, n - s * SEG);
        segmin[s] = SEG_DIRTY;
    }
    __syncthreads();
    u32 zprev = NO_RANK, parity = 0, rparity = 0;
    for (;;)
    {
        // refresh the segments marked in the last iteration, then the minimum over all segments
        u32 best = NO_RANK;
        for (u32 c0 = 0; c0 < S; c0 += CAS_THREADS)
        {
            const u32 s = c0 + t;
            const u32 k = block_list(s < S && segmin[s] == SEG_DIRTY, s, ss);
            for (u32 j = 0; j < k; j++)
                seg_refresh(tok, rk, cnt, segmin, ss->list[j], S, zprev, rt, rparity, ss);
            __syncthreads();
            if (s < S)
                best = min(best, segmin[s]);
        }
        best = __reduce_min_sync(0xFFFFFFFFu, best);
        if (lane == 0)
            sc->red[warp] = best;
        __syncthreads();
#pragma unroll
        for (int w = 0; w < CAS_WARPS; w++)
            best = min(best, sc->red[w]);
        if (best == NO_RANK)
            break;
        // select and compact the segments that hold best, in order.  A selected last pair removes the first token of
        // the next non-empty segment, which is then processed too (with selection bit 1 before it).
        u32 carry_seg = SEG_NONE;
        for (u32 c0 = 0; c0 < S; c0 += CAS_THREADS)
        {
            const u32 s0 = c0 + t;
            const u32 k = block_list(s0 < S && segmin[s0] == best, s0, ss);
            for (u32 j = 0; j < k; j++)
            {
                const u32 s = ss->list[j];
                if (carry_seg != SEG_NONE && carry_seg < s) // a follower without an occurrence of its own
                    seg_select(tok, rk, cnt, segmin, carry_seg, 1, best, parity, sc);
                const u32 out = seg_select(tok, rk, cnt, segmin, s, carry_seg == s, best, parity, sc);
                carry_seg = out ? seg_next(cnt, s, S, ss) : SEG_NONE;
            }
            __syncthreads(); // list[] is rebuilt for the next chunk
        }
        if (carry_seg != SEG_NONE)
            seg_select(tok, rk, cnt, segmin, carry_seg, 1, best, parity, sc);
        zprev = 256 + best;
        __syncthreads();
    }
    // close the gaps: segment by segment to the front (each segment is at most one tile: read, barrier, write)
    u32 m = 0;
    for (u32 s = 0; s < S; s++)
    {
        const u32 c = cnt[s];
        u32 v[CAS_ITEMS];
#pragma unroll
        for (int k = 0; k < CAS_ITEMS; k++)
        {
            const u32 i = t * CAS_ITEMS + k;
            v[k] = i < c ? tok[(u64)s * SEG + i] : 0;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < CAS_ITEMS; k++)
        {
            const u32 i = t * CAS_ITEMS + k;
            if (i < c)
                tok[m + i] = v[k];
        }
        m += c;
        __syncthreads();
    }
    return m;
}

struct CasArgs
{
    const uint8_t *bytes;      // the batch's bytes (offsets relative to offsets[0])
    const u64 *doc_off;        // [n_docs] start of each document in bytes / tok / rk
    const u32 *doc_len;        // [n_docs] length after the NUL cut
    const u32 *order;          // work order: documents longer than WARP_CAP, longest first, then the rest
    u32 n_docs, n_big;         // n_big: documents of the block and global tiers (order[0..n_big))
    u32 n_items;               // n_big + ceil((n_docs - n_big) / CAS_WARPS)
    u32 *tok, *rk;             // [batch bytes] working buffers of the global tier; tok receives every document's ids
    const u32 *seg_base;       // [n_docs] first segment of a global-tier document in seg_cnt / seg_min
    u32 *seg_cnt, *seg_min;    // per segment of the global tier (cascade_segmented)
    u64 *count;                // [n_docs] ids of each document
    u32 *next_item;            // work counter, 0 at launch
    RankTable rt;
};

// E2: persistent; dynamic shared memory CAS_SMEM_BYTES
__global__ void __launch_bounds__(CAS_THREADS, 3) batch_cascade_kernel(CasArgs a)
{
    extern __shared__ u32 s_mem[];
    __shared__ CasScratch sc;
    __shared__ SegScratch ss;
    __shared__ u32 s_item;
    const u32 t = threadIdx.x, lane = t & 31, warp = t >> 5;
    for (;;)
    {
        if (t == 0)
            s_item = atomicAdd(a.next_item, 1u);
        __syncthreads();
        const u32 item = s_item;
        if (item >= a.n_items)
            return;
        if (item < a.n_big)
        {
            const u32 d = a.order[item];
            const u32 n = a.doc_len[d];
            const u64 o = a.doc_off[d];
            u32 m;
            if (n <= BLOCK_CAP)
            {
                u32 *tok = s_mem, *rk = s_mem + CAS_SMEM_WORDS;
                for (u32 p = t; p < n; p += CAS_THREADS)
                    tok[cas_pidx(p)] = a.bytes[o + p];
                __syncthreads();
                m = cascade<CAS_THREADS, true>(tok, rk, n, a.rt, &sc);
                for (u32 p = t; p < m; p += CAS_THREADS)
                    a.tok[o + p] = tok[cas_pidx(p)];
            }
            else
            {
                u32 *tok = a.tok + o, *rk = a.rk + o;
                for (u32 p = t; p < n; p += CAS_THREADS)
                    tok[p] = a.bytes[o + p];
                __syncthreads();
                m = cascade_segmented(tok, rk, n, a.seg_cnt + a.seg_base[d], a.seg_min + a.seg_base[d], a.rt, &sc,
                                      &ss);
            }
            if (t == 0)
                a.count[d] = m;
        }
        else
        {
            const u32 k = a.n_big + (item - a.n_big) * CAS_WARPS + warp;
            if (k < a.n_docs)
            {
                const u32 d = a.order[k];
                const u32 n = a.doc_len[d];
                const u64 o = a.doc_off[d];
                u32 *tok = s_mem + warp * 2 * (cas_pidx(WARP_CAP) + 1), *rk = tok + cas_pidx(WARP_CAP) + 1;
                for (u32 p = lane; p < n; p += 32)
                    tok[cas_pidx(p)] = a.bytes[o + p];
                __syncwarp();
                const u32 m = cascade<32, true>(tok, rk, n, a.rt, nullptr);
                for (u32 p = lane; p < m; p += 32)
                    a.tok[o + p] = tok[cas_pidx(p)];
                if (lane == 0)
                    a.count[d] = m;
            }
        }
        __syncthreads(); // s_item and the shared arrays are reused by the next item
    }
}

// E4: out[tok_off[d] + j] = tok[doc_off[d] + j], one CTA per document at a time
__global__ void __launch_bounds__(256) batch_gather_kernel(const u32 *__restrict__ tok, const u64 *__restrict__ doc_off,
                                                           const u64 *__restrict__ tok_off, u32 n_docs, u32 *__restrict__ out)
{
    for (u32 d = blockIdx.x; d < n_docs; d += gridDim.x)
    {
        const u64 src = doc_off[d], dst = tok_off[d], m = tok_off[d + 1] - dst;
        for (u64 j = threadIdx.x; j < m; j += blockDim.x)
            out[dst + j] = tok[src + j];
    }
}

} // namespace bpe
