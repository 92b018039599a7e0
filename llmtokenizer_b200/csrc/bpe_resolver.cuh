// Exact reproduction of the reference's tie-break when the closed form "max count, then smallest
// murmur3 % B(D)" is not enough:
//   (1) two or more maximal pairs share the winning bucket -> the order inside one chain of the
//       merged hash table decides (hash_table.c:300-302 head insertion, hash_table.c:208-223 every
//       doubling reverses each chain, hash_table.c:146-188 merge order of the 16 worker tables);
//   (2) D sits exactly on a doubling threshold -> whether the merged table doubled depends on
//       whether its very last insert call created a key (hash_table.c:248-254).
// It also maintains the persistent bucket counts of the reference's 16 worker tables
// (hash_table.c:310-338: clear keeps the grown bucket count), which shape that chain order.
//
// Closed form used (validated on the CPU against a literal emulation of the reference's tables,
// oracle/bpe_oracle.c FAST_CF vs FAITHFUL, and against the compiled reference):
//   * in a table that doubles after its thr(B)-th key, a key of first-sight rank r sits in its
//     chain at chain_slot(#doublings still to come after r, r): even -> in front, youngest first;
//     odd -> behind, oldest first;
//   * worker table t lists its keys by (murmur3 % B_t, chain slot); the merged table first sees
//     keys in the order worker 0's list, worker 1's list, ...; that first-sight rank R and the
//     merged table's own doublings give the final chain slot; the smallest one among the tied
//     pairs wins (bpe.c:705-743 walks chains head to tail, dyn_arr.c:163-174 keeps the first max).
//
// Work split: below 1,048,576 tokens the reference cuts the stream into 16 static slices
// (bpe.c:449-477); above it the canonical schedule "worker 0 takes every chunk" is used (see
// DESIGN.md), i.e. one slice.
#pragma once
#include "bpe_kernels.cuh"

namespace bpe
{

constexpr int MAX_CAND = 1024;

struct ResState
{
    u64 census_epoch;
    u32 slices;  // 16 (static) or 1 (dynamic)
    u32 need;    // census: can any worker table grow this iteration?
    u64 per;     // static slice length (tokens)
    u64 npairs;  // n - 1
    u64 Dt[REF_THREADS];
    u32 last_new[REF_THREADS];
    u64 b0[REF_THREADS], b1[REF_THREADS];
    u64 prefixD[REF_THREADS + 1];
    u64 F[REF_THREADS];
    int last_slice;
    u32 pad0;
    u64 last_key;
    u64 bm;
    u32 fmax, wbucket;
    u32 n_cand, overflow;
    u64 cand_slot[MAX_CAND];
    u32 cand_tau[MAX_CAND];
    u64 cand_ord[MAX_CAND];
    u64 cand_before[MAX_CAND];
};

__device__ __forceinline__ u32 slice_of_pos(const ResState *rs, u64 i)
{
    if (rs->slices == 1)
        return 0;
    if (rs->per == 0)
        return REF_THREADS - 1;
    const u64 t = i / rs->per;
    return (u32)(t < REF_THREADS - 1 ? t : REF_THREADS - 1);
}
// last pair position counted by slice t (bpe.c:460-463), or ~0 if the slice is empty
__device__ __forceinline__ u64 slice_last_pos(const ResState *rs, u32 t)
{
    if (rs->npairs == 0)
        return ~0ull;
    if (rs->slices == 1)
        return rs->npairs - 1;
    if (t == REF_THREADS - 1)
        return (rs->per * (REF_THREADS - 1) < rs->npairs) ? rs->npairs - 1 : ~0ull;
    if (rs->per == 0)
        return ~0ull;
    const u64 e = rs->per * (t + 1);
    return (e <= rs->npairs) ? e - 1 : ((rs->per * t < rs->npairs) ? rs->npairs - 1 : ~0ull);
}
__device__ __forceinline__ u64 first_pack(u64 epoch, u64 pos) { return (epoch << 32) | (0xFFFFFFFFull - pos); }
__device__ __forceinline__ u32 cslot31(u32 doublings_to_come, u64 r)
{
    return (doublings_to_come & 1u) ? (0x40000000u | (u32)r) : (0x3FFFFFFFu - (u32)r);
}

// ---- begin: new census epoch, geometry, "is it needed at all" ---------------------------------
__global__ void census_begin_kernel(DevState *st, ResState *rs, int resolver)
{
    const bool active = resolver ? (st->stop == STOP_PAUSE) : (st->stop == STOP_RUN);
    if (!active)
    {
        rs->need = 0;
        return;
    }
    rs->census_epoch++;
    const u64 n = st->n;
    rs->npairs = n ? n - 1 : 0;
    rs->slices = (n < STATIC_LIMIT) ? REF_THREADS : 1;
    rs->per = n / REF_THREADS;
    rs->last_key = 0;
    rs->n_cand = 0;
    rs->overflow = 0;
    rs->wbucket = 0xFFFFFFFFu;
    u32 need = 0;
    const u64 D = (u64)st->distinct;
    for (u32 t = 0; t < REF_THREADS; t++)
    {
        rs->Dt[t] = 0;
        rs->F[t] = 0;
        rs->last_new[t] = 0;
        u64 most;
        if (rs->slices == 1)
            most = (t == 0) ? rs->npairs : 0;
        else
            most = (t == REF_THREADS - 1) ? rs->per + n % REF_THREADS : rs->per;
        if (most > D)
            most = D;
        if (most >= resize_threshold(st->bt[t]))
            need = 1;
    }
    if (rs->slices == 1 && !resolver)
        need = 0; // one worker, D keys: handled without a pass (dynamic_regime_census)
    rs->need = resolver ? 1u : need;
}

// ---- pass 1: first position of every (pair, slice) ---------------------------------------------
__global__ void __launch_bounds__(256) census_mark_kernel(DevState *st, ResState *rs, u64 *first, u32 *pos_slot)
{
    if (!rs->need)
        return;
    const u32 *__restrict__ t = st->tok[st->cur];
    const u64 np = rs->npairs, S = rs->slices, ce = rs->census_epoch;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < np; i += (u64)gridDim.x * blockDim.x)
    {
        const u32 x = t[i], y = t[i + 1];
        const u64 s = table_find(st->tkey, st->tcap, (u64)x | ((u64)y << 32), murmur3_pair(x, y));
        if (s == NO_SLOT)
        {
            atomicOr(&st->err, ERR_MISSING_KEY);
            pos_slot[i] = 0xFFFFFFFFu;
            continue;
        }
        pos_slot[i] = (u32)s;
        atomicMax(first + s * S + slice_of_pos(rs, i), first_pack(ce, i));
    }
}

// ---- pass 2: distinct pairs per slice, and whether each slice's last call created a key -------
__global__ void __launch_bounds__(256) census_count_kernel(DevState *st, ResState *rs, const u64 *first, const u32 *pos_slot)
{
    if (!rs->need)
        return;
    __shared__ u32 s_cnt[REF_THREADS];
    if (threadIdx.x < REF_THREADS)
        s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const u64 np = rs->npairs, S = rs->slices, ce = rs->census_epoch;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < np; i += (u64)gridDim.x * blockDim.x)
    {
        const u32 s = pos_slot[i];
        if (s == 0xFFFFFFFFu)
            continue;
        const u32 tau = slice_of_pos(rs, i);
        const bool is_first = first[(u64)s * S + tau] == first_pack(ce, i);
        if (is_first)
            atomicAdd(&s_cnt[tau], 1u);
        if (i == slice_last_pos(rs, tau))
            rs->last_new[tau] = is_first ? 1u : 0u;
    }
    __syncthreads();
    if (threadIdx.x < REF_THREADS && s_cnt[threadIdx.x])
        atomicAdd(&rs->Dt[threadIdx.x], (u64)s_cnt[threadIdx.x]);
}

// ---- census result: grow the worker tables' persistent bucket counts --------------------------
__global__ void census_update_kernel(DevState *st, ResState *rs)
{
    if (!rs->need)
        return;
    u64 acc = 0;
    int last = -1;
    for (u32 t = 0; t < REF_THREADS; t++)
    {
        rs->b0[t] = st->bt[t];
        rs->b1[t] = grown_buckets(st->bt[t], rs->Dt[t], rs->last_new[t] != 0);
        st->bt[t] = rs->b1[t];
        rs->prefixD[t] = acc;
        acc += rs->Dt[t];
        if (rs->Dt[t])
            last = (int)t;
    }
    rs->prefixD[REF_THREADS] = acc;
    rs->last_slice = last;
}

// ---- resolver: rank of first sight inside each slice (exclusive scan of the first-flags) ------
constexpr int SCAN_TILE = 4096;
__global__ void __launch_bounds__(256) rank_tile_count_kernel(ResState *rs, const u64 *first, const u32 *pos_slot, u32 *tile_cnt)
{
    __shared__ u32 s_c;
    const u64 np = rs->npairs, S = rs->slices, ce = rs->census_epoch;
    const u64 ntiles = (np + SCAN_TILE - 1) / SCAN_TILE;
    for (u64 tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
    {
        if (threadIdx.x == 0)
            s_c = 0;
        __syncthreads();
        u32 c = 0;
        for (int k = threadIdx.x; k < SCAN_TILE; k += blockDim.x)
        {
            const u64 i = tile * SCAN_TILE + k;
            if (i < np)
            {
                const u32 s = pos_slot[i];
                if (s != 0xFFFFFFFFu && first[(u64)s * S + slice_of_pos(rs, i)] == first_pack(ce, i))
                    c++;
            }
        }
        for (int o = 16; o; o >>= 1)
            c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
        if ((threadIdx.x & 31) == 0 && c)
            atomicAdd(&s_c, c);
        __syncthreads();
        if (threadIdx.x == 0)
            tile_cnt[tile] = s_c;
        __syncthreads();
    }
}

// exclusive scan of the per-tile counts (one block; 64-bit running total)
__global__ void __launch_bounds__(1024) rank_tile_scan_kernel(ResState *rs, const u32 *tile_cnt, u64 *tile_off)
{
    __shared__ u64 s_w[32];
    __shared__ u64 s_base;
    const u64 ntiles = (rs->npairs + SCAN_TILE - 1) / SCAN_TILE;
    if (threadIdx.x == 0)
        s_base = 0;
    __syncthreads();
    for (u64 b = 0; b < ntiles; b += blockDim.x)
    {
        const u64 i = b + threadIdx.x;
        const u64 v = (i < ntiles) ? tile_cnt[i] : 0;
        u64 incl = v;
        for (int o = 1; o < 32; o <<= 1)
        {
            const u64 t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if ((threadIdx.x & 31) >= o)
                incl += t;
        }
        if ((threadIdx.x & 31) == 31)
            s_w[threadIdx.x >> 5] = incl;
        __syncthreads();
        u64 woff = 0, tot = 0;
        for (int w = 0; w < 32; w++)
        {
            const u64 t = s_w[w];
            if (w < (int)(threadIdx.x >> 5))
                woff += t;
            tot += t;
        }
        if (i < ntiles)
            tile_off[i] = s_base + woff + incl - v;
        __syncthreads();
        if (threadIdx.x == 0)
            s_base += tot;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256) rank_assign_kernel(ResState *rs, const u64 *first, const u32 *pos_slot, const u64 *tile_off,
                                                          u32 *rank)
{
    __shared__ u32 s_w[8];
    const u64 np = rs->npairs, S = rs->slices, ce = rs->census_epoch;
    const u64 ntiles = (np + SCAN_TILE - 1) / SCAN_TILE;
    constexpr int PER = SCAN_TILE / 256; // 16 consecutive positions per thread
    for (u64 tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
    {
        const u64 i0 = tile * SCAN_TILE + (u64)threadIdx.x * PER;
        u32 flags = 0;
        for (int k = 0; k < PER; k++)
        {
            const u64 i = i0 + k;
            if (i < np)
            {
                const u32 s = pos_slot[i];
                if (s != 0xFFFFFFFFu && first[(u64)s * S + slice_of_pos(rs, i)] == first_pack(ce, i))
                    flags |= 1u << k;
            }
        }
        const u32 c = (u32)__popc(flags);
        u32 incl = c;
        for (int o = 1; o < 32; o <<= 1)
        {
            const u32 t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if ((threadIdx.x & 31) >= o)
                incl += t;
        }
        if ((threadIdx.x & 31) == 31)
            s_w[threadIdx.x >> 5] = incl;
        __syncthreads();
        u32 woff = 0;
        for (int w = 0; w < (int)(threadIdx.x >> 5); w++)
            woff += s_w[w];
        u64 g = tile_off[tile] + woff + incl - c; // flagged positions strictly before my first one
        for (int k = 0; k < PER; k++)
            if ((flags >> k) & 1u)
            {
                const u64 i = i0 + k;
                const u32 tau = slice_of_pos(rs, i);
                rank[(u64)pos_slot[i] * S + tau] = (u32)(g - rs->prefixD[tau] + 1); // 1-based inside the slice
                g++;
            }
        __syncthreads();
    }
}

// is the (slot, tau) entry the first sight of its key in the merge sequence (no lower worker has it)?
__device__ __forceinline__ bool entry_first_seen(const u64 *first, u64 S, u64 ce, u64 slot, u32 tau)
{
    for (u32 q = 0; q < tau; q++)
        if ((first[slot * S + q] >> 32) == ce)
            return false;
    return true;
}

// ---- resolver: keys new to the merge sequence per worker; the last insert call of the merge ---
__global__ void __launch_bounds__(256) entry_pass1_kernel(DevState *st, ResState *rs, const u64 *first, const u32 *pos_slot,
                                                          const u32 *rank)
{
    __shared__ u32 s_f[REF_THREADS];
    if (threadIdx.x < REF_THREADS)
        s_f[threadIdx.x] = 0;
    __syncthreads();
    const u64 np = rs->npairs, S = rs->slices, ce = rs->census_epoch;
    const int last = rs->last_slice;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < np; i += (u64)gridDim.x * blockDim.x)
    {
        const u32 s = pos_slot[i];
        if (s == 0xFFFFFFFFu)
            continue;
        const u32 tau = slice_of_pos(rs, i);
        if (first[(u64)s * S + tau] != first_pack(ce, i))
            continue;
        const bool fs = entry_first_seen(first, S, ce, s, tau);
        if (fs)
            atomicAdd(&s_f[tau], 1u);
        if ((int)tau == last)
        {
            const u32 h = (u32)st->tmeta[s];
            const u64 r = rank[(u64)s * S + tau];
            const u64 key = ((u64)h % rs->b1[tau]) << 32 |
                            ((u64)cslot31(doublings_after(rs->b0[tau], rs->b1[tau], r), r) << 1) | (fs ? 1ull : 0ull);
            atomicMax(&rs->last_key, key);
        }
    }
    __syncthreads();
    if (threadIdx.x < REF_THREADS && s_f[threadIdx.x])
        atomicAdd(&rs->F[threadIdx.x], (u64)s_f[threadIdx.x]);
}

__global__ void resolver_mid_kernel(DevState *st, ResState *rs)
{
    const bool last_call_new = (rs->last_key & 1ull) != 0;
    rs->bm = grown_buckets(65536, (u64)st->distinct, last_call_new);
    rs->fmax = (u32)(st->sel_key >> 32);
    rs->wbucket = 0xFFFFFFFFu;
    rs->n_cand = 0;
}

// ---- resolver: winning bucket under the true bucket count, then the tied pairs in it -----------
__global__ void __launch_bounds__(256) cand_bucket_kernel(DevState *st, ResState *rs)
{
    const u64 cap = st->tcap;
    const u64 bm = rs->bm;
    const u32 fmax = rs->fmax;
    u32 best = 0xFFFFFFFFu;
    for (u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += (u64)gridDim.x * blockDim.x)
    {
        const u64 mv = st->tmeta[s];
        if ((u32)(mv >> 32) == fmax)
        {
            const u32 bk = (u32)((u64)(u32)mv % bm);
            best = bk < best ? bk : best;
        }
    }
    for (int o = 16; o; o >>= 1)
    {
        const u32 t = __shfl_xor_sync(0xFFFFFFFFu, best, o);
        best = t < best ? t : best;
    }
    if ((threadIdx.x & 31) == 0 && best != 0xFFFFFFFFu)
        atomicMin(&rs->wbucket, best);
}

__global__ void __launch_bounds__(256) cand_collect_kernel(DevState *st, ResState *rs, const u64 *first, const u32 *rank)
{
    const u64 cap = st->tcap, S = rs->slices, ce = rs->census_epoch;
    const u64 bm = rs->bm;
    const u32 fmax = rs->fmax, wb = rs->wbucket;
    for (u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += (u64)gridDim.x * blockDim.x)
    {
        const u64 mv = st->tmeta[s];
        if ((u32)(mv >> 32) != fmax || (u32)((u64)(u32)mv % bm) != wb)
            continue;
        const u32 idx = atomicAdd(&rs->n_cand, 1u);
        if (idx >= MAX_CAND)
        {
            rs->overflow = 1;
            continue;
        }
        u32 tau = 0;
        while (tau < S && (first[s * S + tau] >> 32) != ce)
            tau++;
        if (tau >= S)
        {
            atomicOr(&st->err, ERR_MISSING_KEY); // a counted pair that the stream does not contain
            tau = 0;
        }
        const u64 r = rank[s * S + tau];
        rs->cand_slot[idx] = s;
        rs->cand_tau[idx] = tau;
        rs->cand_ord[idx] =
            (((u64)(u32)mv % rs->b1[tau]) << 32) | (u64)cslot31(doublings_after(rs->b0[tau], rs->b1[tau], r), r);
        rs->cand_before[idx] = 0;
    }
}

// ---- resolver: how many keys new to the sequence precede each candidate in its worker's list --
__global__ void __launch_bounds__(256) entry_pass2_kernel(DevState *st, ResState *rs, const u64 *first, const u32 *pos_slot,
                                                          const u32 *rank)
{
    const u64 np = rs->npairs, S = rs->slices, ce = rs->census_epoch;
    const u32 nc = rs->n_cand < MAX_CAND ? rs->n_cand : MAX_CAND;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < np; i += (u64)gridDim.x * blockDim.x)
    {
        const u32 s = pos_slot[i];
        if (s == 0xFFFFFFFFu)
            continue;
        const u32 tau = slice_of_pos(rs, i);
        if (first[(u64)s * S + tau] != first_pack(ce, i))
            continue;
        bool any = false;
        for (u32 c = 0; c < nc; c++)
            any |= (rs->cand_tau[c] == tau);
        if (!any || !entry_first_seen(first, S, ce, s, tau))
            continue;
        const u32 h = (u32)st->tmeta[s];
        const u64 r = rank[(u64)s * S + tau];
        const u64 ord = (((u64)h % rs->b1[tau]) << 32) | (u64)cslot31(doublings_after(rs->b0[tau], rs->b1[tau], r), r);
        for (u32 c = 0; c < nc; c++)
            if (rs->cand_tau[c] == tau && ord < rs->cand_ord[c])
                atomicAdd(&rs->cand_before[c], 1ull);
    }
}

__global__ void resolver_commit_kernel(DevState *st, ResState *rs)
{
    if (st->stop != STOP_PAUSE)
        return;
    if (rs->overflow || rs->n_cand == 0)
    {
        atomicOr(&st->err, ERR_PROBE);
        return;
    }
    u64 prefF[REF_THREADS + 1];
    prefF[0] = 0;
    for (u32 t = 0; t < REF_THREADS; t++)
        prefF[t + 1] = prefF[t] + rs->F[t];
    u64 best_slot = ~0ull, best_cs = ~0ull;
    for (u32 c = 0; c < rs->n_cand; c++)
    {
        const u64 R = prefF[rs->cand_tau[c]] + rs->cand_before[c] + 1;
        const u64 cs = chain_slot(doublings_after(65536, rs->bm, R), R);
        if (cs < best_cs)
        {
            best_cs = cs;
            best_slot = rs->cand_slot[c];
        }
    }
    const u64 key = st->tkey[best_slot];
    commit_merge(st, (u32)(key & 0xFFFFFFFFull), (u32)(key >> 32), rs->fmax, cur_recs(st));
    st->stop = STOP_RUN;
    st->pause = 0;
}

} // namespace bpe
