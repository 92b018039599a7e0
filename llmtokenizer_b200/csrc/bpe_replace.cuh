// K3 for a != b (the overwhelmingly common case): fused replace + prefix-scan compaction + pair-count
// deltas as a TMA-fed, warp-specialised streaming kernel (sm_100a).
//
// Reference loop being replaced: bpe/src/bpe.c:760-772 (greedy left-to-right rewrite) plus the
// recount of the next iteration (bpe.c:460-471), which the delta vectors make unnecessary.
//
// One streaming pass, 4*n_k bytes in, 4*n_{k+1} bytes out.
//
// Layout.  Measured on B200 (profiles/, DESIGN.md): a single-pass scan whose tiles are chained
// through global memory (decoupled look-back, a central scan warp, or row-wise aggregates - all three
// were built and timed) tops out at 2.1-3.3 TB/s on this path, because every store waits for the
// slowest of the ~1,000 tile loads in flight in front of it, while the same kernel with no
// dependency between CTAs streams at 5.7 TB/s.  So the shard is kept RANGED: cut into nr <= 320
// ranges of whole tiles, one CTA per range, each range compacted in place of itself (range c lives at
// tok[buf][c*rcap .. c*rcap + rcnt[buf][c])).  The prefix scan is then local to the CTA - a running
// sum - and CTAs never wait for one another.  What crosses a range boundary is the same
// pair-independent edge information the GPUs exchange at shard boundaries (first three / last two
// tokens of each range, published by the CTA that wrote them), read at the start of the next pass.
// repack_kernel turns the stream back into one dense array when something needs that (a == b merges,
// the exact tie-break kernels, the static regime below 1,048,576 tokens, the final download).
//
// Inside a CTA (18 warps) a ring of shared-memory stages holds one 4,096-token tile (32 "iterations"
// of 128 tokens) each:
//   producer (1 warp)   one 1-D bulk copy (TMA: cp.async.bulk + mbarrier complete_tx) per tile;
//   scanners (8 warps)  4 iterations each: a lane owns one 128-bit chunk (conflict-free LDS.128),
//                       finds the replacements that start on it, counts kept tokens per iteration
//                       (ballots), emits the pair-count deltas;
//   offsets (1 warp)    turns the 32 per-iteration counts into output offsets (running sum), resolves
//                       the range's halos at the start and publishes its edges at the end;
//   storers (8 warps)   re-read the tile from shared memory and write the kept tokens: an iteration
//                       without replacements (the common case once the pair is rarer than ~1 in 1,000
//                       tokens) goes registers -> global with 128-bit stores realigned by warp
//                       shuffles; the others compact through a 136-word per-warp staging buffer.
#pragma once
#include <type_traits>
#include "bpe_kernels.cuh"

namespace bpe
{

#ifndef BPE_V_SCAN_WARPS
#define BPE_V_SCAN_WARPS 8
#endif
#ifndef BPE_V_STORE_WARPS
#define BPE_V_STORE_WARPS 8
#endif
constexpr int V_SCAN_WARPS = BPE_V_SCAN_WARPS;
constexpr int V_STORE_WARPS = BPE_V_STORE_WARPS;
constexpr int V_ITERS = 32;                        // iterations (128 tokens) per tile
constexpr int V_TILE = V_ITERS * 128;              // 4,096 tokens = 16 KB
constexpr int V_THREADS = (V_SCAN_WARPS + V_STORE_WARPS + 2) * 32;
#ifndef BPE_V_STAGES
#define BPE_V_STAGES 4
#endif
constexpr int V_STAGES = BPE_V_STAGES;   // ring depth without the shared-memory delta histogram
constexpr int V_STAGES_HIST = 4;         // with it (a 3-deep ring + a 40 KB histogram so that early merges could share passes
                                         // was tried: slower - those passes are bound by their replacements, not by streaming)
constexpr int V_STAGE_WORDS = V_TILE + 8;          // 4 tokens of halo on either side
constexpr int V_STAGING_WORDS = 136;               // per storer warp: 128 tokens + alignment phase
constexpr u32 V_TILE_BYTES = V_STAGE_WORDS * 4;
constexpr int V_WARP_PRODUCER = V_SCAN_WARPS + V_STORE_WARPS;
constexpr int V_WARP_OFFSETS = V_WARP_PRODUCER + 1;

__host__ __device__ inline size_t stream_smem_bytes(bool hist, u32 z)
{
    return (size_t)(hist ? V_STAGES_HIST : V_STAGES) * V_TILE_BYTES + (size_t)V_STORE_WARPS * V_STAGING_WORDS * 4 +
           (hist ? 16 * ((size_t)z + 1) : (size_t)CLS_SIZE);
}

// ---- mbarrier / bulk-copy wrappers (PTX ISA: mbarrier, cp.async.bulk) --------------------------
__device__ __forceinline__ u32 smem_addr(const void *p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(u64 *bar, u32 count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(u64 *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(u64 *bar, u32 bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(u64 *bar, u32 parity)
{
    u32 ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok)
                 : "r"(smem_addr(bar)), "r"(parity)
                 : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(u64 *bar, u32 parity)
{
    // try_wait with a suspend-time hint: the warp sleeps in hardware instead of burning issue slots in a poll
    // loop (ncu: a third of an early pass's instructions were YIELD / TRYWAIT / BRA of idle roles)
    const u32 addr = smem_addr(bar);
    u32 ok;
    do
    {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok)
                     : "r"(addr), "r"(parity), "r"(2000u)
                     : "memory");
    } while (!ok);
}
__device__ __forceinline__ void bulk_load(void *smem_dst, const void *gmem_src, u32 bytes, u64 *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_addr(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_addr(bar))
                 : "memory");
}
__device__ __forceinline__ void scanner_bar()
{
    asm volatile("bar.sync 1, %0;" ::"n"(V_SCAN_WARPS * 32) : "memory");
}
__device__ __forceinline__ void st_v4(u32 *p, u32 x, u32 y, u32 z, u32 w)
{
    *reinterpret_cast<uint4 *>(p) = make_uint4(x, y, z, w);
}
__device__ __forceinline__ void st_v2(u32 *p, u32 x, u32 y) { *reinterpret_cast<uint2 *>(p) = make_uint2(x, y); }


// per-stage bookkeeping in shared memory
template <bool WIDE> struct StageMetaT
{
    u32 excl;            // output offset of the tile inside the range (running sum)
    u32 slowmask;        // bit j: iteration j has replacements / removals / invalid tokens
    u32 cnt[V_ITERS];    // kept tokens per iteration
    u32 pre[V_ITERS];    // exclusive prefix of cnt
    // what the scanner found, per lane, handed to the storers: iter_bits' five bits (one merge per pass), or
    // those bits << 16 | the four pair nibbles of iter_bits_multi (batched passes, WIDE)
    typename std::conditional<WIDE, u32, unsigned char>::type bits[V_ITERS][32];
};

// Replacements that start on my chunk and whether my first token is removed, for iteration j of the
// tile staged at sin (sin[p] = token at tile position p, p in [-4, V_TILE + 4)).
//   bits 0..3: a replacement starts on token k; bit 4: token 0 is the `b` of one that starts in front
// Returns false (and bits = 0) when the whole warp has nothing to do in this iteration.
__device__ __forceinline__ bool iter_bits(const u32 *sin, int j, int lane, u32 a, u32 b, u32 valid, bool full, const uint4 &c,
                                          u32 &bits, u32 &v)
{
    const u32 nxl = sin[(j + 1) * 128];
    const u32 pvl = sin[j * 128 - 1];
    u32 nx = __shfl_down_sync(0xFFFFFFFFu, c.x, 1);
    if (lane == 31)
        nx = nxl;
    const u32 x0 = __shfl_sync(0xFFFFFFFFu, c.x, 0);
    const u32 carry = (pvl == a && x0 == b) ? 1u : 0u;
    bool m0 = (c.x == a) && (c.y == b);
    bool m1 = (c.y == a) && (c.z == b);
    bool m2 = (c.z == a) && (c.w == b);
    bool m3 = (c.w == a) && (nx == b);
    v = 4;
    if (!full)
    {
        const u32 p = (u32)j * 128u + (u32)lane * 4u;
        v = (p >= valid) ? 0u : ((valid - p < 4u) ? (valid - p) : 4u);
        m0 = m0 && v > 0;
        m1 = m1 && v > 1;
        m2 = m2 && v > 2;
        m3 = m3 && v > 3;
    }
    bits = 0;
    if (!(__any_sync(0xFFFFFFFFu, m0 | m1 | m2 | m3) || carry || !full))
        return false;
    const u32 mb3 = __ballot_sync(0xFFFFFFFFu, m3);
    const u32 r0 = (((mb3 << 1) | carry) >> lane) & 1u;
    bits = (u32)m0 | ((u32)m1 << 1) | ((u32)m2 << 2) | ((u32)m3 << 3) | (r0 << 4);
    return true;
}
__device__ __forceinline__ u32 keep_mask(u32 bits, u32 v) { return ((1u << v) - 1u) & ~((bits >> 4) | ((bits & 7u) << 1)) & 0xFu; }

// Batched pass (nb > 1 merges at once; all 2*nb tokens differ, so at most one pair can match at a position).
// 1 + index of the pair that matches (x, y), 0 if none
__device__ __forceinline__ u32 pair_of(u32 x, u32 y, u32 nb, const u32 *ba, const u32 *bb)
{
    u32 r = 0;
    for (u32 i = 0; i < nb; i++)
        if (x == ba[i] && y == bb[i])
            r = i + 1;
    return r;
}
// pair_of through the class table (see iter_bits_multi)
__device__ __forceinline__ u32 pair_of_cls(u32 x, u32 y, const unsigned char *cls, bool verify, const u32 *ra)
{
    const u32 kx = cls[x & CLS_MASK], ky = cls[y & CLS_MASK];
    u32 m = ((kx & 15u) == (ky >> 4)) ? (kx & 15u) : 0u;
    if (verify && m && (x != ra[2 * (m - 1)] || y != ra[2 * (m - 1) + 1]))
        m = 0;
    return m;
}
// as iter_bits; mi = four nibbles, 1 + index of the pair whose replacement starts on token k.  Which pair a
// token belongs to comes from a byte table in shared memory indexed by (token mod CLS_SIZE): low nibble = 1 +
// index of the pair it is the FIRST token of, high nibble = the pair it is the SECOND token of (the tokens of a
// batch are pairwise different mod CLS_SIZE, see tok_alias).  A replacement starts where the low nibble of a
// token equals the high nibble of the next one and is not zero: the cost does not grow with the batch.  Ids
// beyond CLS_SIZE alias table entries, so candidates are then checked against the real pair (verify).
__device__ __forceinline__ bool iter_bits_multi(const u32 *sin, int j, int lane, const unsigned char *cls, bool verify,
                                                const u32 *ra, u32 valid, bool full, const uint4 &c, u32 &bits, u32 &v, u32 &mi)
{
    const u32 k0 = cls[c.x & CLS_MASK], k1 = cls[c.y & CLS_MASK], k2 = cls[c.z & CLS_MASK], k3 = cls[c.w & CLS_MASK];
    const u32 nxl = sin[(j + 1) * 128];
    const u32 pvl = sin[j * 128 - 1];
    u32 kn = __shfl_down_sync(0xFFFFFFFFu, k0, 1);
    if (lane == 31)
        kn = cls[nxl & CLS_MASK];
    const u32 kx0 = __shfl_sync(0xFFFFFFFFu, k0, 0);
    const u32 kp = cls[pvl & CLS_MASK];
    u32 carry = ((kp & 15u) == (kx0 >> 4)) ? (kp & 15u) : 0u;
    const u32 m0 = ((k0 & 15u) == (k1 >> 4)) ? (k0 & 15u) : 0u;
    const u32 m1 = ((k1 & 15u) == (k2 >> 4)) ? (k1 & 15u) : 0u;
    const u32 m2 = ((k2 & 15u) == (k3 >> 4)) ? (k2 & 15u) : 0u;
    const u32 m3 = ((k3 & 15u) == (kn >> 4)) ? (k3 & 15u) : 0u;
    mi = m0 | (m1 << 4) | (m2 << 8) | (m3 << 12);
    if (verify) // uniform: the vocabulary is larger than the table
    {
        u32 nx = __shfl_down_sync(0xFFFFFFFFu, c.x, 1);
        if (lane == 31)
            nx = nxl;
        const u32 x0 = __shfl_sync(0xFFFFFFFFu, c.x, 0);
        if (mi)
        {
            const u32 tk[5] = {c.x, c.y, c.z, c.w, nx};
#pragma unroll
            for (int k = 0; k < 4; k++)
            {
                const u32 m = (mi >> (4 * k)) & 15u;
                if (m && (tk[k] != ra[2 * (m - 1)] || tk[k + 1] != ra[2 * (m - 1) + 1]))
                    mi &= ~(15u << (4 * k));
            }
        }
        if (carry && (pvl != ra[2 * (carry - 1)] || x0 != ra[2 * (carry - 1) + 1]))
            carry = 0;
    }
    v = 4;
    if (!full)
    {
        const u32 p = (u32)j * 128u + (u32)lane * 4u;
        v = (p >= valid) ? 0u : ((valid - p < 4u) ? (valid - p) : 4u);
        mi &= (v >= 4) ? 0xFFFFu : ((1u << (4 * v)) - 1u);
    }
    bits = 0;
    if (!(__any_sync(0xFFFFFFFFu, mi != 0) || carry || !full))
        return false;
    const bool b3 = (mi >> 12) != 0;
    const u32 mb3 = __ballot_sync(0xFFFFFFFFu, b3);
    const u32 r0 = (((mb3 << 1) | (carry ? 1u : 0u)) >> lane) & 1u;
    bits = ((mi & 0xFu) ? 1u : 0u) | ((mi & 0xF0u) ? 2u : 0u) | ((mi & 0xF00u) ? 4u : 0u) | ((mi & 0xF000u) ? 8u : 0u) | (r0 << 4);
    return true;
}

// ---- a == b on a RANGED stream ---------------------------------------------------------------------------------
// `aaaa -> z z`: replacements pair up from the start of each run of a (bpe.c:760-772 is greedy left to right), so a
// position starts one iff it holds a, its right neighbour holds a, and the number of a right in front of it is
// even.  That parity crosses tiles, ranges and shards, which the warp-specialised pipeline below (every 128-token
// iteration scanned independently) cannot carry; a == b merges are rare (under 1 % of merges on the Zipf corpora),
// so they take this plain path in the same launch instead of pausing the loop for a repack -> dense kernel ->
// re-partition detour (round 1: 5-8 % of a run).  One CTA per range as in the streaming path, tiles one after the
// other (the parity and the output offset are running values of the CTA), every range compacted in place.
//   across ranges: every CTA first publishes the parity of the run that ends its INPUT range (st->rpar, stamped
//                  with the merge epoch) and reads the ranges in front of it as far as the run reaches (all CTAs of
//                  the grid are resident: one per range, two per SM);
//   across shards: st->carry_in, derived from the peers' edge records (resolve_edges).
// The pair-count deltas follow replace_kernel's rules for a == b (each pair INSTANCE charged once).
constexpr int SP_ITEMS = 8, SP_THREADS = V_TILE / SP_ITEMS; // 512 of the CTA's threads hold 8 tokens each
__device__ __noinline__ void same_pair_range(DevState *st, int32_t *gdelta, u32 *smem)
{
    const u32 a = st->a, z = st->z, cta = blockIdx.x, nr = st->nr, epoch = st->epoch;
    const u32 ibuf = st->cur, obuf = st->cur ^ 1u;
    const u64 rcap = st->rcap;
    const u32 n = st->rcnt[ibuf][cta];
    const u32 *in = st->tok[ibuf] + (u64)cta * rcap;
    u32 *out = st->tok[obuf] + (u64)cta * rcap;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    u32 *s_tok = smem + 4; // s_tok[p] = token at tile position p, p in [-2, V_TILE + 3)
    __shared__ u32 s_halo[5], s_carry, s_warp[V_THREADS / 32], s_tail[2];
    const u32 *cnt = st->rcnt[ibuf], *ed = st->redge[ibuf];
    if (cta == 0 && tid == 0)
        st->layout_next = LAYOUT_RANGED;
    if (warp == 0)
    {
        // parity of the run of equal tokens that ends my input range (whatever the token: it only matters if it is a)
        u32 run = 0;
        bool uniform = true;
        if (n)
        {
            const u32 last = in[n - 1];
            u32 pos = n;
            while (pos > 0)
            {
                const int i = (int)pos - 1 - lane;
                const bool eq = (i >= 0) && (in[i] == last);
                const u32 m = __ballot_sync(0xFFFFFFFFu, eq);
                const int c = (m == 0xFFFFFFFFu) ? 32 : (__ffs(~m) - 1);
                run += (u32)c;
                pos -= (u32)c;
                if (c < 32)
                    break;
            }
            uniform = (run == n);
        }
        if (lane == 0)
        {
            *reinterpret_cast<volatile u32 *>(&st->rpar[cta]) = (epoch << 2) | ((u32)uniform << 1) | (run & 1u);
            __threadfence();
            // halos: the two tokens in front of my range and the three behind it (as in the streaming path)
            u32 near[2];
            int got = 0;
            for (int q = (int)cta - 1; q >= 0 && got < 2; q--)
            {
                if (cnt[q] >= 1 && got < 2)
                    near[got++] = ed[q * EDGE_WORDS + 4];
                if (cnt[q] >= 2 && got < 2)
                    near[got++] = ed[q * EDGE_WORDS + 3];
            }
            s_halo[1] = got >= 1 ? near[0] : st->halo_before[1];
            s_halo[0] = got >= 2 ? near[1] : (got == 1 ? st->halo_before[1] : st->halo_before[0]);
            got = 0;
            for (u32 q = cta + 1; q < nr && got < 3; q++)
                for (u32 k = 0; k < 3 && k < cnt[q] && got < 3; k++)
                    s_halo[2 + got++] = ed[q * EDGE_WORDS + k];
            for (int k = 0; got < 3; k++)
                s_halo[2 + got++] = st->halo_after[k];
            // parity of the number of a right in front of my range: back through the ranges while the run goes on
            u32 acc = 0;
            bool open = (s_halo[1] == a);
            int q = (int)cta - 1;
            while (open && q >= 0)
            {
                if (cnt[q] == 0)
                {
                    q--;
                    continue;
                }
                u32 v;
                do
                {
                    v = *reinterpret_cast<volatile u32 *>(&st->rpar[q]);
                } while ((v >> 2) != (epoch & 0x3FFFFFFFu));
                acc ^= v & 1u;
                open = (v & 2u) != 0;
                q--;
            }
            if (open) // the run reaches the start of the shard: the neighbouring GPU's part of it
                acc ^= st->carry_in & 1u;
            s_carry = acc;
        }
    }
    __syncthreads();
    u32 carry = s_carry; // parity of the number of a right in front of the current tile
    u32 out_off = 0;
    const u32 ntiles = (n + V_TILE - 1) / V_TILE;
    for (u32 t = 0; t < ntiles; t++)
    {
        const u32 base = t * V_TILE;
        const u32 tl = (n - base < (u32)V_TILE) ? (n - base) : (u32)V_TILE;
        // ---- stage the tile.  The two tokens in front of it come from the previous tile's copy (their place in the
        // stream may have been overwritten by that tile's output), the ones behind it have not been touched yet.
        for (int p = tid; p < V_TILE + 3; p += V_THREADS)
        {
            const u32 g = base + (u32)p;
            s_tok[p] = (g < n) ? in[g] : ((g - n < 3u) ? s_halo[2 + (g - n)] : SENT);
        }
        if (tid < 2)
            s_tok[tid - 2] = (t == 0) ? s_halo[tid] : s_tail[tid];
        __syncthreads();
        u32 keep = 0, mm = 0, cntk = 0, ea = 0;
        u32 w[SP_ITEMS + 5]; // w[k] = token at tile position p0 + k - 2
        const u32 p0 = (u32)tid * SP_ITEMS;
        const bool worker = tid < SP_THREADS;
        if (worker)
        {
#pragma unroll
            for (int k = 0; k < SP_ITEMS + 5; k++)
                w[k] = s_tok[(int)p0 + k - 2];
            const u32 valid = (p0 >= tl) ? 0u : ((tl - p0 < (u32)SP_ITEMS) ? (tl - p0) : (u32)SP_ITEMS);
            const u32 OWNV = ((1u << valid) - 1u) << 2;
#pragma unroll
            for (int k = 0; k < SP_ITEMS + 5; k++)
                ea |= (u32)(w[k] == a) << k;
            u32 par0 = 0; // parity of the number of a right in front of my first token
            if (valid > 0 && ((ea >> 1) & 1u))
            {
                u32 c = 0;
                int i = (int)p0 - 1;
                while (i >= 0 && s_tok[i] == a)
                {
                    c++;
                    i--;
                }
                par0 = (i < 0) ? ((c ^ carry) & 1u) : (c & 1u);
            }
            u32 m = ((ea >> 1) & (ea >> 2) & 1u & par0) << 1; // does one start at my left neighbour?
            u32 par = par0;
#pragma unroll
            for (int k = 2; k < SP_ITEMS + 2; k++)
            {
                const u32 isa = (ea >> k) & 1u;
                m |= (isa & ((ea >> (k + 1)) & 1u) & (par ^ 1u)) << k;
                par = isa ? (par ^ 1u) : 0u;
            }
            mm = m & OWNV;            // replacements that start on my tokens
            keep = OWNV & ~(m << 1);  // a token goes away iff one starts at its left neighbour
            cntk = (u32)__popc(keep);
        }
        // the carry for the next tile, and this tile's last two tokens, before the tile is overwritten
        if (tid == V_THREADS - 1)
        {
            u32 c = 0;
            int i = (int)tl - 1;
            while (i >= 0 && s_tok[i] == a)
            {
                c++;
                i--;
            }
            s_carry = (i < 0) ? ((c ^ carry) & 1u) : (c & 1u);
            s_tail[0] = s_tok[(int)tl - 2];
            s_tail[1] = s_tok[(int)tl - 1];
        }
        // ---- block-wide exclusive scan of the kept counts
        u32 incl = cntk;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const u32 v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o)
                incl += v;
        }
        if (lane == 31)
            s_warp[warp] = incl;
        __syncthreads(); // every thread has read its window: s_tok may now be overwritten
        u32 woff = 0, total = 0;
#pragma unroll
        for (int i = 0; i < V_THREADS / 32; i++)
        {
            const u32 v = s_warp[i];
            woff += (i < warp) ? v : 0u;
            total += v;
        }
        carry = s_carry;
        if (worker)
        {
            u32 r = woff + incl - cntk;
#pragma unroll
            for (int k = 2; k < SP_ITEMS + 2; k++)
                if ((keep >> k) & 1u)
                    s_tok[r++] = ((mm >> k) & 1u) ? z : w[k];
            // ---- pair-count deltas (replace_kernel's rules for a == b)
            if (mm)
            {
#pragma unroll
                for (int k = 2; k < SP_ITEMS + 2; k++)
                    if ((mm >> k) & 1u)
                    {
                        const u32 x = w[k - 1], y = w[k + 2];
                        const u32 pm = (ea >> (k - 1)) & 1u;                      // a replacement ends right in front
                        const u32 nm = (ea >> (k + 2)) & (ea >> (k + 3)) & 1u;    // another one starts right behind
                        if (x != SENT)
                        {
                            if (x != a)
                                delta_add(st, gdelta, (u64)x * 4 + 0, 1);
                            delta_add(st, gdelta, (u64)(pm ? z : x) * 4 + 2, 1);
                        }
                        if (y != SENT && !nm)
                        {
                            if (y != a)
                                delta_add(st, gdelta, (u64)y * 4 + 1, 1);
                            delta_add(st, gdelta, (u64)y * 4 + 3, 1);
                        }
                    }
            }
        }
        __syncthreads();
        for (u32 i = tid; i < total; i += V_THREADS)
            out[out_off + i] = s_tok[i];
        out_off += total;
        __syncthreads();
    }
    __syncthreads();
    if (tid == 0)
    {
        __threadfence_block();
        u32 *oe = st->redge[obuf] + cta * EDGE_WORDS;
        const volatile u32 *o = out;
        for (u32 k = 0; k < 3; k++)
            oe[k] = (k < out_off) ? o[k] : SENT;
        oe[3] = out_off >= 2 ? o[out_off - 2] : SENT;
        oe[4] = out_off >= 1 ? o[out_off - 1] : SENT;
        st->rcnt[obuf][cta] = out_off;
        atomicAdd(&st->n_next, (u64)out_off);
    }
}

template <bool SMEM_HIST>
__global__ void __launch_bounds__(V_THREADS, 2) replace_stream_kernel(DevState *st, int32_t *delta, u32 hist_words)
{
    constexpr int NST = SMEM_HIST ? V_STAGES_HIST : V_STAGES;
    pdl_wait();
    pdl_launch_dependents();
    if (st->stop != STOP_RUN || st->skip)
        return;
    // Two specialisations keep each variant's code small (the kernel is instruction-bound on replacement-heavy
    // passes and ncu shows instruction-cache misses): <true> = one merge, deltas privatised in shared memory (the
    // host launches it only while ids are below hist_max, where passes are never batched); <false> = up to BATCH_MAX
    // merges, deltas straight to global memory.
    const u32 a = st->a, b = st->b, z = st->z;
    const u32 nb = SMEM_HIST ? 1u : st->nb;
    const u32 VS = z + nb; // delta block stride, see apply_deltas
    const u32 hist_need = 4 * VS;
    constexpr bool use_hist = SMEM_HIST;
    if (SMEM_HIST && (st->nb != 1 || hist_need > hist_words))
    {
        if (threadIdx.x == 0)
            atomicOr(&st->err, ERR_PROBE); // host / device disagree about the regime: fail loudly
        return;
    }
    const u32 cta = blockIdx.x, nr = st->nr;
    if (st->layout != LAYOUT_RANGED)
    {
        if (threadIdx.x == 0)
            atomicOr(&st->err, ERR_PROBE); // host logic error: this kernel only takes passes of a RANGED stream
        return;
    }
    if (cta >= nr)
        return;
    extern __shared__ __align__(16) u32 smem[];
    if (a == b)
    {
        same_pair_range(st, delta + HDR_INTS, smem);
        return;
    }
    const u32 ibuf = st->cur, obuf = st->cur ^ 1u;
    const u64 rcap = st->rcap;
    const u32 n = st->rcnt[ibuf][cta]; // tokens of my range
    if (cta == 0 && threadIdx.x == 0)
        st->layout_next = LAYOUT_RANGED;

    u32 *s_in = smem;                                       // NST x V_STAGE_WORDS
    u32 *s_staging = smem + NST * V_STAGE_WORDS;       // V_STORE_WARPS x V_STAGING_WORDS
    int32_t *s_hist = reinterpret_cast<int32_t *>(s_staging + V_STORE_WARPS * V_STAGING_WORDS);
    unsigned char *s_cls = reinterpret_cast<unsigned char *>(s_hist); // <false> only: token -> pair table of a batched pass
    const bool cls_verify = (z + nb > CLS_SIZE);
    __shared__ __align__(8) u64 s_full[NST], s_scanned[NST], s_ready[NST], s_empty[NST], s_halo_ready;
    using StageMeta = StageMetaT<!SMEM_HIST>;
    __shared__ StageMeta s_meta[NST];
    __shared__ u32 s_halo[5]; // tokens at range positions -2, -1, n, n+1, n+2
    __shared__ u32 s_ba[BATCH_MAX], s_bb[BATCH_MAX];
    __shared__ __align__(16) u32 s_ab[2 * BATCH_MAX]; // the same pairs interleaved (a0, b0, a1, b1, ...)

    // in and out are the same array (the stream is compacted in place, see partition_kernel): every tile is
    // written at or below where it was read, and the storers wait for the next tile's load (whose front
    // halo is the only part of it a store of this tile can reach) before they write
    const u32 *in = st->tok[ibuf] + (u64)cta * rcap;
    u32 *out = st->tok[obuf] + (u64)cta * rcap;
    const u32 ntiles = (n + V_TILE - 1) / V_TILE;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int32_t *gdelta = delta + HDR_INTS;

    if (tid == 0)
    {
        for (int s = 0; s < NST; s++)
        {
            mbar_init(&s_full[s], 1);
            mbar_init(&s_scanned[s], V_SCAN_WARPS);
            mbar_init(&s_ready[s], 1);
            mbar_init(&s_empty[s], V_STORE_WARPS);
            s_meta[s].slowmask = 0;
        }
        mbar_init(&s_halo_ready, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (use_hist)
        for (u32 i = tid; i < hist_need; i += V_THREADS)
            s_hist[i] = 0;
    if (tid < BATCH_MAX)
    {
        s_ba[tid] = (tid < (int)nb) ? st->ba[tid] : SENT;
        s_bb[tid] = (tid < (int)nb) ? st->bb[tid] : SENT;
        s_ab[2 * tid] = s_ba[tid];
        s_ab[2 * tid + 1] = s_bb[tid];
    }
    // <false> always matches through the class table, a single merge included: one code path keeps the
    // variant small (ncu: 18 % of the stall samples of batched passes were instruction-cache misses)
    if (!SMEM_HIST)
        for (u32 i = tid; i < CLS_SIZE / 4; i += V_THREADS)
            reinterpret_cast<u32 *>(s_cls)[i] = 0;
    __syncthreads();
    if (!SMEM_HIST)
    {
        // every byte has one writer: the tokens of a batch differ mod CLS_SIZE (tok_alias in the selection); a
        // single merge whose two tokens alias each other (ids beyond CLS_SIZE, verified) shares one byte
        if (tid < (int)nb)
        {
            s_cls[s_ba[tid] & CLS_MASK] |= (unsigned char)(tid + 1);
            s_cls[s_bb[tid] & CLS_MASK] |= (unsigned char)((tid + 1) << 4);
        }
        __syncthreads();
    }

    if (warp == V_WARP_PRODUCER)
    {
        // ---------------- producer ----------------
        if (lane == 0)
        {
            for (u32 t = 0; t < ntiles; t++)
            {
                const u32 s = t % NST;
                if (t >= NST)
                    mbar_wait(&s_empty[s], ((t / NST) & 1u) ^ 1u);
                s_meta[s].slowmask = 0; // every storer is done with the previous tile of this stage
                mbar_arrive_expect_tx(&s_full[s], V_TILE_BYTES);
                bulk_load(s_in + s * V_STAGE_WORDS, in + (u64)t * V_TILE - 4, V_TILE_BYTES, &s_full[s]);
            }
        }
    }
    else if (warp == V_WARP_OFFSETS)
    {
        // ---------------- halos, output offsets (the range-local prefix scan), new edges ----------------
        if (lane == 0)
        {
            // the two tokens in front of my range and the three behind it, skipping empty ranges; beyond
            // the shard: the neighbouring GPUs' tokens (SENT at the true ends of the corpus)
            const u32 *cnt = st->rcnt[ibuf], *ed = st->redge[ibuf];
            u32 near[2];
            int got = 0;
            for (int q = (int)cta - 1; q >= 0 && got < 2; q--)
            {
                if (cnt[q] >= 1 && got < 2)
                    near[got++] = ed[q * EDGE_WORDS + 4];
                if (cnt[q] >= 2 && got < 2)
                    near[got++] = ed[q * EDGE_WORDS + 3];
            }
            s_halo[1] = got >= 1 ? near[0] : st->halo_before[1];
            s_halo[0] = got >= 2 ? near[1] : (got == 1 ? st->halo_before[1] : st->halo_before[0]);
            got = 0;
            for (u32 q = cta + 1; q < nr && got < 3; q++)
                for (u32 k = 0; k < 3 && k < cnt[q] && got < 3; k++)
                    s_halo[2 + got++] = ed[q * EDGE_WORDS + k];
            for (int k = 0; got < 3; k++)
                s_halo[2 + got++] = st->halo_after[k];
            mbar_arrive(&s_halo_ready);
        }
        __syncwarp();
        u32 run = 0; // kept tokens of the tiles in front, i.e. the output offset inside the range
        for (u32 t = 0; t < ntiles; t++)
        {
            const u32 s = t % NST;
            StageMeta &sm = s_meta[s];
            mbar_wait(&s_scanned[s], (t / NST) & 1u);
            const u32 cnt = sm.cnt[lane];
            u32 incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1)
            {
                const u32 v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                if (lane >= o)
                    incl += v;
            }
            sm.pre[lane] = incl - cnt;
            __syncwarp();
            if (lane == 0)
            {
                sm.excl = run;
                mbar_arrive(&s_ready[s]);
            }
            run += __shfl_sync(0xFFFFFFFFu, incl, 31);
        }
        // wait for the storers of the last tiles, then publish the range's new length and edges
        for (u32 t = (ntiles > (u32)NST ? ntiles - NST : 0); t < ntiles; t++)
            mbar_wait(&s_empty[t % NST], (t / NST) & 1u);
        __threadfence_block();
        if (lane == 0)
        {
            u32 *oe = st->redge[obuf] + cta * EDGE_WORDS;
            const volatile u32 *o = out;
            for (u32 k = 0; k < 3; k++)
                oe[k] = (k < run) ? o[k] : SENT;
            oe[3] = run >= 2 ? o[run - 2] : SENT;
            oe[4] = run >= 1 ? o[run - 1] : SENT;
            st->rcnt[obuf][cta] = run;
            atomicAdd(&st->n_next, (u64)run);
        }
    }
    else if (warp < V_SCAN_WARPS)
    {
        // ---------------- scanners ----------------
        constexpr int PER = V_ITERS / V_SCAN_WARPS;
        for (u32 t = 0; t < ntiles; t++)
        {
            const u32 s = t % NST;
            StageMeta &sm = s_meta[s];
            mbar_wait(&s_full[s], (t / NST) & 1u);
            const u32 base = t * V_TILE;
            const u32 valid = (n - base < (u32)V_TILE) ? (n - base) : (u32)V_TILE;
            const bool full = (valid == (u32)V_TILE);
            u32 *sin = s_in + s * V_STAGE_WORDS + 4;
            if (t == 0 || n < base + (u32)V_TILE + 4u)
            {
                // The tile's window reaches over an end of the range: those positions come from the
                // neighbouring ranges.  (Not only the last tile: when the last one holds fewer than
                // three tokens, the window of the tile in front of it sees past the end as well.)
                if (warp == 0)
                {
                    mbar_wait(&s_halo_ready, 0);
                    if (lane == 0)
                    {
                        if (t == 0)
                        {
                            sin[-2] = s_halo[0];
                            sin[-1] = s_halo[1];
                        }
                        for (u32 k = 0; k < 3; k++)
                        {
                            const u32 local = n + k - base; // n >= base + 1
                            if (local < (u32)V_TILE + 4u)
                                sin[local] = s_halo[2 + k];
                        }
                    }
                }
                scanner_bar();
            }
            u32 slow = 0;
#pragma unroll 2
            for (int jj = 0; jj < PER; jj++)
            {
                const int j = warp * PER + jj;
                const uint4 c = *reinterpret_cast<const uint4 *>(sin + j * 128 + lane * 4);
                u32 bits, v, mi = 0, ktj = 128;
                const bool slow_it = SMEM_HIST ? iter_bits(sin, j, lane, a, b, valid, full, c, bits, v)
                                               : iter_bits_multi(sin, j, lane, s_cls, cls_verify, s_ab, valid, full, c, bits, v, mi);
                if (slow_it)
                {
                    slow |= 1u << j;
                    ktj = __reduce_add_sync(0xFFFFFFFFu, (u32)__popc(keep_mask(bits, v)));
                    // ---- pair-count deltas of the replacements that start on my tokens
                    if (SMEM_HIST)
                        sm.bits[j][lane] = (unsigned char)bits;
                    else
                        sm.bits[j][lane] = (bits << 16) | mi;
                    if (bits & 0xFu)
                    {
                        const int p0 = j * 128 + lane * 4;
                        // one trip per replacement (a lane has at most two), not one per token position
                        for (u32 todo = bits & 0xFu; todo; todo &= todo - 1u)
                            {
                                const int k = __ffs(todo) - 1;
                                const int p = p0 + k;
                                const u32 xl = sin[p - 1], yr = sin[p + 2];
                                if (SMEM_HIST)
                                {
                                    const bool pm = (sin[p - 2] == a) && (xl == b); // a replacement ends right in front
                                    const bool nm = (yr == a) && (sin[p + 3] == b); // another one starts right behind
                                    if (xl != SENT)
                                    {
                                        const u32 xn = pm ? z : xl;
                                        if (use_hist)
                                        {
                                            atomicAdd(&s_hist[xl * 4 + 0], 1);
                                            atomicAdd(&s_hist[xn * 4 + 2], 1);
                                        }
                                        else
                                        {
                                            delta_add(st, gdelta, (u64)xl * 4 + 0, 1);
                                            delta_add(st, gdelta, (u64)xn * 4 + 2, 1);
                                        }
                                    }
                                    if (yr != SENT && !nm)
                                    {
                                        if (use_hist)
                                        {
                                            atomicAdd(&s_hist[yr * 4 + 1], 1);
                                            atomicAdd(&s_hist[yr * 4 + 3], 1);
                                        }
                                        else
                                        {
                                            delta_add(st, gdelta, (u64)yr * 4 + 1, 1);
                                            delta_add(st, gdelta, (u64)yr * 4 + 3, 1);
                                        }
                                    }
                                }
                                else
                                {
                                    // batched: the same ownership rule, with "a replacement" meaning one of any pair
                                    const u32 i = ((mi >> (4 * k)) & 15u) - 1u;
                                    const u32 pm = pair_of_cls(sin[p - 2], xl, s_cls, cls_verify, s_ab);
                                    const bool nm = pair_of_cls(yr, sin[p + 3], s_cls, cls_verify, s_ab) != 0;
                                    const u64 off = (u64)i * 4 * VS;
                                    if (xl != SENT)
                                    {
                                        const u32 xn = pm ? (z + pm - 1u) : xl;
                                        if (use_hist)
                                        {
                                            atomicAdd(&s_hist[off + xl * 4 + 0], 1);
                                            atomicAdd(&s_hist[off + xn * 4 + 2], 1);
                                        }
                                        else
                                        {
                                            delta_add(st, gdelta, off + (u64)xl * 4 + 0, 1);
                                            delta_add(st, gdelta, off + (u64)xn * 4 + 2, 1);
                                        }
                                    }
                                    if (yr != SENT && !nm)
                                    {
                                        if (use_hist)
                                        {
                                            atomicAdd(&s_hist[off + yr * 4 + 1], 1);
                                            atomicAdd(&s_hist[off + yr * 4 + 3], 1);
                                        }
                                        else
                                        {
                                            delta_add(st, gdelta, off + (u64)yr * 4 + 1, 1);
                                            delta_add(st, gdelta, off + (u64)yr * 4 + 3, 1);
                                        }
                                    }
                                }
                            }
                    }
                    // the delta loop is lane-divergent: reconverge here, or every shuffle / ballot of the next
                    // iteration runs through the slow divergent-warp path (measured: a third of all instructions)
                    __syncwarp();
                }
                if (lane == 0)
                    sm.cnt[j] = ktj;
            }
            __syncwarp(); // every lane's sm.bits are written before lane 0 publishes the tile
            if (lane == 0)
            {
                if (slow)
                    atomicOr(&sm.slowmask, slow);
                mbar_arrive(&s_scanned[s]);
            }
        }
    }
    else
    {
        // ---------------- storers ----------------
        const int sw = warp - V_SCAN_WARPS;
        u32 *stg = s_staging + sw * V_STAGING_WORDS;
        for (u32 t = 0; t < ntiles; t++)
        {
            const u32 s = t % NST;
            StageMeta &sm = s_meta[s];
            mbar_wait(&s_ready[s], (t / NST) & 1u);
            if (t + 1 < ntiles)
                mbar_wait(&s_full[(t + 1) % NST], ((t + 1) / NST) & 1u); // in place: see the note at `in`/`out`
            const u32 base = t * V_TILE;
            const u32 valid = (n - base < (u32)V_TILE) ? (n - base) : (u32)V_TILE;
            const bool full = (valid == (u32)V_TILE);
            const u32 *sin = s_in + s * V_STAGE_WORDS + 4;
            const u32 excl = sm.excl;
            const u32 slowmask = sm.slowmask;
#pragma unroll 2
            for (int j = sw; j < V_ITERS; j += V_STORE_WARPS)
            {
                const uint4 c = *reinterpret_cast<const uint4 *>(sin + j * 128 + lane * 4);
                const u32 g = excl + sm.pre[j];
                if (!((slowmask >> j) & 1u))
                {
                    // 128 kept tokens, contiguous in the output: 128-bit stores realigned by shuffles
                    u32 *o = out + g + 4 * lane;
                    const u32 ph = g & 3u;
                    if (ph == 0)
                        st_v4(o, c.x, c.y, c.z, c.w);
                    else if (ph == 1)
                    {
                        const u32 t0 = __shfl_down_sync(0xFFFFFFFFu, c.x, 1), t1 = __shfl_down_sync(0xFFFFFFFFu, c.y, 1),
                                  t2 = __shfl_down_sync(0xFFFFFFFFu, c.z, 1);
                        if (lane < 31)
                            st_v4(o + 3, c.w, t0, t1, t2);
                        else
                            o[3] = c.w;
                        if (lane == 0)
                        {
                            o[0] = c.x;
                            o[1] = c.y;
                            o[2] = c.z;
                        }
                    }
                    else if (ph == 2)
                    {
                        const u32 t0 = __shfl_down_sync(0xFFFFFFFFu, c.x, 1), t1 = __shfl_down_sync(0xFFFFFFFFu, c.y, 1);
                        if (lane < 31)
                            st_v4(o + 2, c.z, c.w, t0, t1);
                        else
                            st_v2(o + 2, c.z, c.w);
                        if (lane == 0)
                            st_v2(o, c.x, c.y);
                    }
                    else
                    {
                        const u32 t0 = __shfl_down_sync(0xFFFFFFFFu, c.x, 1);
                        if (lane < 31)
                            st_v4(o + 1, c.y, c.z, c.w, t0);
                        else
                        {
                            o[1] = c.y;
                            o[2] = c.z;
                            o[3] = c.w;
                        }
                        if (lane == 0)
                            o[0] = c.x;
                    }
                }
                else
                {
                    // compaction through the per-warp staging buffer
                    u32 bits, v, mi = 0x1111u; // single merge: every replacement is pair 0
                    if (SMEM_HIST)
                    {
                        // what the scanner found (the barrier chain scanned -> ready orders the accesses)
                        bits = sm.bits[j][lane];
                        const u32 p = (u32)j * 128u + (u32)lane * 4u;
                        v = full ? 4u : ((p >= valid) ? 0u : ((valid - p < 4u) ? (valid - p) : 4u));
                    }
                    else
                    {
                        const u32 w = sm.bits[j][lane];
                        bits = w >> 16;
                        mi = w & 0xFFFFu;
                        const u32 p = (u32)j * 128u + (u32)lane * 4u;
                        v = full ? 4u : ((p >= valid) ? 0u : ((valid - p < 4u) ? (valid - p) : 4u));
                    }
                    const u32 keep = keep_mask(bits, v);
                    const u32 kc = (u32)__popc(keep);
                    // exclusive prefix of the kept counts (0..4 each) from three ballots
                    const u32 lt = (1u << lane) - 1u;
                    const u32 incl = kc + (u32)__popc(__ballot_sync(0xFFFFFFFFu, kc & 1u) & lt) +
                                     2u * (u32)__popc(__ballot_sync(0xFFFFFFFFu, kc & 2u) & lt) +
                                     4u * (u32)__popc(__ballot_sync(0xFFFFFFFFu, kc & 4u) & lt);
                    const u32 ktj = sm.cnt[j];
                    const u32 ph = g & 3u;
                    u32 rk = ph + incl - kc;
                    const u32 tk[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
                    for (int k = 0; k < 4; k++)
                        if ((keep >> k) & 1u)
                            stg[rk++] = ((bits >> k) & 1u) ? (z + ((mi >> (4 * k)) & 15u) - 1u) : tk[k];
                    __syncwarp();
                    // stg[ph + i] <-> out[g + i], i in [0, ktj): aligned 16 B chunks line up on both sides
                    u32 *ob = out + (g - ph); // 16 B aligned
                    const u32 lo = ph, hi = ph + ktj;
                    for (u32 q = lane; q * 4 < hi; q += 32)
                    {
                        const u32 w0 = q * 4;
                        if (w0 >= lo && w0 + 4 <= hi)
                            *reinterpret_cast<uint4 *>(ob + w0) = *reinterpret_cast<const uint4 *>(stg + w0);
                        else
                        {
#pragma unroll
                            for (int k = 0; k < 4; k++)
                                if (w0 + k >= lo && w0 + k < hi)
                                    ob[w0 + k] = stg[w0 + k];
                        }
                    }
                    __syncwarp();
                }
            }
            __syncwarp();
            if (lane == 0)
                mbar_arrive(&s_empty[s]);
        }
    }

    if (use_hist)
    {
        __syncthreads();
        for (u32 i = tid; i < hist_need; i += V_THREADS)
        {
            const int32_t v = s_hist[i];
            if (v)
                delta_add(st, gdelta, i, v);
        }
    }
}



// ---------------------------------------------------------------------------------------------
// DENSE -> RANGED: cut tok[cur][0..n) into ranges of whole tiles, in place (a dense stream is a ranged
// stream whose ranges are full).  One block.
__global__ void __launch_bounds__(RANGE_MAX) partition_kernel(DevState *st)
{
    if (st->stop != STOP_RUN || st->layout != LAYOUT_DENSE)
        return;
    const u64 n = st->n;
    const u64 tiles = (n + V_TILE - 1) / V_TILE;
    u64 want = st->rmax ? st->rmax : 1;
    if (want > tiles)
        want = tiles;
    const u64 per = want ? (tiles + want - 1) / want : 0; // tiles per range
    const u64 rcap = per * V_TILE;
    const u32 nr = per ? (u32)((tiles + per - 1) / per) : 0;
    const u32 c = threadIdx.x;
    if (c < nr)
    {
        const u32 *t = st->tok[st->cur] + (u64)c * rcap;
        const u64 left = n - (u64)c * rcap;
        const u32 cnt = (u32)(left < rcap ? left : rcap);
        st->rcnt[st->cur][c] = cnt;
        u32 *e = st->redge[st->cur] + c * EDGE_WORDS;
        for (u32 k = 0; k < 3; k++)
            e[k] = (k < cnt) ? t[k] : SENT;
        e[3] = cnt >= 2 ? t[cnt - 2] : SENT;
        e[4] = cnt >= 1 ? t[cnt - 1] : SENT;
    }
    __syncthreads();
    if (c == 0)
    {
        st->nr = nr;
        st->rcap = rcap;
        st->layout = LAYOUT_RANGED;
        // passes now read and write the same array (half the working set: late streams stay in L2 from pass to pass)
        st->tok[st->cur ^ 1u] = st->tok[st->cur];
    }
}

// RANGED -> DENSE: range c is copied to its place in the dense stream of the other buffer (its offset
// is the sum of the lower ranges' lengths: <= 320 numbers, summed by every CTA for itself).  The last
// CTA to finish flips the buffers.  Runs whatever the loop state is (the host asks for it on pauses
// and before the final download).
__global__ void __launch_bounds__(1024) repack_kernel(DevState *st)
{
    if (st->layout != LAYOUT_RANGED)
        return;
    __shared__ u64 s_off;
    __shared__ u64 s_w[32];
    const u32 nr = st->nr, c = blockIdx.x;
    const u32 *cnt = st->rcnt[st->cur];
    if (c < nr)
    {
        u64 part = 0;
        for (u32 q = threadIdx.x; q < c; q += blockDim.x)
            part += cnt[q];
        // block sum (counts fit 32 bits per range; the sum may not)
        for (int o = 16; o; o >>= 1)
            part += __shfl_xor_sync(0xFFFFFFFFu, part, o);
        if ((threadIdx.x & 31) == 0)
            s_w[threadIdx.x >> 5] = part;
        __syncthreads();
        if (threadIdx.x == 0)
        {
            u64 t = 0;
            for (u32 w = 0; w < blockDim.x / 32; w++)
                t += s_w[w];
            s_off = t;
        }
        __syncthreads();
        const u32 *src = st->tok[st->cur] + (u64)c * st->rcap;
        u32 *dst = (st->tok_real[0] == st->tok[st->cur] ? st->tok_real[1] : st->tok_real[0]) + s_off;
        const u32 m = cnt[c];
        // four independent loads per thread and trip: a copy lives on the bytes it keeps in flight
        const u32 B = blockDim.x;
        u32 i = threadIdx.x;
        for (; i + 3 * B < m; i += 4 * B)
        {
            const u32 v0 = src[i], v1 = src[i + B], v2 = src[i + 2 * B], v3 = src[i + 3 * B];
            dst[i] = v0;
            dst[i + B] = v1;
            dst[i + 2 * B] = v2;
            dst[i + 3 * B] = v3;
        }
        for (; i < m; i += B)
            dst[i] = src[i];
    }
    __syncthreads();
    if (threadIdx.x == 0)
    {
        __threadfence();
        if (atomicAdd(&st->rp_done, 1u) == gridDim.x - 1)
        {
            st->rp_done = 0;
            // every block has read its pointers (it counted itself in after copying): un-alias the buffers
            st->tok[st->cur ^ 1u] = (st->tok_real[0] == st->tok[st->cur]) ? st->tok_real[1] : st->tok_real[0];
            st->cur ^= 1u;
            st->layout = LAYOUT_DENSE;
        }
    }
}

} // namespace bpe
