// bpe_decode.cuh — ids -> bytes on the GPU (SURVEY.md §8f rank 2).
//
// What it computes is what the reference's decompress()/resolve_pair() compute (bpe/src/bpe.c:23-92,
// 341-394): every id is replaced by the byte string its pair expands to, recursively.  The reference
// memoises the expansions as NUL-terminated strings in a hash table; here the host flattens the
// vocabulary once (id -> offset/length into one byte blob, O(sum of lengths)), and the stream is
// expanded in three launches:
//   D1 decode_len_kernel     per tile of DEC_TILE ids: sum of expansion lengths
//   D2 decode_scan_kernel    exclusive scan of the tile sums (one block; the tile count is n/2048)
//   D3 decode_expand_kernel  per tile: block scan of the lengths, bytes gathered from the blob into
//                            shared memory, written out as aligned 16-byte vectors
// HBM traffic per id: 4 B read twice (D1, D3) + its expansion written once; the blob (a few hundred
// KB) stays in L1/L2.  Byte-exact and NUL-safe (lengths are explicit), unlike the char* original.
// A batch of documents (D4) runs decode_batch_tiles_kernel, D1, D2 and decode_expand_kernel<true>, which also writes
// the byte offset of every document: O(1) per document and per tile on top of the plain decode.
#pragma once
#include "bpe_kernels.cuh"

namespace bpe
{

constexpr int DEC_THREADS = 256;
constexpr int DEC_PER_THREAD = 8;
constexpr int DEC_TILE = DEC_THREADS * DEC_PER_THREAD; // ids per block
constexpr u32 DEC_STAGE_BYTES = 32 * 1024;             // tile outputs up to this size are staged in shared memory

struct DecodeVocab
{
    const u32 *len;  // [vocab] expansion length of each id
    const u32 *off;  // [vocab] offset of the expansion in blob
    const uint8_t *blob;
    u32 vocab;
};

__device__ inline u64 dec_block_sum(u64 v, u64 *s_warp)
{
    for (int o = 16; o > 0; o >>= 1)
        v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    if ((threadIdx.x & 31) == 0)
        s_warp[threadIdx.x >> 5] = v;
    __syncthreads();
    u64 t = 0;
    for (int w = 0; w < DEC_THREADS / 32; w++)
        t += s_warp[w];
    __syncthreads();
    return t;
}

// D1: tile_sum[t] = bytes the ids of tile t expand to.  An id outside the vocabulary sets *err.
__global__ void __launch_bounds__(DEC_THREADS) decode_len_kernel(const u32 *__restrict__ tok, u64 n, DecodeVocab v,
                                                                 u64 *__restrict__ tile_sum, u32 *err)
{
    __shared__ u64 s_warp[DEC_THREADS / 32];
    const u64 base = (u64)blockIdx.x * DEC_TILE;
    u64 sum = 0;
#pragma unroll
    for (int k = 0; k < DEC_PER_THREAD; k++)
    {
        const u64 i = base + (u64)k * DEC_THREADS + threadIdx.x;
        if (i < n)
        {
            const u32 t = tok[i];
            if (t < v.vocab)
                sum += v.len[t];
            else
                atomicOr(err, 1u);
        }
    }
    sum = dec_block_sum(sum, s_warp);
    if (threadIdx.x == 0)
        tile_sum[blockIdx.x] = sum;
}

// D2: in-place exclusive scan of tile_sum[0..nt), total to tile_sum[nt].  One block.
__global__ void __launch_bounds__(1024) decode_scan_kernel(u64 *tile_sum, u64 nt)
{
    __shared__ u64 s_warp[32];
    __shared__ u64 s_carry;
    if (threadIdx.x == 0)
        s_carry = 0;
    __syncthreads();
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (u64 base = 0; base < nt; base += 1024)
    {
        const u64 i = base + threadIdx.x;
        const u64 x = i < nt ? tile_sum[i] : 0;
        u64 incl = x;
        for (int o = 1; o < 32; o <<= 1)
        {
            const u64 y = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= (u32)o)
                incl += y;
        }
        if (lane == 31)
            s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0)
        {
            u64 w = s_warp[lane], wi = w;
            for (int o = 1; o < 32; o <<= 1)
            {
                const u64 y = __shfl_up_sync(0xFFFFFFFFu, wi, o);
                if (lane >= (u32)o)
                    wi += y;
            }
            s_warp[lane] = wi - w; // exclusive over warps
        }
        __syncthreads();
        const u64 carry = s_carry;
        if (i < nt)
            tile_sum[i] = carry + s_warp[warp] + incl - x;
        __syncthreads();
        if (threadIdx.x == 1023)
            s_carry = carry + s_warp[warp] + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0)
        tile_sum[nt] = s_carry;
}

// D4 (batch decode): the documents of a batch, for decode_expand_kernel<true>.  Entry i of tok_off (i <= n_docs, the
// last one being the batch's end) starts at id tok_off[i] - base; the ones that start inside tile t are
// tile_doc[t] .. tile_doc[t+1]-1, and the last tile also takes those that start at the end of the batch.
struct DecodeDocs
{
    const u64 *tok_off; // [n_docs + 1]
    u64 base;           // tok_off[0]
    u32 *tile_doc;       // [tiles + 1], written by decode_batch_tiles_kernel
    u64 *byte_off;       // [n_docs + 1] out
};

// D4 helper: tile_doc[t] = first entry of tok_off that starts at or after tile t (one binary search per tile);
// tile_doc[nt] = n_docs + 1.
__global__ void __launch_bounds__(256) decode_batch_tiles_kernel(const u64 *__restrict__ tok_off, u32 n_ends, u64 base,
                                                                 u64 nt, u32 *__restrict__ tile_doc)
{
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t > nt)
        return;
    u32 lo = t < nt ? 0 : n_ends, hi = n_ends;
    if (t < nt)
    {
        const u64 start = base + t * DEC_TILE;
        while (lo < hi)
        {
            const u32 mid = lo + (hi - lo) / 2;
            if (tok_off[mid] < start)
                lo = mid + 1;
            else
                hi = mid;
        }
    }
    tile_doc[t] = lo;
}

// D3: expand the ids of one tile.  Thread t owns DEC_PER_THREAD CONSECUTIVE ids so that its bytes are
// one contiguous run.  The body stays in the kernel (not an inlined helper) so that <false> compiles to the same code
// as before D4 existed.  With DOCS (D4), also the byte offset of every document that starts in the tile: the thread
// that owns its first id knows where that thread's bytes start (s_pos), plus at most DEC_PER_THREAD - 1 lengths.
template <bool DOCS>
__global__ void __launch_bounds__(DEC_THREADS) decode_expand_kernel(const u32 *__restrict__ tok, u64 n, DecodeVocab v,
                                                                    const u64 *__restrict__ tile_off,
                                                                    uint8_t *__restrict__ out, DecodeDocs d)
{
    __shared__ u64 s_warp[DEC_THREADS / 32];
    __shared__ __align__(16) uint8_t s_stage[DEC_STAGE_BYTES + 16];
    const u64 base = (u64)blockIdx.x * DEC_TILE + (u64)threadIdx.x * DEC_PER_THREAD;
    u32 t[DEC_PER_THREAD];
    u64 mine = 0;
#pragma unroll
    for (int k = 0; k < DEC_PER_THREAD; k++)
    {
        t[k] = (base + k < n) ? tok[base + k] : 0xFFFFFFFFu;
        if (t[k] < v.vocab)
            mine += v.len[t[k]];
    }
    // block-wide exclusive scan of `mine`
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u64 incl = mine;
    for (int o = 1; o < 32; o <<= 1)
    {
        const u64 y = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= (u32)o)
            incl += y;
    }
    if (lane == 31)
        s_warp[warp] = incl;
    __syncthreads();
    u64 before = 0;
    for (u32 w = 0; w < warp; w++)
        before += s_warp[w];
    u64 pos = before + incl - mine; // offset inside the tile's output
    const u64 o0 = tile_off[blockIdx.x];
    const u64 tile_bytes = tile_off[blockIdx.x + 1] - o0;
    if constexpr (DOCS)
    {
        __shared__ u64 s_pos[DEC_THREADS];
        s_pos[threadIdx.x] = pos;
        __syncthreads();
        const u64 lo = (u64)blockIdx.x * DEC_TILE;
        const u64 tile_ids = n - lo < (u64)DEC_TILE ? n - lo : (u64)DEC_TILE;
        const u64 end = d.tile_doc[blockIdx.x + 1];
        for (u64 i = d.tile_doc[blockIdx.x] + threadIdx.x; i < end; i += DEC_THREADS)
        {
            const u64 j = d.tok_off[i] - d.base - lo; // first id of document i, inside the tile
            u64 b = tile_bytes;                       // (j == tile_ids: it starts at the end of the batch)
            if (j < tile_ids)
            {
                const u32 th = (u32)(j / DEC_PER_THREAD);
                b = s_pos[th];
                for (u64 k = lo + (u64)th * DEC_PER_THREAD; k < lo + j; k++)
                    b += v.len[tok[k]];
            }
            d.byte_off[i] = o0 + b;
        }
    }
    if (tile_bytes <= DEC_STAGE_BYTES)
    {
        // stage with the same 16-byte phase as the destination, then store whole vectors
        const u32 phase = (u32)((uintptr_t)(out + o0) & 15);
#pragma unroll
        for (int k = 0; k < DEC_PER_THREAD; k++)
            if (t[k] < v.vocab)
            {
                const u32 l = v.len[t[k]];
                const uint8_t *src = v.blob + v.off[t[k]];
                for (u32 j = 0; j < l; j++)
                    s_stage[phase + pos + j] = src[j];
                pos += l;
            }
        __syncthreads();
        const u32 total = phase + (u32)tile_bytes;
        uint8_t *dst = out + o0 - phase; // 16-byte aligned
        for (u32 q = threadIdx.x * 16; q < total; q += DEC_THREADS * 16)
        {
            if (q >= phase && q + 16 <= total)
                *reinterpret_cast<uint4 *>(dst + q) = *reinterpret_cast<const uint4 *>(s_stage + q);
            else
                for (u32 j = (q < phase ? phase : q); j < q + 16 && j < total; j++)
                    dst[j] = s_stage[j];
        }
    }
    else
    {
        // long expansions (pathological vocabularies): straight to global memory
#pragma unroll
        for (int k = 0; k < DEC_PER_THREAD; k++)
            if (t[k] < v.vocab)
            {
                const u32 l = v.len[t[k]];
                const uint8_t *src = v.blob + v.off[t[k]];
                for (u32 j = 0; j < l; j++)
                    out[o0 + pos + j] = src[j];
                pos += l;
            }
    }
}

// round-trip check without leaving the device: *diff = number of bytes that differ (both buffers come
// from cudaMalloc, so 8-byte words are aligned)
__global__ void decode_compare_kernel(const uint8_t *__restrict__ x, const uint8_t *__restrict__ y, u64 n, u64 *diff)
{
    u64 bad = 0;
    const u64 words = n / 8;
    const u64 *xw = reinterpret_cast<const u64 *>(x), *yw = reinterpret_cast<const u64 *>(y);
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < words; i += (u64)gridDim.x * blockDim.x)
    {
        const u64 d = xw[i] ^ yw[i];
        if (d)
            for (int k = 0; k < 8; k++)
                bad += ((d >> (8 * k)) & 0xFF) != 0;
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 7))
        bad += x[words * 8 + threadIdx.x] != y[words * 8 + threadIdx.x];
    for (int o = 16; o > 0; o >>= 1)
        bad += __shfl_xor_sync(0xFFFFFFFFu, bad, o);
    if ((threadIdx.x & 31) == 0 && bad)
        atomicAdd((unsigned long long *)diff, (unsigned long long)bad);
}
} // namespace bpe
