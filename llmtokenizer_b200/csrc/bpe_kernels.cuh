// Device side of the B200 BPE merge-loop engine (sm_100a).
//
// Reference path being replaced (file:line relative to the reference tree):
//   widen            bpe/src/bpe.c:580-584
//   pair count       bpe/src/bpe.c:428-527 (get_freq) + hash_table/src/hash_table.c:109-193 (merge)
//   argmax           bpe/src/bpe.c:705-750 + dyn_arr/src/dyn_arr.c:136-181 (first maximum wins)
//   rewrite          bpe/src/bpe.c:760-779
//
// Everything here is integer work bounded by HBM bandwidth; nothing is a dense contraction, so
// tensor cores / TMEM are deliberately unused (see DESIGN.md).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace bpe
{

typedef unsigned long long u64;
typedef long long i64;
typedef uint32_t u32;

constexpr u32 SENT = 0xFFFFFFFFu; // "no token": stream start / end inside halo windows
constexpr u64 EMPTY_KEY = ~0ull;
constexpr u64 NO_SLOT = ~0ull;

constexpr int MAX_RANKS = 8;
#ifndef BPE_BATCH_MAX
#define BPE_BATCH_MAX 12
#endif
constexpr int BATCH_MAX = BPE_BATCH_MAX; // merges per pass (at most 15: a nibble holds 1 + the pair index)
// batched passes look tokens up in a byte table indexed by (token mod CLS_SIZE): the tokens of a batch must
// differ mod CLS_SIZE (a stronger form of "pairwise different")
constexpr u32 CLS_SIZE = 8192, CLS_MASK = CLS_SIZE - 1;
__host__ __device__ inline bool tok_alias(u32 x, u32 y) { return ((x ^ y) & CLS_MASK) == 0; }
constexpr int REC_INTS = 8;                    // one edge record
constexpr int HDR_INTS = MAX_RANKS * REC_INTS; // edge records sit in front of the delta vectors

constexpr u64 STATIC_LIMIT = 65536ull * 16ull; // bpe.c:423,449: below this the reference slices statically
constexpr int REF_THREADS = 16;                // bpe.c:409

enum : u32
{
    STOP_RUN = 0,
    STOP_DONE = 1,
    STOP_PAUSE = 2,
    STOP_ERROR = 3
};
enum : u32
{
    PAUSE_TIE = 1,    // >= 2 maximal pairs share the winning bucket: chain order decides
    PAUSE_EDGE = 2,   // D sits exactly on a doubling threshold of the merged table
    PAUSE_STATIC = 4, // stream fell below 1,048,576 tokens: reference switches to static slicing
    PAUSE_REBUILD = 16 // the best candidate fell below the list's threshold: the list must be rebuilt
};
enum : u32
{
    LAYOUT_DENSE = 0,
    LAYOUT_RANGED = 1,
    LAYOUT_SPARSE = 2 // one GPU, late phase: tokens at their byte offsets, never compacted (bpe_sparse.cuh)
};
constexpr u64 SPARSE_PASS_MARK = 1ull << 63; // n_hist[k] of a merge whose pass ran on the SPARSE layout
constexpr int RANGE_MAX = 320;  // ranges per shard (= CTAs of the streaming kernel)
constexpr int EDGE_WORDS = 8;   // per range: [0..2] first three tokens, [3] second to last, [4] last (SENT where absent)
enum : u32
{
    ERR_TABLE_FULL = 1,
    ERR_MISSING_KEY = 2,
    ERR_NEGATIVE = 4,
    ERR_PROBE = 8,
    ERR_XCHG_OVERFLOW = 16, // a rank's list of touched counters outgrew its slot in the peers' inboxes
    ERR_XCHG_TIMEOUT = 32   // a peer's flag did not arrive (a rank died or fell out of step)
};

// Multi-GPU exchange over NVLink peer memory (DESIGN.md, row (e)).  Every rank owns one INBOX buffer that all
// peers can write: after a pass each rank pushes the pair-count deltas its shard produced - as a compact list
// of (counter index, value) entries, a few thousand whatever the vocabulary size - and its pair-independent edge
// record into its slot of every peer's inbox, then raises its flag there.  Every rank folds all P lists into
// its replica of the pair table (integer adds commute, so all replicas end up identical); nothing is reduced
// in between and no collective is launched.  Two parities: a rank can be at most one pass ahead of a peer.
//   inbox layout (u32 words): flags[MAX_RANKS] | counts[2][MAX_RANKS] | recs[2][MAX_RANKS][REC_INTS] | pad to
//   XCHG_HDR_WORDS | entries[2][MAX_RANKS][xcap] (u64: index | value << 32)
constexpr u32 XCHG_FLAGS = 0, XCHG_COUNTS = 64, XCHG_RECS = 128, XCHG_HDR_WORDS = 256;
struct Xchg
{
    u32 *local;             // my inbox
    u32 *peer[MAX_RANKS];   // every rank's inbox as mapped into my address space (peer[rank] == local)
    u64 xcap;               // entries per (parity, sender) slot
};
__host__ __device__ inline size_t xchg_bytes(u64 xcap) { return (size_t)XCHG_HDR_WORDS * 4 + (size_t)2 * MAX_RANKS * xcap * 8; }
__device__ __forceinline__ u64 *xchg_entries(u32 *inbox, u64 xcap, u32 par, u32 sender)
{
    return reinterpret_cast<u64 *>(inbox + XCHG_HDR_WORDS) + ((u64)par * MAX_RANKS + sender) * xcap;
}
__device__ __forceinline__ u32 *xchg_recs(u32 *inbox, u32 par) { return inbox + XCHG_RECS + par * MAX_RANKS * REC_INTS; }

// Device-resident control block.  Everything a merge step needs lives here, so a step is a fixed
// sequence of launches with no host round trip.
struct DevState
{
    // token stream, ping-pong (pointers are 16 B aligned; 4 readable slots in front of each)
    u32 *tok[2];
    u32 cur;
    u32 epoch;  // bumped per merge; stamps tile descriptors so they never need clearing
    u64 n;      // tokens in tok[cur] (this rank's shard)
    u64 n_next; // written by the replace kernel
    u64 n_global;
    // selected merge(s): a pass may carry a BATCH of nb merges (a_i, b_i) -> z + i whose 2*nb tokens are
    // all different and which are provably the next nb merges of the sequential algorithm (DESIGN.md)
    u32 a, b, z, freq;
    u32 nb, batch_max;
    u32 batch_min_z, pad_bz;  // no batching below this id (test / tuning knob)
    u32 hist_max, hist_words; // ids below hist_max run with a shared-memory delta histogram of hist_words counters
    u32 ba[BATCH_MAX], bb[BATCH_MAX];
    u64 batch_merges, batch_passes; // statistics: merges that rode along in a batch / passes with nb > 1
    u32 skip; // encode: this rank's pair does not occur anywhere -> no pass
    // loop control
    u32 stop, pause, err, static_mode;
    u64 merges_done, max_merges;
    // Stream layout.  DENSE: tok[cur][0..n).  RANGED: the shard is cut into nr ranges that are compacted
    // independently (one CTA each, no prefix scan across CTAs): range c lives at tok[buf][c*rcap ..
    // c*rcap + rcnt[buf][c]); redge[buf][8c..] holds its first three and last two tokens.
    u32 layout, layout_next;
    u32 want_ranged, pad_wr; // the host runs this run's passes above the static limit with replace_stream_kernel
    u32 nr, rmax;
    u64 rcap;
    u32 *rcnt[2];
    u32 *redge[2];
    u32 rp_done, pad_rp;
    u32 rpar[RANGE_MAX];  // a == b passes: per range, epoch << 2 | whole range is one run << 1 | parity of its trailing run
    u32 *tok_real[2];     // the two allocations; tok[] aliases one of them while RANGED (tok[0] == tok[1])
    u64 ext_why[8];       // debug statistics: why batch extensions ended (see apply_select_kernel)
    u64 probe_key, probe_slot; // last pair of the stream and its table slot, looked up while the deltas are applied
    u64 dbg[8]; // phase timers of the fused apply+select kernel (ns, summed; BPE_CUDA_DEBUG prints them)
    // pair table: open addressing, key = a | b<<32, meta = murmur3 | count<<32
    u64 *tkey;
    u64 *tmeta;
    u64 tcap;
    i64 distinct; // D: keys with count > 0
    u64 occupied; // claimed slots (dead keys included)
    // argmax candidates: every table slot whose count is >= cand_T is in cand[] (cflag = membership
    // bits), so the maximum over cand[] is the maximum over the table.  cand_T == 0: no list, the
    // selection scans the whole table.
    u32 *cand;
    u32 *cflag;
    u32 ncand, cand_cap, cand_T, cand_overflow;
    u32 cand_big_ok, pad_cb; // the host found no threshold that keeps the list within CAND_FIT entries: do not ask again
    u32 pending, pad_pend; // a merge is committed and its pass / delta application is still to come
    // scheduling counters
    u32 ticket, sel_done;
    // selection result (kept for the resolver)
    u64 sel_key, sel_slot;
    u32 sel_mult, sel_pad;
    // statistics
    u64 same_bucket_ties, threshold_edges;
    // shard edges (single GPU: SENT / 0)
    u32 halo_before[2], halo_after[3], carry_in;
    u32 rank, world;
    // peer-memory exchange (world > 1): sequence number of the last exchange this rank completed, scratch counters
    Xchg x;
    u32 xseq, x_count, x_done, x_bar;
    u64 x_timeout_ns; // how long a rank waits for a peer's flag before it stops the run with an error
    // the reference's 16 worker tables keep their grown bucket count across iterations
    u64 bt[REF_THREADS];
    // logs
    u32 *merges; // pairs, 2 u32 each
    u64 *n_hist; // global token count before merge k
    // encode
    const u32 *enc_merges;
    u64 enc_total;
    u64 ranks_applied;
    // LAYOUT_SPARSE (bpe_sparse.cuh): tok[0] == tok[1] holds the id that starts at each byte offset (SENT at every
    // other byte), start_of[e] the start of the token whose last byte is e; slen = byte length per id
    u32 *start_of;
    u32 *slen;
    u64 n0;      // byte positions of the sparse stream
    u32 zsw;     // ids below zsw existed when the frozen index was built
    const u64 *ikey; // frozen index: copy of the table keys at the switch, per slot its positions ipos[ioff[s] ..]
    u64 icap;
    const u32 *ioff;
    u32 *ipos;
    u32 *cl_off, *cl_cnt, *pool; // creation lists: positions where id z was written, pool[cl_off[z] ..][cl_cnt[z]]
    u64 pool_top;
    // replacements of the current pass, merge by merge: merge i's sp_cnt[i] positions at pass_buf[sp_ent[i] ..], where
    // sp_ent[i] is the number of list entries of the merges before it (a merge replaces at most one pair instance per
    // entry, and the lists of one pass are disjoint: the frozen lists of different pairs and the creation lists of
    // different ids; so 2 n + 2 words hold any pass)
    u32 *pass_buf;
    u32 sp_cnt[BATCH_MAX], sp_ent[BATCH_MAX];
    u64 sparse_passes, sparse_bytes;
    u64 sparse_entries; // list entries the sparse scans checked
};

// ---------------------------------------------------------------------------------------------
// hash_table.c:8-53 on the 8-byte key {u32 a; u32 b}
// Programmatic dependent launch: a kernel launched with the "programmatic stream serialization" attribute may be
// scheduled while its predecessor is still running; pdl_wait() blocks until the predecessor has completed and its
// writes are visible (a no-op for a normal launch), pdl_launch_dependents() lets the successor's CTAs be scheduled.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

__device__ __forceinline__ u64 gtime()
{
    u64 t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
__host__ __device__ __forceinline__ u32 rotl32(u32 x, int r) { return (x << r) | (x >> (32 - r)); }

// system-scope release / acquire on a flag another GPU reads / writes through NVLink peer memory
__device__ __forceinline__ void st_release_sys(u32 *p, u32 v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ u32 ld_acquire_sys(const u32 *p)
{
    u32 v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ u64 ld_relaxed_sys_u64(const u64 *p)
{
    u64 v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ u32 ld_relaxed_sys_u32(const u32 *p)
{
    u32 v;
    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__host__ __device__ __forceinline__ u32 murmur3_pair(u32 a, u32 b)
{
    u32 h = 0x9747b28cu;
    u32 k = a;
    k *= 0xcc9e2d51u;
    k = rotl32(k, 15);
    k *= 0x1b873593u;
    h ^= k;
    h = rotl32(h, 13);
    h = h * 5u + 0xe6546b64u;
    k = b;
    k *= 0xcc9e2d51u;
    k = rotl32(k, 15);
    k *= 0x1b873593u;
    h ^= k;
    h = rotl32(h, 13);
    h = h * 5u + 0xe6546b64u;
    h ^= 8u;
    h ^= h >> 16;
    h *= 0x85ebca6bu;
    h ^= h >> 13;
    h *= 0xc2b2ae35u;
    h ^= h >> 16;
    return h;
}

// hash_table.c:6,248: a table doubles at the top of an insert call once nodes >= 0.3 * buckets
__host__ __device__ __forceinline__ bool resize_due(u64 nodes, u64 buckets)
{
    return (double)nodes >= 0.3 * (double)buckets;
}
__host__ __device__ inline u64 resize_threshold_exact(u64 buckets)
{
    u64 t = (u64)(0.3 * (double)buckets);
    while (!resize_due(t, buckets))
        t++;
    while (t > 0 && resize_due(t - 1, buckets))
        t--;
    return t;
}
// Every table of the reference has a power-of-two bucket count (256 * 2^j workers, 65,536 * 2^k merged), and the
// selection asks for thresholds on its critical path (bucket order B(D), the exact-threshold edge, batch margins):
// on the device they come from a table filled once by the host with the function above.
constexpr int THR_LOG2_MIN = 8, THR_ENTRIES = 48;
__constant__ u64 c_resize_thr[THR_ENTRIES];
__host__ __device__ inline u64 resize_threshold(u64 buckets)
{
#ifdef __CUDA_ARCH__
    const int lg = 63 - __clzll((long long)buckets);
    if ((buckets & (buckets - 1)) == 0 && lg >= THR_LOG2_MIN && lg < THR_LOG2_MIN + THR_ENTRIES)
        return c_resize_thr[lg - THR_LOG2_MIN];
#endif
    return resize_threshold_exact(buckets);
}
// bucket count of the merged table (fresh 65,536 buckets every iteration, bpe.c:611,684) once D
// keys went in, away from the exact-threshold edge (handled by the resolver)
__host__ __device__ inline u64 merged_buckets(u64 distinct)
{
    u64 b = 65536;
    while (distinct > resize_threshold(b))
        b *= 2;
    return b;
}
__host__ __device__ inline bool on_threshold(u64 distinct)
{
    for (u64 b = 65536;; b *= 2)
    {
        const u64 t = resize_threshold(b);
        if (t == distinct)
            return true;
        if (t > distinct)
            return false;
    }
}
// growth of a table that starts an iteration with b0 buckets, sees d distinct keys, and whose
// very last insert call did / did not create the d-th key
__host__ __device__ inline u64 grown_buckets(u64 b0, u64 d, bool last_call_is_new)
{
    u64 b = b0;
    for (;;)
    {
        const u64 th = resize_threshold(b);
        if (d > th || (d == th && !last_call_is_new))
            b *= 2;
        else
            return b;
    }
}
__host__ __device__ inline u32 doublings_after(u64 b0, u64 bfinal, u64 r)
{
    u32 c = 0;
    for (u64 b = b0; b < bfinal; b *= 2)
        if (resize_threshold(b) >= r)
            c++;
    return c;
}
// position inside one chain as a sortable number (each doubling reverses every chain)
__host__ __device__ __forceinline__ u64 chain_slot(u32 doublings_to_come, u64 r)
{
    return (doublings_to_come & 1u) ? ((1ull << 40) | r) : ((1ull << 40) - 1 - r);
}

// ---------------------------------------------------------------------------------------------
// pair table
__device__ __forceinline__ u64 probe_start(u32 h, u64 cap) { return (((u64)h * 0x9E3779B97F4A7C15ull) >> 20) & (cap - 1); }
__device__ __forceinline__ u32 *cnt_ptr(u64 *meta, u64 slot) { return reinterpret_cast<u32 *>(meta + slot) + 1; }
__device__ __forceinline__ u32 *hsh_ptr(u64 *meta, u64 slot) { return reinterpret_cast<u32 *>(meta + slot); }

// add to a global delta counter (fire and forget: compiles to RED)
__device__ __forceinline__ void delta_add(DevState *, int32_t *gdelta, u64 idx, int32_t v) { atomicAdd(&gdelta[idx], v); }

__device__ __forceinline__ u64 table_find(const u64 *tkey, u64 cap, u64 key, u32 h)
{
    u64 s = probe_start(h, cap);
    for (u64 i = 0; i < cap; i++)
    {
        const u64 k = tkey[s];
        if (k == key)
            return s;
        if (k == EMPTY_KEY)
            return NO_SLOT;
        s = (s + 1) & (cap - 1);
    }
    return NO_SLOT;
}

__device__ __forceinline__ u64 table_insert(DevState *st, u64 key, u32 h)
{
    u64 *tkey = st->tkey;
    const u64 cap = st->tcap;
    u64 s = probe_start(h, cap);
    for (u64 i = 0; i < cap; i++)
    {
        u64 k = tkey[s];
        if (k == EMPTY_KEY)
        {
            k = atomicCAS(tkey + s, EMPTY_KEY, key);
            if (k == EMPTY_KEY)
            {
                *hsh_ptr(st->tmeta, s) = h;
                atomicAdd(&st->occupied, 1ull);
                return s;
            }
        }
        if (k == key)
            return s;
        s = (s + 1) & (cap - 1);
    }
    return NO_SLOT;
}

// ---------------------------------------------------------------------------------------------
// Stream views that work for both layouts (ends of the shard only; the bulk is never touched here).
struct StreamEnds
{
    u32 first[3]; // first three tokens (SENT where the shard is shorter)
    u32 last2[2]; // second to last, last
};
__device__ inline void stream_ends(const DevState *st, u32 buf, u32 layout, u64 n, StreamEnds &e)
{
    for (int k = 0; k < 3; k++)
        e.first[k] = SENT;
    e.last2[0] = e.last2[1] = SENT;
    const u32 *t = st->tok[buf];
    if (layout == LAYOUT_SPARSE)
    {
        u64 p = 0;
        for (int k = 0; k < 3 && p < st->n0; k++)
        {
            e.first[k] = t[p];
            p += st->slen[t[p]];
        }
        if (n >= 1)
        {
            const u32 lp = st->start_of[st->n0 - 1];
            e.last2[1] = t[lp];
            if (n >= 2)
                e.last2[0] = t[st->start_of[lp - 1]];
        }
        return;
    }
    if (layout == LAYOUT_DENSE)
    {
        for (u64 k = 0; k < 3 && k < n; k++)
            e.first[k] = t[k];
        if (n >= 1)
            e.last2[1] = t[n - 1];
        if (n >= 2)
            e.last2[0] = t[n - 2];
        return;
    }
    const u32 *cnt = st->rcnt[buf], *ed = st->redge[buf];
    int got = 0;
    for (u32 q = 0; q < st->nr && got < 3; q++)
        for (u32 k = 0; k < 3 && k < cnt[q] && got < 3; k++)
            e.first[got++] = ed[q * EDGE_WORDS + k];
    got = 0;
    for (int q = (int)st->nr - 1; q >= 0 && got < 2; q--)
    {
        if (cnt[q] >= 1 && got < 2)
            e.last2[1 - got++] = ed[q * EDGE_WORDS + 4];
        if (cnt[q] >= 2 && got < 2)
            e.last2[1 - got++] = ed[q * EDGE_WORDS + 3];
    }
}

// ---------------------------------------------------------------------------------------------
// K0 + K1: widen bytes to u32 tokens (bpe.c:580-584) and histogram all adjacent byte pairs into
// a dense 256x256 table (every overlapping occurrence counts, bpe.c:460-471).  While all ids are
// < 256 the dense table replaces the hash table.  16 bytes per thread: one 128-bit load, four
// 128-bit stores.  The launch covers the byte positions [lo, hi) (lo a multiple of 16) and counts the pair
// that ENDS on each of them, so the corpus can be widened and counted chunk by chunk while later chunks are
// still on their way from the host (file ingest): every pair is counted by exactly one launch, and only bytes in
// front of `hi` are looked at.
__global__ void __launch_bounds__(256) widen_count_kernel(const uint8_t *__restrict__ bytes, u64 lo, u64 hi, u32 *__restrict__ tok,
                                                          u32 *__restrict__ dense)
{
    extern __shared__ __align__(16) u32 s_lo[]; // 128*128 privatised counts for pairs of 7-bit bytes (ASCII text)
    for (int i = threadIdx.x; i < 128 * 128; i += blockDim.x)
        s_lo[i] = 0;
    __syncthreads();
    const u64 v0 = lo / 16, nvec = (hi + 15) / 16;
    for (u64 v = v0 + (u64)blockIdx.x * blockDim.x + threadIdx.x; v < nvec; v += (u64)gridDim.x * blockDim.x)
    {
        const u64 base = v * 16;
        const uint4 q = __ldg(reinterpret_cast<const uint4 *>(bytes) + v);
        u32 c[17]; // c[k + 1] = byte at base + k, c[0] = the byte in front
        const u32 qq[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int k = 0; k < 16; k++)
            c[k + 1] = (qq[k >> 2] >> ((k & 3) * 8)) & 0xFFu;
        c[0] = base ? (u32)bytes[base - 1] : 0u;
        uint4 *o = reinterpret_cast<uint4 *>(tok + base);
        o[0] = make_uint4(c[1], c[2], c[3], c[4]);
        o[1] = make_uint4(c[5], c[6], c[7], c[8]);
        o[2] = make_uint4(c[9], c[10], c[11], c[12]);
        o[3] = make_uint4(c[13], c[14], c[15], c[16]);
#pragma unroll
        for (int k = 0; k < 16; k++)
        {
            if (base + k < hi && base + k >= 1)
            {
                const u32 x = c[k], y = c[k + 1];
                if ((x | y) < 128u)
                    atomicAdd(&s_lo[x * 128 + y], 1u);
                else
                    atomicAdd(&dense[x * 256 + y], 1u);
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 128 * 128; i += blockDim.x)
    {
        const u32 v = s_lo[i];
        if (v)
            atomicAdd(&dense[(i >> 7) * 256 + (i & 127)], v);
    }
}

// the pair that straddles two shards is counted by the left shard (its first token is the left
// shard's last): one thread, after the edge records are known
__global__ void boundary_pair_kernel(DevState *st, u32 *dense)
{
    if (st->n == 0 || st->halo_after[0] == SENT)
        return;
    const u32 x = st->tok[st->cur][st->n - 1], y = st->halo_after[0];
    atomicAdd(&dense[x * 256 + y], 1u);
}

__global__ void table_from_dense_kernel(DevState *st, const u32 *__restrict__ dense)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 65536)
        return;
    const u32 c = dense[i];
    if (!c)
        return;
    const u32 a = i >> 8, b = i & 255u;
    const u64 s = table_insert(st, (u64)a | ((u64)b << 32), murmur3_pair(a, b));
    if (s == NO_SLOT)
    {
        atomicOr(&st->err, ERR_TABLE_FULL);
        return;
    }
    atomicAdd(cnt_ptr(st->tmeta, s), c);
    atomicAdd(reinterpret_cast<u64 *>(&st->distinct), 1ull);
}

// ---------------------------------------------------------------------------------------------
// table maintenance: copy the live entries into a fresh (larger or purged) table
__global__ void rehash_kernel(const u64 *__restrict__ okey, const u64 *__restrict__ ometa, u64 ocap, u64 *nkey, u64 *nmeta,
                              u64 ncap, u32 *err)
{
    for (u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x; s < ocap; s += (u64)gridDim.x * blockDim.x)
    {
        const u64 k = okey[s];
        const u64 m = ometa[s];
        if (k == EMPTY_KEY || (m >> 32) == 0)
            continue;
        u64 p = probe_start((u32)m, ncap);
        bool placed = false;
        for (u64 i = 0; i < ncap; i++)
        {
            if (atomicCAS(nkey + p, EMPTY_KEY, k) == EMPTY_KEY)
            {
                nmeta[p] = m;
                placed = true;
                break;
            }
            p = (p + 1) & (ncap - 1);
        }
        if (!placed)
            atomicOr(err, ERR_TABLE_FULL);
    }
}

__global__ void table_swap_kernel(DevState *st, u64 *nkey, u64 *nmeta, u64 ncap, u32 *cflag)
{
    st->tkey = nkey;
    st->tmeta = nmeta;
    st->tcap = ncap;
    st->cflag = cflag;
    st->occupied = (u64)st->distinct;
    st->ncand = 0;
    st->cand_T = 0; // slots moved: the host rebuilds the candidate list
}

// ---------------------------------------------------------------------------------------------
// Multi-GPU shard edges.  After every pass each rank publishes a pair-independent record of its
// shard (length, first three tokens, last two tokens, parity of its trailing run of equal tokens
// and whether the whole shard is that one run) in its slot of the buffer that the per-merge
// all-reduce sums; disjoint slots make the sum an all-gather, so there is ONE collective per merge.
//   rec[0..1] = length (lo, hi)   rec[2..4] = first tokens   rec[5..6] = last two tokens
//   rec[7]    = trailing-run parity | uniform<<1
// (32 lanes; the record is complete in lane 0)
__device__ inline void edge_record_compute(const DevState *st, bool nxt, u32 rec[REC_INTS])
{
    const u32 buf = nxt ? (st->cur ^ 1u) : st->cur;
    const u32 layout = nxt ? st->layout_next : st->layout;
    const u64 len = nxt ? st->n_next : st->n;
    const u32 *s = st->tok[buf];
    const int lane = threadIdx.x & 31;
    StreamEnds e;
    stream_ends(st, buf, layout, len, e);
    // trailing run of the last token, 32 tokens per step, range by range from the back
    u64 run = 0;
    bool uniform = false;
    if (len)
    {
        const u32 last = e.last2[1];
        const int nseg = (layout == LAYOUT_DENSE) ? 1 : (int)st->nr;
        bool open = true; // the run may still extend further to the left
        for (int q = nseg - 1; q >= 0 && open; q--)
        {
            const u32 *p = (layout == LAYOUT_DENSE) ? s : s + (u64)q * st->rcap;
            const u64 cnt = (layout == LAYOUT_DENSE) ? len : (u64)st->rcnt[buf][q];
            u64 pos = cnt; // tokens [pos, cnt) of this piece are known to equal `last`
            while (pos > 0)
            {
                const i64 i = (i64)pos - 1 - lane;
                const bool eq = (i >= 0) && (p[i] == last);
                const u32 m = __ballot_sync(0xFFFFFFFFu, eq);
                const int c = (m == 0xFFFFFFFFu) ? 32 : (__ffs(~m) - 1);
                run += (u64)c;
                pos -= (u64)c;
                if (c < 32)
                    break;
            }
            open = (pos == 0); // the whole piece is part of the run: it may continue in the piece in front
        }
        uniform = (run == len);
    }
    rec[0] = (u32)len;
    rec[1] = (u32)(len >> 32);
    for (int k = 0; k < 3; k++)
        rec[2 + k] = e.first[k];
    rec[5] = e.last2[0];
    rec[6] = e.last2[1];
    rec[7] = (u32)(run & 1ull) | ((u32)uniform << 1);
}

// ---- peer-memory exchange primitives (see struct Xchg) ----------------------------------------------
// the records every rank pushed in exchange `seq` (the latest one this rank completed: st->xseq)
__device__ __forceinline__ const u32 *cur_recs(const DevState *st)
{
    return st->world > 1 ? xchg_recs(st->x.local, st->xseq & 1u) : nullptr;
}
// lane 0 of the calling warp: publish my record for exchange `seq` in every inbox (mine included)
__device__ inline void xchg_push_record(DevState *st, u32 seq, const u32 rec[REC_INTS])
{
    for (u32 p = 0; p < st->world; p++)
    {
        u32 *dst = xchg_recs(st->x.peer[p], seq & 1u) + st->rank * REC_INTS;
        for (int k = 0; k < REC_INTS; k++)
            dst[k] = rec[k];
    }
}
// one thread, after every write of this rank for exchange `seq` is fenced: tell the peers how many entries my list
// holds and raise my flag in their inboxes
__device__ inline void xchg_signal(DevState *st, u32 seq, u32 count)
{
    for (u32 p = 0; p < st->world; p++)
        if (p != st->rank)
            st->x.peer[p][XCHG_COUNTS + (seq & 1u) * MAX_RANKS + st->rank] = count;
    __threadfence_system();
    for (u32 p = 0; p < st->world; p++) // (my own inbox too: this rank's blocks wait for "my list is complete" there)
        st_release_sys(st->x.peer[p] + XCHG_FLAGS + st->rank, seq);
}
// one thread: wait until `sender` has raised its flag for exchange `seq` in my inbox.  Peers run the same launch
// sequence on their own GPUs; a flag that does not arrive within x_timeout_ns (20 s) means a rank died or fell out of step:
// the run is stopped with an error instead of spinning for ever.
__device__ inline bool xchg_wait(DevState *st, u32 sender, u32 seq, u64 timeout_ns = 0)
{
    if (!timeout_ns)
        timeout_ns = st->x_timeout_ns;
    const u32 *f = st->x.local + XCHG_FLAGS + sender;
    const u64 t0 = gtime();
    u32 spins = 0;
    while ((int)(ld_acquire_sys(f) - seq) < 0)
    {
        if ((++spins & 1023u) == 0 && gtime() - t0 > timeout_ns)
        {
            atomicOr(&st->err, ERR_XCHG_TIMEOUT);
            st->stop = STOP_ERROR;
            return false;
        }
    }
    return true;
}

// Exchange of the edge records alone (start of a run: nothing has been merged yet, or after the host changed the
// stream).  One warp.  Afterwards every rank knows every shard's length and edge tokens.
__global__ void edge_exchange_kernel(DevState *st, int use_next)
{
    if (st->world <= 1 || (st->stop != STOP_RUN && use_next))
        return;
    u32 rec[REC_INTS];
    edge_record_compute(st, use_next && !st->skip, rec);
    const u32 seq = st->xseq + 1u;
    if (threadIdx.x == 0)
    {
        xchg_push_record(st, seq, rec);
        __threadfence_system();
        xchg_signal(st, seq, 0u);
        bool ok = true;
        // (the ranks of a job start their runs when their callers get there - corpus generation, file reads - not in
        // lockstep: the first exchange of a run waits 30 times longer than the per-pass ones)
        for (u32 p = 0; p < st->world && ok; p++)
            if (p != st->rank)
                ok = xchg_wait(st, p, seq, 30 * st->x_timeout_ns);
        st->xseq = seq;
    }
}

// derive this rank's halos from all records (device function, used once a pair is chosen)
__device__ inline void resolve_edges(DevState *st, const u32 *rec_all, u32 a, bool same)
{
    const int P = (int)st->world, me = (int)st->rank;
    u64 total = 0;
    for (int r = 0; r < P; r++)
        total += (u64)rec_all[r * REC_INTS] | ((u64)rec_all[r * REC_INTS + 1] << 32);
    st->n_global = total;
    u32 before[2] = {SENT, SENT};
    int got = 0;
    for (int q = me - 1; q >= 0 && got < 2; q--)
    {
        const u32 *rc = rec_all + q * REC_INTS;
        const u64 len = (u64)rc[0] | ((u64)rc[1] << 32);
        if (len >= 1 && got < 2)
            before[1 - got++] = rc[6];
        if (len >= 2 && got < 2)
            before[1 - got++] = rc[5];
    }
    u32 after[3] = {SENT, SENT, SENT};
    got = 0;
    for (int q = me + 1; q < P && got < 3; q++)
    {
        const u32 *rc = rec_all + q * REC_INTS;
        const u64 len = (u64)rc[0] | ((u64)rc[1] << 32);
        for (int k = 0; k < 3 && got < 3; k++)
            if ((u64)k < len)
                after[got++] = rc[2 + k];
    }
    u32 carry = 0;
    if (same)
        for (int q = me - 1; q >= 0; q--)
        {
            const u32 *rc = rec_all + q * REC_INTS;
            const u64 len = (u64)rc[0] | ((u64)rc[1] << 32);
            if (!len)
                continue;
            if (rc[6] != a)
                break;
            carry ^= (rc[7] & 1u);
            if (!(rc[7] & 2u))
                break;
        }
    st->halo_before[0] = before[0];
    st->halo_before[1] = before[1];
    st->halo_after[0] = after[0];
    st->halo_after[1] = after[1];
    st->halo_after[2] = after[2];
    st->carry_in = carry;
}

// ---------------------------------------------------------------------------------------------
// K2: most frequent pair with the reference's order (bpe.c:705-750).  The merged table is walked
// bucket 0.., so among equal frequencies the smallest `murmur3 % B(D)` wins: one packed 64-bit key
// (count << 32 | ~bucket) turns that into a plain max.  Warp shuffles, then a block tree, then the
// last block folds the per-block partials.  The multiplicity of the maximal key is carried along:
// > 1 means chain order inside one bucket decides (resolver).
struct SelPart
{
    u64 key;
    u64 slot;
    u32 mult;
    u32 pad;
};

__device__ __forceinline__ void sel_combine(u64 &k, u64 &s, u32 &m, u64 k2, u64 s2, u32 m2)
{
    if (k2 > k)
    {
        k = k2;
        s = s2;
        m = m2;
    }
    else if (k2 == k)
    {
        m += m2;
        s = (s2 < s) ? s2 : s;
    }
}

__device__ __forceinline__ void sel_block_reduce(u64 &k, u64 &s, u32 &m, SelPart *sm)
{
#pragma unroll
    for (int o = 16; o; o >>= 1)
    {
        const u64 k2 = __shfl_xor_sync(0xFFFFFFFFu, k, o);
        const u64 s2 = __shfl_xor_sync(0xFFFFFFFFu, s, o);
        const u32 m2 = __shfl_xor_sync(0xFFFFFFFFu, m, o);
        // xor butterflies visit each lane once, so multiplicities add exactly once
        if (k2 > k)
        {
            k = k2;
            s = s2;
            m = m2;
        }
        else if (k2 == k)
        {
            m += m2;
            s = (s2 < s) ? s2 : s;
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    __syncthreads();
    if (lane == 0)
    {
        sm[warp].key = k;
        sm[warp].slot = s;
        sm[warp].mult = m;
    }
    __syncthreads();
    if (warp == 0)
    {
        k = (lane < nw) ? sm[lane].key : 0ull;
        s = (lane < nw) ? sm[lane].slot : NO_SLOT;
        m = (lane < nw) ? sm[lane].mult : 0u;
#pragma unroll
        for (int o = 16; o; o >>= 1)
        {
            const u64 k2 = __shfl_xor_sync(0xFFFFFFFFu, k, o);
            const u64 s2 = __shfl_xor_sync(0xFFFFFFFFu, s, o);
            const u32 m2 = __shfl_xor_sync(0xFFFFFFFFu, m, o);
            if (k2 > k)
            {
                k = k2;
                s = s2;
                m = m2;
            }
            else if (k2 == k)
            {
                m += m2;
                s = (s2 < s) ? s2 : s;
            }
        }
    }
}

// Above 1,048,576 tokens the canonical schedule gives every chunk to worker 0 (DESIGN.md): its
// table sees all D keys, and its last insert call creates a key iff the stream's last pair occurs
// exactly once.  That keeps the worker's persistent bucket count exact without touching the stream.
// Does the stream's last pair occur exactly once?  (independent of which pair gets merged next, so
// the fused apply+select kernel asks this while the candidates are still being scanned)
__device__ inline u64 last_pair_key(const DevState *st, const u32 *rec_all, u32 buf, u32 layout, u64 n)
{
    u32 x = SENT, y = SENT;
    if (st->world > 1)
    {
        int got = 0;
        u32 last2[2] = {SENT, SENT};
        for (int q = (int)st->world - 1; q >= 0 && got < 2; q--)
        {
            const u32 *rc = rec_all + q * REC_INTS;
            const u64 len = (u64)rc[0] | ((u64)rc[1] << 32);
            if (len >= 1 && got < 2)
                last2[1 - got++] = rc[6];
            if (len >= 2 && got < 2)
                last2[1 - got++] = rc[5];
        }
        x = last2[0];
        y = last2[1];
    }
    else if (n >= 2)
    {
        StreamEnds e;
        stream_ends(st, buf, layout, n, e);
        x = e.last2[0];
        y = e.last2[1];
    }
    if (x == SENT || y == SENT)
        return EMPTY_KEY;
    return (u64)x | ((u64)y << 32);
}
__device__ inline bool census_probe(const DevState *st, const u32 *rec_all, u32 buf, u32 layout, u64 n)
{
    u32 x = SENT, y = SENT;
    if (st->world > 1)
    {
        int got = 0;
        u32 last2[2] = {SENT, SENT};
        for (int q = (int)st->world - 1; q >= 0 && got < 2; q--)
        {
            const u32 *rc = rec_all + q * REC_INTS;
            const u64 len = (u64)rc[0] | ((u64)rc[1] << 32);
            if (len >= 1 && got < 2)
                last2[1 - got++] = rc[6];
            if (len >= 2 && got < 2)
                last2[1 - got++] = rc[5];
        }
        x = last2[0];
        y = last2[1];
    }
    else if (n >= 2)
    {
        StreamEnds e;
        stream_ends(st, buf, layout, n, e);
        x = e.last2[0];
        y = e.last2[1];
    }
    if (x == SENT || y == SENT)
        return false;
    const u64 s = table_find(st->tkey, st->tcap, (u64)x | ((u64)y << 32), murmur3_pair(x, y));
    return (s != NO_SLOT) && (*reinterpret_cast<volatile u32 *>(cnt_ptr(st->tmeta, s)) == 1u);
}

// what the last block of the fused kernel works out next to the candidate scan
struct PreDecide
{
    u32 valid;    // the two fields below are filled in
    u32 last_new; // census_probe()
    u32 edge;     // on_threshold(D)
};

// record the chosen pair and prepare the pass (single thread)
__device__ inline void commit_merge(DevState *st, u32 a, u32 b, u32 freq, const u32 *rec_all, bool encode = false,
                                    const PreDecide *pre = nullptr)
{
    const u64 k = st->merges_done;
    st->a = a;
    st->b = b;
    st->z = (u32)(256 + k);
    st->freq = freq;
    st->skip = 0;
    st->nb = 1;
    st->ba[0] = a;
    st->bb[0] = b;
    st->merges[2 * k] = a;
    st->merges[2 * k + 1] = b;
    if (st->world > 1)
        resolve_edges(st, rec_all, a, a == b);
    else
        st->n_global = st->n;
    if (!encode && st->n_global >= STATIC_LIMIT)
    {
        const bool last_new = (pre && pre->valid) ? (pre->last_new != 0) : census_probe(st, rec_all, st->cur, st->layout, st->n);
        st->bt[0] = grown_buckets(st->bt[0], (u64)st->distinct, last_new);
    }
    st->n_next = 0; // the ranged streaming kernel accumulates its ranges' new lengths here
    st->pending = 1;
    st->n_hist[k] = st->n_global;
    st->merges_done = k + 1;
    st->epoch = st->epoch + 1;
    st->ticket = 0;
}

// one more merge for the pass that is already committed (single thread)
__device__ inline void extend_batch(DevState *st, u32 a, u32 b)
{
    const u64 k = st->merges_done;
    const u32 i = st->nb;
    st->ba[i] = a;
    st->bb[i] = b;
    st->nb = i + 1;
    st->merges[2 * k] = a;
    st->merges[2 * k + 1] = b;
    st->n_hist[k] = ~0ull; // rides along: no pass of its own
    st->merges_done = k + 1;
    st->batch_merges++;
}

constexpr int SEL_THREADS = 512;
// candidates the last block of apply_select_kernel keeps in registers (8 per thread); batches are only formed
// from such a list, so the host aims below it and the device asks for a new threshold when the list outgrows it
constexpr u32 CAND_FIT = SEL_THREADS * 8, CAND_TARGET = 3072;

// What the batch extension needs to know about the merge decide_list() has just committed (shared memory)
struct Committed
{
    u32 ok;             // a merge was committed and the pass may take more merges along
    u32 a, b, freq, z;  // the committed merge
    u32 cand_T, batch_max, hist_max, hist_words;
    u64 merges_done;    // after the commit
    u64 max_merges;
    u64 bt0;            // worker-table buckets after the commit
    u64 n_stream;       // tokens in the (global) stream the committed merge is applied to
    u32 *merges;
    u64 *n_hist;
};

// decide() for the list mode on one GPU (the per-pass critical path): the same decisions, but every
// field is loaded up front in one burst (the loads overlap; in decide()/commit_merge() each load waits for the
// stores in front of it, five serial round trips to L2) and the merge is committed from registers.
__device__ inline void decide_list(DevState *st, u64 k, u64 s, u32 m, const PreDecide *pre, Committed *out, u32 ncand)
{
    const u64 D = (u64)st->distinct, md = st->merges_done, mm = st->max_merges, n_local = st->n, bt0 = st->bt[0];
    const u32 cand_T = st->cand_T, stat = st->static_mode, wr = st->want_ranged, epoch = st->epoch;
    const u32 batch_max = st->batch_max, batch_min_z = st->batch_min_z, hist_max = st->hist_max, hist_words = st->hist_words;
    const u32 big_ok = st->cand_big_ok;
    u32 *merges = st->merges;
    u64 *n_hist = st->n_hist;
    const u64 key = (s != NO_SLOT) ? __ldcg(st->tkey + s) : 0ull;
    out->ok = 0;
    st->sel_key = k;
    st->sel_slot = s;
    st->sel_mult = m;
    st->n_global = n_local;
    const u32 freq = (u32)(k >> 32);
    if (cand_T && D != 0 && freq < cand_T && md < mm)
    {
        st->pause = PAUSE_REBUILD; // see decide()
        st->stop = STOP_PAUSE;
        return;
    }
    if (D == 0 || m == 0 || freq <= 1 || md >= mm) // bpe.c:730, bpe.c:745, cap
    {
        st->stop = STOP_DONE;
        return;
    }
    if (cand_T && ncand > CAND_FIT && !big_ok && batch_max > 1 && wr && !stat)
    {
        // the list has outgrown the registers of this block (no batches, and a gather per entry): the host
        // rebuilds it with a higher threshold (k is the true maximum here, so nothing is lost)
        st->pause = PAUSE_REBUILD;
        st->stop = STOP_PAUSE;
        return;
    }
    if (!stat && n_local < STATIC_LIMIT)
    {
        st->static_mode = 1;
        st->pause = PAUSE_STATIC;
        st->stop = STOP_PAUSE;
        return;
    }
    const bool tie = (m > 1), edge = pre->edge != 0;
    if (tie || edge)
    {
        if (tie)
            st->same_bucket_ties++;
        if (edge)
            st->threshold_edges++;
        st->pause = (tie ? PAUSE_TIE : 0u) | (edge ? PAUSE_EDGE : 0u);
        st->stop = STOP_PAUSE;
        return;
    }
    // commit_merge(), from registers
    const u32 a = (u32)(key & 0xFFFFFFFFull), b = (u32)(key >> 32), z = (u32)(256 + md);
    st->a = a;
    st->b = b;
    st->z = z;
    st->freq = freq;
    st->skip = 0;
    st->nb = 1;
    st->ba[0] = a;
    st->bb[0] = b;
    merges[2 * md] = a;
    merges[2 * md + 1] = b;
    u64 bt_new = bt0;
    if (n_local >= STATIC_LIMIT)
    {
        bt_new = grown_buckets(bt0, D, pre->last_new != 0);
        st->bt[0] = bt_new;
    }
    st->n_next = 0;
    st->pending = 1;
    n_hist[md] = n_local;
    st->merges_done = md + 1;
    st->epoch = epoch + 1;
    st->ticket = 0;
    out->ok = (batch_max > 1 && cand_T && wr && !stat && !tok_alias(a, b) && z >= batch_min_z && z >= hist_max && md + 1 < mm) ? 1u : 0u;
    out->a = a;
    out->b = b;
    out->freq = freq;
    out->z = z;
    out->cand_T = cand_T;
    out->batch_max = batch_max;
    out->hist_max = hist_max;
    out->hist_words = hist_words;
    out->merges_done = md + 1;
    out->max_merges = mm;
    out->bt0 = bt_new;
    out->n_stream = n_local;
    out->merges = merges;
    out->n_hist = n_hist;
}

// The decision once the best packed key (count << 32 | ~bucket), its multiplicity and a slot holding
// it are known: stop / pause / commit (bpe.c:730-758).  One thread.
__device__ inline void decide(DevState *st, u64 k, u64 s, u32 m, const u32 *rec_all, const PreDecide *pre = nullptr)
{
    const u64 D = (u64)st->distinct;
    st->sel_key = k;
    st->sel_slot = s;
    st->sel_mult = m;
    if (st->world > 1)
    {
        u64 total = 0;
        for (u32 r = 0; r < st->world; r++)
            total += (u64)rec_all[r * REC_INTS] | ((u64)rec_all[r * REC_INTS + 1] << 32);
        st->n_global = total;
    }
    else
        st->n_global = st->n;
    const u32 freq = (u32)(k >> 32);
    if (st->cand_T && D != 0 && freq < st->cand_T && st->merges_done < st->max_merges)
    {
        // every count >= cand_T is in the list, and nothing in the list reaches cand_T any more:
        // the true maximum is somewhere below; the host rebuilds the list with a lower threshold
        st->pause = PAUSE_REBUILD;
        st->stop = STOP_PAUSE;
        return;
    }
    if (D == 0 || m == 0 || freq <= 1 || st->merges_done >= st->max_merges) // bpe.c:730, bpe.c:745, cap
    {
        st->stop = STOP_DONE;
        return;
    }
    if (!st->static_mode && st->n_global < STATIC_LIMIT)
    {
        st->static_mode = 1;
        st->pause = PAUSE_STATIC;
        st->stop = STOP_PAUSE;
        return;
    }
    const bool tie = (m > 1), edge = (pre && pre->valid) ? (pre->edge != 0) : on_threshold(D);
    if (tie || edge)
    {
        if (tie)
            st->same_bucket_ties++;
        if (edge)
            st->threshold_edges++;
        st->pause = (tie ? PAUSE_TIE : 0u) | (edge ? PAUSE_EDGE : 0u);
        st->stop = STOP_PAUSE;
        return;
    }
    const u64 key = st->tkey[s];
    commit_merge(st, (u32)(key & 0xFFFFFFFFull), (u32)(key >> 32), freq, rec_all, false, pre);
    // (a == b on a RANGED stream: replace_stream_kernel takes its run-parity path, same_pair_range)
}

// encode: the "selection" is simply the next rank of the given merge list; a rank whose pair does
// not occur (count 0 in the replicated table) costs no pass.  One thread.
__device__ inline void decide_rank(DevState *st, const u32 *rec_all)
{
    const u64 r = st->merges_done;
    if (st->world > 1)
    {
        u64 total = 0; // (kept current for the statistics of a run that ends here)
        for (u32 q = 0; q < st->world; q++)
            total += (u64)rec_all[q * REC_INTS] | ((u64)rec_all[q * REC_INTS + 1] << 32);
        st->n_global = total;
    }
    if (r >= st->enc_total)
    {
        st->stop = STOP_DONE;
        return;
    }
    const u32 a = st->enc_merges[2 * r], b = st->enc_merges[2 * r + 1];
    const u64 slot = table_find(st->tkey, st->tcap, (u64)a | ((u64)b << 32), murmur3_pair(a, b));
    const u32 cnt = (slot == NO_SLOT) ? 0u : *cnt_ptr(st->tmeta, slot);
    commit_merge(st, a, b, cnt, rec_all, true);
    if (cnt == 0)
        st->skip = 1;
    else
    {
        st->ranks_applied++;
        if (!tok_alias(a, b) && st->batch_max > 1 && st->want_ranged && !st->static_mode && st->z >= st->batch_min_z &&
                 st->z >= st->hist_max)
        {
            // The following ranks can share this pass as long as nothing connects them: pairwise different tokens,
            // none of them an id that this very pass creates, no a == a pair.  (No counts are involved here: the
            // merge list is given, only the ORDER of application must not matter.)
            const u32 z_first = st->z;
            u32 jcap = min(st->batch_max, (u32)BATCH_MAX);
            for (u64 r2 = r + 1; r2 < st->enc_total && st->nb < jcap; r2++)
            {
                const u32 a2 = st->enc_merges[2 * r2], b2 = st->enc_merges[2 * r2 + 1];
                bool ok = !tok_alias(a2, b2) && a2 < z_first && b2 < z_first;
                for (u32 i = 0; ok && i < st->nb; i++)
                    ok = !tok_alias(a2, st->ba[i]) && !tok_alias(a2, st->bb[i]) && !tok_alias(b2, st->ba[i]) &&
                         !tok_alias(b2, st->bb[i]);
                if (!ok)
                    break;
                extend_batch(st, a2, b2);
                st->ranks_applied++;
            }
            if (st->nb > 1)
                st->batch_passes++;
        }
    }
}

// K2, whole-table form (no candidate list: start of training, tiny counts near exhaustion).
__global__ void __launch_bounds__(SEL_THREADS) select_kernel(DevState *st, SelPart *part)
{
    if (st->stop != STOP_RUN || st->pending)
        return;
    __shared__ SelPart sm[SEL_THREADS / 32];
    __shared__ bool s_last;
    const u64 cap = st->tcap;
    const u64 *__restrict__ meta = st->tmeta;
    const u64 D = (u64)st->distinct;
    const u64 B = merged_buckets(D);
    const u32 bmask = (u32)(B - 1);
    u64 k = 0, s = NO_SLOT;
    u32 m = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += (u64)gridDim.x * blockDim.x)
    {
        const u64 mv = meta[i];
        if (mv >> 32)
        {
            const u64 kk = (mv & 0xFFFFFFFF00000000ull) | (u64)(0xFFFFFFFFu - ((u32)mv & bmask));
            sel_combine(k, s, m, kk, i, 1u);
        }
    }
    sel_block_reduce(k, s, m, sm);
    if (threadIdx.x == 0)
    {
        part[blockIdx.x].key = k;
        part[blockIdx.x].slot = s;
        part[blockIdx.x].mult = m;
        __threadfence();
        const u32 done = atomicAdd(&st->sel_done, 1u);
        s_last = (done == gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last)
        return;
    __threadfence();
    k = 0;
    s = NO_SLOT;
    m = 0;
    for (u32 i = threadIdx.x; i < gridDim.x; i += blockDim.x)
    {
        const volatile SelPart *p = part + i;
        sel_combine(k, s, m, p->key, p->slot, p->mult);
    }
    sel_block_reduce(k, s, m, sm);
    if (threadIdx.x != 0)
        return;
    st->sel_done = 0;
    decide(st, k, s, m, cur_recs(st));
}

__global__ void select_rank_kernel(DevState *st)
{
    if (st->stop != STOP_RUN || st->pending)
        return;
    decide_rank(st, cur_recs(st));
}

// ---------------------------------------------------------------------------------------------
// K3: fused replace + prefix-scan compaction + pair-count deltas — the hot kernel.
//
// One streaming pass: 4*n_k bytes in, 4*n_{k+1} bytes out.  Persistent CTAs take tiles in ticket
// order; a tile is staged in shared memory with 128-bit coalesced loads (two tokens of halo in
// front, three behind), every thread then owns 15 consecutive tokens (odd stride: conflict-free
// shared-memory access), finds the replacements that start in its window, and the kept tokens
// are compacted through shared memory and written out coalesced.  Tile offsets come from a
// single-pass decoupled look-back over 64-bit descriptors stamped with the merge epoch (no
// clearing between merges).
//
// Replacements are greedy left to right (bpe.c:760-772).  For a != b they cannot overlap, so a
// position starts one iff it holds a and its right neighbour holds b.  For a == b they pair up
// from the start of each run of a, so a position starts one iff the number of a right in front of
// it is even; that parity is carried across tiles through a second descriptor array (and across
// shards through the edge records).
//
// Every replacement also reports which pair INSTANCES vanish and appear around it, into four
// dense vectors indexed by the free token: (x,a)-, (b,y)-, (x',z)+, (z,y)+.  A replacement always
// owns its left neighbour pair and owns its right one unless another replacement starts right
// behind it, so each instance is charged once (abab -> zz: one (b,a) gone, one (z,z) new).  The
// vectors live in shared memory while the vocabulary is small (hot early merges), else in global
// memory; the table is updated from them afterwards, so the stream is never recounted.
constexpr int R_THREADS = 256;
constexpr int R_ITEMS = 15;
constexpr int R_TILE = R_THREADS * R_ITEMS; // 3840 tokens, a multiple of 4

constexpr u64 DESC_AGG = 1ull << 62;
constexpr u64 DESC_INCL = 2ull << 62;
constexpr u64 DESC_COUNT_MASK = (1ull << 40) - 1;
__device__ __forceinline__ u64 desc_pack(u64 status, u32 epoch, u64 count)
{
    return status | ((u64)(epoch & 0x3FFFFFu) << 40) | (count & DESC_COUNT_MASK);
}
__device__ __forceinline__ bool desc_ready(u64 d, u32 epoch)
{
    return (d >> 62) != 0 && ((u32)(d >> 40) & 0x3FFFFFu) == (epoch & 0x3FFFFFu);
}
// run-parity descriptor: status(2) | all_a(1) | parity(1) | epoch(22)
constexpr u32 PD_LOCAL = 1u << 30;
constexpr u32 PD_RESOLVED = 2u << 30;
__device__ __forceinline__ u32 pd_pack(u32 status, u32 epoch, u32 all_a, u32 par)
{
    return status | (all_a << 29) | (par << 28) | (epoch & 0x3FFFFFu);
}

template <bool SMEM_HIST>
__global__ void __launch_bounds__(R_THREADS) replace_kernel(DevState *st, u64 *desc, u32 *pdesc, int32_t *delta)
{
    if (st->stop != STOP_RUN || st->skip)
        return;
    if (blockIdx.x == 0 && threadIdx.x == 0)
        st->layout_next = LAYOUT_DENSE;
    extern __shared__ __align__(16) u32 smem[];
    u32 *s_tok = smem;                                             // R_TILE + 8 tokens
    int32_t *s_hist = reinterpret_cast<int32_t *>(smem + R_TILE + 8); // 4*(z+1) counters when SMEM_HIST
    __shared__ u32 s_warp[R_THREADS / 32];
    __shared__ u64 s_excl;
    __shared__ u32 s_tile, s_carry;

    const u32 a = st->a, b = st->b, z = st->z;
    const bool same = (a == b);
    const u64 n = st->n;
    const u32 *__restrict__ in = st->tok[st->cur];
    u32 *__restrict__ out = st->tok[st->cur ^ 1];
    const u32 epoch = st->epoch;
    const u64 ntiles = (n + R_TILE - 1) / R_TILE;
    const u32 hb0 = st->halo_before[0], hb1 = st->halo_before[1];
    const u32 ha0 = st->halo_after[0], ha1 = st->halo_after[1], ha2 = st->halo_after[2];
    const u32 carry_in = st->carry_in;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int32_t *gdelta = delta + HDR_INTS;

    if (n == 0)
    {
        if (blockIdx.x == 0 && tid == 0)
            st->n_next = 0;
        return;
    }
    if (SMEM_HIST)
        for (u32 i = tid; i < 4 * (z + 1); i += R_THREADS)
            s_hist[i] = 0;

    for (;;)
    {
        __syncthreads();
        if (tid == 0)
            s_tile = atomicAdd(&st->ticket, 1u);
        __syncthreads();
        const u64 tile = s_tile;
        if (tile >= ntiles)
            break;
        const u64 base = tile * R_TILE;
        const u32 tl = (u32)((n - base < (u64)R_TILE) ? (n - base) : (u64)R_TILE);

        // ---- stage the tile: s_tok[4 + p] = token at local position p, p in [-4, R_TILE + 4)
        {
            const uint4 *in4 = reinterpret_cast<const uint4 *>(in);
            uint4 *s4 = reinterpret_cast<uint4 *>(s_tok);
            for (int v = tid; v < R_TILE / 4 + 2; v += R_THREADS)
            {
                const i64 g0 = (i64)base + 4 * (i64)v - 4;
                uint4 q;
                if (g0 >= 0 && (u64)g0 + 4 <= n)
                    q = __ldg(in4 + (g0 >> 2));
                else
                {
                    u32 e[4];
#pragma unroll
                    for (int k = 0; k < 4; k++)
                    {
                        const i64 g = g0 + k;
                        u32 val;
                        if (g < 0)
                            val = (g == -1) ? hb1 : ((g == -2) ? hb0 : SENT);
                        else if ((u64)g < n)
                            val = in[g];
                        else
                        {
                            const u64 o = (u64)g - n;
                            val = (o == 0) ? ha0 : ((o == 1) ? ha1 : ((o == 2) ? ha2 : SENT));
                        }
                        e[k] = val;
                    }
                    q = make_uint4(e[0], e[1], e[2], e[3]);
                }
                s4[v] = q;
            }
        }
        __syncthreads();

        // ---- my window: w[k] = token at local position p0 + k - 2
        const u32 p0 = (u32)tid * R_ITEMS;
        u32 w[R_ITEMS + 5];
#pragma unroll
        for (int k = 0; k < R_ITEMS + 5; k++)
            w[k] = s_tok[p0 + k + 2];
        const u32 valid = (p0 >= tl) ? 0u : ((tl - p0 < (u32)R_ITEMS) ? (tl - p0) : (u32)R_ITEMS);
        const u32 vmask = (1u << valid) - 1u;
        const u32 OWNV = vmask << 2;
        u32 ea = 0, eb = 0;
#pragma unroll
        for (int k = 0; k < R_ITEMS + 5; k++)
        {
            ea |= (u32)(w[k] == a) << k;
            eb |= (u32)(w[k] == b) << k;
        }

        u32 m; // bit k: a replacement starts at window index k
        if (!same)
            m = ea & (eb >> 1);
        else
        {
            const int all_a = __syncthreads_and(((ea >> 2) & vmask) == vmask);
            if (tid == 0)
            {
                u32 lp; // parity of the run of a that ends at the tile's last token
                if (all_a)
                    lp = tl & 1u;
                else
                {
                    u32 c = 0;
                    int i = (int)tl - 1;
                    while (i >= 0 && s_tok[4 + i] == a)
                    {
                        c++;
                        i--;
                    }
                    lp = c & 1u;
                }
                *reinterpret_cast<volatile u32 *>(pdesc + tile) = pd_pack(PD_LOCAL, epoch, (u32)all_a, lp);
                u32 carry;
                if (tile == 0)
                    carry = carry_in;
                else if (s_tok[3] != a)
                    carry = 0;
                else
                {
                    u32 acc = 0;
                    i64 q = (i64)tile - 1;
                    for (;;)
                    {
                        u32 d;
                        do
                        {
                            d = *reinterpret_cast<volatile u32 *>(pdesc + q);
                        } while ((d >> 30) == 0 || (d & 0x3FFFFFu) != (epoch & 0x3FFFFFu));
                        const u32 par = (d >> 28) & 1u;
                        if ((d >> 30) == 2u || !((d >> 29) & 1u))
                        {
                            carry = acc ^ par;
                            break;
                        }
                        acc ^= par;
                        if (q == 0)
                        {
                            carry = acc ^ carry_in;
                            break;
                        }
                        q--;
                    }
                }
                *reinterpret_cast<volatile u32 *>(pdesc + tile) =
                    pd_pack(PD_RESOLVED, epoch, (u32)all_a, all_a ? (carry ^ (tl & 1u)) : lp);
                s_carry = carry;
            }
            __syncthreads();
            const u32 carry = s_carry;
            u32 par0 = 0; // parity of the number of a right in front of my first token
            if (valid > 0 && ((ea >> 1) & 1u))
            {
                if (p0 == 0)
                    par0 = carry;
                else
                {
                    u32 c = 0;
                    int i = (int)p0 - 1;
                    while (i >= 0 && s_tok[4 + i] == a)
                    {
                        c++;
                        i--;
                    }
                    par0 = (i < 0) ? ((c ^ carry) & 1u) : (c & 1u);
                }
            }
            m = ((ea >> 1) & (ea >> 2) & 1u & par0) << 1; // does one start at my left neighbour?
            u32 par = par0;
#pragma unroll
            for (int k = 2; k < R_ITEMS + 2; k++)
            {
                const u32 isa = (ea >> k) & 1u;
                m |= (isa & ((ea >> (k + 1)) & 1u) & (par ^ 1u)) << k;
                par = isa ? (par ^ 1u) : 0u;
            }
        }
        const u32 mm = m & OWNV;                 // replacements that start on my tokens
        const u32 keep = OWNV & ~(m << 1);       // a token goes away iff one starts at its left neighbour
        const u32 cnt = (u32)__popc(keep);

        // ---- block-wide exclusive scan of the kept counts
        u32 incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const u32 t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o)
                incl += t;
        }
        if (lane == 31)
            s_warp[warp] = incl;
        __syncthreads(); // every thread has read its window: s_tok may now be overwritten
        u32 woff = 0, total = 0;
#pragma unroll
        for (int i = 0; i < R_THREADS / 32; i++)
        {
            const u32 t = s_warp[i];
            woff += (i < warp) ? t : 0u;
            total += t;
        }
        if (tid == 0)
            *reinterpret_cast<volatile u64 *>(desc + tile) = desc_pack(tile == 0 ? DESC_INCL : DESC_AGG, epoch, total);

        // ---- compact into shared memory
        u32 *s_out = s_tok + 4;
        {
            u32 r = woff + incl - cnt;
#pragma unroll
            for (int k = 2; k < R_ITEMS + 2; k++)
                if ((keep >> k) & 1u)
                    s_out[r++] = ((mm >> k) & 1u) ? z : w[k];
        }

        // ---- pair-count deltas
        if (mm)
        {
#pragma unroll
            for (int k = 2; k < R_ITEMS + 2; k++)
                if ((mm >> k) & 1u)
                {
                    const u32 x = w[k - 1], y = w[k + 2];
                    const u32 pm = same ? ((ea >> (k - 1)) & 1u) : ((m >> (k - 2)) & 1u);
                    const u32 nm = (ea >> (k + 2)) & (eb >> (k + 3)) & 1u;
                    if (x != SENT)
                    {
                        if (!(same && x == a))
                        {
                            if (SMEM_HIST)
                                atomicAdd(&s_hist[x * 4 + 0], 1);
                            else
                                delta_add(st, gdelta, (u64)x * 4 + 0, 1);
                        }
                        const u32 xn = pm ? z : x;
                        if (SMEM_HIST)
                            atomicAdd(&s_hist[xn * 4 + 2], 1);
                        else
                            delta_add(st, gdelta, (u64)xn * 4 + 2, 1);
                    }
                    if (y != SENT && !nm)
                    {
                        if (!(same && y == a))
                        {
                            if (SMEM_HIST)
                                atomicAdd(&s_hist[y * 4 + 1], 1);
                            else
                                delta_add(st, gdelta, (u64)y * 4 + 1, 1);
                        }
                        if (SMEM_HIST)
                            atomicAdd(&s_hist[y * 4 + 3], 1);
                        else
                            delta_add(st, gdelta, (u64)y * 4 + 3, 1);
                    }
                }
        }

        // ---- decoupled look-back: where does this tile's output start?
        if (warp == 0)
        {
            u64 excl = 0;
            if (tile > 0)
            {
                i64 q = (i64)tile - 1 - lane;
                for (;;)
                {
                    u64 d;
                    bool ok;
                    do
                    {
                        d = (q >= 0) ? *reinterpret_cast<volatile u64 *>(desc + q) : desc_pack(DESC_INCL, epoch, 0);
                        ok = desc_ready(d, epoch);
                    } while (!__all_sync(0xFFFFFFFFu, ok));
                    const u32 incl_mask = __ballot_sync(0xFFFFFFFFu, (d >> 62) == 2ull);
                    u64 c = d & DESC_COUNT_MASK;
                    if (incl_mask && lane > (__ffs(incl_mask) - 1))
                        c = 0;
#pragma unroll
                    for (int o = 16; o; o >>= 1)
                        c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
                    excl += c;
                    if (incl_mask)
                        break;
                    q -= 32;
                }
                if (lane == 0)
                    *reinterpret_cast<volatile u64 *>(desc + tile) = desc_pack(DESC_INCL, epoch, excl + total);
            }
            if (lane == 0)
                s_excl = excl;
        }
        __syncthreads();
        const u64 excl = s_excl;
        for (u32 i = tid; i < total; i += R_THREADS)
            out[excl + i] = s_out[i];
        if (tile == ntiles - 1 && tid == 0)
            st->n_next = excl + total;
    }

    if (SMEM_HIST)
    {
        // all threads left the loop through the same barrier pair; publish the privatised deltas
        for (u32 i = tid; i < 4 * (z + 1); i += R_THREADS)
        {
            const int32_t v = s_hist[i];
            if (v)
                delta_add(st, gdelta, i, v);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// K4: fold the (all-reduced) delta vectors into the replicated pair table, zero the merged pair,
// keep D exact and the candidate list complete.
__device__ __forceinline__ void cand_offer(DevState *st, u64 slot, u32 newcount)
{
    const u32 T = st->cand_T;
    if (!T || newcount < T)
        return;
    const u32 bit = 1u << (slot & 31);
    if (atomicOr(&st->cflag[slot >> 5], bit) & bit)
        return; // already listed
    const u32 i = atomicAdd(&st->ncand, 1u);
    if (i < st->cand_cap)
        st->cand[i] = (u32)slot;
    else
        st->cand_overflow = 1;
}

// D and the slot occupancy are kept in shared memory while a block works and published once per block:
// thousands of same-address atomics would otherwise queue up in front of the fence that ends the phase.
__device__ __forceinline__ u64 table_insert_counted(DevState *st, u64 *tkey, u64 *tmeta, u64 cap, u64 key, u32 h, int *s_occ)
{
    u64 s = probe_start(h, cap);
    for (u64 i = 0; i < cap; i++)
    {
        u64 k = tkey[s];
        if (k == EMPTY_KEY)
        {
            k = atomicCAS(tkey + s, EMPTY_KEY, key);
            if (k == EMPTY_KEY)
            {
                *hsh_ptr(tmeta, s) = h;
                atomicAdd(s_occ, 1);
                return s;
            }
        }
        if (k == key)
            return s;
        s = (s + 1) & (cap - 1);
    }
    return NO_SLOT;
}

// One delta counter -> the pair table.  Entry e of the delta vectors: merge i of the batch owns the block
// [i * 4 * VS, (i + 1) * 4 * VS), VS = z + nb (one slot per token id that exists after the pass); inside a block,
// token t holds {-(t,a_i), -(b_i,t), +(t,z_i), +(z_i,t)}.
// Every update is a chain of dependent, cache-missing accesses (probe the key, then the atomic on its count; the
// table has long outgrown L2), so the chains of up to N entries are started together: all first probes are issued
// before any of them is waited for.
struct EntryProbe
{
    u64 key, s, k; // pair key, first probe slot, key found there
    u32 h, vec;
};
__device__ __forceinline__ void entry_probe(const DevState *st, const u64 *tkey, u64 cap, u32 e, u32 VS, u32 z0, EntryProbe &p)
{
    const u32 bi = e / (4 * VS), r = e - bi * 4 * VS;
    const u32 a = st->ba[bi], b = st->bb[bi], z = z0 + bi;
    const u32 t = r >> 2, vec = r & 3u;
    const u32 ka = (vec == 1) ? b : ((vec == 3) ? z : t);
    const u32 kb = (vec == 0) ? a : ((vec == 2) ? z : t);
    p.key = (u64)ka | ((u64)kb << 32);
    p.h = murmur3_pair(ka, kb);
    p.vec = vec;
    p.s = probe_start(p.h, cap);
    p.k = tkey[p.s];
}
__device__ __forceinline__ void entry_finish(DevState *st, u64 *tkey, u64 *tmeta, u64 cap, const EntryProbe &p, u32 d, int *s_dD, int *s_occ)
{
    u64 s = p.s, k = p.k;
    if (p.vec >= 2)
    {
        // a pair that contains a new id: claim a slot if it is not in the table yet
        bool found = false;
        for (u64 i = 0; i < cap; i++)
        {
            if (k == EMPTY_KEY)
            {
                k = atomicCAS(tkey + s, EMPTY_KEY, p.key);
                if (k == EMPTY_KEY)
                {
                    *hsh_ptr(tmeta, s) = p.h;
                    atomicAdd(s_occ, 1);
                    k = p.key;
                }
            }
            if (k == p.key)
            {
                found = true;
                break;
            }
            s = (s + 1) & (cap - 1);
            k = tkey[s];
        }
        if (!found)
        {
            atomicOr(&st->err, ERR_TABLE_FULL);
            return;
        }
        const u32 old = atomicAdd(cnt_ptr(tmeta, s), d);
        if (old == 0)
            atomicAdd(s_dD, 1);
        cand_offer(st, s, old + d);
    }
    else
    {
        bool found = false;
        for (u64 i = 0; i < cap; i++)
        {
            if (k == p.key)
            {
                found = true;
                break;
            }
            if (k == EMPTY_KEY)
                break;
            s = (s + 1) & (cap - 1);
            k = tkey[s];
        }
        if (!found)
        {
            atomicOr(&st->err, ERR_MISSING_KEY);
            return;
        }
        const u32 old = atomicSub(cnt_ptr(tmeta, s), d);
        if (old < d)
            atomicOr(&st->err, ERR_NEGATIVE);
        if (old == d)
            atomicAdd(s_dD, -1);
    }
}
template <int N>
__device__ __forceinline__ void apply_entries(DevState *st, u64 *tkey, u64 *tmeta, u64 cap, const u32 (&e)[N], const u32 (&d)[N], u32 VS,
                                              u32 z0, int *s_dD, int *s_occ)
{
    EntryProbe p[N];
#pragma unroll
    for (int j = 0; j < N; j++)
        if (d[j])
            entry_probe(st, tkey, cap, e[j], VS, z0, p[j]);
#pragma unroll
    for (int j = 0; j < N; j++)
        if (d[j])
            entry_finish(st, tkey, tmeta, cap, p[j], d[j], s_dD, s_occ);
}

// Several GPUs, step 1 of a pass's exchange: push every non-zero counter of this rank's delta vectors as one
// (index, value) entry into my slot of every peer's inbox (the counters themselves stay where they are).
__device__ __noinline__ void push_deltas(DevState *st, const int32_t *delta, u32 gtid, u32 gsize, u32 xpar)
{
    const u32 nb = st->nb, z0 = st->z;
    const u32 quads = nb * (z0 + nb);
    const u32 lane = threadIdx.x & 31u, me = st->rank, P = st->world;
    const u64 xcap = st->x.xcap;
    const int4 *dq = reinterpret_cast<const int4 *>(delta + HDR_INTS);
    for (u32 q0 = gtid - lane; q0 < quads; q0 += gsize) // (warp-uniform trip count: the list positions come from a warp scan)
    {
        const u32 q = q0 + lane;
        int4 v = make_int4(0, 0, 0, 0);
        if (q < quads)
            v = __ldcg(dq + q);
        const u32 d[4] = {(u32)v.x, (u32)v.y, (u32)v.z, (u32)v.w};
        const u32 c = (d[0] ? 1u : 0u) + (d[1] ? 1u : 0u) + (d[2] ? 1u : 0u) + (d[3] ? 1u : 0u);
        if (!__any_sync(0xFFFFFFFFu, c != 0))
            continue;
        u32 incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const u32 t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if ((int)lane >= o)
                incl += t;
        }
        u32 base = 0;
        if (lane == 31)
            base = atomicAdd(&st->x_count, incl);
        base = __shfl_sync(0xFFFFFFFFu, base, 31);
        u64 pos = (u64)base + incl - c;
#pragma unroll
        for (int j = 0; j < 4; j++)
            if (d[j])
            {
                if (pos < xcap)
                {
                    const u64 pk = (u64)(4 * q + j) | ((u64)d[j] << 32);
                    for (u32 p = 0; p < P; p++)
                        if (p != me)
                            xchg_entries(st->x.peer[p], xcap, xpar, me)[pos] = pk; // store into the peer's HBM over NVLink
                }
                else
                    atomicOr(&st->err, ERR_XCHG_OVERFLOW);
                pos++;
            }
    }
}

// Several GPUs, step 2: add the peers' lists for exchange `seq` to my own delta vectors as they arrive in my inbox
// (starting with the right-hand neighbour so that the ranks do not all wait for the same sender first).  The
// vectors are L2-resident, so this is cheap; folding every list into the (cache-missing) pair table separately
// would cost P times the table accesses.  Afterwards the vectors hold the sum over all ranks - the same numbers on
// every rank - and apply_deltas() runs exactly as on one GPU.
__device__ __noinline__ void add_peer_lists(DevState *st, int32_t *delta, u32 gtid, u32 gsize, u32 seq)
{
    __shared__ u32 s_cnt;
    const u64 xcap = st->x.xcap;
    const u32 me = st->rank, P = st->world, par = seq & 1u;
    // Nothing may be added to the vectors while a block of THIS rank is still reading them for its pushes
    // (push_deltas): my own flag goes up when the last of them is done.
    if (threadIdx.x == 0)
        xchg_wait(st, me, seq);
    for (u32 k = 1; k < P; k++)
    {
        const u32 sender = (me + k) % P;
        __syncthreads();
        if (threadIdx.x == 0)
            s_cnt = xchg_wait(st, sender, seq) ? ld_relaxed_sys_u32(st->x.local + XCHG_COUNTS + par * MAX_RANKS + sender) : 0u;
        __syncthreads();
        const u32 cnt = s_cnt;
        const u64 *ent = xchg_entries(st->x.local, xcap, par, sender);
        for (u32 i = gtid; i < cnt; i += gsize)
        {
            const u64 pk = ld_relaxed_sys_u64(ent + i); // written by the peer: not through this SM's L1
            atomicAdd(delta + HDR_INTS + (u32)pk, (int32_t)(u32)(pk >> 32));
        }
    }
}

// Fold the delta vectors into the pair table and clear them.  D is kept exact by the 0 <-> non-0 transitions of
// the individual adds.  A thread takes one token's four counters (one 128-bit load) per trip.
__device__ __noinline__ void apply_deltas(DevState *st, int32_t *delta, u32 gtid, u32 gsize)
{
    __shared__ int s_dD, s_occ;
    if (threadIdx.x == 0)
    {
        s_dD = 0;
        s_occ = 0;
    }
    __syncthreads();
    const u32 nb = st->nb, z0 = st->z;
    const u32 VS = z0 + nb;
    const u32 quads = nb * VS;
    u64 *tmeta = st->tmeta, *tkey = st->tkey;
    const u64 cap = st->tcap;
    if (gtid + nb >= gsize && gtid < gsize)
    {
        // SURVEY.md A.5.1: the merged pairs are gone (their own threads, so the probes overlap the others)
        const u32 i = gsize - 1 - gtid;
        const u32 a = st->ba[i], b = st->bb[i];
        const u64 s = table_find(tkey, cap, (u64)a | ((u64)b << 32), murmur3_pair(a, b));
        if (s != NO_SLOT)
        {
            const u32 old = atomicExch(cnt_ptr(tmeta, s), 0u);
            if (old)
                atomicAdd(&s_dD, -1);
        }
    }
    int4 *dq = reinterpret_cast<int4 *>(delta + HDR_INTS);
    for (u32 q = gtid; q < quads; q += gsize)
    {
        const int4 v = __ldcg(dq + q);
        const u32 d[4] = {(u32)v.x, (u32)v.y, (u32)v.z, (u32)v.w};
        if (!(d[0] | d[1] | d[2] | d[3]))
            continue;
        dq[q] = make_int4(0, 0, 0, 0);
        const u32 e[4] = {4 * q, 4 * q + 1, 4 * q + 2, 4 * q + 3};
        apply_entries<4>(st, tkey, tmeta, cap, e, d, VS, z0, &s_dD, &s_occ);
    }
    __syncthreads();
    if (threadIdx.x == 0)
    {
        if (s_dD)
            atomicAdd(reinterpret_cast<u64 *>(&st->distinct), (u64)(i64)s_dD);
        if (s_occ)
            atomicAdd(&st->occupied, (u64)s_occ);
    }
}

// LAYOUT_SPARSE (bpe_sparse.cuh): the write half of a pass, run by the blocks that apply its deltas (the scan that
// recorded the replacements in pass_buf is complete, and the table and the stream are disjoint).  Every block calls it.
// Replacement r of the pass (counted merge by merge) goes to pool[pool_top + r]: the creation list of z + i is
// pool[pool_top + sum of sp_cnt[j < i] ..], as finish_pass records it.
__device__ inline void sparse_rewrite(DevState *st, u32 gtid, u32 gsize)
{
    __shared__ u32 s_la[BATCH_MAX], s_lb[BATCH_MAX], s_ent[BATCH_MAX], s_cum[BATCH_MAX + 1];
    const u32 nb = st->nb, z = st->z;
    u32 *tok = st->tok[st->cur], *so = st->start_of, *pool = st->pool + st->pool_top;
    if (threadIdx.x == 0)
    {
        u32 r = 0;
        for (u32 i = 0; i < nb; i++)
        {
            s_la[i] = st->slen[st->ba[i]];
            s_lb[i] = st->slen[st->bb[i]];
            s_ent[i] = st->sp_ent[i];
            s_cum[i] = r;
            r += st->sp_cnt[i];
        }
        s_cum[nb] = r;
    }
    __syncthreads();
    const u32 total = s_cum[nb];
    for (u32 r = gtid; r < total; r += gsize)
    {
        u32 i = 0;
        while (r >= s_cum[i + 1])
            i++;
        const u32 p = st->pass_buf[s_ent[i] + (r - s_cum[i])];
        const u32 q = p + s_la[i];
        tok[p] = z + i;
        tok[q] = SENT;
        so[q + s_lb[i] - 1] = p;
        pool[r] = p;
    }
}

// the pass is over: its output becomes the current stream (one thread, after every delta is applied - and on the
// sparse layout, after the whole grid has rewritten the stream)
__device__ __forceinline__ void finish_pass(DevState *st)
{
    if (!st->skip)
    {
        if (st->layout == LAYOUT_SPARSE)
        {
            // the creation lists of the new ids, and the counters the next pass's scan adds to back at zero
            const u32 nb = st->nb, z = st->z;
            u64 top = st->pool_top, r = 0;
            for (u32 i = 0; i < nb; i++)
            {
                const u32 c = st->sp_cnt[i];
                st->cl_off[z + i] = (u32)top;
                st->cl_cnt[z + i] = c;
                top += c;
                r += c;
                st->sp_cnt[i] = 0;
            }
            st->pool_top = top;
            st->sparse_passes++;
            st->n_hist[st->merges_done - nb] |= SPARSE_PASS_MARK;
            st->n_next = st->n - r; // every replacement removes one token
        }
        st->n = st->n_next;
        st->cur ^= 1u;
        st->layout = st->layout_next;
    }
    st->pending = 0;
}

// whole-table mode: K4 alone (select_kernel follows)
__global__ void __launch_bounds__(256) apply_kernel(DevState *st, int32_t *delta)
{
    if (st->stop != STOP_RUN || !st->pending)
        return;
    if (!st->skip && st->layout == LAYOUT_SPARSE)
        sparse_rewrite(st, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
    if (!st->skip)
        apply_deltas(st, delta, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
    __syncthreads();
    if (threadIdx.x == 0)
    {
        __threadfence();
        if (atomicAdd(&st->sel_done, 1u) == gridDim.x - 1)
        {
            st->sel_done = 0;
            finish_pass(st);
        }
    }
}

// list mode: K4 + K2 in one launch.  Every block applies its share of the deltas; the last block to
// finish then owns a consistent table, takes the maximum over the candidate list (one gather per
// candidate, warp shuffles + block tree with the multiplicity of the maximal key carried along) and
// decides.  mode: AS_TRAIN; AS_ENCODE = the next rank of the given merge list instead of the maximum;
// AS_APPLY_ONLY = no decision (select_kernel follows: whole-table selection on several GPUs).
// Several GPUs: the same launch also carries the exchange (struct Xchg): own deltas are pushed into the peers'
// inboxes while they are applied, the last block to finish raises this rank's flag, and every block then
// folds in the peers' lists as their flags arrive - no collective, no extra launch.
enum : int
{
    AS_TRAIN = 0,
    AS_ENCODE = 1,
    AS_APPLY_ONLY = 2
};
__global__ void __launch_bounds__(SEL_THREADS) apply_select_kernel(DevState *st, int32_t *delta, int mode)
{
    pdl_wait();
    pdl_launch_dependents();
    if (st->stop != STOP_RUN)
        return;
    const bool encode = (mode == AS_ENCODE);
    __shared__ SelPart sm[SEL_THREADS / 32];
    __shared__ bool s_last;
    __shared__ u32 s_recs[MAX_RANKS * REC_INTS]; // every rank's edge record (last block and the probe block)
    const u64 t0 = gtime();
    const bool pending = st->pending != 0;
    const u32 world = st->world;
    const bool xch = world > 1 && pending && !st->skip; // this launch carries an exchange
    const u32 seq = st->xseq + (xch ? 1u : 0u);          // the exchange whose records describe the stream from now on
    const bool sparse = pending && !st->skip && st->layout == LAYOUT_SPARSE; // the apply blocks also rewrite the stream
    const u32 nb_apply = gridDim.x - 1; // the last block of the grid only looks up the stream's last pair
    if (blockIdx.x == nb_apply)
    {
        // While the other blocks fold the deltas in, this one asks for the candidates' table lines: the table has
        // long outgrown L2 (2 GB on the 1 GB corpus), and the last block's gathers are on the critical path.
        if (mode == AS_TRAIN && st->cand_T)
        {
            const u32 ncp = min(*reinterpret_cast<volatile u32 *>(&st->ncand), min(st->cand_cap, CAND_FIT));
            const u64 *pm = st->tmeta, *pk = st->tkey;
            for (u32 i = threadIdx.x; i < ncp; i += blockDim.x)
            {
                const u32 sl = __ldcg(st->cand + i);
                asm volatile("prefetch.global.L2 [%0];" ::"l"(pm + sl));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(pk + sl));
            }
        }
        if (xch && threadIdx.x < 32)
        {
            u32 rec[REC_INTS];
            edge_record_compute(st, true, rec);
            if (threadIdx.x == 0)
                xchg_push_record(st, seq, rec);
        }
    }
    else if (xch)
        push_deltas(st, delta, blockIdx.x * blockDim.x + threadIdx.x, nb_apply * blockDim.x, seq & 1u);
    else if (pending && !st->skip)
    {
        if (sparse)
            sparse_rewrite(st, blockIdx.x * blockDim.x + threadIdx.x, nb_apply * blockDim.x);
        apply_deltas(st, delta, blockIdx.x * blockDim.x + threadIdx.x, nb_apply * blockDim.x);
    }
    if (xch)
    {
        __syncthreads();
        if (threadIdx.x == 0)
        {
            __threadfence_system();
            if (atomicAdd(&st->x_done, 1u) == gridDim.x - 1)
            {
                // every block of this rank has pushed its entries: my list is complete
                st->x_done = 0;
                const u32 cnt = atomicExch(&st->x_count, 0u);
                xchg_signal(st, seq, cnt < st->x.xcap ? cnt : (u32)st->x.xcap);
            }
        }
        if (blockIdx.x != nb_apply)
        {
            add_peer_lists(st, delta, blockIdx.x * blockDim.x + threadIdx.x, nb_apply * blockDim.x, seq);
            // every block has added its share of every list before anybody folds the sums into the table (all
            // blocks of this grid are resident: at most one per SM, and the pass kernel in front of it is over)
            __syncthreads();
            if (threadIdx.x == 0)
            {
                __threadfence();
                atomicAdd(&st->x_bar, 1u);
                while (*reinterpret_cast<volatile u32 *>(&st->x_bar) < nb_apply)
                    ;
                __threadfence();
            }
            __syncthreads();
            apply_deltas(st, delta, blockIdx.x * blockDim.x + threadIdx.x, nb_apply * blockDim.x);
        }
        else if (threadIdx.x == 0)
        {
            bool ok = true;
            for (u32 p = 0; p < world && ok; p++)
                if (p != st->rank)
                    ok = xchg_wait(st, p, seq);
        }
        __syncthreads();
    }
    if (world > 1 && (blockIdx.x == nb_apply) && threadIdx.x < MAX_RANKS * REC_INTS)
        s_recs[threadIdx.x] = ld_relaxed_sys_u32(xchg_recs(st->x.local, seq & 1u) + threadIdx.x);
    __syncthreads();
    if (blockIdx.x == nb_apply && threadIdx.x == 0 && mode == AS_TRAIN && !sparse)
    {
        const bool flip0 = pending && !st->skip;
        const u64 key = last_pair_key(st, s_recs, flip0 ? (st->cur ^ 1u) : st->cur, flip0 ? st->layout_next : st->layout,
                                      flip0 ? st->n_next : st->n);
        st->probe_key = key;
        st->probe_slot = (key == EMPTY_KEY) ? NO_SLOT : table_find(st->tkey, st->tcap, key, murmur3_pair((u32)key, (u32)(key >> 32)));
    }
    __syncthreads();
    const u64 t1 = gtime();
    if (threadIdx.x == 0)
    {
        __threadfence();
        s_last = atomicAdd(&st->sel_done, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last)
        return;
    __threadfence();
    const u64 t2 = gtime();
    // ---- last block: the table is final.  Side jobs (flip the buffers, census probe, threshold test)
    // run on three different warps while everybody scans the candidates.
    __shared__ PreDecide s_pre;
    if (world > 1 && threadIdx.x < MAX_RANKS * REC_INTS)
        s_recs[threadIdx.x] = ld_relaxed_sys_u32(xchg_recs(st->x.local, seq & 1u) + threadIdx.x);
    const u64 D = (u64) * reinterpret_cast<volatile i64 *>(&st->distinct);
    __syncthreads();
    if (threadIdx.x == 0)
    {
        st->sel_done = 0;
        st->xseq = seq;
        st->x_bar = 0;
        if (pending)
            finish_pass(st);
    }
    if (sparse)
        __syncthreads(); // (thread 32 below reads the stream length finish_pass has just set)
    if (mode == AS_APPLY_ONLY)
        return;
    if (encode)
    {
        if (threadIdx.x == 0)
            decide_rank(st, s_recs);
        return;
    }
    if (threadIdx.x == 32)
    {
        // the key and (unless this very apply created it) its slot were looked up while the deltas were applied.
        // A sparse pass's stream is rewritten by the same blocks that apply the deltas, so the probe block could not
        // read its last pair; this block can: every other block passed the sel_done handshake after its share of the
        // rewrite (L2 loads: lines cached in this SM's L1 before the rewrite must not be read).
        u64 key, slot;
        if (sparse)
        {
            key = EMPTY_KEY;
            slot = NO_SLOT;
            if (st->n >= 2)
            {
                const u32 *t = st->tok[st->cur], *so = st->start_of;
                const u32 lp = __ldcg(so + st->n0 - 1);
                const u32 x = __ldcg(t + __ldcg(so + lp - 1)), y = __ldcg(t + lp);
                if (x != SENT && y != SENT)
                    key = (u64)x | ((u64)y << 32);
            }
        }
        else
        {
            key = *reinterpret_cast<volatile u64 *>(&st->probe_key);
            slot = *reinterpret_cast<volatile u64 *>(&st->probe_slot);
        }
        if (key != EMPTY_KEY && slot == NO_SLOT)
            slot = table_find(st->tkey, st->tcap, key, murmur3_pair((u32)key, (u32)(key >> 32)));
        s_pre.last_new = (key != EMPTY_KEY && slot != NO_SLOT && __ldcg(cnt_ptr(st->tmeta, slot)) == 1u) ? 1u : 0u;
    }
    if (threadIdx.x == 64)
    {
        s_pre.edge = on_threshold(D) ? 1u : 0u;
        s_pre.valid = 1;
    }
    const u64 t3 = gtime();
    const u64 *meta = st->tmeta;
    const u64 *tkeys = st->tkey;
    const u64 B = merged_buckets(D);
    const u32 bmask = (u32)(B - 1);
    const u32 ncr = *reinterpret_cast<volatile u32 *>(&st->ncand);
    const u32 nc = ncr < st->cand_cap ? ncr : st->cand_cap;
    const u32 *cand = st->cand;
    u64 k = 0, s = NO_SLOT;
    u32 m = 0;
    constexpr int UNR = 8; // independent gathers in flight per thread
    // the first trip's candidates stay in registers: when the whole list fits (it almost always does) the
    // batch extension below works on them without touching memory again
    u32 sl[UNR];
    u64 pk[UNR], kk[UNR]; // pair key (a | b << 32), packed order key (count << 32 | ~bucket), 0 = none / taken
    const bool fits = nc <= (u32)(SEL_THREADS * UNR);
#pragma unroll
    for (int j = 0; j < UNR; j++)
    {
        const u32 i = j * SEL_THREADS + threadIdx.x;
        sl[j] = (i < nc) ? __ldcg(cand + i) : 0xFFFFFFFFu;
    }
#pragma unroll
    for (int j = 0; j < UNR; j++)
    {
        const u64 mv = (sl[j] != 0xFFFFFFFFu) ? __ldcg(meta + sl[j]) : 0ull;
        pk[j] = (sl[j] != 0xFFFFFFFFu) ? __ldcg(tkeys + sl[j]) : 0ull;
        kk[j] = (mv >> 32) ? ((mv & 0xFFFFFFFF00000000ull) | (u64)(0xFFFFFFFFu - ((u32)mv & bmask))) : 0ull;
        if (kk[j])
            sel_combine(k, s, m, kk[j], (u64)sl[j], 1u);
    }
    for (u32 base = SEL_THREADS * UNR; base < nc; base += SEL_THREADS * UNR)
    {
        u32 sl2[UNR];
        u64 mv2[UNR];
#pragma unroll
        for (int j = 0; j < UNR; j++)
        {
            const u32 i = base + j * SEL_THREADS + threadIdx.x;
            sl2[j] = (i < nc) ? __ldcg(cand + i) : 0xFFFFFFFFu;
        }
#pragma unroll
        for (int j = 0; j < UNR; j++)
            mv2[j] = (sl2[j] != 0xFFFFFFFFu) ? __ldcg(meta + sl2[j]) : 0ull;
#pragma unroll
        for (int j = 0; j < UNR; j++)
            if (mv2[j] >> 32)
            {
                const u64 k2 = (mv2[j] & 0xFFFFFFFF00000000ull) | (u64)(0xFFFFFFFFu - ((u32)mv2[j] & bmask));
                sel_combine(k, s, m, k2, (u64)sl2[j], 1u);
            }
    }
    const u64 t4 = gtime();
    sel_block_reduce(k, s, m, sm); // (its barriers also publish s_pre)
    __shared__ u64 s_win;          // slot of the pair chosen last (NO_SLOT: stop extending the batch)
    __shared__ Committed s_cm;
    u64 t5 = 0, t6 = 0;
    if (threadIdx.x == 0)
    {
        t5 = gtime();
        bool extend = false;
        if (st->world == 1 && s_pre.valid)
        {
            decide_list(st, k, s, m, &s_pre, &s_cm, ncr);
            extend = fits && s_cm.ok;
        }
        else
        {
            decide(st, k, s, m, s_recs, &s_pre); // several GPUs: the general form
            extend = fits && st->stop == STOP_RUN && st->pending && st->batch_max > 1 && st->cand_T && st->want_ranged &&
                     !st->static_mode && !tok_alias(st->a, st->b) && st->z >= st->batch_min_z && st->z >= st->hist_max &&
                     st->merges_done < st->max_merges;
            if (extend)
            {
                s_cm.a = st->a;
                s_cm.b = st->b;
                s_cm.freq = st->freq;
                s_cm.z = st->z;
                s_cm.cand_T = st->cand_T;
                s_cm.batch_max = st->batch_max;
                s_cm.hist_max = st->hist_max;
                s_cm.hist_words = st->hist_words;
                s_cm.merges_done = st->merges_done;
                s_cm.max_merges = st->max_merges;
                s_cm.bt0 = st->bt[0];
                s_cm.n_stream = st->n_global;
                s_cm.merges = st->merges;
                s_cm.n_hist = st->n_hist;
            }
        }
        t6 = gtime();
        s_win = extend ? s : NO_SLOT;
    }
    __syncthreads();
    if (s_win != NO_SLOT)
    {
        // Which candidates come next in exact selection order?  Every warp extracts its own four best (warp
        // shuffles only, everything is in registers); warp 0 then merges the sixteen sorted lists and accepts a
        // candidate while it is certain to be the next merge of the sequential algorithm:
        //   * its two tokens occur in none of the accepted pairs (so its count cannot change, and the pass can
        //     replace all accepted pairs at once without interaction);
        //   * it is not involved in a same-bucket tie and is not an a == a pair;
        //   * its count is strictly above the count of the first candidate that was NOT accepted (every pair
        //     whose count the accepted merges can change or create ranks at or below that one: new pairs never
        //     exceed the old pairs they come from, SURVEY.md A.5.4);
        //   * D stays far enough from every table-doubling threshold that the bucket order B(D) and the
        //     workers' bucket counts cannot change inside the batch.
        // Several GPUs: every rank must form the SAME batch, but the candidate list is in a different order on every
        // rank (it is filled by atomics), so which warp holds which candidate differs.  With as many entries per warp
        // list as a batch has merges no list can be used up before the cap ends the walk, and the walk depends on
        // the SET of candidates only.  (One GPU: four per warp are cheaper to extract, and any prefix of the
        // sequential merges is a correct batch.)
        constexpr int NW = SEL_THREADS / 32, TOPK_MAX = BATCH_MAX > 4 ? BATCH_MAX : 4;
        const int TOPK = (world > 1) ? TOPK_MAX : 4;
        __shared__ u64 s_wk[NW][TOPK_MAX], s_wp[NW][TOPK_MAX];
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const u64 first = s_win;
#pragma unroll
        for (int j = 0; j < UNR; j++)
            if ((u64)sl[j] == first)
                kk[j] = 0;
        for (int r = 0; r < TOPK; r++)
        {
            u64 bk = 0, bp = 0;
            u32 bs = 0xFFFFFFFFu;
#pragma unroll
            for (int j = 0; j < UNR; j++)
                if (kk[j] > bk || (kk[j] == bk && bk && sl[j] < bs))
                {
                    bk = kk[j];
                    bs = sl[j];
                    bp = pk[j];
                }
#pragma unroll
            for (int o = 16; o; o >>= 1)
            {
                const u64 k2 = __shfl_xor_sync(0xFFFFFFFFu, bk, o), p2 = __shfl_xor_sync(0xFFFFFFFFu, bp, o);
                const u32 s2 = __shfl_xor_sync(0xFFFFFFFFu, bs, o);
                if (k2 > bk || (k2 == bk && s2 < bs))
                {
                    bk = k2;
                    bs = s2;
                    bp = p2;
                }
            }
#pragma unroll
            for (int j = 0; j < UNR; j++)
                if (bk && sl[j] == bs)
                    kk[j] = 0;
            if (lane == 0)
            {
                s_wk[warp][r] = bk;
                s_wp[warp][r] = bp;
            }
        }
        __syncthreads();
        __shared__ u32 s_acc_a[BATCH_MAX], s_acc_b[BATCH_MAX];
        __shared__ u32 s_resc[4]; // bound, merges the walk accepted, merges strictly above the bound, rescue result
        const Committed cm = s_cm; // (one burst of shared-memory loads)
        u32 my_a = SENT, my_b = SENT, my_c = 0, nacc = 1, bound = 0, why = 0, nacc_walk = 1, nacc_bound = 1;
        if (warp == 0)
        {
            const u64 room = cm.max_merges - cm.merges_done + 1; // merges the cap still allows, this pass included
            u32 jcap = (u32)min((u64)min(cm.batch_max, (u32)BATCH_MAX), room);
            // while replacements are frequent their deltas are privatised in shared memory: keep the batch small
            // enough for that histogram (one block of 4 vectors per merge) until the ids outgrow it
            // (beyond hist_max ids a pass makes few enough replacements for global atomics)
            if (cm.z < cm.hist_max)
                while (jcap > 1 && jcap * 4 * (cm.z + jcap) > cm.hist_words)
                    jcap--;
            // lane i keeps accepted pair i; lane w < NW walks warp w's list
            if (lane == 0)
            {
                my_a = cm.a;
                my_b = cm.b;
                my_c = cm.freq;
            }
            u32 ptr = 0; // why: 0 cap, 1 below cand_T, 2 tie, 3 overlap, 4 a==b/alias/cnt<2, 5 list used up
            bool stop = false;
            for (u32 r = 1; r <= jcap && !stop; r++)
            {
                const u64 hk = (lane < NW && ptr < (u32)TOPK) ? s_wk[lane][ptr] : 0ull;
                u64 bk = hk;
                u32 bl = (u32)lane;
#pragma unroll
                for (int o = 16; o; o >>= 1)
                {
                    const u64 k2 = __shfl_xor_sync(0xFFFFFFFFu, bk, o);
                    const u32 l2 = __shfl_xor_sync(0xFFFFFFFFu, bl, o);
                    if (k2 > bk || (k2 == bk && l2 < bl))
                    {
                        bk = k2;
                        bl = l2;
                    }
                }
                if (bk == 0 || (u32)(bk >> 32) < cm.cand_T)
                {
                    // The list is only complete for counts >= cand_T: entries that have decayed below the threshold
                    // say nothing about the pairs that were never listed.  Everything else is below the threshold.
                    bound = cm.cand_T - 1;
                    why = 1;
                    break;
                }
                // same-bucket tie: another list's head, or the winner list's next entry, has the same packed key
                const u32 wptr = __shfl_sync(0xFFFFFFFFu, ptr, bl);
                const u64 nextk = (wptr + 1 < (u32)TOPK) ? s_wk[bl][wptr + 1] : 0ull;
                const bool tie = __ballot_sync(0xFFFFFFFFu, lane != (int)bl && hk == bk) != 0 || nextk == bk;
                const u64 pay = s_wp[bl][wptr];
                const u32 cnt = (u32)(bk >> 32), a = (u32)pay, b = (u32)(pay >> 32);
                const bool overlap =
                    __ballot_sync(0xFFFFFFFFu, (u32)lane < nacc && (tok_alias(a, my_a) || tok_alias(a, my_b) || tok_alias(b, my_a) ||
                                                                    tok_alias(b, my_b))) != 0;
                const bool ok = !tie && cnt >= 2 && !tok_alias(a, b) && !overlap && r < jcap;
                if (!ok)
                {
                    bound = cnt;
                    why = tie ? 2u : (overlap ? 3u : (r >= jcap ? 0u : 4u));
                    break;
                }
                if ((u32)lane == nacc)
                {
                    my_a = a;
                    my_b = b;
                    my_c = cnt;
                }
                nacc++;
                if ((u32)lane == bl)
                    ptr++;
                // a list that is used up may hide further candidates of its warp: nothing beyond is certain
                if (wptr + 1 == (u32)TOPK)
                {
                    bound = cnt;
                    stop = true;
                    why = 5;
                }
            }
            nacc_walk = nacc; // accepted before the bound / margin rules trim the batch
            // Strictly above the bound: every pair whose count the accepted merges can change, or that they create,
            // ranks at or below the first candidate that was not accepted (count `bound`).
            while (nacc > 1 && __shfl_sync(0xFFFFFFFFu, my_c, nacc - 1) <= bound)
                nacc--;
            if ((u32)lane < (u32)BATCH_MAX)
            {
                s_acc_a[lane] = ((u32)lane < nacc_walk) ? my_a : SENT;
                s_acc_b[lane] = ((u32)lane < nacc_walk) ? my_b : SENT;
            }
            if (lane == 0)
            {
                s_resc[0] = bound;
                s_resc[1] = nacc_walk;
                s_resc[2] = (why == 0 || why == 3 || why == 4) ? nacc : nacc_walk; // (no rescue after a tie / a used-up list)
                s_resc[3] = 0xFFFFFFFFu;
            }
        }
        __syncthreads();
        if (s_resc[2] < s_resc[1])
        {
            // Accepted merges whose count EQUALS the bound: merge i is still certain to be next unless a pair with
            // exactly that count contains a token of the merges in front of it (only such a pair can turn into a new
            // pair (x, z_j) of the same count that the bucket order might put first).  Every pair with that count is
            // in the list (bound >= cand_T here): each thread looks at its own candidates, and the first threads at
            // the entries that were moved to the warps' lists.  Result: the smallest merge index any of them touches.
            const u32 bnd = s_resc[0], nw = s_resc[1];
            u32 jm = 0xFFFFFFFFu;
            auto look = [&](u64 key, u64 pair) {
                if ((u32)(key >> 32) != bnd)
                    return;
                const u32 a = (u32)pair, b = (u32)(pair >> 32);
                for (u32 i = 0; i < nw; i++)
                {
                    const u32 xa = s_acc_a[i], xb = s_acc_b[i];
                    if (a == xa && b == xb)
                        return; // an accepted merge itself
                    if (a == xa || a == xb || b == xa || b == xb)
                    {
                        jm = min(jm, i);
                        return; // (indices only grow from here)
                    }
                }
            };
#pragma unroll
            for (int j = 0; j < UNR; j++)
                if (kk[j])
                    look(kk[j], pk[j]);
            if ((int)threadIdx.x < NW * TOPK)
                look(s_wk[threadIdx.x / TOPK][threadIdx.x % TOPK], s_wp[threadIdx.x / TOPK][threadIdx.x % TOPK]);
#pragma unroll
            for (int o = 16; o; o >>= 1)
                jm = min(jm, __shfl_xor_sync(0xFFFFFFFFu, jm, o));
            if (lane == 0 && jm != 0xFFFFFFFFu)
                atomicMin(&s_resc[3], jm);
            __syncthreads();
            if (warp == 0)
            {
                // merges 0 .. jm are safe (nothing in front of them is touched); at least the strictly-above ones
                const u32 jmin = s_resc[3];
                const u32 safe = (jmin >= nw) ? nw : jmin + 1;
                nacc = max(nacc, min(nw, safe));
            }
        }
        if (warp == 0)
        {
            nacc_bound = nacc;
            // How far can D move before merge i of the batch is selected (i.e. through merges 0 .. i-1)?  A merge
            // with c replacements creates at most min(2c, 2V) new keys ((x,z) and (z,y), one of each per
            // replacement, V token ids) and empties at most that many old ones ((x,a), (b,y)) plus (a,b) itself.
            // The merged table is rebuilt from 65,536 buckets every iteration: no doubling threshold may lie within
            // reach on either side (so B(D), the exact-threshold edge and the tie-break order stay what this walk
            // assumed); the worker table only ever grows: its next threshold must stay out of reach.  The batch is
            // cut in front of the first merge for which that cannot be promised.
            const u64 vb = 2ull * (cm.z + BATCH_MAX);
            const u64 mine = ((u32)lane < nacc) ? min(2ull * my_c, vb) : 0ull;
            u64 up = mine, down = mine + (((u32)lane < nacc) ? 1ull : 0ull); // inclusive prefix sums below
#pragma unroll
            for (int o = 1; o < 32; o <<= 1)
            {
                const u64 u2 = __shfl_up_sync(0xFFFFFFFFu, up, o), d2 = __shfl_up_sync(0xFFFFFFFFu, down, o);
                if (lane >= o)
                {
                    up += u2;
                    down += d2;
                }
            }
            up = __shfl_up_sync(0xFFFFFFFFu, up, 1); // merges 0 .. lane-1
            down = __shfl_up_sync(0xFFFFFFFFu, down, 1);
            // tokens the merges in front of this one remove (a != b: one per occurrence, SURVEY.md A.5.5)
            u64 gone = ((u32)lane < nacc) ? (u64)my_c : 0ull;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1)
            {
                const u64 g2 = __shfl_up_sync(0xFFFFFFFFu, gone, o);
                if (lane >= o)
                    gone += g2;
            }
            gone = __shfl_up_sync(0xFFFFFFFFu, gone, 1);
            bool clear = true;
            if (lane >= 1 && (u32)lane < nacc)
            {
                // The reference switches to its 16 static slices in the first iteration that starts below
                // 1,048,576 tokens (bpe.c:449), and from then on the worker tables grow with their slices'
                // contents: that iteration must be selected on its own (census), not ride along in this pass.
                if (cm.n_stream < STATIC_LIMIT + gone)
                    clear = false;
                for (u64 bsz = 65536; bsz <= (1ull << 40); bsz *= 2)
                {
                    const u64 thr = resize_threshold(bsz);
                    if (thr + down >= D && thr <= D + up)
                        clear = false;
                    if (thr > D + up)
                        break;
                }
                if (D + up + 1 >= resize_threshold(cm.bt0))
                    clear = false;
            }
            const u32 blocked = __ballot_sync(0xFFFFFFFFu, !clear);
            if (blocked)
                nacc = min(nacc, (u32)__ffs(blocked) - 1u);
            // extend_batch() for merges 1 .. nacc-1, every lane its own merge, nothing read back
            if (lane >= 1 && (u32)lane < nacc)
            {
                const u64 km = cm.merges_done + (u32)lane - 1;
                st->ba[lane] = my_a;
                st->bb[lane] = my_b;
                cm.merges[2 * km] = my_a;
                cm.merges[2 * km + 1] = my_b;
                cm.n_hist[km] = ~0ull; // rides along: no pass of its own
            }
            if (lane == 0)
            {
                // 0-5: why the walk ended; 6: merges lost to the strictly-above-the-bound rule; 7: to the D margin
                atomicAdd(reinterpret_cast<unsigned long long *>(&st->ext_why[why]), 1ull);
                if (nacc_walk > nacc_bound)
                    atomicAdd(reinterpret_cast<unsigned long long *>(&st->ext_why[6]), (unsigned long long)(nacc_walk - nacc_bound));
                if (nacc_bound > nacc)
                    atomicAdd(reinterpret_cast<unsigned long long *>(&st->ext_why[7]), (unsigned long long)(nacc_bound - nacc));
            }
            if (lane == 0 && nacc > 1)
            {
                st->nb = nacc;
                st->merges_done = cm.merges_done + nacc - 1;
                atomicAdd(reinterpret_cast<unsigned long long *>(&st->batch_merges), (unsigned long long)(nacc - 1));
                atomicAdd(reinterpret_cast<unsigned long long *>(&st->batch_passes), 1ull);
            }
        }
    }
    if (threadIdx.x == 0)
    {
        st->dbg[0] += t1 - t0;
        st->dbg[1] += t2 - t1;
        st->dbg[2] += t3 - t2;
        st->dbg[3] += t4 - t3;
        st->dbg[4] += t5 - t4;
        st->dbg[5] += t6 - t5;
        st->dbg[6] += 1;
        st->dbg[7] += gtime() - t6;
    }
}

__global__ void cand_reset_kernel(DevState *st)
{
    st->ncand = 0;
    st->cand_overflow = 0;
    st->cand_big_ok = 0;
    st->cand_T = 0;
}

// (re)build the candidate list for threshold T (cflag cleared by the host, then cand_reset_kernel)
__global__ void __launch_bounds__(256) cand_rebuild_kernel(DevState *st, u32 T)
{
    const u64 cap = st->tcap;
    const u64 *__restrict__ meta = st->tmeta;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += (u64)gridDim.x * blockDim.x)
        if ((u32)(meta[i] >> 32) >= T)
        {
            atomicOr(&st->cflag[i >> 5], 1u << (i & 31));
            const u32 j = atomicAdd(&st->ncand, 1u);
            if (j < st->cand_cap)
                st->cand[j] = (u32)i;
            else
                st->cand_overflow = 1;
        }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        st->cand_T = T;
}

__global__ void cand_big_ok_kernel(DevState *st) { st->cand_big_ok = 1; }

// halos of the untouched stream (before the first merge), for the shard-straddling byte pair
__global__ void resolve_edges_kernel(DevState *st)
{
    if (st->world > 1)
        resolve_edges(st, cur_recs(st), SENT, false);
    else
        st->n_global = st->n;
}

// host cleared a pause: resume the step sequence
__global__ void resume_kernel(DevState *st)
{
    if (st->stop == STOP_PAUSE)
    {
        st->stop = STOP_RUN;
        st->pause = 0;
    }
}

// a skipped encode rank still has to advance (no pass, no deltas): nothing to do, the stream and
// the table are unchanged.  Paused / finished steps fall through every kernel above.

} // namespace bpe
