// Host side of the B200 BPE merge-loop engine + the C ABI of include/bpe_cuda.h.
//
// One context per GPU.  A merge step is a fixed sequence of launches driven entirely by a
// device-resident control block (bpe::DevState): select -> replace(+scan+deltas) -> [edge record,
// ncclAllReduce] -> apply.  The host enqueues steps in batches and polls the control block once
// per batch (stop / pause / table occupancy), so there is no host round trip per merge.
//
// There is no CPU fallback anywhere in this file: without a CUDA device every entry point fails.
#include "../../include/bpe_cuda.h"
#include "bpe_kernels.cuh"
#include "bpe_replace.cuh"
#include "bpe_resolver.cuh"
#include "bpe_decode.cuh"
#include "bpe_encode_batch.cuh"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <mutex>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

using namespace bpe;

// ---------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static char g_err_global[512] = "";

static void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    memcpy(g_err_global, g_err, sizeof g_err);
}

#define CU(call)                                                                                                       \
    do                                                                                                                 \
    {                                                                                                                  \
        cudaError_t e_ = (call);                                                                                       \
        if (e_ != cudaSuccess)                                                                                         \
        {                                                                                                              \
            set_error("CUDA error %s at %s:%d (%s)", cudaGetErrorString(e_), __FILE__, __LINE__, #call);               \
            return BPE_CUDA_ERR_CUDA;                                                                                  \
        }                                                                                                              \
    } while (0)

// NCCL is resolved at run time (dlopen) so that the single-GPU path carries no link dependency.
struct NcclApi
{
    void *lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Broadcast)(const void *, void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;

static int nccl_load()
{
    if (g_nccl.lib)
        return 0;
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    void *h = nullptr;
    for (const char *nm : names)
        if ((h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL)))
            break;
    if (!h)
    {
        set_error("cannot load NCCL: %s", dlerror());
        return BPE_CUDA_ERR_CUDA;
    }
    g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))dlsym(h, "ncclGetUniqueId");
    g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))dlsym(h, "ncclCommInitRank");
    g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))dlsym(h, "ncclCommDestroy");
    g_nccl.AllReduce = (decltype(g_nccl.AllReduce))dlsym(h, "ncclAllReduce");
    g_nccl.AllGather = (decltype(g_nccl.AllGather))dlsym(h, "ncclAllGather");
    g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))dlsym(h, "ncclGetErrorString");
    g_nccl.Broadcast = (decltype(g_nccl.Broadcast))dlsym(h, "ncclBroadcast");
    g_nccl.GroupStart = (decltype(g_nccl.GroupStart))dlsym(h, "ncclGroupStart");
    g_nccl.GroupEnd = (decltype(g_nccl.GroupEnd))dlsym(h, "ncclGroupEnd");
    if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce || !g_nccl.AllGather || !g_nccl.CommDestroy ||
        !g_nccl.Broadcast || !g_nccl.GroupStart || !g_nccl.GroupEnd)
    {
        set_error("NCCL library lacks required symbols");
        return BPE_CUDA_ERR_CUDA;
    }
    g_nccl.lib = h;
    return 0;
}

#define NC(call)                                                                                                       \
    do                                                                                                                 \
    {                                                                                                                  \
        ncclResult_t r_ = (call);                                                                                      \
        if (r_ != ncclSuccess)                                                                                         \
        {                                                                                                              \
            set_error("NCCL error %s at %s:%d", g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "?", __FILE__,     \
                      __LINE__);                                                                                       \
            return BPE_CUDA_ERR_CUDA;                                                                                  \
        }                                                                                                              \
    } while (0)

// ---------------------------------------------------------------------------------------------
struct bpe_cuda_ctx
{
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    // resident input shard
    uint8_t *d_bytes = nullptr;
    size_t bytes_cap = 0, n_bytes = 0;
    // file ingest / result download: two pinned staging buffers, a copy stream, "buffer is free again" events
    uint8_t *h_stage[2] = {nullptr, nullptr};
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t stage_ev[2] = {nullptr, nullptr};
    bool prewidened = false; // the ingest has already widened and counted the resident shard (consumed by the next run)
    // token stream ping-pong
    u32 *d_tok_alloc[2] = {nullptr, nullptr};
    size_t tok_cap = 0;
    // control block
    DevState *d_st = nullptr;
    DevState *h_st = nullptr;              // the latest copy of the control block (one of h_buf)
    DevState *h_buf[2] = {nullptr, nullptr}; // pinned
    cudaEvent_t poll_ev[2] = {nullptr, nullptr};
    // ranged layout: per buffer, length and edge tokens of every range
    u32 *d_rcnt[2] = {nullptr, nullptr};
    u32 *d_redge[2] = {nullptr, nullptr};
    int rmax = 296;
    // tile descriptors
    u64 *d_desc = nullptr;
    u32 *d_pdesc = nullptr;
    size_t desc_cap = 0;
    // delta vectors (+ edge-record header)
    int32_t *d_delta = nullptr;
    size_t delta_cap = 0;
    // pair table
    u64 *d_tkey = nullptr, *d_tmeta = nullptr;
    u64 tcap = 0;
    u32 *d_cflag = nullptr;  // candidate-membership bit per table slot
    struct Arena
    {
        u64 *key = nullptr, *meta = nullptr;
        u32 *cflag = nullptr;
        u64 cap = 0;
    } arena[2];
    int arena_cur = 0;
    double host_ms[6] = {0, 0, 0, 0, 0, 0}; // wall clock of host-side phases (debug): rehash, candidates, pause, poll wait, enqueue, setup
    u32 *d_cand = nullptr;   // candidate slots of the argmax (fixed capacity)
    SelPart *d_part = nullptr;
    u32 cand_T = 0;          // host copy of the list threshold we asked for (0 = whole-table selection)
    int batch_max = BATCH_MAX; // merges per pass (1 = off)
    int batch_min_z = -1;      // (-1: where the shared-memory delta histogram ends)
    bool run_encode = false;   // the current run applies a given merge list
    u64 run_max_merges = 0;    // its merge cap (0 = none)
    int ranges_opt = 0;      // test knob: number of ranges (0 = two per SM)
    int want_ranged = 0;     // this run uses the streaming kernel (RANGED layout) for its passes
    u32 list_retry_below = ~0u; // whole-table mode: try a list again once the best count is below this
    bool fresh_select = false;  // the candidate list ran empty: one whole-table selection must say what the maximum is now
                                // before any new list is chosen (the control block's `freq` is stale until then)
    bool debug = false;         // BPE_CUDA_DEBUG (read once per context)
    // logs
    u32 *d_merges = nullptr;
    u64 *d_nhist = nullptr;
    size_t merges_cap = 0;
    u32 *d_enc_merges = nullptr;
    size_t enc_cap = 0;
    // dense byte-pair histogram
    int sel_grid = 0;
    u32 *d_dense = nullptr;
    // exact tie-break machinery (bpe_resolver.cuh)
    ResState *d_rs = nullptr;
    u64 *d_first = nullptr;
    // decode: flattened vocabulary, tile offsets, output bytes
    u32 *d_dec_len = nullptr, *d_dec_off = nullptr;
    uint8_t *d_dec_blob = nullptr, *d_dec_out = nullptr;
    u64 *d_dec_tiles = nullptr;
    size_t dec_vocab_cap = 0, dec_blob_cap = 0, dec_out_cap = 0, dec_tiles_cap = 0, dec_n_out = 0;
    bool dec_valid = false;                 // the vocabulary on the device is the flattening of dec_merges
    std::vector<bpe_pair_t> dec_merges;
    // batch decode: the batch's ids and token offsets, first document per tile, byte offsets
    u32 *d_dbtok = nullptr, *d_dbtile = nullptr;
    u64 *d_dbtoff = nullptr, *d_dbboff = nullptr;
    size_t dbtok_cap = 0, dbtile_cap = 0, dbtoff_cap = 0, dbboff_cap = 0;
    u32 *d_rank = nullptr;
    size_t first_cap = 0; // entries (slots * slices)
    u32 *d_pos_slot = nullptr;
    size_t pos_cap = 0;
    u32 *d_tile_cnt = nullptr;
    u64 *d_tile_off = nullptr;
    size_t tile_cap = 0;
    // batch encode (bpe_encode_batch.cuh): buffers of its own, so the resident shard and the last run's results stay
    uint8_t *d_bb = nullptr;          // the batch's bytes
    u32 *d_btok = nullptr, *d_brk = nullptr; // per byte: ids at the document's offset / pair ranks; d_brk then holds the
                                      // compacted ids
    u64 *d_bdoc = nullptr, *d_btoff = nullptr; // per document: start, then count -> tok_offsets (n_docs + 1)
    u32 *d_blen = nullptr, *d_border = nullptr;
    u32 *d_bseg = nullptr, *d_bsegs = nullptr; // global tier: first segment per document; per segment: count, min rank
    size_t bb_cap = 0, btok_cap = 0, brk_cap = 0, bdoc_cap = 0, btoff_cap = 0, blen_cap = 0, border_cap = 0, bseg_cap = 0,
           bsegs_cap = 0;
    u64 *d_rt_key = nullptr;          // pair -> smallest rank (open addressing), kept for the next batch
    u32 *d_rt_rank = nullptr, *d_bnext = nullptr;
    size_t rt_key_cap = 0, rt_rank_cap = 0;
    u32 rt_mask = 0;
    bool rt_valid = false;
    std::vector<bpe_pair_t> rt_merges; // the list the table was built from
    uint2 *d_bmerges = nullptr;
    size_t bmerges_cap = 0;
    int cas_grid = 0;                 // persistent CTAs of batch_cascade_kernel (0: not set up yet)
    // communicator (bootstrap + the two collectives of a run's start) and the peer-memory exchange (struct Xchg)
    int rank = 0, world = 1;
    ncclComm_t comm = nullptr;
    bool solo = false;                // this run has been CONSOLIDATED: the global stream fell below 1,048,576 tokens, every
                                      // rank now holds all of it and runs the single-GPU algorithm (exact 16-slice census
                                      // and chain-order resolver); no exchange any more
    u32 *d_gather = nullptr;          // the whole stream on this rank, for the exact tie-break above the static limit
    size_t gather_cap = 0;
    Xchg hx{};                        // host copy of the exchange descriptor (goes into DevState at the start of a run)
    u32 xseq = 0;                     // exchanges completed so far (continues from run to run: the flags are never reset)
    size_t xcap_opt = 0;              // test knob: initial entries per inbox slot
    u64 x_timeout_ms = 20000;         // BPE_CUDA_XCHG_TIMEOUT_MS
    int agrid_max = 120;              // blocks of apply_select_kernel that fold deltas into the table (BPE_CUDA_AGRID_MAX)
    void *d_hello = nullptr;          // staging of the handle exchange
    std::vector<void *> x_owned;      // every inbox this context ever allocated (freed with the context: a peer may still
                                      // have an old one mapped)
    std::vector<void *> x_mapped;     // peers' inboxes opened through CUDA IPC
    // options
    int profile_replace = 0;
    int batch_steps = 64;
    int smem_hist_max_vocab = 448;  // ids below this: one merge per pass, deltas privatised in shared memory (7 KB); above: batched
                                    // passes with global RED.  Measured on config 2 (final batching rules): 320 -> 138.8 ms,
                                    // 448 -> 137.3, 512 -> 139.3, 640 -> 141.8 (with the first rules: 1792 -> 209, 640 -> 182)
    int replace_occ[2] = {0, 0};
    int stream_occ[2] = {0, 0}; // CTAs per SM of replace_stream_kernel<false>, <true> at the largest histogram
    // profiling events
    std::vector<cudaEvent_t> prof;
    std::vector<unsigned char> prof_tag;
    size_t prof_used = 0;
    // results
    size_t res_n_merges = 0, res_n_tokens = 0;
    bpe_cuda_stats_t stats;
    uint64_t launches = 0;
};

static inline size_t round_up(size_t x, size_t m) { return (x + m - 1) / m * m; }
// the stream of this run is cut into shards that exchange deltas and edge records
static inline bool sharded(const bpe_cuda_ctx *c) { return c->world > 1 && !c->solo; }
// Merges that may share one pass (the exchange between GPUs carries the touched counters only, so its cost does not
// depend on the batch size or the vocabulary: the same limit for every world size).
static inline size_t eff_batch(const bpe_cuda_ctx *c)
{
    return (size_t)std::max(1, std::min(c->batch_max, (int)BATCH_MAX));
}

struct HostTimer
{
    double *acc;
    std::chrono::steady_clock::time_point t0;
    explicit HostTimer(double *a) : acc(a), t0(std::chrono::steady_clock::now()) {}
    ~HostTimer() { *acc += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); }
};

static int ensure_bytes(bpe_cuda_ctx *c, size_t n)
{
    const size_t need = round_up(n, 16) + 64;
    if (need > c->bytes_cap)
    {
        if (c->d_bytes)
            CU(cudaFree(c->d_bytes));
        c->d_bytes = nullptr;
        CU(cudaMalloc(&c->d_bytes, need));
        c->bytes_cap = need;
    }
    return 0;
}

static int ensure_stream_buffers(bpe_cuda_ctx *c, size_t n)
{
    // 4 slots in front; behind: the streaming kernel copies whole tiles (+ halo) and the halos are written in place
    const size_t need = round_up(n, V_TILE) + V_TILE + 64;
    if (need > c->tok_cap)
    {
        for (int i = 0; i < 2; i++)
        {
            if (c->d_tok_alloc[i])
                CU(cudaFree(c->d_tok_alloc[i]));
            c->d_tok_alloc[i] = nullptr;
            CU(cudaMalloc(&c->d_tok_alloc[i], need * sizeof(u32)));
        }
        c->tok_cap = need;
    }
    const size_t tiles = n / R_TILE + 2;
    if (tiles > c->desc_cap)
    {
        if (c->d_desc)
            CU(cudaFree(c->d_desc));
        if (c->d_pdesc)
            CU(cudaFree(c->d_pdesc));
        c->d_desc = nullptr;
        c->d_pdesc = nullptr;
        CU(cudaMalloc(&c->d_desc, tiles * sizeof(u64)));
        CU(cudaMalloc(&c->d_pdesc, tiles * sizeof(u32)));
        c->desc_cap = tiles;
    }
    return 0;
}

// merges that may share one pass in this run (decides how far the device can run ahead of the host's id estimate)
static inline size_t eff_batch(const bpe_cuda_ctx *c);
// words of the delta buffer when ids up to z_ub exist: one block of 4 vectors per merge of a batch
static inline size_t delta_need(const bpe_cuda_ctx *c, size_t z_ub) { return HDR_INTS + eff_batch(c) * 4 * (z_ub + eff_batch(c) + 1); }

static int ensure_delta(bpe_cuda_ctx *c, size_t vocab)
{
    const size_t need = delta_need(c, vocab);
    if (need <= c->delta_cap)
        return 0;
    size_t cap = c->delta_cap ? c->delta_cap : (size_t)HDR_INTS + 4 * 8192;
    while (cap < need)
        cap *= 2;
    // the vectors are all-zero between steps and the stream is idle when this is called
    int32_t *nd = nullptr;
    CU(cudaMalloc(&nd, cap * sizeof(int32_t)));
    CU(cudaMemsetAsync(nd, 0, cap * sizeof(int32_t), c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (c->d_delta)
        CU(cudaFree(c->d_delta));
    c->d_delta = nd;
    c->delta_cap = cap;
    return 0;
}

// ---- peer-memory exchange: inbox allocation and the handle exchange (struct Xchg in bpe_kernels.cuh) ------------
// 256 Ki entries per (parity, sender) slot = 32 MB per rank; grown (ensure_xchg) when a pass could touch more counters
constexpr size_t XCAP_DEFAULT = 1u << 18;
struct XchgHello
{
    unsigned long long pid, ptr, xcap;
    int device, pad;
    cudaIpcMemHandle_t handle;
};

// Allocate an inbox of `xcap` entries per slot and learn every peer's.  Called by all ranks at the same point of
// their (replicated) host logic with their streams drained: from set_comm, and from ensure_xchg when the lists may
// outgrow the slots.  Ranks of one process (bpe_cuda_train with n_gpus > 1: one thread per GPU) use each other's
// pointers directly with peer access enabled; ranks in separate processes (one per GPU, e.g. under torchrun) map
// each other's inbox through CUDA IPC.  The handles travel through one ncclAllGather (bootstrap, not data path).
static int xchg_setup(bpe_cuda_ctx *c, size_t xcap)
{
    CU(cudaSetDevice(c->device));
    void *buf = nullptr;
    CU(cudaMalloc(&buf, xchg_bytes(xcap)));
    c->x_owned.push_back(buf);
    CU(cudaMemsetAsync(buf, 0, xchg_bytes(xcap), c->stream));
    if (c->hx.local) // flags, counts and edge records of the exchanges so far stay valid
        CU(cudaMemcpyAsync(buf, c->hx.local, XCHG_HDR_WORDS * sizeof(u32), cudaMemcpyDeviceToDevice, c->stream));
    XchgHello mine;
    memset(&mine, 0, sizeof mine);
    mine.pid = (unsigned long long)getpid();
    mine.ptr = (unsigned long long)buf;
    mine.xcap = xcap;
    mine.device = c->device;
    CU(cudaIpcGetMemHandle(&mine.handle, buf));
    if (!c->d_hello)
        CU(cudaMalloc(&c->d_hello, MAX_RANKS * sizeof(XchgHello)));
    char *hello = static_cast<char *>(c->d_hello);
    CU(cudaMemcpyAsync(hello + (size_t)c->rank * sizeof mine, &mine, sizeof mine, cudaMemcpyHostToDevice, c->stream));
    NC(g_nccl.AllGather(hello + (size_t)c->rank * sizeof mine, hello, sizeof mine, ncclChar, c->comm, c->stream));
    std::vector<XchgHello> all((size_t)c->world);
    CU(cudaMemcpyAsync(all.data(), hello, (size_t)c->world * sizeof mine, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    Xchg nx{};
    nx.local = static_cast<u32 *>(buf);
    nx.xcap = xcap;
    for (int r = 0; r < c->world; r++)
    {
        const XchgHello &h = all[(size_t)r];
        if (h.xcap != xcap)
        {
            set_error("exchange setup: rank %d allocated %llu entries per slot, rank %d %zu (ranks out of step)", r, h.xcap, c->rank, xcap);
            return BPE_CUDA_ERR_STATE;
        }
        if (r == c->rank)
            nx.peer[r] = nx.local;
        else if (h.pid == mine.pid)
        {
            int can = 0;
            CU(cudaDeviceCanAccessPeer(&can, c->device, h.device));
            if (!can)
            {
                set_error("device %d cannot access device %d's memory (no NVLink / PCIe peer path)", c->device, h.device);
                return BPE_CUDA_ERR_CUDA;
            }
            const cudaError_t e = cudaDeviceEnablePeerAccess(h.device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
            {
                set_error("cudaDeviceEnablePeerAccess(%d) from device %d: %s", h.device, c->device, cudaGetErrorString(e));
                return BPE_CUDA_ERR_CUDA;
            }
            cudaGetLastError();
            nx.peer[r] = reinterpret_cast<u32 *>(h.ptr);
        }
        else
        {
            void *p = nullptr;
            CU(cudaIpcOpenMemHandle(&p, h.handle, cudaIpcMemLazyEnablePeerAccess));
            c->x_mapped.push_back(p);
            nx.peer[r] = static_cast<u32 *>(p);
        }
    }
    c->hx = nx;
    // (a run in progress reads the descriptor from its control block)
    CU(cudaMemcpyAsync(&c->d_st->x, &c->hx, sizeof(Xchg), cudaMemcpyHostToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

// Entries one pass can put into a slot: a counter per (merge of the batch, vector, token id), and no more than four
// per replacement - the best count never grows (SURVEY.md A.5.4), so `freq_bound` (the count of the last committed
// merge, 0 = unknown) bounds every later merge's replacements.  Every rank calls this with the same arguments.
static int ensure_xchg(bpe_cuda_ctx *c, size_t z_ub, u64 freq_bound)
{
    if (!sharded(c))
        return 0;
    const size_t bm = eff_batch(c);
    size_t need = bm * 4 * (z_ub + bm + 1);
    if (freq_bound)
        need = (size_t)std::min<u64>(need, 4ull * bm * freq_bound);
    if (need <= c->hx.xcap)
        return 0;
    size_t cap = (size_t)c->hx.xcap;
    while (cap < need)
        cap *= 2;
    if (c->debug)
        fprintf(stderr, "[bpe_cuda r%d] exchange inbox grows to %zu entries per slot\n", c->rank, cap);
    return xchg_setup(c, cap);
}

static int ensure_logs(bpe_cuda_ctx *c, size_t merges)
{
    if (merges <= c->merges_cap)
        return 0;
    size_t cap = c->merges_cap ? c->merges_cap : 8192;
    while (cap < merges)
        cap *= 2;
    u32 *nm = nullptr;
    u64 *nh = nullptr;
    CU(cudaMalloc(&nm, cap * 2 * sizeof(u32)));
    CU(cudaMalloc(&nh, (cap + 1) * sizeof(u64)));
    if (c->d_merges)
    {
        CU(cudaMemcpyAsync(nm, c->d_merges, c->merges_cap * 2 * sizeof(u32), cudaMemcpyDeviceToDevice, c->stream));
        CU(cudaMemcpyAsync(nh, c->d_nhist, (c->merges_cap + 1) * sizeof(u64), cudaMemcpyDeviceToDevice, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        CU(cudaFree(c->d_merges));
        CU(cudaFree(c->d_nhist));
    }
    c->d_merges = nm;
    c->d_nhist = nh;
    c->merges_cap = cap;
    // the control block holds the pointers
    CU(cudaMemcpyAsync(&c->d_st->merges, &c->d_merges, sizeof(u32 *), cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(&c->d_st->n_hist, &c->d_nhist, sizeof(u64 *), cudaMemcpyHostToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

constexpr u32 CAND_CAP = 65536;

// Pair-table memory comes from two arenas that only ever grow and live as long as the context: a
// rehash builds the new table in the arena the current one does not use.  (cudaMalloc / cudaFree
// inside a run cost milliseconds and synchronise the device.)
typedef bpe_cuda_ctx::Arena TableMem;

static int table_alloc(bpe_cuda_ctx *c, u64 cap, int arena)
{
    TableMem &t = c->arena[arena];
    if (t.cap < cap)
    {
        cudaFree(t.key); // one allocation: keys, then meta, then the candidate bits
        t = TableMem();
        CU(cudaMalloc(&t.key, cap * 2 * sizeof(u64) + cap / 8));
        t.cap = cap;
    }
    // (the sub-arrays are placed for the capacity in use, so that the live table is one contiguous window)
    t.meta = t.key + cap;
    t.cflag = reinterpret_cast<u32 *>(t.meta + cap);
    CU(cudaMemsetAsync(t.key, 0xFF, cap * sizeof(u64), c->stream));
    CU(cudaMemsetAsync(t.meta, 0, cap * sizeof(u64) + cap / 8, c->stream));
    return 0;
}

static void table_free(bpe_cuda_ctx *c)
{
    for (int i = 0; i < 2; i++)
    {
        cudaFree(c->arena[i].key);
        c->arena[i] = TableMem();
    }
    c->d_tkey = c->d_tmeta = nullptr;
    c->d_cflag = nullptr;
}

static void table_adopt(bpe_cuda_ctx *c, int arena, u64 cap)
{
    c->arena_cur = arena;
    c->d_tkey = c->arena[arena].key;
    c->d_tmeta = c->arena[arena].meta;
    c->d_cflag = c->arena[arena].cflag;
    c->tcap = cap;
}

static int table_rehash(bpe_cuda_ctx *c, u64 new_cap)
{
    HostTimer ht(&c->host_ms[0]);
    const int other = c->arena_cur ^ 1;
    int rc = table_alloc(c, new_cap, other);
    if (rc)
        return rc;
    const TableMem &t = c->arena[other];
    const int grid = (int)std::min<u64>((c->tcap + 255) / 256, (u64)c->sm_count * 8);
    rehash_kernel<<<grid, 256, 0, c->stream>>>(c->d_tkey, c->d_tmeta, c->tcap, t.key, t.meta, new_cap, &c->d_st->err);
    table_swap_kernel<<<1, 1, 0, c->stream>>>(c->d_st, t.key, t.meta, new_cap, t.cflag);
    c->launches += 2;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(c->stream));
    table_adopt(c, other, new_cap);
    c->stats.table_rehashes++;
    return 0;
}

static int check_state(bpe_cuda_ctx *c)
{
    if (c->debug)
        fprintf(stderr, "[bpe_cuda r%d] merges=%llu n=%llu n_global=%llu D=%lld occ=%llu cap=%llu stop=%u pause=%u static=%u err=%u a=%u b=%u f=%u mult=%u\n",
                c->rank, c->h_st->merges_done, c->h_st->n, c->h_st->n_global, c->h_st->distinct, c->h_st->occupied, c->h_st->tcap,
                c->h_st->stop, c->h_st->pause, c->h_st->static_mode, c->h_st->err, c->h_st->a, c->h_st->b, c->h_st->freq,
                c->h_st->sel_mult),
        fprintf(stderr, "            layout=%u nr=%u pending=%u cand_T=%u ncand=%u\n", c->h_st->layout, c->h_st->nr, c->h_st->pending,
                c->h_st->cand_T, c->h_st->ncand);
    if (c->h_st->err)
    {
        set_error("device reported error flags 0x%x (1=table full 2=missing key 4=negative count 8=probe/logic 16=exchange slot overflow 32=peer flag timeout)", c->h_st->err);
        return BPE_CUDA_ERR_STATE;
    }
    return 0;
}

static int poll_state(bpe_cuda_ctx *c)
{
    c->h_st = c->h_buf[0];
    CU(cudaMemcpyAsync(c->h_st, c->d_st, sizeof(DevState), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return check_state(c);
}

// ---------------------------------------------------------------------------------------------
static size_t replace_smem_bytes(bool hist, u32 z) { return (R_TILE + 8) * sizeof(u32) + (hist ? 16 * ((size_t)z + 1) : 0); }

static int setup_kernels(bpe_cuda_ctx *c)
{
    {
        u64 thr[THR_ENTRIES];
        for (int i = 0; i < THR_ENTRIES; i++)
            thr[i] = resize_threshold_exact(1ull << (THR_LOG2_MIN + i));
        CU(cudaMemcpyToSymbol(c_resize_thr, thr, sizeof thr));
    }
    CU(cudaFuncSetAttribute(replace_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    CU(cudaFuncSetAttribute(replace_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    CU(cudaFuncSetAttribute(widen_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    int occ = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, replace_kernel<false>, R_THREADS, replace_smem_bytes(false, 0)));
    c->replace_occ[0] = std::max(1, occ);
    CU(cudaFuncSetAttribute(replace_stream_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    CU(cudaFuncSetAttribute(replace_stream_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, replace_stream_kernel<false>, V_THREADS, stream_smem_bytes(false, 0)));
    c->stream_occ[0] = std::max(1, occ);
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, replace_stream_kernel<true>, V_THREADS,
                                                     stream_smem_bytes(true, (u32)std::max(1, c->smem_hist_max_vocab) - 1)));
    c->stream_occ[1] = std::max(1, occ);
    return 0;
}

// scratch of the census / resolver: first position and first-sight rank per (table slot, slice),
// table slot per stream position, scan scratch.  Stamped with a census epoch, never cleared.
static int ensure_resolver(bpe_cuda_ctx *c, u64 n, u32 slices)
{
    if (!c->d_rs)
    {
        CU(cudaMalloc(&c->d_rs, sizeof(ResState)));
        CU(cudaMemsetAsync(c->d_rs, 0, sizeof(ResState), c->stream));
    }
    const size_t ent = (size_t)c->tcap * slices;
    if (ent > c->first_cap)
    {
        if (c->d_first)
            CU(cudaFree(c->d_first));
        if (c->d_rank)
            CU(cudaFree(c->d_rank));
        c->d_first = nullptr;
        c->d_rank = nullptr;
        CU(cudaMalloc(&c->d_first, ent * sizeof(u64)));
        CU(cudaMalloc(&c->d_rank, ent * sizeof(u32)));
        CU(cudaMemsetAsync(c->d_first, 0, ent * sizeof(u64), c->stream));
        c->first_cap = ent;
    }
    if (n + 16 > c->pos_cap)
    {
        if (c->d_pos_slot)
            CU(cudaFree(c->d_pos_slot));
        c->d_pos_slot = nullptr;
        CU(cudaMalloc(&c->d_pos_slot, (n + 16) * sizeof(u32)));
        c->pos_cap = n + 16;
    }
    const size_t tiles = n / SCAN_TILE + 2;
    if (tiles > c->tile_cap)
    {
        if (c->d_tile_cnt)
            CU(cudaFree(c->d_tile_cnt));
        if (c->d_tile_off)
            CU(cudaFree(c->d_tile_off));
        c->d_tile_cnt = nullptr;
        c->d_tile_off = nullptr;
        CU(cudaMalloc(&c->d_tile_cnt, tiles * sizeof(u32)));
        CU(cudaMalloc(&c->d_tile_off, tiles * sizeof(u64)));
        c->tile_cap = tiles;
    }
    return 0;
}

// Launch with the programmatic-stream-serialization attribute (see pdl_wait in bpe_kernels.cuh): the step kernels
// follow one another, so each may be scheduled while its predecessor drains.
template <typename... KArgs, typename... Args>
static cudaError_t launch_chained(bpe_cuda_ctx *c, void (*kernel)(KArgs...), int grid, int block, size_t smem, Args... args)
{
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = c->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// profiling marks: the interval that ends at a mark is charged to the mark's class
enum
{
    PT_GAP = 0,
    PT_SELECT = 1,
    PT_REPLACE = 2,
    PT_APPLY = 3
};
static inline void prof_mark(bpe_cuda_ctx *c, int tag)
{
    if (!c->profile_replace || c->prof_used >= c->prof.size())
        return;
    c->prof_tag[c->prof_used] = (unsigned char)tag;
    cudaEventRecord(c->prof[c->prof_used++], c->stream);
}

static int pos_grid(bpe_cuda_ctx *c, u64 n) { return (int)std::max<u64>(1, std::min<u64>((n + 255) / 256, (u64)c->sm_count * 8)); }

// the 16-slice distinct-pair census that keeps the worker tables' bucket counts exact
static int enqueue_census(bpe_cuda_ctx *c, u64 n_upper, int resolver)
{
    const int g = pos_grid(c, n_upper);
    census_begin_kernel<<<1, 1, 0, c->stream>>>(c->d_st, c->d_rs, resolver);
    census_mark_kernel<<<g, 256, 0, c->stream>>>(c->d_st, c->d_rs, c->d_first, c->d_pos_slot);
    census_count_kernel<<<g, 256, 0, c->stream>>>(c->d_st, c->d_rs, c->d_first, c->d_pos_slot);
    census_update_kernel<<<1, 1, 0, c->stream>>>(c->d_st, c->d_rs);
    c->launches += 4;
    return 0;
}

// ---- argmax candidates ---------------------------------------------------------------------------
// (re)build the list of table slots whose count is >= T; T == 0 switches to whole-table selection
static int rebuild_candidates(bpe_cuda_ctx *c, u32 T)
{
    CU(cudaMemsetAsync(c->d_cflag, 0, c->tcap / 8, c->stream));
    cand_reset_kernel<<<1, 1, 0, c->stream>>>(c->d_st);
    c->launches++;
    if (T)
    {
        const int grid = (int)std::min<u64>((c->tcap + 255) / 256, (u64)c->sm_count * 8);
        cand_rebuild_kernel<<<grid, 256, 0, c->stream>>>(c->d_st, T);
        c->launches++;
    }
    c->cand_T = T;
    CU(cudaGetLastError());
    return 0;
}

// Pick the threshold from the best count seen: the list then holds every pair within a factor two of
// the maximum, and stays valid until the maximum itself has halved.  Tiny counts (many ties, lists as
// long as the table) and overflowing lists fall back to whole-table selection.
static int choose_candidates(bpe_cuda_ctx *c, u32 best)
{
    HostTimer ht(&c->host_ms[1]);
    int rc;
    if (best >= 8)
    {
        // Start at half the maximum and move the threshold up until the list fits the registers of the
        // selecting block (CAND_TARGET leaves room for the pairs that will cross the threshold later); a
        // threshold closer to the maximum is outlived sooner, so stop at 15/16.  If the counts are too flat
        // for that, any list that fits the buffer will do (whole-list gathers, no batches).
        u32 T = best / 2, T_usable = 0, T_small = 0;
        int downs = 0;
        for (int tries = 0; tries < 4 && T < best && T >= 4;)
        {
            if ((rc = rebuild_candidates(c, T)))
                return rc;
            if ((rc = poll_state(c)))
                return rc;
            const bool usable = !c->h_st->cand_overflow && c->h_st->ncand <= CAND_CAP / 2;
            if (c->debug)
                fprintf(stderr, "[bpe_cuda] candidate list: best %u threshold %u -> %u entries%s\n", best, T, c->h_st->ncand,
                        c->h_st->cand_overflow ? " (overflow)" : "");
            if (c->h_st->ncand == 0)
            {
                // Nothing reaches T: `best` did not describe the table (the maximum has dropped by more than half
                // since it was read).  An empty list can never be accepted - the next selection would find nothing,
                // ask for a rebuild and land here again: whole-table selection until a real maximum is known.
                if (T_small)
                    break;
                c->list_retry_below = T;
                if ((rc = rebuild_candidates(c, 0)))
                    return rc;
                return poll_state(c);
            }
            if (usable && c->h_st->ncand <= CAND_TARGET)
            {
                // a list of a handful of pairs (steep counts: the first merges of a byte-level corpus) is used up
                // after a few merges and costs a pause each time: look further down while the list stays small
                if (c->h_st->ncand >= 128 || downs >= 3 || tries > 0 || T < 64)
                    return 0;
                T_small = T;
                T /= 4;
                downs++;
                continue;
            }
            if (T_small)
                break; // one step too far down: the previous (short) list it is
            if (usable && !T_usable)
                T_usable = T; // the lowest threshold whose list fits the buffer: it lives longest
            T += (best - T + 1) / 2;
            tries++;
        }
        if (T_small)
        {
            if ((rc = rebuild_candidates(c, T_small)))
                return rc;
            return poll_state(c);
        }
        if (T_usable)
        {
            if ((rc = rebuild_candidates(c, T_usable)))
                return rc;
            cand_big_ok_kernel<<<1, 1, 0, c->stream>>>(c->d_st);
            c->launches++;
            return poll_state(c);
        }
    }
    c->list_retry_below = best / 2;
    if ((rc = rebuild_candidates(c, 0)))
        return rc;
    return poll_state(c);
}

// K2 alone (no deltas pending): start of a run, after a pause that did not commit a merge
static int enqueue_select(bpe_cuda_ctx *c, bool encode)
{
    if (encode)
        apply_select_kernel<<<2, SEL_THREADS, 0, c->stream>>>(c->d_st, c->d_delta, AS_ENCODE);
    else if (c->cand_T == 0)
        select_kernel<<<c->sel_grid, SEL_THREADS, 0, c->stream>>>(c->d_st, c->d_part);
    else
        apply_select_kernel<<<2, SEL_THREADS, 0, c->stream>>>(c->d_st, c->d_delta, AS_TRAIN);
    c->launches++;
    return 0;
}

// One merge step for the committed merge that creates id z: [census] -> replace (+scan+deltas) ->
// [edge record, ncclAllReduce] -> apply deltas + select the next merge.
static int enqueue_step(bpe_cuda_ctx *c, u32 z, u64 n_upper, bool encode, bool census, bool ranged, u64 z_ub = 0)
{
    if (z_ub < z)
        z_ub = z;
    prof_mark(c, PT_GAP);
    if (census)
    {
        int rc = enqueue_census(c, n_upper, 0);
        if (rc)
            return rc;
        c->stats.census_runs++;
    }
    const bool hist = ((int)z + 1 <= c->smem_hist_max_vocab);
    if (ranged)
    {
        // RANGED stream: one CTA per range (a == b runs same_pair_range inside the same kernel)
        // the histogram always gets its full budget: the device may be ahead of this id estimate, or batch merges
        const size_t vsmem = stream_smem_bytes(hist, hist ? (u32)c->smem_hist_max_vocab - 1 : 0);
        if (hist)
            CU(launch_chained(c, replace_stream_kernel<true>, c->rmax, V_THREADS, vsmem, c->d_st, c->d_delta,
                              (u32)(4 * c->smem_hist_max_vocab)));
        else
            CU(launch_chained(c, replace_stream_kernel<false>, c->rmax, V_THREADS, vsmem, c->d_st, c->d_delta, 0u));
    }
    else
    {
        const size_t smem = replace_smem_bytes(hist, z);
        int occ = c->replace_occ[0];
        if (hist)
        {
            const size_t per_sm = 220 * 1024;
            occ = (int)std::max<size_t>(1, std::min<size_t>((size_t)occ, per_sm / (smem + 1024)));
        }
        const u64 tiles = std::max<u64>(1, (n_upper + R_TILE - 1) / R_TILE);
        const int grid = (int)std::min<u64>(tiles, (u64)c->sm_count * (u64)occ);
        if (hist)
            replace_kernel<true><<<grid, R_THREADS, smem, c->stream>>>(c->d_st, c->d_desc, c->d_pdesc, c->d_delta);
        else
            replace_kernel<false><<<grid, R_THREADS, smem, c->stream>>>(c->d_st, c->d_desc, c->d_pdesc, c->d_delta);
    }
    prof_mark(c, PT_REPLACE);
    c->launches++;
    c->stats.replace_launches++;
    // every thread looks at one token's four counters (128 bits) per trip; 32 blocks keep the "last block" wait short
    // (batches are mostly short: size the grid for two merges, the loop is grid-stride).  Several GPUs: the same
    // launch pushes this rank's touched counters into the peers' inboxes and folds theirs in (struct Xchg).
    // (a thread takes one token's four counters per trip: aim at two trips for a pass of four merges; at least 64
    // blocks - few chains per thread - and at most 120, so that the whole grid is resident next to the pass kernel)
    const int agrid = (int)std::max<u64>(64, std::min<u64>((std::min<u64>(eff_batch(c), 4) * (u64)(z + 1)) / (2 * SEL_THREADS), (u64)c->agrid_max));
    if (encode || c->cand_T)
    {
        CU(launch_chained(c, apply_select_kernel, agrid + 1, SEL_THREADS, 0, c->d_st, c->d_delta, encode ? (int)AS_ENCODE : (int)AS_TRAIN));
        c->launches++;
        prof_mark(c, PT_APPLY);
    }
    else
    {
        if (sharded(c))
            CU(launch_chained(c, apply_select_kernel, agrid + 1, SEL_THREADS, 0, c->d_st, c->d_delta, (int)AS_APPLY_ONLY));
        else
        {
            const int g1 = (int)std::min<u64>((4ull * (z + 1) + 255) / 256, (u64)c->sm_count * 4);
            apply_kernel<<<g1, 256, 0, c->stream>>>(c->d_st, c->d_delta);
        }
        prof_mark(c, PT_APPLY);
        select_kernel<<<c->sel_grid, SEL_THREADS, 0, c->stream>>>(c->d_st, c->d_part);
        c->launches += 2;
        prof_mark(c, PT_SELECT);
    }
    return 0;
}

// ---- the host side of the loop -------------------------------------------------------------------
// The host never takes part in a merge step; it enqueues steps in batches and looks at the control
// block once per batch.  To keep the GPU fed while the host looks (or is descheduled), the NEXT batch
// is enqueued before the poll of the current one is waited for: it is planned on the assumption
// that the current batch runs to its end, and if that batch stops or pauses instead, every kernel of
// the speculative batch falls through (they all test the control block first).
struct BatchPlan
{
    u64 m1 = 0;     // merges_done the batch starts from
    u64 z0 = 0;     // id created by its first pass
    u64 G = 0;      // steps
    u64 n_upper = 0;
    u64 margin = 0; // table slots it may claim
    u64 zub0 = 0;   // upper bound of the id created by its first pass (the device may be ahead of z0)
    bool pending = false, census = false, ranged = false;
};

// table slots a batch of G steps may claim: every replacement creates at most two new pair instances, and a
// pass replaces at most bm * freq occurrences (the best count never grows, SURVEY.md A.5.4)
static u64 batch_margin(u64 G, u64 z0, u64 bm, u64 freq)
{
    const u64 per_merge = std::min<u64>(2 * (z0 + G * bm + 1), freq ? 2 * freq : ~0ull);
    return G * bm * per_merge;
}

static u64 batch_steps_for(bpe_cuda_ctx *c, const DevState *h, bool encode, u64 m1, u64 z0)
{
    u64 G = (u64)std::max(1, c->batch_steps);
    if (!encode && h->max_merges != ~0ull)
        G = (h->max_merges + 1 > m1) ? std::min<u64>(G, h->max_merges - m1 + 1) : 0;
    if (encode)
        G = (h->enc_total + 1 > m1) ? std::min<u64>(G, h->enc_total - m1 + 1) : 0;
    while (G > 4 && batch_margin(G, z0, eff_batch(c), encode ? 0 : h->freq) > c->tcap / 4)
        G /= 2;
    return G;
}

static int enqueue_batch(bpe_cuda_ctx *c, const BatchPlan &p, bool encode)
{
    HostTimer ht(&c->host_ms[4]);
    int rc;
    if (!p.pending && (rc = enqueue_select(c, encode)))
        return rc;
    for (u64 g = 0; g < p.G; g++)
        if ((rc = enqueue_step(c, (u32)(p.z0 + g), p.n_upper, encode, p.census, p.ranged, p.zub0 + (g + 1) * eff_batch(c))))
            return rc;
    CU(cudaGetLastError());
    return 0;
}

static int poll_async(bpe_cuda_ctx *c, int slot)
{
    CU(cudaMemcpyAsync(c->h_buf[slot], c->d_st, sizeof(DevState), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaEventRecord(c->poll_ev[slot], c->stream));
    return 0;
}

static int poll_wait(bpe_cuda_ctx *c, int slot)
{
    HostTimer ht(&c->host_ms[3]);
    CU(cudaEventSynchronize(c->poll_ev[slot]));
    c->h_st = c->h_buf[slot];
    return check_state(c);
}

// Same-bucket ties / exact-threshold iterations / layout changes / candidate rebuilds.
static int resolve_pause(bpe_cuda_ctx *c, bool encode);
static int consolidate(bpe_cuda_ctx *c);

static int run_loop(bpe_cuda_ctx *c, bool encode)
{
    int rc;
    c->list_retry_below = ~0u;
    c->fresh_select = false;
    if ((rc = poll_state(c)))
        return rc;
    // watchdog: every trip through this loop must commit a merge (or a rank) sooner or later; a run of trips
    // that leaves merges_done where it was is a host-side logic error and must end as one, not spin
    u64 wd_merges = ~0ull;
    int wd_trips = 0;
    for (;;)
    {
        // ---- the queue is drained and c->h_st is current
        DevState *h = c->h_st;
        if (h->stop == STOP_DONE)
            break;
        if (h->merges_done != wd_merges)
        {
            wd_merges = h->merges_done;
            wd_trips = 0;
        }
        else if (++wd_trips > 24)
        {
            set_error("no progress after %d host round trips at merge %llu (stop %u pause 0x%x pending %u list threshold %u, "
                      "%u candidates, best count %u)", wd_trips, (unsigned long long)h->merges_done, h->stop, h->pause, h->pending,
                      h->cand_T, h->ncand, (u32)(h->sel_key >> 32));
            return BPE_CUDA_ERR_STATE;
        }
        if (h->stop == STOP_PAUSE)
        {
            if ((rc = resolve_pause(c, encode)))
                return rc;
            if ((rc = poll_state(c)))
                return rc;
            continue;
        }
        if (!encode && !h->pending && (h->merges_done == 0 || c->fresh_select))
        {
            // The very first selection, or the first one after the candidate list ran empty: on the whole table.
            // Only its count says what the maximum is now, so only it may size the next candidate list (the
            // control block's `freq` still holds the count of the last COMMITTED merge, bpe.c:737-743).
            c->fresh_select = false;
            if ((rc = ensure_logs(c, (size_t)h->merges_done + 2)))
                return rc;
            if (c->cand_T && (rc = rebuild_candidates(c, 0)))
                return rc;
            if ((rc = enqueue_select(c, encode)))
                return rc;
            CU(cudaGetLastError());
            if ((rc = poll_state(c)))
                return rc;
            if (!(c->h_st->stop == STOP_RUN && c->h_st->pending))
                continue; // stopped or paused instead of committing
            if ((rc = choose_candidates(c, c->h_st->freq)))
                return rc;
            h = c->h_st;
        }
        BatchPlan X;
        X.m1 = h->merges_done;
        X.pending = h->pending != 0;
        X.z0 = 256 + X.m1 - (X.pending ? 1 : 0);
        X.zub0 = X.z0;
        X.G = batch_steps_for(c, h, encode, X.m1, X.z0);
        const u64 bm = eff_batch(c);
        X.margin = batch_margin(X.G, X.z0, bm, encode ? 0 : h->freq);
        X.n_upper = h->n;
        // table growth: bounded by the headroom two batches may consume (<= 2*(V+1) new keys a step)
        if (h->occupied + 2 * X.margin > c->tcap / 2 + c->tcap / 8)
        {
            u64 want = 1ull << 20;
            while (want < 3 * ((u64)h->distinct + 2 * X.margin))
                want *= 2;
            if ((rc = table_rehash(c, want)))
                return rc;
            if (c->cand_T && (rc = choose_candidates(c, std::max<u32>(h->freq, 2 * c->cand_T))))
                return rc;
            if ((rc = poll_state(c)))
                return rc;
            continue;
        }
        const u64 batch = (u64)std::max(1, c->batch_steps);
        if ((rc = ensure_delta(c, (size_t)(X.z0 + 3 * batch * bm + 4))))
            return rc;
        if ((rc = ensure_xchg(c, (size_t)(X.z0 + 3 * batch * bm + 4), (!encode && h->merges_done) ? h->freq : 0)))
            return rc;
        if ((rc = ensure_logs(c, (size_t)(X.m1 + 3 * batch * bm + 4))))
            return rc;
        u64 z_ub = X.z0 + X.G * bm, m_ub = X.m1 + X.G * bm; // how far the device may have got when X is done
        // candidate list upkeep: try a list when selection runs on the whole table, shrink a bloated one
        if (!encode)
        {
            const u32 T0 = c->cand_T;
            if (T0 == 0 && h->pending && h->freq >= 16 && h->freq < c->list_retry_below)
                rc = choose_candidates(c, h->freq); // (pending: `freq` is the count of a merge that is still in the table)
            else if (T0 && (h->cand_overflow || h->ncand > CAND_CAP * 3 / 4))
                rc = choose_candidates(c, std::max<u32>(h->freq, T0 + 1));
            if (rc)
                return rc;
            h = c->h_st;
        }
        // Worker-table growth is only possible while some slice can still hold thr(B_t) distinct pairs.
        // (every rank must take the same decisions about what it enqueues - the collectives have to
        // match - so anything that steers the batch structure looks at replicated state only)
        const bool stat = (sharded(c) ? h->n_global : h->n) < STATIC_LIMIT;
        if (!encode && !sharded(c))
        {
            if (stat)
            {
                const u64 dmax = (u64)h->distinct + X.margin;
                for (int t = 0; t < REF_THREADS; t++)
                    if (std::min<u64>(h->n / REF_THREADS + 32, dmax) >= resize_threshold(h->bt[t]))
                        X.census = true;
            }
            if (X.census && (rc = ensure_resolver(c, h->n, stat ? REF_THREADS : 1)))
                return rc;
        }
        // The streaming kernel works on the RANGED layout; everything that needs positions in one dense
        // array (static regime, census) keeps the stream dense and uses the general kernel.
        X.ranged = c->want_ranged && !X.census && !h->static_mode && h->n > 0;
        if (X.ranged && h->layout == LAYOUT_DENSE)
        {
            partition_kernel<<<1, RANGE_MAX, 0, c->stream>>>(c->d_st);
            c->launches++;
        }
        else if (!X.ranged && h->layout == LAYOUT_RANGED)
        {
            repack_kernel<<<RANGE_MAX, 1024, 0, c->stream>>>(c->d_st);
            c->launches++;
        }
        if ((rc = enqueue_batch(c, X, encode)))
            return rc;
        // ---- one batch in flight, its poll pending in slot ps
        DevState snap = *h; // the state X was planned from (a copy: the pinned buffers are rewritten by the polls)
        const DevState *prev = &snap;
        u64 occ_bound = snap.occupied + X.margin;
        int ps = 0;
        if ((rc = poll_async(c, ps)))
            return rc;
        for (;;)
        {
            BatchPlan Y;
            Y.m1 = X.m1 + X.G;
            Y.z0 = X.z0 + X.G;
            Y.zub0 = z_ub;
            Y.pending = true;
            Y.G = batch_steps_for(c, prev, encode, Y.m1, Y.z0);
            Y.margin = batch_margin(Y.G, Y.z0, bm, encode ? 0 : prev->freq);
            Y.n_upper = X.n_upper;
            Y.census = false;
            Y.ranged = X.ranged;
            const bool spec = Y.G > 0 && !X.census && !stat && !prev->static_mode &&
                              (encode || prev->n_global >= STATIC_LIMIT) &&
                              occ_bound + Y.margin <= c->tcap / 2 + c->tcap / 8 &&
                              delta_need(c, z_ub + Y.G * bm + 2) <= c->delta_cap && m_ub + Y.G * bm + 2 <= c->merges_cap;
            if (spec)
            {
                if ((rc = enqueue_batch(c, Y, encode)))
                    return rc;
                if ((rc = poll_async(c, ps ^ 1)))
                    return rc;
            }
            if ((rc = poll_wait(c, ps)))
                return rc;
            if (!spec)
                break;
            if (c->h_st->stop != STOP_RUN)
            {
                // X stopped or paused: Y fell through; drain it and handle the state it left
                if ((rc = poll_wait(c, ps ^ 1)))
                    return rc;
                break;
            }
            snap = *c->h_st;
            occ_bound = snap.occupied + Y.margin;
            X = Y;
            // the poll tells where the device really is; re-anchor the plan on it
            X.m1 = snap.merges_done;
            X.z0 = 256 + X.m1 - (snap.pending ? 1 : 0);
            X.zub0 = X.z0;
            z_ub = X.z0 + X.G * bm;
            m_ub = X.m1 + X.G * bm;
            ps ^= 1;
        }
    }
    if (c->h_st->layout == LAYOUT_RANGED)
    {
        repack_kernel<<<RANGE_MAX, 1024, 0, c->stream>>>(c->d_st);
        c->launches++;
        CU(cudaGetLastError());
        if ((rc = poll_state(c)))
            return rc;
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------
static int init_state(bpe_cuda_ctx *c, u64 n_local, u64 max_merges, size_t enc_total)
{
    DevState s;
    memset(&s, 0, sizeof s);
    s.tok[0] = c->d_tok_alloc[0] + 4;
    s.tok[1] = c->d_tok_alloc[1] + 4;
    s.tok_real[0] = s.tok[0];
    s.tok_real[1] = s.tok[1];
    s.cur = 0;
    s.epoch = 1;
    s.n = n_local;
    s.n_global = n_local;
    s.max_merges = max_merges ? max_merges : ~0ull;
    s.tkey = c->d_tkey;
    s.tmeta = c->d_tmeta;
    s.tcap = c->tcap;
    s.cand = c->d_cand;
    s.cflag = c->d_cflag;
    s.cand_cap = CAND_CAP;
    s.cand_T = 0;
    s.halo_before[0] = s.halo_before[1] = SENT;
    s.halo_after[0] = s.halo_after[1] = s.halo_after[2] = SENT;
    s.rank = (u32)c->rank;
    s.world = (u32)c->world;
    s.x = c->hx;
    s.xseq = c->xseq;
    s.x_timeout_ns = c->x_timeout_ms * 1000000ull;
    for (int t = 0; t < REF_THREADS; t++)
        s.bt[t] = 256; // bpe.c:610,615
    s.merges = c->d_merges;
    s.n_hist = c->d_nhist;
    s.enc_merges = c->d_enc_merges;
    s.enc_total = enc_total;
    s.static_mode = 0;
    c->want_ranged = (u64)c->n_bytes * (u64)c->world >= STATIC_LIMIT;
    s.want_ranged = (u32)c->want_ranged;
    s.batch_max = (u32)eff_batch(c);
    s.hist_max = (u32)std::max(0, c->smem_hist_max_vocab);
    s.hist_words = 4 * s.hist_max;
    s.batch_min_z = c->batch_min_z >= 0 ? (u32)c->batch_min_z : s.hist_max;
    s.nb = 1;
    s.layout = s.layout_next = LAYOUT_DENSE;
    s.rmax = (u32)c->rmax;
    for (int i = 0; i < 2; i++)
    {
        s.rcnt[i] = c->d_rcnt[i];
        s.redge[i] = c->d_redge[i];
    }
    CU(cudaMemcpyAsync(c->d_st, &s, sizeof s, cudaMemcpyHostToDevice, c->stream));
    return 0;
}

static int run_common(bpe_cuda_ctx *c, u64 max_merges, const bpe_pair_t *enc_merges, size_t n_enc, bool encode,
                      bpe_cuda_stats_t *stats_out)
{
    int rc;
    CU(cudaSetDevice(c->device));
    const auto t0 = std::chrono::steady_clock::now();
    c->run_encode = encode;
    c->solo = false;
    c->run_max_merges = encode ? 0 : max_merges;
    memset(&c->stats, 0, sizeof c->stats);
    for (double &x : c->host_ms)
        x = 0;
    c->launches = 0;
    c->prof_used = 0;
    const u64 n = c->n_bytes;
    if (c->world == 1 && n < 2 && !encode)
    {
        set_error("Error: File contains less than 2 characters"); // bpe.c:560
        return BPE_CUDA_ERR_SHORT;
    }
    if ((rc = ensure_stream_buffers(c, n)))
        return rc;
    if (!c->d_dense)
        CU(cudaMalloc(&c->d_dense, 65536 * sizeof(u32)));
    for (int i = 0; i < 2; i++)
        if (!c->d_rcnt[i])
        {
            CU(cudaMalloc(&c->d_rcnt[i], RANGE_MAX * sizeof(u32)));
            CU(cudaMalloc(&c->d_redge[i], RANGE_MAX * EDGE_WORDS * sizeof(u32)));
        }
    c->rmax = c->ranges_opt > 0 ? std::min(RANGE_MAX, c->ranges_opt) : std::min(RANGE_MAX, c->sm_count * c->stream_occ[0]);
    c->sel_grid = c->sm_count * 2;
    if (!c->d_part)
    {
        CU(cudaMalloc(&c->d_part, (size_t)c->sel_grid * sizeof(SelPart)));
        CU(cudaMalloc(&c->d_cand, CAND_CAP * sizeof(u32)));
    }
    c->cand_T = 0;
    // fresh table (in the arena the last run left unused, so a big arena stays available for the rehashes)
    {
        const int arena = c->arena[0].cap <= c->arena[1].cap ? 0 : 1;
        if ((rc = table_alloc(c, 1ull << 20, arena)))
            return rc;
        table_adopt(c, arena, 1ull << 20);
    }
    if (c->merges_cap == 0)
    {
        c->merges_cap = 8192;
        CU(cudaMalloc(&c->d_merges, c->merges_cap * 2 * sizeof(u32)));
        CU(cudaMalloc(&c->d_nhist, (c->merges_cap + 1) * sizeof(u64)));
    }
    if (encode)
    {
        if (n_enc + 1 > c->enc_cap)
        {
            if (c->d_enc_merges)
                CU(cudaFree(c->d_enc_merges));
            c->d_enc_merges = nullptr;
            CU(cudaMalloc(&c->d_enc_merges, (n_enc + 1) * 2 * sizeof(u32)));
            c->enc_cap = n_enc + 1;
        }
        if (n_enc)
            CU(cudaMemcpyAsync(c->d_enc_merges, enc_merges, n_enc * sizeof(bpe_pair_t), cudaMemcpyHostToDevice, c->stream));
    }
    if ((rc = ensure_delta(c, 8192)))
        return rc;
    CU(cudaMemsetAsync(c->d_delta, 0, c->delta_cap * sizeof(int32_t), c->stream));
    CU(cudaMemsetAsync(c->d_desc, 0, c->desc_cap * sizeof(u64), c->stream));
    CU(cudaMemsetAsync(c->d_pdesc, 0, c->desc_cap * sizeof(u32), c->stream));
    const bool prewidened = c->prewidened;
    c->prewidened = false;
    if (!prewidened)
        CU(cudaMemsetAsync(c->d_dense, 0, 65536 * sizeof(u32), c->stream));
    if (c->profile_replace && c->prof.empty())
    {
        c->prof.resize(4 * 70000);
        c->prof_tag.resize(c->prof.size());
        for (auto &e : c->prof)
            CU(cudaEventCreate(&e));
    }
    if ((rc = init_state(c, n, max_merges, n_enc)))
        return rc;

    cudaEvent_t ev0, ev1;
    CU(cudaEventCreate(&ev0));
    CU(cudaEventCreate(&ev1));
    CU(cudaEventRecord(ev0, c->stream));

    // K0 + K1: widen and count byte pairs (already done chunk by chunk when the shard came in through the file ingest)
    if (n && !prewidened)
    {
        const u64 nvec = (n + 15) / 16;
        const int grid = (int)std::min<u64>((nvec + 255) / 256, (u64)c->sm_count * 3);
        widen_count_kernel<<<grid, 256, 128 * 128 * sizeof(u32), c->stream>>>(c->d_bytes, 0, n, c->d_tok_alloc[0] + 4, c->d_dense);
        c->launches++;
    }
    if (c->world > 1)
    {
        // every rank's edge record (one exchange over peer memory), this rank's halos, the byte pair that straddles
        // the shard boundary (counted by the left shard), and the one real collective of a run: the sum of the dense
        // 256 x 256 byte-pair histograms
        edge_exchange_kernel<<<1, 32, 0, c->stream>>>(c->d_st, 0);
        resolve_edges_kernel<<<1, 1, 0, c->stream>>>(c->d_st);
        boundary_pair_kernel<<<1, 1, 0, c->stream>>>(c->d_st, c->d_dense);
        NC(g_nccl.AllReduce(c->d_dense, c->d_dense, 65536, ncclUint32, ncclSum, c->comm, c->stream));
        c->launches += 3;
    }
    table_from_dense_kernel<<<65536 / 256, 256, 0, c->stream>>>(c->d_st, c->d_dense);
    c->launches++;
    CU(cudaGetLastError());

    // the reference slices statically below 1,048,576 tokens (bpe.c:449): known up front for small inputs
    if ((rc = poll_state(c)))
        return rc;
    {
        u64 n_global = c->h_st->n_global;
        if (c->world > 1)
        {
            // the records of the exchange that has just completed hold every rank's length
            std::vector<u32> hdr(HDR_INTS);
            CU(cudaMemcpyAsync(hdr.data(), c->hx.local + XCHG_RECS + (c->h_st->xseq & 1u) * MAX_RANKS * REC_INTS,
                               HDR_INTS * sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
            CU(cudaStreamSynchronize(c->stream));
            n_global = 0;
            for (int r = 0; r < c->world; r++)
                n_global += (u64)hdr[r * REC_INTS] | ((u64)hdr[r * REC_INTS + 1] << 32);
        }
        c->stats.n_input = n_global;
        if (!encode && n_global < 2)
        {
            set_error("Error: File contains less than 2 characters");
            return BPE_CUDA_ERR_SHORT;
        }
        if (!encode && n_global < STATIC_LIMIT)
        {
            const u32 one = 1;
            CU(cudaMemcpyAsync(&c->d_st->static_mode, &one, sizeof one, cudaMemcpyHostToDevice, c->stream));
            c->h_st->static_mode = 1;
            if (c->world > 1)
            {
                // a corpus that small is not worth sharding, and the static slices need the whole stream anyway
                if ((rc = consolidate(c)))
                    return rc;
                if ((rc = poll_state(c)))
                    return rc;
            }
        }
    }

    if ((rc = run_loop(c, encode)))
        return rc;

    CU(cudaEventRecord(ev1, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, ev0, ev1));
    CU(cudaEventDestroy(ev0));
    CU(cudaEventDestroy(ev1));

    DevState *h = c->h_st;
    c->xseq = h->xseq;
    if (c->debug)
        fprintf(stderr, "[bpe_cuda] host ms: rehash %.1f | candidates %.1f | pauses %.1f | poll waits %.1f | enqueue %.1f\n", c->host_ms[0],
                c->host_ms[1], c->host_ms[2], c->host_ms[3], c->host_ms[4]);
    if (c->debug && h->dbg[6])
        fprintf(stderr, "[bpe_cuda] apply+select phases, avg ns over %llu launches: apply %.0f | done-atomic %.0f | last-block setup %.0f | "
                        "candidate scan %.0f | reduce %.0f | decide %.0f | batch extension %.0f\n",
                h->dbg[6], (double)h->dbg[0] / h->dbg[6], (double)h->dbg[1] / h->dbg[6], (double)h->dbg[2] / h->dbg[6],
                (double)h->dbg[3] / h->dbg[6], (double)h->dbg[4] / h->dbg[6], (double)h->dbg[5] / h->dbg[6],
                (double)h->dbg[7] / h->dbg[6]);
    if (c->debug)
        fprintf(stderr, "[bpe_cuda] batch walks ended by: cap %llu | below cand_T %llu | tie %llu | overlap %llu | a==b/alias %llu | list used up %llu | merges trimmed by the bound %llu, by the D margin %llu\n",
                (unsigned long long)h->ext_why[0], (unsigned long long)h->ext_why[1], (unsigned long long)h->ext_why[2],
                (unsigned long long)h->ext_why[3], (unsigned long long)h->ext_why[4], (unsigned long long)h->ext_why[5], (unsigned long long)h->ext_why[6], (unsigned long long)h->ext_why[7]);
    c->res_n_merges = (size_t)h->merges_done;
    // (consolidated run: every rank holds the whole stream; rank 0 reports it, so that the ranks' results still
    // concatenate to the stream)
    c->res_n_tokens = (c->solo && c->rank != 0) ? 0 : (size_t)h->n;
    c->stats.n_merges = h->merges_done;
    c->stats.n_tokens = sharded(c) ? h->n_global : h->n;
    c->stats.ranks_applied = h->ranks_applied;
    c->stats.same_bucket_ties = h->same_bucket_ties;
    c->stats.threshold_edges = h->threshold_edges;
    c->stats.table_capacity = c->tcap;
    c->stats.final_distinct = (u64)h->distinct;
    c->stats.batch_merges = h->batch_merges;
    c->stats.batch_passes = h->batch_passes;
    c->stats.kernel_launches = c->launches;
    c->stats.ms_device = ms;
    for (int t = 0; t < REF_THREADS; t++)
        c->stats.worker_buckets[t] = h->bt[t];
    // algorithmic bytes of the replace passes: 4*(n_k + n_{k+1}) per merge that ran a pass
    if (h->merges_done)
    {
        std::vector<u64> nh(h->merges_done);
        CU(cudaMemcpy(nh.data(), c->d_nhist, h->merges_done * sizeof(u64), cudaMemcpyDeviceToHost));
        u64 bytes = 0;
        // one pass per entry that is not marked "rode along in a batch"
        std::vector<u64> pass_n;
        for (u64 k = 0; k < h->merges_done; k++)
            if (nh[k] != ~0ull)
                pass_n.push_back(nh[k]);
        for (size_t k = 0; k < pass_n.size(); k++)
        {
            const u64 nk = pass_n[k], nk1 = (k + 1 < pass_n.size()) ? pass_n[k + 1] : c->stats.n_tokens;
            if (!encode || nk1 != nk)
                bytes += 4 * (nk + nk1);
        }
        c->stats.replace_passes = pass_n.size();
        c->stats.replace_bytes = bytes;
    }
    if (c->profile_replace)
    {
        double tot[4] = {0, 0, 0, 0};
        for (size_t i = 0; i + 1 < c->prof_used; i++)
        {
            float e = 0;
            CU(cudaEventElapsedTime(&e, c->prof[i], c->prof[i + 1]));
            tot[c->prof_tag[i + 1] & 3] += e;
        }
        c->stats.gap_ms = tot[PT_GAP];
        c->stats.select_ms = tot[PT_SELECT];
        c->stats.replace_ms = tot[PT_REPLACE];
        c->stats.apply_ms = tot[PT_APPLY];
    }
    c->stats.ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (stats_out)
        *stats_out = c->stats;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// Exactness on several GPUs (hash_table.c:208-223,248-254,300-338; bpe.c:449-477).  The chain order inside one
// bucket and the 16 worker tables' bucket counts depend on WHERE in the stream a pair is first seen, i.e. on
// positions in the whole stream.  Two rare situations need them, and both are handled by giving every rank the whole
// stream and letting it run the single-GPU kernels (all ranks compute the same thing, nothing has to be agreed on):
//   * the global stream falls below 1,048,576 tokens (the reference's static slicing, at most 4 MB): the run is
//     CONSOLIDATED for good - sharding a stream that fits in L2 many times over buys nothing;
//   * a same-bucket tie / an exact-threshold iteration above that limit: the stream is gathered into a scratch
//     buffer for the resolver kernels only, and the shards carry on afterwards.
// The gathers are NCCL broadcasts (rare, off the per-pass path).
static int read_shard_lengths(bpe_cuda_ctx *c, std::vector<u64> &lens, u64 *total)
{
    std::vector<u32> hdr(HDR_INTS);
    CU(cudaMemcpyAsync(hdr.data(), c->hx.local + XCHG_RECS + (c->h_st->xseq & 1u) * MAX_RANKS * REC_INTS, HDR_INTS * sizeof(u32),
                       cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    lens.assign((size_t)c->world, 0);
    *total = 0;
    for (int r = 0; r < c->world; r++)
    {
        lens[(size_t)r] = (u64)hdr[r * REC_INTS] | ((u64)hdr[r * REC_INTS + 1] << 32);
        *total += lens[(size_t)r];
    }
    return 0;
}

// dst[0 .. n_global) = the ranks' dense streams in rank order, on every rank (c->h_st must be current and DENSE)
static int gather_stream(bpe_cuda_ctx *c, u32 *dst, const std::vector<u64> &lens)
{
    const u32 *mine = c->h_st->tok[c->h_st->cur];
    NC(g_nccl.GroupStart());
    u64 off = 0;
    for (int r = 0; r < c->world; r++)
    {
        if (lens[(size_t)r])
            NC(g_nccl.Broadcast(r == c->rank ? (const void *)mine : (const void *)(dst + off), dst + off, (size_t)lens[(size_t)r], ncclUint32,
                                r, c->comm, c->stream));
        off += lens[(size_t)r];
    }
    NC(g_nccl.GroupEnd());
    return 0;
}

__global__ void consolidate_kernel(DevState *st, u32 *t0, u32 *t1, u64 n)
{
    st->tok[0] = st->tok_real[0] = t0;
    st->tok[1] = st->tok_real[1] = t1;
    st->cur = 0;
    st->n = st->n_global = n;
    st->layout = st->layout_next = LAYOUT_DENSE;
    st->world = 1;
    st->rank = 0;
    st->halo_before[0] = st->halo_before[1] = SENT;
    st->halo_after[0] = st->halo_after[1] = st->halo_after[2] = SENT;
    st->carry_in = 0;
    st->static_mode = 1;
}

// the resolver kernels read the stream through tok[cur] / n: point them at the gathered copy, and back
__global__ void stream_view_kernel(DevState *st, u32 *view, u64 n)
{
    if (view)
    {
        st->probe_slot = (u64)st->tok[st->cur]; // (scratch fields: nothing else uses them during a pause)
        st->probe_key = st->n;
        st->tok[st->cur] = view;
        st->n = n;
    }
    else
    {
        st->tok[st->cur] = reinterpret_cast<u32 *>(st->probe_slot);
        st->n = st->probe_key;
    }
}

static int consolidate(bpe_cuda_ctx *c)
{
    int rc;
    if ((rc = poll_state(c)))
        return rc;
    if (c->h_st->layout != LAYOUT_DENSE)
    {
        set_error("consolidate: the stream is not dense");
        return BPE_CUDA_ERR_STATE;
    }
    std::vector<u64> lens;
    u64 total = 0;
    if ((rc = read_shard_lengths(c, lens, &total)))
        return rc;
    const size_t cap = round_up((size_t)total, V_TILE) + V_TILE + 64;
    u32 *nt[2] = {nullptr, nullptr};
    for (int i = 0; i < 2; i++)
    {
        CU(cudaMalloc(&nt[i], cap * sizeof(u32)));
        CU(cudaMemsetAsync(nt[i], 0xFF, 16, c->stream)); // the 4 readable slots in front
    }
    if ((rc = gather_stream(c, nt[0] + 4, lens)))
        return rc;
    consolidate_kernel<<<1, 1, 0, c->stream>>>(c->d_st, nt[0] + 4, nt[1] + 4, total);
    c->launches++;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < 2; i++)
    {
        CU(cudaFree(c->d_tok_alloc[i]));
        c->d_tok_alloc[i] = nt[i];
    }
    c->tok_cap = cap;
    const size_t tiles = (size_t)total / R_TILE + 2;
    if (tiles > c->desc_cap)
    {
        CU(cudaFree(c->d_desc));
        CU(cudaFree(c->d_pdesc));
        c->d_desc = nullptr;
        c->d_pdesc = nullptr;
        CU(cudaMalloc(&c->d_desc, tiles * sizeof(u64)));
        CU(cudaMalloc(&c->d_pdesc, tiles * sizeof(u32)));
        c->desc_cap = tiles;
    }
    CU(cudaMemsetAsync(c->d_desc, 0, c->desc_cap * sizeof(u64), c->stream));
    CU(cudaMemsetAsync(c->d_pdesc, 0, c->desc_cap * sizeof(u32), c->stream));
    c->solo = true;
    c->want_ranged = 0;
    if (c->debug)
        fprintf(stderr, "[bpe_cuda r%d] consolidated: %llu tokens on every rank from here on\n", c->rank, (unsigned long long)total);
    return 0;
}

// ---------------------------------------------------------------------------------------------
// pause handling
static int resolve_pause(bpe_cuda_ctx *c, bool encode)
{
    HostTimer ht(&c->host_ms[2]);
    DevState *h = c->h_st;
    int rc;
    const u32 pause = h->pause;
    const u64 merges_done = h->merges_done, n = h->n;
    const u32 best = (u32)(h->sel_key >> 32);
    if (pause & PAUSE_REBUILD)
    {
        // nothing was committed: new list (or whole-table mode), then select again
        if (best == 0 && c->cand_T)
        {
            // the list ran EMPTY (every listed pair was merged or decayed): nothing says what the maximum is now.
            // run_loop makes ONE whole-table selection and builds the next list from the count it finds.
            if ((rc = rebuild_candidates(c, 0)))
                return rc;
            c->list_retry_below = ~0u;
            c->fresh_select = true;
        }
        else if ((rc = choose_candidates(c, best)))
            return rc;
        resume_kernel<<<1, 1, 0, c->stream>>>(c->d_st);
        c->launches++;
        return 0;
    }
    if (h->layout == LAYOUT_RANGED)
    {
        // everything below works on positions of one dense array
        repack_kernel<<<RANGE_MAX, 1024, 0, c->stream>>>(c->d_st);
        c->launches++;
    }
    if (pause & PAUSE_STATIC)
    {
        // the select kernel latched static_mode; several GPUs: from here on every rank works on the whole stream;
        // then resume (and select again)
        if (sharded(c) && !encode && (rc = consolidate(c)))
            return rc;
        resume_kernel<<<1, 1, 0, c->stream>>>(c->d_st);
        c->launches++;
        return 0;
    }
    c->stats.resolver_runs++;
    if ((rc = ensure_delta(c, (size_t)(256 + merges_done + 2))))
        return rc;
    if ((rc = ensure_xchg(c, (size_t)(256 + merges_done + 2), 0)))
        return rc;
    if ((rc = ensure_logs(c, (size_t)(merges_done + 2))))
        return rc;
    u64 n_res = n; // tokens the resolver kernels look at
    if (sharded(c))
    {
        // chain order needs positions in the WHOLE stream: gather it on every rank (scratch) for the resolver kernels
        if ((rc = poll_state(c))) // (the repack above moved the stream)
            return rc;
        std::vector<u64> lens;
        if ((rc = read_shard_lengths(c, lens, &n_res)))
            return rc;
        if (n_res >= 0xFFFFFFF0ull)
        {
            set_error("a same-bucket tie on a sharded stream of %llu tokens: first-sight positions are kept in 32 bits",
                      (unsigned long long)n_res);
            return BPE_CUDA_ERR_STATE;
        }
        if (n_res + 16 > c->gather_cap)
        {
            CU(cudaFree(c->d_gather));
            c->d_gather = nullptr;
            c->gather_cap = 0;
            CU(cudaMalloc(&c->d_gather, (n_res + 16) * sizeof(u32)));
            c->gather_cap = n_res + 16;
        }
        if ((rc = gather_stream(c, c->d_gather, lens)))
            return rc;
        stream_view_kernel<<<1, 1, 0, c->stream>>>(c->d_st, c->d_gather, n_res);
        c->launches++;
    }
    const u32 slices = (n_res < STATIC_LIMIT) ? REF_THREADS : 1;
    if ((rc = ensure_resolver(c, n_res, slices)))
        return rc;
    if ((rc = enqueue_census(c, n_res, 1)))
        return rc;
    const int g = pos_grid(c, n_res);
    const int tg = (int)std::max<u64>(1, std::min<u64>(n_res / SCAN_TILE + 1, (u64)c->sm_count * 8));
    const int sg = (int)std::min<u64>((c->tcap + 255) / 256, (u64)c->sm_count * 8);
    rank_tile_count_kernel<<<tg, 256, 0, c->stream>>>(c->d_rs, c->d_first, c->d_pos_slot, c->d_tile_cnt);
    rank_tile_scan_kernel<<<1, 1024, 0, c->stream>>>(c->d_rs, c->d_tile_cnt, c->d_tile_off);
    rank_assign_kernel<<<tg, 256, 0, c->stream>>>(c->d_rs, c->d_first, c->d_pos_slot, c->d_tile_off, c->d_rank);
    entry_pass1_kernel<<<g, 256, 0, c->stream>>>(c->d_st, c->d_rs, c->d_first, c->d_pos_slot, c->d_rank);
    resolver_mid_kernel<<<1, 1, 0, c->stream>>>(c->d_st, c->d_rs);
    cand_bucket_kernel<<<sg, 256, 0, c->stream>>>(c->d_st, c->d_rs);
    cand_collect_kernel<<<sg, 256, 0, c->stream>>>(c->d_st, c->d_rs, c->d_first, c->d_rank);
    entry_pass2_kernel<<<g, 256, 0, c->stream>>>(c->d_st, c->d_rs, c->d_first, c->d_pos_slot, c->d_rank);
    if (sharded(c))
    {
        stream_view_kernel<<<1, 1, 0, c->stream>>>(c->d_st, nullptr, 0); // back to this rank's shard
        c->launches++;
    }
    resolver_commit_kernel<<<1, 1, 0, c->stream>>>(c->d_st, c->d_rs);
    c->launches += 9;
    CU(cudaGetLastError());
    return enqueue_step(c, (u32)(256 + merges_done), n, encode, false, false);
}

// ---------------------------------------------------------------------------------------------
// C ABI
extern "C"
{

const char *bpe_cuda_last_error(void) { return g_err[0] ? g_err : g_err_global; }

void bpe_cuda_free(void *p) { free(p); }

int bpe_cuda_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess)
        return 0;
    return n;
}

int bpe_cuda_ctx_create(int device, bpe_cuda_ctx_t **out)
{
    if (!out)
        return BPE_CUDA_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    CU(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev)
    {
        set_error("no CUDA device %d (%d visible); this engine has no CPU fallback", device, ndev);
        return BPE_CUDA_ERR_CUDA;
    }
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
    {
        set_error("device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
        return BPE_CUDA_ERR_CUDA;
    }
    bpe_cuda_ctx *c = new bpe_cuda_ctx();
    c->device = device;
    c->debug = getenv("BPE_CUDA_DEBUG") != nullptr;
    c->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaMalloc(&c->d_st, sizeof(DevState)) != cudaSuccess ||
        cudaMallocHost(&c->h_buf[0], sizeof(DevState)) != cudaSuccess ||
        cudaMallocHost(&c->h_buf[1], sizeof(DevState)) != cudaSuccess ||
        cudaEventCreateWithFlags(&c->poll_ev[0], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&c->poll_ev[1], cudaEventDisableTiming) != cudaSuccess)
    {
        set_error("context allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
        delete c;
        return BPE_CUDA_ERR_CUDA;
    }
    memset(&c->stats, 0, sizeof c->stats);
    int rc = setup_kernels(c);
    if (rc)
    {
        delete c;
        return rc;
    }
    if (const char *e = getenv("BPE_CUDA_BATCH_STEPS"))
        c->batch_steps = std::max(1, atoi(e));
    if (const char *e = getenv("BPE_CUDA_SMEM_HIST_MAX_VOCAB"))
    {
        c->smem_hist_max_vocab = atoi(e);
        if ((rc = setup_kernels(c)))
        {
            delete c;
            return rc;
        }
    }
    if (const char *e = getenv("BPE_CUDA_BATCH_MAX"))
        c->batch_max = atoi(e);
    if (const char *e = getenv("BPE_CUDA_RANGES"))
        c->ranges_opt = atoi(e);
    if (const char *e = getenv("BPE_CUDA_AGRID_MAX"))
        c->agrid_max = std::max(64, atoi(e));
    if (const char *e = getenv("BPE_CUDA_XCHG_TIMEOUT_MS"))
        c->x_timeout_ms = (u64)std::max(1, atoi(e));
    if (const char *e = getenv("BPE_CUDA_XCHG_CAP"))
        c->xcap_opt = (size_t)std::max(64, atoi(e));
    *out = c;
    return 0;
}

void bpe_cuda_ctx_destroy(bpe_cuda_ctx_t *c)
{
    if (!c)
        return;
    cudaSetDevice(c->device);
    if (c->stream)
        cudaStreamSynchronize(c->stream);
    if (c->comm && g_nccl.CommDestroy)
        g_nccl.CommDestroy(c->comm);
    for (auto &e : c->prof)
        cudaEventDestroy(e);
    cudaFree(c->d_bytes);
    cudaFree(c->d_tok_alloc[0]);
    cudaFree(c->d_tok_alloc[1]);
    cudaFree(c->d_st);
    for (int i = 0; i < 2; i++)
    {
        cudaFreeHost(c->h_buf[i]);
        if (c->poll_ev[i])
            cudaEventDestroy(c->poll_ev[i]);
    }
    cudaFree(c->d_desc);
    cudaFree(c->d_pdesc);
    for (int i = 0; i < 2; i++)
    {
        cudaFree(c->d_rcnt[i]);
        cudaFree(c->d_redge[i]);
    }
    cudaFree(c->d_delta);
    cudaFree(c->d_hello);
    cudaFree(c->d_gather);
    for (int i = 0; i < 2; i++)
    {
        cudaFreeHost(c->h_stage[i]);
        if (c->stage_ev[i])
            cudaEventDestroy(c->stage_ev[i]);
    }
    if (c->copy_stream)
        cudaStreamDestroy(c->copy_stream);
    for (void *p : c->x_mapped)
        cudaIpcCloseMemHandle(p);
    for (void *p : c->x_owned)
        cudaFree(p);
    table_free(c);
    cudaFree(c->d_part);
    cudaFree(c->d_cand);
    cudaFree(c->d_merges);
    cudaFree(c->d_nhist);
    cudaFree(c->d_enc_merges);
    cudaFree(c->d_dense);
    cudaFree(c->d_rs);
    cudaFree(c->d_first);
    cudaFree(c->d_dec_len);
    cudaFree(c->d_dec_off);
    cudaFree(c->d_dec_blob);
    cudaFree(c->d_dec_out);
    cudaFree(c->d_dec_tiles);
    cudaFree(c->d_rank);
    cudaFree(c->d_pos_slot);
    cudaFree(c->d_tile_cnt);
    cudaFree(c->d_tile_off);
    for (void *p : {(void *)c->d_bb, (void *)c->d_btok, (void *)c->d_brk, (void *)c->d_bdoc, (void *)c->d_btoff,
                    (void *)c->d_blen, (void *)c->d_border, (void *)c->d_bseg, (void *)c->d_bsegs, (void *)c->d_rt_key, (void *)c->d_rt_rank,
                    (void *)c->d_bnext, (void *)c->d_bmerges, (void *)c->d_dbtok, (void *)c->d_dbtile, (void *)c->d_dbtoff,
                    (void *)c->d_dbboff})
        cudaFree(p);
    if (c->stream)
        cudaStreamDestroy(c->stream);
    delete c;
}

int bpe_cuda_nccl_unique_id(void *id128)
{
    if (!id128)
        return BPE_CUDA_ERR_ARG;
    int rc = nccl_load();
    if (rc)
        return rc;
    ncclUniqueId id;
    NC(g_nccl.GetUniqueId(&id));
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
    memcpy(id128, &id, 128);
    return 0;
}

int bpe_cuda_ctx_set_comm(bpe_cuda_ctx_t *c, int rank, int world, const void *id128)
{
    if (!c || !id128 || world < 1 || world > MAX_RANKS || rank < 0 || rank >= world)
        return BPE_CUDA_ERR_ARG;
    if (world == 1)
    {
        c->rank = 0;
        c->world = 1;
        return 0;
    }
    int rc = nccl_load();
    if (rc)
        return rc;
    CU(cudaSetDevice(c->device));
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    NC(g_nccl.CommInitRank(&c->comm, world, id, rank));
    c->rank = rank;
    c->world = world;
    return xchg_setup(c, c->xcap_opt ? c->xcap_opt : XCAP_DEFAULT);
}

int bpe_cuda_ctx_upload(bpe_cuda_ctx_t *c, const uint8_t *shard, size_t n)
{
    if (!c || (!shard && n))
        return BPE_CUDA_ERR_ARG;
    CU(cudaSetDevice(c->device));
    int rc = ensure_bytes(c, n);
    if (rc)
        return rc;
    if (n)
        CU(cudaMemcpyAsync(c->d_bytes, shard, n, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemsetAsync(c->d_bytes + n, 0, c->bytes_cap - n, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->n_bytes = n;
    c->prewidened = false;
    return 0;
}

int bpe_cuda_ctx_upload_device(bpe_cuda_ctx_t *c, const void *dev, size_t n)
{
    if (!c || (!dev && n))
        return BPE_CUDA_ERR_ARG;
    CU(cudaSetDevice(c->device));
    int rc = ensure_bytes(c, n);
    if (rc)
        return rc;
    if (n)
        CU(cudaMemcpyAsync(c->d_bytes, dev, n, cudaMemcpyDeviceToDevice, c->stream));
    CU(cudaMemsetAsync(c->d_bytes + n, 0, c->bytes_cap - n, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->n_bytes = n;
    c->prewidened = false;
    return 0;
}

// ---- file ingest (SURVEY.md §8f rank 3; reference get_file bpe.c:130-180, strlen cut bpe.c:555, widen bpe.c:580-584) ----
constexpr size_t STAGE_BYTES = 32u << 20; // per pinned staging buffer (a multiple of 16)

static int ensure_staging(bpe_cuda_ctx *c)
{
    if (c->h_stage[0])
        return 0;
    for (int i = 0; i < 2; i++)
    {
        CU(cudaMallocHost(&c->h_stage[i], STAGE_BYTES));
        CU(cudaEventCreateWithFlags(&c->stage_ev[i], cudaEventDisableTiming));
    }
    CU(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    return 0;
}

// Bytes [offset, offset + max_len) of the file become this context's resident shard, cut at the first 0x00 like the
// reference's strlen (bpe.c:555).  The file is read in 32 MB pieces into two pinned buffers: while piece i+1 is being
// read, piece i travels to the GPU on a copy stream and the pieces in front of it are widened to tokens and counted
// (widen_count_kernel on [lo, hi)), so the next train / encode starts from a stream that is already widened and counted.
int bpe_cuda_ctx_upload_file(bpe_cuda_ctx_t *c, const char *path, uint64_t offset, uint64_t max_len, size_t *n_shard, int *nul_found)
{
    if (!c || !path)
        return BPE_CUDA_ERR_ARG;
    CU(cudaSetDevice(c->device));
    const int fd = open(path, O_RDONLY);
    if (fd < 0)
    {
        set_error("fopen: %s", strerror(errno)); // bpe.c:133-137
        return BPE_CUDA_ERR_ARG;
    }
    struct stat sb;
    if (fstat(fd, &sb) != 0)
    {
        set_error("fstat: %s", strerror(errno));
        close(fd);
        return BPE_CUDA_ERR_ARG;
    }
    const u64 fsize = (u64)sb.st_size;
    const u64 lo = std::min<u64>(offset, fsize), hi = (max_len > fsize - lo) ? fsize : lo + max_len;
    const size_t want = (size_t)(hi - lo);
    int rc;
    auto fail = [&](int r) {
        close(fd);
        return r;
    };
    if ((rc = ensure_staging(c)) || (rc = ensure_bytes(c, want)) || (rc = ensure_stream_buffers(c, want)))
        return fail(rc);
    if (!c->d_dense && cudaMalloc(&c->d_dense, 65536 * sizeof(u32)) != cudaSuccess)
    {
        set_error("out of device memory");
        return fail(BPE_CUDA_ERR_NOMEM);
    }
    if (cudaMemsetAsync(c->d_dense, 0, 65536 * sizeof(u32), c->stream) != cudaSuccess)
        return fail(BPE_CUDA_ERR_CUDA);
    size_t n = 0;
    bool nul = false;
    for (int i = 0; n < want && !nul; i ^= 1)
    {
        // buffer i is free again once the copy that last used it is over
        if (cudaEventSynchronize(c->stage_ev[i]) != cudaSuccess)
            return fail(BPE_CUDA_ERR_CUDA);
        const size_t ask = std::min(STAGE_BYTES, want - n);
        size_t got = 0;
        while (got < ask)
        {
            const ssize_t r = pread(fd, c->h_stage[i] + got, ask - got, (off_t)(lo + n + got));
            if (r < 0)
            {
                set_error("fread: %s", strerror(errno));
                return fail(BPE_CUDA_ERR_ARG);
            }
            if (r == 0)
                break;
            got += (size_t)r;
        }
        if (got == 0)
            break;
        if (const void *z = memchr(c->h_stage[i], 0, got))
        {
            got = (size_t)((const uint8_t *)z - c->h_stage[i]);
            nul = true;
        }
        if (got)
        {
            if (cudaMemcpyAsync(c->d_bytes + n, c->h_stage[i], got, cudaMemcpyHostToDevice, c->copy_stream) != cudaSuccess ||
                cudaEventRecord(c->stage_ev[i], c->copy_stream) != cudaSuccess ||
                cudaStreamWaitEvent(c->stream, c->stage_ev[i], 0) != cudaSuccess)
                return fail(BPE_CUDA_ERR_CUDA);
            const u64 nvec = (got + 15) / 16;
            const int grid = (int)std::min<u64>((nvec + 255) / 256, (u64)c->sm_count * 3);
            widen_count_kernel<<<grid, 256, 128 * 128 * sizeof(u32), c->stream>>>(c->d_bytes, n, n + got, c->d_tok_alloc[0] + 4, c->d_dense);
            c->launches++;
        }
        n += got;
        if (got < ask)
            break;
    }
    close(fd);
    CU(cudaStreamSynchronize(c->copy_stream));
    CU(cudaMemsetAsync(c->d_bytes + n, 0, c->bytes_cap - n, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    CU(cudaGetLastError());
    c->n_bytes = n;
    c->prewidened = (n > 0);
    if (n_shard)
        *n_shard = n;
    if (nul_found)
        *nul_found = nul ? 1 : 0;
    return 0;
}

// (a shard that has to be shortened after the ingest - a lower rank found the corpus' NUL - is widened again by the run)
int bpe_cuda_ctx_truncate(bpe_cuda_ctx_t *c, size_t n)
{
    if (!c || n > c->n_bytes)
        return BPE_CUDA_ERR_ARG;
    if (n == c->n_bytes)
        return 0;
    CU(cudaSetDevice(c->device));
    CU(cudaMemsetAsync(c->d_bytes + n, 0, c->bytes_cap - n, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->n_bytes = n;
    c->prewidened = false;
    return 0;
}

int bpe_cuda_ctx_train(bpe_cuda_ctx_t *c, uint64_t max_merges, bpe_cuda_stats_t *stats)
{
    if (!c)
        return BPE_CUDA_ERR_ARG;
    return run_common(c, max_merges, nullptr, 0, false, stats);
}

int bpe_cuda_ctx_encode(bpe_cuda_ctx_t *c, const bpe_pair_t *merges, size_t n_merges, bpe_cuda_stats_t *stats)
{
    if (!c || (!merges && n_merges))
        return BPE_CUDA_ERR_ARG;
    for (size_t r = 0; r < n_merges; r++)
        if (merges[r].a >= 256 + r || merges[r].b >= 256 + r)
        {
            set_error("merge %zu refers to an id that does not exist yet", r);
            return BPE_CUDA_ERR_ARG;
        }
    return run_common(c, n_merges, merges, n_merges, true, stats);
}

int bpe_cuda_ctx_result_sizes(bpe_cuda_ctx_t *c, size_t *n_merges, size_t *n_tokens_local)
{
    if (!c)
        return BPE_CUDA_ERR_ARG;
    if (n_merges)
        *n_merges = c->res_n_merges;
    if (n_tokens_local)
        *n_tokens_local = c->res_n_tokens;
    return 0;
}

const uint32_t *bpe_cuda_ctx_device_tokens(bpe_cuda_ctx_t *c)
{
    if (!c || !c->h_st)
        return nullptr;
    return c->h_st->tok[c->h_st->cur];
}

int bpe_cuda_ctx_download(bpe_cuda_ctx_t *c, bpe_pair_t *merges, uint32_t *tokens)
{
    if (!c)
        return BPE_CUDA_ERR_ARG;
    CU(cudaSetDevice(c->device));
    if (merges && c->res_n_merges)
        CU(cudaMemcpyAsync(merges, c->d_merges, c->res_n_merges * sizeof(bpe_pair_t), cudaMemcpyDeviceToHost, c->stream));
    if (tokens && c->res_n_tokens)
        CU(cudaMemcpyAsync(tokens, c->h_st->tok[c->h_st->cur], c->res_n_tokens * sizeof(u32), cudaMemcpyDeviceToHost,
                           c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

// The same into PAGEABLE memory (malloc'd results of the one-call entry points, SURVEY.md §8f rank 4): 32 MB pieces
// through the two pinned staging buffers, the host copy of piece i overlapping the DMA of piece i+1 (a plain
// cudaMemcpy into pageable memory stages through one small driver buffer and runs at a fraction of the link).
static int download_staged(bpe_cuda_ctx *c, void *dst, const void *src_dev, size_t bytes)
{
    int rc;
    if ((rc = ensure_staging(c)))
        return rc;
    // The destination is fresh malloc'd memory: its pages are faulted in on first touch, which a single copying
    // thread does at ~2 GB/s (measured: 0.55 s for the 1.17 GB of ids of the 1 GB corpus).  Helper threads touch the
    // pages ahead of the copy.
    std::vector<std::thread> toucher;
    if (bytes >= (64u << 20))
    {
        const int T = 3;
        for (int t = 0; t < T; t++)
            toucher.emplace_back([=] {
                // (an atomic add of zero: faults the page in for writing without changing what the copy may already
                // have put there)
                char *p = (char *)dst;
                const size_t lo = bytes / T * (size_t)t, hi = (t == T - 1) ? bytes : bytes / T * (size_t)(t + 1);
                for (size_t o = (lo + 4095) & ~(size_t)4095; o < hi; o += 4096)
                    __atomic_fetch_add(p + o, (char)0, __ATOMIC_RELAXED);
            });
    }
    struct Joiner
    {
        std::vector<std::thread> &v;
        ~Joiner()
        {
            for (auto &t : v)
                t.join();
        }
    } joiner{toucher};
    size_t issued = 0, copied = 0, len[2] = {0, 0};
    int head = 0, next = 0, inflight = 0; // head: the buffer that holds the oldest piece still on its way
    while (copied < bytes)
    {
        while (inflight < 2 && issued < bytes)
        {
            len[next] = std::min(STAGE_BYTES, bytes - issued);
            CU(cudaMemcpyAsync(c->h_stage[next], (const char *)src_dev + issued, len[next], cudaMemcpyDeviceToHost, c->copy_stream));
            CU(cudaEventRecord(c->stage_ev[next], c->copy_stream));
            issued += len[next];
            next ^= 1;
            inflight++;
        }
        CU(cudaEventSynchronize(c->stage_ev[head]));
        memcpy((char *)dst + copied, c->h_stage[head], len[head]);
        copied += len[head];
        head ^= 1;
        inflight--;
    }
    return 0;
}

int bpe_cuda_ctx_download_pageable(bpe_cuda_ctx_t *c, bpe_pair_t *merges, uint32_t *tokens)
{
    if (!c)
        return BPE_CUDA_ERR_ARG;
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    if (merges && c->res_n_merges)
        CU(cudaMemcpy(merges, c->d_merges, c->res_n_merges * sizeof(bpe_pair_t), cudaMemcpyDeviceToHost));
    if (tokens && c->res_n_tokens)
        return download_staged(c, tokens, c->h_st->tok[c->h_st->cur], c->res_n_tokens * sizeof(u32));
    return 0;
}

int bpe_cuda_ctx_set_option(bpe_cuda_ctx_t *c, const char *name, long long value)
{
    if (!c || !name)
        return BPE_CUDA_ERR_ARG;
    if (!strcmp(name, "profile_replace"))
        c->profile_replace = (int)value;
    else if (!strcmp(name, "batch_steps"))
        c->batch_steps = (int)std::max<long long>(1, value);
    else if (!strcmp(name, "smem_hist_max_vocab"))
    {
        c->smem_hist_max_vocab = (int)std::min<long long>(value, 8192);
        return setup_kernels(c);
    }
    else if (!strcmp(name, "batch_min_z"))
        c->batch_min_z = (int)value;
    else if (!strcmp(name, "batch_max"))
        c->batch_max = (int)value;
    else if (!strcmp(name, "ranges"))
        c->ranges_opt = (int)value;
    else if (!strcmp(name, "xchg_cap")) // entries per inbox slot at set_comm (test knob: small values force growth)
        c->xcap_opt = (size_t)std::max<long long>(64, value);
    else
        return BPE_CUDA_ERR_ARG;
    return 0;
}

// ---- decode (SURVEY.md §8f rank 2; reference bpe/src/bpe.c:23-92, 341-394) --------------------
// Flatten the vocabulary on the host: id < 256 is its own byte, id 256+r is expansion(a) ++ expansion(b)
// (resolve_pair, bpe.c:23-92, without the NUL-terminated strings).
static int decode_flatten(const bpe_pair_t *merges, size_t n_merges, std::vector<u32> &len, std::vector<u32> &off,
                          std::vector<uint8_t> &blob)
{
    const size_t V = 256 + n_merges;
    len.resize(V);
    off.resize(V);
    u64 total = 256;
    for (size_t i = 0; i < 256; i++)
    {
        len[i] = 1;
        off[i] = (u32)i;
    }
    for (size_t r = 0; r < n_merges; r++)
    {
        const u32 a = merges[r].a, b = merges[r].b;
        if (a >= 256 + r || b >= 256 + r)
        {
            set_error("merge %zu refers to an id that does not exist yet", r);
            return BPE_CUDA_ERR_ARG;
        }
        const u64 l = (u64)len[a] + len[b];
        if (total + l > (1ull << 30))
        {
            set_error("decode: the flattened vocabulary exceeds 1 GiB");
            return BPE_CUDA_ERR_NOMEM;
        }
        len[256 + r] = (u32)l;
        off[256 + r] = (u32)total;
        total += l;
    }
    blob.resize(total);
    for (size_t i = 0; i < 256; i++)
        blob[i] = (uint8_t)i;
    for (size_t r = 0; r < n_merges; r++)
    {
        const u32 a = merges[r].a, b = merges[r].b;
        memcpy(&blob[off[256 + r]], &blob[off[a]], len[a]);
        memcpy(&blob[off[256 + r] + len[a]], &blob[off[b]], len[b]);
    }
    return 0;
}

extern "C++"
{
template <class T> static int dec_reserve(T *&p, size_t &cap, size_t need)
{
    if (need <= cap)
        return 0;
    if (p)
        CU(cudaFree(p));
    p = nullptr;
    cap = 0;
    const size_t want = need + need / 8 + 256;
    CU(cudaMalloc(&p, want * sizeof(T)));
    cap = want;
    return 0;
}
}

// The flattened vocabulary of the merge list on the device (d_dec_len, d_dec_off, d_dec_blob).  It is rebuilt only
// when the list differs from the one it was built from, so a stream of decodes with one vocabulary flattens and
// uploads it once.  *rebuilt says whether this call did.
static int dec_vocab(bpe_cuda_ctx *c, const bpe_pair_t *merges, size_t n_merges, bool *rebuilt)
{
    *rebuilt = false;
    if (c->dec_valid && c->dec_merges.size() == n_merges &&
        (!n_merges || !memcmp(c->dec_merges.data(), merges, n_merges * sizeof(bpe_pair_t))))
        return 0;
    int rc;
    c->dec_valid = false; // until the upload has completed
    std::vector<u32> len, off;
    std::vector<uint8_t> blob;
    if ((rc = decode_flatten(merges, n_merges, len, off, blob)))
        return rc;
    const size_t V = len.size();
    size_t cap2 = c->dec_vocab_cap;
    if ((rc = dec_reserve(c->d_dec_len, c->dec_vocab_cap, V)) || (rc = dec_reserve(c->d_dec_off, cap2, V)) ||
        (rc = dec_reserve(c->d_dec_blob, c->dec_blob_cap, blob.size())))
        return rc;
    CU(cudaMemcpyAsync(c->d_dec_len, len.data(), V * sizeof(u32), cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->d_dec_off, off.data(), V * sizeof(u32), cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->d_dec_blob, blob.data(), blob.size(), cudaMemcpyHostToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->dec_merges.assign(merges, merges + n_merges);
    c->dec_valid = true;
    *rebuilt = true;
    return 0;
}

// Expand d_tok[0..n) (device) into c->d_dec_out through the vocabulary dec_vocab() left on the device; *n_bytes = size
// of the expansion, *ms = device time of the kernels (CUDA events, without the host round trip between D2 and D3).
// With docs (batch decode, n > 0), also the byte offset of each of its n_ends entries.  An id outside the vocabulary
// returns BPE_CUDA_ERR_ARG before anything is expanded.
static int decode_run(bpe_cuda_ctx *c, const u32 *d_tok, u64 n, const DecodeDocs *docs, u64 n_ends, size_t *n_bytes, float *ms)
{
    int rc;
    const size_t V = 256 + c->dec_merges.size();
    const u64 nt = (n + DEC_TILE - 1) / DEC_TILE;
    if ((rc = dec_reserve(c->d_dec_tiles, c->dec_tiles_cap, nt + 2)))
        return rc;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    struct EvGuard
    {
        cudaEvent_t *e;
        ~EvGuard()
        {
            for (int k = 0; k < 4; k++)
                if (e[k])
                    cudaEventDestroy(e[k]);
        }
    } ev_guard{ev};
    for (int k = 0; k < 4; k++)
        CU(cudaEventCreate(&ev[k]));
    u64 *d_total = c->d_dec_tiles + nt;     // written by the scan
    u32 *d_err = reinterpret_cast<u32 *>(c->d_dec_tiles + nt + 1);
    CU(cudaMemsetAsync(c->d_dec_tiles + nt, 0, 2 * sizeof(u64), c->stream));
    DecodeVocab v{c->d_dec_len, c->d_dec_off, c->d_dec_blob, (u32)V};
    c->dec_n_out = 0;
    CU(cudaEventRecord(ev[0], c->stream));
    if (n)
    {
        if (docs)
        {
            decode_batch_tiles_kernel<<<(unsigned)((nt + 1 + 255) / 256), 256, 0, c->stream>>>(docs->tok_off, (u32)n_ends,
                                                                                               docs->base, nt, docs->tile_doc);
            c->launches++;
        }
        decode_len_kernel<<<(unsigned)nt, DEC_THREADS, 0, c->stream>>>(d_tok, n, v, c->d_dec_tiles, d_err);
        decode_scan_kernel<<<1, 1024, 0, c->stream>>>(c->d_dec_tiles, nt);
        c->launches += 2;
    }
    CU(cudaEventRecord(ev[1], c->stream));
    u64 h[2] = {0, 0};
    CU(cudaMemcpyAsync(h, d_total, sizeof h, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if ((u32)h[1])
    {
        set_error("decode: the stream holds an id outside the vocabulary (%zu entries)", V);
        return BPE_CUDA_ERR_ARG;
    }
    if ((rc = dec_reserve(c->d_dec_out, c->dec_out_cap, (size_t)h[0] + 16)))
        return rc;
    CU(cudaEventRecord(ev[2], c->stream));
    if (n)
    {
        if (docs)
            decode_expand_kernel<true><<<(unsigned)nt, DEC_THREADS, 0, c->stream>>>(d_tok, n, v, c->d_dec_tiles, c->d_dec_out,
                                                                                  *docs);
        else
            decode_expand_kernel<false><<<(unsigned)nt, DEC_THREADS, 0, c->stream>>>(d_tok, n, v, c->d_dec_tiles, c->d_dec_out,
                                                                                   DecodeDocs{});
        c->launches++;
    }
    CU(cudaGetLastError());
    CU(cudaEventRecord(ev[3], c->stream));
    CU(cudaStreamSynchronize(c->stream));
    float m01 = 0, m23 = 0;
    CU(cudaEventElapsedTime(&m01, ev[0], ev[1]));
    CU(cudaEventElapsedTime(&m23, ev[2], ev[3]));
    *ms = m01 + m23;
    c->dec_n_out = (size_t)h[0];
    *n_bytes = (size_t)h[0];
    return 0;
}

// Expand d_tok[0..n) (device) into c->d_dec_out; *n_bytes = size of the expansion, *ms = its device time.
static int decode_device(bpe_cuda_ctx *c, const u32 *d_tok, u64 n, const bpe_pair_t *merges, size_t n_merges, size_t *n_bytes,
                         float *ms = nullptr)
{
    int rc;
    CU(cudaSetDevice(c->device));
    bool rebuilt;
    if ((rc = dec_vocab(c, merges, n_merges, &rebuilt)))
        return rc;
    size_t nb = 0;
    float t = 0;
    if ((rc = decode_run(c, d_tok, n, nullptr, 0, &nb, &t)))
        return rc;
    if (n_bytes)
        *n_bytes = nb;
    if (ms)
        *ms = t;
    return 0;
}

int bpe_cuda_ctx_decode(bpe_cuda_ctx_t *c, const bpe_pair_t *merges, size_t n_merges, size_t *n_bytes)
{
    if (!c || (!merges && n_merges) || !c->h_st)
        return BPE_CUDA_ERR_ARG;
    return decode_device(c, c->h_st->tok[c->h_st->cur], c->res_n_tokens, merges, n_merges, n_bytes);
}

int bpe_cuda_ctx_decode_download(bpe_cuda_ctx_t *c, uint8_t *bytes)
{
    if (!c || (!bytes && c->dec_n_out))
        return BPE_CUDA_ERR_ARG;
    CU(cudaSetDevice(c->device));
    if (c->dec_n_out)
        CU(cudaMemcpyAsync(bytes, c->d_dec_out, c->dec_n_out, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

int bpe_cuda_ctx_decode_compare(bpe_cuda_ctx_t *c, uint64_t *n_diff)
{
    if (!c || !n_diff)
        return BPE_CUDA_ERR_ARG;
    CU(cudaSetDevice(c->device));
    if (c->dec_n_out != c->n_bytes)
    {
        *n_diff = UINT64_MAX; // different lengths
        return 0;
    }
    if (!c->n_bytes)
    {
        *n_diff = 0;
        return 0;
    }
    u64 *d_diff = c->d_dec_tiles; // free again after the expansion
    CU(cudaMemsetAsync(d_diff, 0, sizeof(u64), c->stream));
    decode_compare_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>(c->d_dec_out, c->d_bytes, c->n_bytes, d_diff);
    c->launches++;
    CU(cudaMemcpyAsync(n_diff, d_diff, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

const uint8_t *bpe_cuda_ctx_device_decoded(bpe_cuda_ctx_t *c)
{
    return c ? c->d_dec_out : nullptr;
}

int bpe_cuda_decode(const uint32_t *tokens, size_t n_tokens, const bpe_pair_t *merges, size_t n_merges, uint8_t **bytes_out,
                    size_t *n_bytes, bpe_cuda_stats_t *stats)
{
    if ((!tokens && n_tokens) || (!merges && n_merges) || !bytes_out || !n_bytes)
    {
        set_error("invalid argument");
        return BPE_CUDA_ERR_ARG;
    }
    *bytes_out = nullptr;
    *n_bytes = 0;
    bpe_cuda_ctx_t *c = nullptr;
    int rc = bpe_cuda_ctx_create(0, &c);
    if (rc)
        return rc;
    const auto t0 = std::chrono::steady_clock::now();
    u32 *d_tok = nullptr;
    uint8_t *out = nullptr;
    size_t nb = 0;
    float ms = 0;
    auto body = [&]() -> int {
        if (n_tokens)
        {
            CU(cudaMalloc(&d_tok, n_tokens * sizeof(u32)));
            CU(cudaMemcpyAsync(d_tok, tokens, n_tokens * sizeof(u32), cudaMemcpyHostToDevice, c->stream));
        }
        int r = decode_device(c, d_tok, n_tokens, merges, n_merges, &nb, &ms);
        if (r)
            return r;
        out = (uint8_t *)malloc(nb + 1); // +1: room for the terminator decompress() appends (bpe.c:390)
        if (!out)
        {
            set_error("out of host memory");
            return BPE_CUDA_ERR_NOMEM;
        }
        out[nb] = 0;
        return bpe_cuda_ctx_decode_download(c, out);
    };
    rc = body();
    if (d_tok)
        cudaFree(d_tok);
    if (stats)
    {
        memset(stats, 0, sizeof *stats);
        stats->n_input = n_tokens;
        stats->n_merges = n_merges;
        stats->n_tokens = nb;
        stats->kernel_launches = c->launches;
        stats->ms_device = ms;
        stats->ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
    bpe_cuda_ctx_destroy(c);
    if (rc)
    {
        free(out);
        return rc;
    }
    *bytes_out = out;
    *n_bytes = nb;
    return 0;
}

// ---- batch encode (bpe_encode_batch.cuh) ------------------------------------------------------
static int check_merges(const bpe_pair_t *merges, size_t n_merges)
{
    for (size_t r = 0; r < n_merges; r++)
        if (merges[r].a >= 256 + r || merges[r].b >= 256 + r)
        {
            set_error("merge %zu refers to an id that does not exist yet", r);
            return BPE_CUDA_ERR_ARG;
        }
    return 0;
}

// Every argument is checked before any device call, so that a bad call fails the same way with or without a GPU.
static int batch_check(const uint8_t *bytes, const uint64_t *offsets, size_t n_docs, const bpe_pair_t *merges,
                       size_t n_merges)
{
    if (!offsets || (!merges && n_merges))
    {
        set_error("invalid argument: NULL offsets or merges");
        return BPE_CUDA_ERR_ARG;
    }
    if (n_docs >= 0xFFFFFFFFu)
    {
        set_error("invalid argument: %zu documents (at most 4,294,967,294 in one batch)", n_docs);
        return BPE_CUDA_ERR_ARG;
    }
    for (size_t i = 0; i < n_docs; i++)
    {
        if (offsets[i + 1] < offsets[i])
        {
            set_error("invalid argument: offsets[%zu] < offsets[%zu] (offsets must not decrease)", i + 1, i);
            return BPE_CUDA_ERR_ARG;
        }
        if (offsets[i + 1] - offsets[i] >= 0xFFFFFFFFull)
        {
            set_error("invalid argument: document %zu is 4 GiB or longer (encode it with bpe_cuda_encode)", i);
            return BPE_CUDA_ERR_ARG;
        }
    }
    if (!bytes && offsets[n_docs] > offsets[0])
    {
        set_error("invalid argument: NULL bytes");
        return BPE_CUDA_ERR_ARG;
    }
    return check_merges(merges, n_merges);
}

// Encode the batch on the device.  On success the ids are c->d_brk[0 .. *n_tokens) and the offsets c->d_btoff[0 ..
// n_docs]; stats gets every field but ms_d2h (the caller's copies) and ms_total.
static int batch_run(bpe_cuda_ctx *c, const uint8_t *bytes, const uint64_t *offsets, size_t n_docs, const bpe_pair_t *merges,
                     size_t n_merges, size_t *n_tokens, bpe_cuda_stats_t *st)
{
    int rc;
    CU(cudaSetDevice(c->device));
    memset(st, 0, sizeof *st);
    const u64 base = offsets[0], N = offsets[n_docs] - base;
    // lengths after the NUL cut; work order: longest first among the documents of the block and global tiers (an exact
    // sort for the global tier, 64-byte buckets below it: O(n_docs)), then the warp tier in input order
    std::vector<u64> doc(n_docs);
    std::vector<u32> len(n_docs), order;
    order.reserve(n_docs);
    u64 n_input = 0;
    std::vector<u32> global_docs;
    std::vector<u32> bucket_cnt(BLOCK_CAP / 64 + 2, 0);
    for (size_t i = 0; i < n_docs; i++)
    {
        const uint8_t *p = bytes + offsets[i];
        const size_t span = offsets[i + 1] - offsets[i];
        const void *nul = span ? memchr(p, 0, span) : nullptr;
        doc[i] = offsets[i] - base;
        len[i] = (u32)(nul ? (const uint8_t *)nul - p : span);
        n_input += len[i];
        if (len[i] > BLOCK_CAP)
            global_docs.push_back((u32)i);
        else if (len[i] > WARP_CAP)
            bucket_cnt[len[i] / 64]++;
    }
    std::sort(global_docs.begin(), global_docs.end(), [&](u32 x, u32 y) { return len[x] > len[y] || (len[x] == len[y] && x < y); });
    order = global_docs;
    {
        std::vector<u32> start(bucket_cnt.size());
        u32 acc = (u32)order.size();
        for (size_t b = bucket_cnt.size(); b-- > 0;)
        {
            start[b] = acc;
            acc += bucket_cnt[b];
        }
        order.resize(acc);
        for (size_t i = 0; i < n_docs; i++)
            if (len[i] > WARP_CAP && len[i] <= BLOCK_CAP)
                order[start[len[i] / 64]++] = (u32)i;
    }
    const u32 n_big = (u32)order.size();
    for (size_t i = 0; i < n_docs; i++)
        if (len[i] <= WARP_CAP)
            order.push_back((u32)i);
    // global tier: segments of SEG positions per document (cascade_segmented)
    std::vector<u32> seg_base(n_docs, 0);
    size_t n_segs = 0;
    for (u32 i : global_docs)
    {
        seg_base[i] = (u32)n_segs;
        n_segs += (len[i] + SEG - 1) / SEG;
    }
    // device memory: 9 B per input byte (bytes, ids, ranks) + 32 B per document + 8 B per 4 KB segment + the rank
    // table, each buffer with the 1/8 headroom dec_reserve() gives it
    size_t rt_cap = 64; // a power of two, at least twice the merges: short probe chains
    while (rt_cap < 2 * n_merges)
        rt_cap <<= 1;
    {
        size_t free_b = 0, total_b = 0;
        CU(cudaMemGetInfo(&free_b, &total_b));
        auto grown = [](size_t n) { return n + n / 8 + 256; };
        const size_t have = c->bb_cap + 4 * (c->btok_cap + c->brk_cap) + 8 * (c->bdoc_cap + c->btoff_cap) +
                            4 * (c->blen_cap + c->border_cap + c->bseg_cap + c->bsegs_cap);
        const size_t need = grown((size_t)N + 16) + 8 * grown((size_t)N + 1) + 16 * grown(n_docs + 1) +
                            12 * grown(n_docs + 1) + 4 * grown(2 * n_segs + 1) + 12 * rt_cap + (64u << 20);
        if (need > free_b + have)
        {
            set_error("batch of %llu bytes needs about %zu MB of device memory (about 10 B per input byte), %zu MB are free",
                      (unsigned long long)N, need >> 20, (free_b + have) >> 20);
            return BPE_CUDA_ERR_NOMEM;
        }
    }
    if ((rc = dec_reserve(c->d_bb, c->bb_cap, (size_t)N + 16)) || (rc = dec_reserve(c->d_btok, c->btok_cap, (size_t)N + 1)) ||
        (rc = dec_reserve(c->d_brk, c->brk_cap, (size_t)N + 1)) || (rc = dec_reserve(c->d_bdoc, c->bdoc_cap, n_docs + 1)) ||
        (rc = dec_reserve(c->d_btoff, c->btoff_cap, n_docs + 1)) || (rc = dec_reserve(c->d_blen, c->blen_cap, n_docs + 1)) ||
        (rc = dec_reserve(c->d_border, c->border_cap, n_docs + 1)) || (rc = dec_reserve(c->d_bseg, c->bseg_cap, n_docs + 1)) ||
        (rc = dec_reserve(c->d_bsegs, c->bsegs_cap, 2 * n_segs + 1)))
        return rc;
    if (!c->d_bnext)
        CU(cudaMalloc(&c->d_bnext, sizeof(u32)));
    if (!c->cas_grid)
    {
        CU(cudaFuncSetAttribute(batch_cascade_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CAS_SMEM_BYTES));
        int occ = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, batch_cascade_kernel, CAS_THREADS, CAS_SMEM_BYTES));
        c->cas_grid = c->sm_count * std::max(1, occ);
    }
    {
        const auto h0 = std::chrono::steady_clock::now();
        if (N)
            CU(cudaMemcpyAsync(c->d_bb, bytes + base, N, cudaMemcpyHostToDevice, c->stream));
        if (n_docs)
        {
            CU(cudaMemcpyAsync(c->d_bdoc, doc.data(), n_docs * sizeof(u64), cudaMemcpyHostToDevice, c->stream));
            CU(cudaMemcpyAsync(c->d_blen, len.data(), n_docs * sizeof(u32), cudaMemcpyHostToDevice, c->stream));
            CU(cudaMemcpyAsync(c->d_border, order.data(), n_docs * sizeof(u32), cudaMemcpyHostToDevice, c->stream));
            CU(cudaMemcpyAsync(c->d_bseg, seg_base.data(), n_docs * sizeof(u32), cudaMemcpyHostToDevice, c->stream));
        }
        CU(cudaStreamSynchronize(c->stream));
        st->ms_h2d = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - h0).count();
    }
    cudaEvent_t ev[2] = {nullptr, nullptr};
    CU(cudaEventCreate(&ev[0]));
    if (cudaEventCreate(&ev[1]) != cudaSuccess)
    {
        cudaEventDestroy(ev[0]);
        set_error("cudaEventCreate failed");
        return BPE_CUDA_ERR_CUDA;
    }
    struct EvGuard
    {
        cudaEvent_t *e;
        ~EvGuard()
        {
            cudaEventDestroy(e[0]);
            cudaEventDestroy(e[1]);
        }
    } ev_guard{ev};
    u64 launches = 0;
    CU(cudaEventRecord(ev[0], c->stream));
    // the rank table: rebuilt only when the merge list differs from the one it was built from
    const bool rebuild = !c->rt_valid || c->rt_merges.size() != n_merges ||
                         (n_merges && memcmp(c->rt_merges.data(), merges, n_merges * sizeof(bpe_pair_t)));
    if (rebuild)
    {
        c->rt_valid = false; // until the batch that builds it has completed
        if ((rc = dec_reserve(c->d_rt_key, c->rt_key_cap, rt_cap)) || (rc = dec_reserve(c->d_rt_rank, c->rt_rank_cap, rt_cap)) ||
            (rc = dec_reserve(c->d_bmerges, c->bmerges_cap, n_merges + 1)))
            return rc;
        c->rt_mask = (u32)(rt_cap - 1);
        CU(cudaMemsetAsync(c->d_rt_key, 0xFF, rt_cap * sizeof(u64), c->stream));
        CU(cudaMemsetAsync(c->d_rt_rank, 0xFF, rt_cap * sizeof(u32), c->stream));
        if (n_merges)
            CU(cudaMemcpyAsync(c->d_bmerges, merges, n_merges * sizeof(bpe_pair_t), cudaMemcpyHostToDevice, c->stream));
        const int grid = (int)std::max<size_t>(1, std::min<size_t>((n_merges + 255) / 256, (size_t)c->sm_count * 4));
        batch_rank_table_kernel<<<grid, 256, 0, c->stream>>>(c->d_bmerges, (u32)n_merges, c->d_rt_key, c->d_rt_rank, c->rt_mask);
        launches++;
    }
    CasArgs a;
    a.bytes = c->d_bb;
    a.doc_off = c->d_bdoc;
    a.doc_len = c->d_blen;
    a.order = c->d_border;
    a.n_docs = (u32)n_docs;
    a.n_big = n_big;
    a.n_items = n_big + (u32)((n_docs - n_big + CAS_WARPS - 1) / CAS_WARPS);
    a.tok = c->d_btok;
    a.rk = c->d_brk;
    a.seg_base = c->d_bseg;
    a.seg_cnt = c->d_bsegs;
    a.seg_min = c->d_bsegs + n_segs;
    a.count = c->d_btoff;
    a.next_item = c->d_bnext;
    a.rt = RankTable{c->d_rt_key, c->d_rt_rank, c->rt_mask};
    CU(cudaMemsetAsync(c->d_bnext, 0, sizeof(u32), c->stream));
    batch_cascade_kernel<<<c->cas_grid, CAS_THREADS, CAS_SMEM_BYTES, c->stream>>>(a);
    decode_scan_kernel<<<1, 1024, 0, c->stream>>>(c->d_btoff, n_docs);
    batch_gather_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>(c->d_btok, c->d_bdoc, c->d_btoff, (u32)n_docs, c->d_brk);
    launches += 3;
    CU(cudaGetLastError());
    CU(cudaEventRecord(ev[1], c->stream));
    u64 m = 0;
    CU(cudaMemcpyAsync(&m, c->d_btoff + n_docs, sizeof m, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, ev[0], ev[1]));
    if (rebuild)
    {
        c->rt_merges.assign(merges, merges + n_merges);
        c->rt_valid = true;
    }
    st->n_input = n_input;
    st->n_merges = n_merges;
    st->n_tokens = m;
    st->kernel_launches = launches;
    st->ms_device = ms;
    *n_tokens = (size_t)m;
    return 0;
}

int bpe_cuda_ctx_encode_batch(bpe_cuda_ctx_t *c, const uint8_t *bytes, const uint64_t *offsets, size_t n_docs,
                              const bpe_pair_t *merges, size_t n_merges, uint32_t *tokens, uint64_t *tok_offsets,
                              bpe_cuda_stats_t *stats)
{
    if (!c || !tok_offsets || (!tokens && offsets && offsets[n_docs] > offsets[0]))
    {
        set_error("invalid argument: NULL context or output buffer");
        return BPE_CUDA_ERR_ARG;
    }
    int rc = batch_check(bytes, offsets, n_docs, merges, n_merges);
    if (rc)
        return rc;
    const auto t0 = std::chrono::steady_clock::now();
    bpe_cuda_stats_t st;
    size_t m = 0;
    if ((rc = batch_run(c, bytes, offsets, n_docs, merges, n_merges, &m, &st)))
        return rc;
    const auto h0 = std::chrono::steady_clock::now();
    CU(cudaMemcpyAsync(tok_offsets, c->d_btoff, (n_docs + 1) * sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (m && (rc = download_staged(c, tokens, c->d_brk, m * sizeof(u32))))
        return rc;
    const auto t1 = std::chrono::steady_clock::now();
    st.ms_d2h = std::chrono::duration<double, std::milli>(t1 - h0).count();
    st.ms_total = std::chrono::duration<double, std::milli>(t1 - t0).count();
    if (stats)
        *stats = st;
    return 0;
}

int bpe_cuda_encode_batch(const uint8_t *bytes, const uint64_t *offsets, size_t n_docs, const bpe_pair_t *merges,
                          size_t n_merges, uint32_t **tokens_out, uint64_t **tok_offsets_out, size_t *n_tokens,
                          bpe_cuda_stats_t *stats)
{
    if (!tokens_out || !tok_offsets_out || !n_tokens)
    {
        set_error("invalid argument: NULL output pointer");
        return BPE_CUDA_ERR_ARG;
    }
    *tokens_out = nullptr;
    *tok_offsets_out = nullptr;
    *n_tokens = 0;
    int rc = batch_check(bytes, offsets, n_docs, merges, n_merges);
    if (rc)
        return rc;
    const auto t0 = std::chrono::steady_clock::now();
    bpe_cuda_ctx_t *c = nullptr;
    if ((rc = bpe_cuda_ctx_create(0, &c)))
        return rc;
    bpe_cuda_stats_t st;
    size_t m = 0;
    uint32_t *tok = nullptr;
    uint64_t *toff = nullptr;
    auto body = [&]() -> int {
        int r = batch_run(c, bytes, offsets, n_docs, merges, n_merges, &m, &st);
        if (r)
            return r;
        tok = (uint32_t *)malloc(std::max<size_t>(1, m) * sizeof(uint32_t));
        toff = (uint64_t *)malloc((n_docs + 1) * sizeof(uint64_t));
        if (!tok || !toff)
        {
            set_error("out of host memory");
            return BPE_CUDA_ERR_NOMEM;
        }
        const auto h0 = std::chrono::steady_clock::now();
        CU(cudaMemcpyAsync(toff, c->d_btoff, (n_docs + 1) * sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        if (m && (r = download_staged(c, tok, c->d_brk, m * sizeof(u32))))
            return r;
        st.ms_d2h = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - h0).count();
        return 0;
    };
    rc = body();
    bpe_cuda_ctx_destroy(c);
    if (rc)
    {
        free(tok);
        free(toff);
        return rc;
    }
    st.ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (stats)
        *stats = st;
    *tokens_out = tok;
    *tok_offsets_out = toff;
    *n_tokens = m;
    return 0;
}

// ---- batch decode (D4 in bpe_decode.cuh) ------------------------------------------------------
// Every argument is checked before any device call, as batch_check() does for encode.
static int decode_batch_check(const uint32_t *tokens, const uint64_t *tok_offsets, size_t n_docs, const bpe_pair_t *merges,
                              size_t n_merges)
{
    if (!tok_offsets || (!merges && n_merges))
    {
        set_error("invalid argument: NULL tok_offsets or merges");
        return BPE_CUDA_ERR_ARG;
    }
    if (n_docs >= 0xFFFFFFFFu) // n_docs + 1 entries are indexed with 32 bits on the device
    {
        set_error("invalid argument: %zu documents (at most 4,294,967,294 in one batch)", n_docs);
        return BPE_CUDA_ERR_ARG;
    }
    for (size_t i = 0; i < n_docs; i++)
        if (tok_offsets[i + 1] < tok_offsets[i])
        {
            set_error("invalid argument: tok_offsets[%zu] < tok_offsets[%zu] (offsets must not decrease)", i + 1, i);
            return BPE_CUDA_ERR_ARG;
        }
    if (!tokens && tok_offsets[n_docs] > tok_offsets[0])
    {
        set_error("invalid argument: NULL tokens");
        return BPE_CUDA_ERR_ARG;
    }
    return check_merges(merges, n_merges);
}

// Decode the batch on the device: the bytes go to c->d_dec_out[0 .. *n_bytes), the byte offsets to the host array
// byte_offsets[0 .. n_docs].  st gets every field of the result but ms_total; its ms_d2h covers the offsets.
static int decode_batch_run(bpe_cuda_ctx *c, const uint32_t *tokens, const uint64_t *tok_offsets, size_t n_docs,
                            const bpe_pair_t *merges, size_t n_merges, uint64_t *byte_offsets, size_t *n_bytes,
                            bpe_cuda_stats_t *st)
{
    int rc;
    CU(cudaSetDevice(c->device));
    memset(st, 0, sizeof *st);
    const u64 base = tok_offsets[0], N = tok_offsets[n_docs] - base;
    st->n_input = N;
    st->n_merges = n_merges;
    c->dec_n_out = 0;
    *n_bytes = 0;
    if (!N) // no id at all: every document is empty, and nothing is launched
    {
        memset(byte_offsets, 0, (n_docs + 1) * sizeof(uint64_t));
        return 0;
    }
    const u64 nt = (N + DEC_TILE - 1) / DEC_TILE;
    bool rebuilt = false;
    {
        const auto h0 = std::chrono::steady_clock::now();
        if ((rc = dec_vocab(c, merges, n_merges, &rebuilt)) || (rc = dec_reserve(c->d_dbtok, c->dbtok_cap, (size_t)N)) ||
            (rc = dec_reserve(c->d_dbtoff, c->dbtoff_cap, n_docs + 1)) ||
            (rc = dec_reserve(c->d_dbboff, c->dbboff_cap, n_docs + 1)) || (rc = dec_reserve(c->d_dbtile, c->dbtile_cap, nt + 1)))
            return rc;
        CU(cudaMemcpyAsync(c->d_dbtok, tokens + base, N * sizeof(u32), cudaMemcpyHostToDevice, c->stream));
        CU(cudaMemcpyAsync(c->d_dbtoff, tok_offsets, (n_docs + 1) * sizeof(u64), cudaMemcpyHostToDevice, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        st->ms_h2d = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - h0).count();
    }
    const DecodeDocs d{c->d_dbtoff, base, c->d_dbtile, c->d_dbboff};
    const u64 l0 = c->launches;
    size_t nb = 0;
    float ms = 0;
    rc = decode_run(c, c->d_dbtok, N, &d, n_docs + 1, &nb, &ms);
    if (rc == BPE_CUDA_ERR_ARG)
    {
        // the device only says that some id is outside the vocabulary; the host still holds the ids
        const size_t V = 256 + n_merges;
        const uint32_t *t = tokens + base;
        u64 k = 0;
        while (k < N && t[k] < V)
            k++;
        if (k < N)
        {
            const size_t doc = (size_t)(std::upper_bound(tok_offsets, tok_offsets + n_docs + 1, base + k) - tok_offsets) - 1;
            set_error("decode_batch: document %zu holds id %u, outside the vocabulary (%zu entries)", doc, t[k], V);
        }
    }
    if (rc)
        return rc;
    const auto h0 = std::chrono::steady_clock::now();
    CU(cudaMemcpyAsync(byte_offsets, c->d_dbboff, (n_docs + 1) * sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    st->ms_d2h = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - h0).count();
    st->n_tokens = nb;
    st->kernel_launches = c->launches - l0;
    st->table_rehashes = rebuilt;
    st->ms_device = ms;
    *n_bytes = nb;
    return 0;
}

int bpe_cuda_ctx_decode_batch(bpe_cuda_ctx_t *c, const uint32_t *tokens, const uint64_t *tok_offsets, size_t n_docs,
                              const bpe_pair_t *merges, size_t n_merges, uint64_t *byte_offsets, size_t *n_bytes,
                              bpe_cuda_stats_t *stats)
{
    int rc = decode_batch_check(tokens, tok_offsets, n_docs, merges, n_merges);
    if (rc)
        return rc;
    if (!byte_offsets || !n_bytes)
    {
        set_error("invalid argument: NULL output buffer");
        return BPE_CUDA_ERR_ARG;
    }
    if (!c)
    {
        set_error("invalid argument: NULL context");
        return BPE_CUDA_ERR_ARG;
    }
    const auto t0 = std::chrono::steady_clock::now();
    bpe_cuda_stats_t st;
    if ((rc = decode_batch_run(c, tokens, tok_offsets, n_docs, merges, n_merges, byte_offsets, n_bytes, &st)))
        return rc;
    st.ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (stats)
        *stats = st;
    return 0;
}

int bpe_cuda_decode_batch(const uint32_t *tokens, const uint64_t *tok_offsets, size_t n_docs, const bpe_pair_t *merges,
                          size_t n_merges, uint8_t **bytes_out, uint64_t **byte_offsets_out, size_t *n_bytes,
                          bpe_cuda_stats_t *stats)
{
    if (!bytes_out || !byte_offsets_out || !n_bytes)
    {
        set_error("invalid argument: NULL output pointer");
        return BPE_CUDA_ERR_ARG;
    }
    *bytes_out = nullptr;
    *byte_offsets_out = nullptr;
    *n_bytes = 0;
    int rc = decode_batch_check(tokens, tok_offsets, n_docs, merges, n_merges);
    if (rc)
        return rc;
    const auto t0 = std::chrono::steady_clock::now();
    bpe_cuda_ctx_t *c = nullptr;
    if ((rc = bpe_cuda_ctx_create(0, &c)))
        return rc;
    bpe_cuda_stats_t st;
    size_t nb = 0;
    uint8_t *out = nullptr;
    uint64_t *boff = nullptr;
    auto body = [&]() -> int {
        boff = (uint64_t *)malloc((n_docs + 1) * sizeof(uint64_t));
        if (!boff)
        {
            set_error("out of host memory");
            return BPE_CUDA_ERR_NOMEM;
        }
        int r = decode_batch_run(c, tokens, tok_offsets, n_docs, merges, n_merges, boff, &nb, &st);
        if (r)
            return r;
        out = (uint8_t *)malloc(nb + 1); // +1: the terminator bpe_cuda_decode() appends too
        if (!out)
        {
            set_error("out of host memory");
            return BPE_CUDA_ERR_NOMEM;
        }
        out[nb] = 0;
        const auto h0 = std::chrono::steady_clock::now();
        if ((r = bpe_cuda_ctx_decode_download(c, out)))
            return r;
        st.ms_d2h += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - h0).count();
        return 0;
    };
    rc = body();
    bpe_cuda_ctx_destroy(c);
    if (rc)
    {
        free(out);
        free(boff);
        return rc;
    }
    st.ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (stats)
        *stats = st;
    *bytes_out = out;
    *byte_offsets_out = boff;
    *n_bytes = nb;
    return 0;
}

// ---- one-call entry points -------------------------------------------------------------------
// What the ranks of one call share: meeting points (after the ingest, after the run) and the result buffers.
struct HostJob
{
    int world = 1;
    std::mutex mu;
    std::condition_variable cv;
    int arrived[3] = {0, 0, 0};
    bool failed = false;
    std::vector<size_t> rank_bytes, rank_tokens;
    std::vector<int> rank_nul;
    u32 *tokens = nullptr;       // malloc'd, all ranks' ids in rank order (the caller free()s it, main.c:22)
    bpe_pair_t *merges = nullptr; // malloc'd (rank 0's copy)
    size_t n_merges = 0, total_tokens = 0;
    // every rank arrives; false if some rank has failed (nobody waits for it any longer)
    bool meet(int phase)
    {
        std::unique_lock<std::mutex> lk(mu);
        arrived[phase]++;
        cv.notify_all();
        cv.wait(lk, [&] { return failed || arrived[phase] >= world; });
        return !failed;
    }
    void abort()
    {
        std::lock_guard<std::mutex> lk(mu);
        failed = true;
        cv.notify_all();
    }
};

struct RankJob
{
    int rank, world, rc;
    HostJob *job;
    const uint8_t *bytes; // host shard, or
    const char *path;     // the file and this rank's byte range of it
    uint64_t foff, flen;
    size_t n;
    ncclUniqueId id;
    uint64_t max_merges;
    const bpe_pair_t *enc;
    size_t n_enc;
    bool encode;
    bpe_cuda_stats_t stats;
    char err[512];
};

static void rank_body(RankJob *j);
static void rank_main(RankJob *j)
{
    // (a C++ exception escaping a thread would terminate the process)
    try
    {
        rank_body(j);
    }
    catch (const std::exception &e)
    {
        j->rc = BPE_CUDA_ERR_NOMEM;
        snprintf(j->err, sizeof j->err, "rank %d: %s", j->rank, e.what());
        j->job->abort();
    }
}

static void rank_body(RankJob *j)
{
    bpe_cuda_ctx_t *c = nullptr;
    HostJob *job = j->job;
    j->err[0] = 0;
    auto fail = [&](int rc) {
        j->rc = rc;
        snprintf(j->err, sizeof j->err, "%s", bpe_cuda_last_error());
        job->abort();
        if (c)
            bpe_cuda_ctx_destroy(c);
    };
    auto peer_failed = [&]() {
        j->rc = BPE_CUDA_ERR_STATE;
        snprintf(j->err, sizeof j->err, "another rank failed");
        if (c)
            bpe_cuda_ctx_destroy(c);
    };
    int rc = bpe_cuda_ctx_create(j->rank, &c);
    if (rc)
        return fail(rc);
    if (j->world > 1 && (rc = bpe_cuda_ctx_set_comm(c, j->rank, j->world, &j->id)))
        return fail(rc);
    const auto t0 = std::chrono::steady_clock::now();
    if (j->path)
    {
        size_t got = 0;
        int nul = 0;
        if ((rc = bpe_cuda_ctx_upload_file(c, j->path, j->foff, j->flen, &got, &nul)))
            return fail(rc);
        job->rank_bytes[(size_t)j->rank] = got;
        job->rank_nul[(size_t)j->rank] = nul;
        if (j->world > 1)
        {
            // strlen semantics (bpe.c:555): the corpus ends at the FIRST 0x00 of the file; shards behind it are empty
            if (!job->meet(0))
                return peer_failed();
            for (int q = 0; q < j->rank; q++)
                if (job->rank_nul[(size_t)q] && (rc = bpe_cuda_ctx_truncate(c, 0)))
                    return fail(rc);
        }
    }
    else if ((rc = bpe_cuda_ctx_upload(c, j->bytes, j->n)))
        return fail(rc);
    const double ms_h2d = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    rc = j->encode ? bpe_cuda_ctx_encode(c, j->enc, j->n_enc, &j->stats) : bpe_cuda_ctx_train(c, j->max_merges, &j->stats);
    if (rc)
        return fail(rc);
    size_t nm = 0, nt = 0;
    bpe_cuda_ctx_result_sizes(c, &nm, &nt);
    job->rank_tokens[(size_t)j->rank] = nt;
    if (!job->meet(1))
        return peer_failed();
    // results go straight into the caller's malloc'd buffers: rank 0 allocates once every rank's size is known
    if (j->rank == 0)
    {
        size_t total = 0;
        for (size_t v : job->rank_tokens)
            total += v;
        job->total_tokens = total;
        job->n_merges = nm;
        job->tokens = (u32 *)malloc((total ? total : 1) * sizeof(u32));
        job->merges = (bpe_pair_t *)malloc((nm ? nm : 1) * sizeof(bpe_pair_t));
        if (!job->tokens || !job->merges)
        {
            set_error("out of host memory");
            return fail(BPE_CUDA_ERR_NOMEM);
        }
    }
    if (!job->meet(2))
        return peer_failed();
    size_t off = 0;
    for (int q = 0; q < j->rank; q++)
        off += job->rank_tokens[(size_t)q];
    const auto t1 = std::chrono::steady_clock::now();
    if ((rc = bpe_cuda_ctx_download_pageable(c, j->rank == 0 ? job->merges : nullptr, job->tokens + off)))
        return fail(rc);
    j->stats.ms_h2d = ms_h2d;
    j->stats.ms_d2h = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t1).count();
    j->rc = 0;
    bpe_cuda_ctx_destroy(c);
}

// bytes != NULL: the corpus is in host memory; else `path` names the file it is read from (chunked, pinned, overlapped
// with the copy and the widening: bpe_cuda_ctx_upload_file)
static int run_host(const uint8_t *bytes, size_t n_in, const char *path, uint64_t max_merges, const bpe_pair_t *enc, size_t n_enc,
                    bool encode, int n_gpus, bpe_pair_t **merges_out, size_t *n_merges, uint32_t **tokens_out, size_t *n_tokens,
                    bpe_cuda_stats_t *stats)
{
    if ((!bytes && !path) || !tokens_out || !n_tokens || (!encode && (!merges_out || !n_merges)) || n_gpus < 1 || n_gpus > MAX_RANKS)
    {
        set_error("invalid argument");
        return BPE_CUDA_ERR_ARG;
    }
    const auto t0 = std::chrono::steady_clock::now();
    size_t n = 0;
    if (bytes)
    {
        const void *z = memchr(bytes, 0, n_in); // strlen semantics, bpe.c:555
        n = z ? (size_t)((const uint8_t *)z - bytes) : n_in;
        if (!encode && n < 2)
        {
            set_error("Error: File contains less than 2 characters");
            return BPE_CUDA_ERR_SHORT;
        }
    }
    else
    {
        struct stat sb;
        if (stat(path, &sb) != 0)
        {
            set_error("fopen: %s", strerror(errno)); // bpe.c:133-137
            return BPE_CUDA_ERR_ARG;
        }
        n = (size_t)sb.st_size; // (the first NUL, if any, is found while the file is read)
    }
    {
        // a rank without a device would fail at once and leave its peers waiting in the communicator setup
        const int ndev = bpe_cuda_device_count();
        if (n_gpus > ndev)
        {
            set_error("n_gpus = %d but only %d CUDA device(s) are visible", n_gpus, ndev);
            return BPE_CUDA_ERR_CUDA;
        }
    }
    HostJob job;
    job.world = n_gpus;
    job.rank_bytes.assign((size_t)n_gpus, 0);
    job.rank_tokens.assign((size_t)n_gpus, 0);
    job.rank_nul.assign((size_t)n_gpus, 0);
    std::vector<RankJob> jobs((size_t)n_gpus);
    ncclUniqueId id;
    memset(&id, 0, sizeof id);
    if (n_gpus > 1)
    {
        int rc = bpe_cuda_nccl_unique_id(&id);
        if (rc)
            return rc;
    }
    for (int r = 0; r < n_gpus; r++)
    {
        RankJob &j = jobs[(size_t)r];
        // (shard borders on multiples of 16 bytes: the ingest widens 16 bytes per thread)
        size_t lo = (size_t)((unsigned __int128)n * (unsigned)r / (unsigned)n_gpus);
        size_t hi = (size_t)((unsigned __int128)n * (unsigned)(r + 1) / (unsigned)n_gpus);
        if (path)
        {
            lo = (r == 0) ? 0 : (lo & ~(size_t)15);
            hi = (r == n_gpus - 1) ? n : (hi & ~(size_t)15);
        }
        j.rank = r;
        j.world = n_gpus;
        j.rc = -1;
        j.job = &job;
        j.bytes = bytes ? bytes + lo : nullptr;
        j.path = bytes ? nullptr : path;
        j.foff = lo;
        j.flen = hi - lo;
        j.n = hi - lo;
        j.id = id;
        j.max_merges = max_merges;
        j.enc = enc;
        j.n_enc = n_enc;
        j.encode = encode;
    }
    if (n_gpus == 1)
        rank_main(&jobs[0]);
    else
    {
        std::vector<std::thread> th;
        for (int r = 0; r < n_gpus; r++)
            th.emplace_back(rank_main, &jobs[(size_t)r]);
        for (auto &t : th)
            t.join();
    }
    int first_rc = 0;
    for (auto &j : jobs)
        if (j.rc && (!first_rc || first_rc == BPE_CUDA_ERR_STATE))
        {
            set_error(n_gpus > 1 ? "rank %d: %s" : "%.0d%s", n_gpus > 1 ? j.rank : 0, j.err);
            first_rc = j.rc;
        }
    if (first_rc)
    {
        free(job.tokens);
        free(job.merges);
        return first_rc;
    }
    if (merges_out)
    {
        *merges_out = job.merges;
        *n_merges = job.n_merges;
    }
    else
        free(job.merges);
    *tokens_out = job.tokens;
    *n_tokens = job.total_tokens;
    if (stats)
    {
        *stats = jobs[0].stats;
        for (auto &j : jobs)
        {
            stats->ms_device = std::max(stats->ms_device, j.stats.ms_device);
            stats->ms_h2d = std::max(stats->ms_h2d, j.stats.ms_h2d);
            stats->ms_d2h = std::max(stats->ms_d2h, j.stats.ms_d2h);
        }
        stats->n_tokens = job.total_tokens;
        stats->ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
    return 0;
}

int bpe_cuda_train(const uint8_t *bytes, size_t n, uint64_t max_merges, int n_gpus, bpe_pair_t **merges_out, size_t *n_merges,
                   uint32_t **tokens_out, size_t *n_tokens, bpe_cuda_stats_t *stats)
{
    if (!bytes)
    {
        set_error("invalid argument");
        return BPE_CUDA_ERR_ARG;
    }
    return run_host(bytes, n, nullptr, max_merges, nullptr, 0, false, n_gpus, merges_out, n_merges, tokens_out, n_tokens, stats);
}

int bpe_cuda_encode(const uint8_t *bytes, size_t n, const bpe_pair_t *merges, size_t n_merges, int n_gpus,
                    uint32_t **tokens_out, size_t *n_tokens, bpe_cuda_stats_t *stats)
{
    if ((!merges && n_merges) || !bytes)
        return BPE_CUDA_ERR_ARG;
    return run_host(bytes, n, nullptr, 0, merges, n_merges, true, n_gpus, nullptr, nullptr, tokens_out, n_tokens, stats);
}

int bpe_cuda_train_file(const char *path, uint64_t max_merges, int n_gpus, bpe_pair_t **merges_out, size_t *n_merges,
                        uint32_t **tokens_out, size_t *n_tokens, bpe_cuda_stats_t *stats)
{
    if (!path)
    {
        set_error("invalid argument");
        return BPE_CUDA_ERR_ARG;
    }
    return run_host(nullptr, 0, path, max_merges, nullptr, 0, false, n_gpus, merges_out, n_merges, tokens_out, n_tokens, stats);
}

int bpe_cuda_encode_file(const char *path, const bpe_pair_t *merges, size_t n_merges, int n_gpus, uint32_t **tokens_out,
                         size_t *n_tokens, bpe_cuda_stats_t *stats)
{
    if ((!merges && n_merges) || !path)
        return BPE_CUDA_ERR_ARG;
    return run_host(nullptr, 0, path, 0, merges, n_merges, true, n_gpus, nullptr, nullptr, tokens_out, n_tokens, stats);
}

} // extern "C"
