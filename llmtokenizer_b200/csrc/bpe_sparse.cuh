// LAYOUT_SPARSE: the late phase of a one-GPU run, where a pass replaces a tiny share of the stream (DESIGN.md §3, §4).
//
// A token lives at the byte offset where it starts: tok[p] is the id that starts at byte p, SENT at every byte
// that starts no token.  start_of[e] is the start of the token whose last byte is e (meaningful at token ends).
// With len[] = byte length per id:
//   next(p) = p + len[tok[p]],   prev(p) = start_of[p - 1],
//   replacing (a at p, b at q) by z:  tok[p] = z, tok[q] = SENT, start_of[q + len[b] - 1] = p.
// Nothing is ever compacted, so a pass costs in proportion to the occurrences it looks at, not to the stream.
//
// Occurrences come from two structures.  Once (a, b) is merged no new instance of it can appear: a new adjacency
// always involves the id the merge that made it created.  So
//   * the FROZEN INDEX, built at the switch, lists every pair instance that exists then, bucketed by the slot of its
//     pair in a copy of the pair table's keys (later rehashes move the live table's slots, not the copy's); it
//     serves every pair whose two ids both existed at the switch (ids < zsw), and each of its lists is read once;
//   * CREATION LISTS: the pass that makes id z appends the positions where it wrote z.  A pair with a younger id
//     reads the list of that id (the shorter one if both are young) and checks every entry against the stream.
// Every entry is checked (tok[p] == a and tok[next(p)] == b), so entries whose token has since been merged away, on
// either side, are skipped: the replaced right-hand token is overwritten with SENT.
//
// A pass is two launches, both chained with programmatic dependent launch: sparse_scan_kernel (plans the lists of the
// pass's merges, checks the entries, finds the replacements and emits exactly the pair-count deltas
// replace_stream_kernel emits; it reads the stream only), then the delta application, whose blocks also rewrite the
// stream and fill the creation lists (sparse_rewrite, bpe_kernels.cuh).  Splitting the read from the write keeps every
// neighbour a replacement looks at the one of the stream before the pass.
namespace bpe
{

constexpr int SPX_THREADS = 256;
constexpr int SPX_ITEMS = 16;
constexpr u32 SPX_TILE = SPX_THREADS * SPX_ITEMS; // elements per block-tile of the conversions and scans

// exclusive block scan over SPX_THREADS threads; s_w holds SPX_THREADS / 32 words
__device__ __forceinline__ u32 spx_block_scan(u32 v, u32 *s_w, u32 &total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u32 incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const u32 x = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o)
            incl += x;
    }
    if (lane == 31)
        s_w[warp] = incl;
    __syncthreads();
    u32 woff = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < SPX_THREADS / 32; w++)
    {
        const u32 x = s_w[w];
        woff += (w < warp) ? x : 0u;
        tot += x;
    }
    __syncthreads();
    total = tot;
    return woff + incl - v;
}

// ---- generic exclusive scan of u32 (in place allowed): tile sums, one-block scan of the sums, apply ----------------
__global__ void __launch_bounds__(SPX_THREADS) spx_tile_sums_kernel(const u32 *in, u64 n, u32 *tsum)
{
    __shared__ u32 s_w[SPX_THREADS / 32];
    const u64 base = (u64)blockIdx.x * SPX_TILE + (u64)threadIdx.x * SPX_ITEMS;
    u32 s = 0;
    for (int k = 0; k < SPX_ITEMS; k++)
        s += (base + k < n) ? in[base + k] : 0u;
    u32 total;
    spx_block_scan(s, s_w, total);
    if (threadIdx.x == 0)
        tsum[blockIdx.x] = total;
}

__global__ void __launch_bounds__(1024) spx_top_scan_kernel(u32 *v, u32 m)
{
    __shared__ u32 s_w[32];
    __shared__ u32 s_carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0)
        s_carry = 0;
    __syncthreads();
    for (u32 base = 0; base < m; base += 1024)
    {
        const u32 i = base + threadIdx.x;
        const u32 x = i < m ? v[i] : 0u;
        u32 incl = x;
        for (int o = 1; o < 32; o <<= 1)
        {
            const u32 y = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o)
                incl += y;
        }
        if (lane == 31)
            s_w[warp] = incl;
        __syncthreads();
        u32 woff = 0, tot = 0;
        for (int w = 0; w < 32; w++)
        {
            woff += (w < warp) ? s_w[w] : 0u;
            tot += s_w[w];
        }
        const u32 carry = s_carry;
        if (i < m)
            v[i] = carry + woff + incl - x;
        __syncthreads();
        if (threadIdx.x == 0)
            s_carry = carry + tot;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(SPX_THREADS) spx_apply_scan_kernel(const u32 *in, u32 *out, u64 n, const u32 *tsum)
{
    __shared__ u32 s_w[SPX_THREADS / 32];
    const u64 base = (u64)blockIdx.x * SPX_TILE + (u64)threadIdx.x * SPX_ITEMS;
    u32 v[SPX_ITEMS], s = 0;
    for (int k = 0; k < SPX_ITEMS; k++)
    {
        v[k] = (base + k < n) ? in[base + k] : 0u;
        s += v[k];
    }
    u32 total;
    u32 r = tsum[blockIdx.x] + spx_block_scan(s, s_w, total);
    for (int k = 0; k < SPX_ITEMS; k++)
        if (base + k < n)
        {
            out[base + k] = r;
            r += v[k];
        }
}

// ---- DENSE -> SPARSE ------------------------------------------------------------------------------------------------
// Pass 1 over the dense stream tok[cur][0..n): per tile the byte length of its tokens, and per pair instance one
// count in the slot of its pair (the frozen index is keyed by a copy of the table's keys, ikey).
__global__ void __launch_bounds__(SPX_THREADS) sparse_count_kernel(DevState *st, u32 *tsum, u32 *icnt)
{
    __shared__ u32 s_w[SPX_THREADS / 32];
    const u32 *t = st->tok[st->cur];
    const u64 n = st->n;
    const u64 base = (u64)blockIdx.x * SPX_TILE + (u64)threadIdx.x * SPX_ITEMS;
    u32 s = 0;
    for (int k = 0; k < SPX_ITEMS; k++)
    {
        const u64 i = base + k;
        if (i >= n)
            break;
        const u32 x = t[i];
        s += st->slen[x];
        if (i + 1 < n)
        {
            const u32 y = t[i + 1];
            const u64 slot = table_find(st->ikey, st->icap, (u64)x | ((u64)y << 32), murmur3_pair(x, y));
            if (slot == NO_SLOT)
                atomicOr(&st->err, ERR_MISSING_KEY);
            else
                atomicAdd(&icnt[slot], 1u);
        }
    }
    u32 total;
    spx_block_scan(s, s_w, total);
    if (threadIdx.x == 0)
        tsum[blockIdx.x] = total;
}

// Pass 2: every token to its byte offset in the other buffer (filled with SENT beforehand), every pair instance's
// position into its list of the frozen index (ioff = exclusive scan of the counts, icur = cursors).
__global__ void __launch_bounds__(SPX_THREADS) sparse_scatter_kernel(DevState *st, const u32 *tsum, u32 *icur)
{
    __shared__ u32 s_w[SPX_THREADS / 32];
    const u32 *t = st->tok[st->cur];
    u32 *out = st->tok[st->cur ^ 1u];
    const u64 n = st->n;
    const u64 base = (u64)blockIdx.x * SPX_TILE + (u64)threadIdx.x * SPX_ITEMS;
    u32 s = 0;
    for (int k = 0; k < SPX_ITEMS; k++)
        if (base + k < n)
            s += st->slen[t[base + k]];
    u32 total;
    u32 pos = tsum[blockIdx.x] + spx_block_scan(s, s_w, total);
    for (int k = 0; k < SPX_ITEMS; k++)
    {
        const u64 i = base + k;
        if (i >= n)
            break;
        const u32 x = t[i];
        out[pos] = x;
        if (i + 1 < n)
        {
            const u32 y = t[i + 1];
            const u64 slot = table_find(st->ikey, st->icap, (u64)x | ((u64)y << 32), murmur3_pair(x, y));
            if (slot != NO_SLOT)
                st->ipos[st->ioff[slot] + atomicAdd(&icur[slot], 1u)] = pos;
        }
        pos += st->slen[x];
    }
}

// Pass 3: start_of over the sparse tokens, into the buffer that held the dense stream; then the layout flips.
__global__ void __launch_bounds__(SPX_THREADS) sparse_start_kernel(DevState *st)
{
    const u32 *t = st->tok[st->cur ^ 1u];
    u32 *so = st->tok[st->cur];
    const u64 n0 = st->n0;
    for (u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x; p < n0; p += (u64)gridDim.x * blockDim.x)
    {
        const u32 x = t[p];
        if (x != SENT)
            so[p + st->slen[x] - 1] = (u32)p;
    }
}

__global__ void sparse_enter_kernel(DevState *st)
{
    u32 *so = st->tok[st->cur], *t = st->tok[st->cur ^ 1u];
    st->start_of = so;
    st->tok[0] = st->tok[1] = t;
    st->layout = st->layout_next = LAYOUT_SPARSE;
    st->pool_top = 0;
    for (int i = 0; i < BATCH_MAX; i++)
        st->sp_cnt[i] = 0;
}

// ---- SPARSE -> DENSE: the live starts in byte order ---------------------------------------------------------------
__global__ void __launch_bounds__(SPX_THREADS) sparse_live_count_kernel(DevState *st, u32 *bcnt)
{
    __shared__ u32 s_w[SPX_THREADS / 32];
    const u32 *t = st->tok[st->cur];
    const u64 n0 = st->n0;
    const u64 base = (u64)blockIdx.x * SPX_TILE + (u64)threadIdx.x * SPX_ITEMS;
    u32 s = 0;
    for (int k = 0; k < SPX_ITEMS; k++)
        s += (base + k < n0 && t[base + k] != SENT) ? 1u : 0u;
    u32 total;
    spx_block_scan(s, s_w, total);
    if (threadIdx.x == 0)
        bcnt[blockIdx.x] = total;
}

__global__ void __launch_bounds__(SPX_THREADS) sparse_compact_kernel(DevState *st, const u32 *boff)
{
    __shared__ u32 s_w[SPX_THREADS / 32];
    const u32 *t = st->tok[st->cur];
    u32 *out = st->start_of;
    const u64 n0 = st->n0;
    const u64 base = (u64)blockIdx.x * SPX_TILE + (u64)threadIdx.x * SPX_ITEMS;
    u32 v[SPX_ITEMS], s = 0;
    for (int k = 0; k < SPX_ITEMS; k++)
    {
        v[k] = (base + k < n0) ? t[base + k] : SENT;
        s += (v[k] != SENT) ? 1u : 0u;
    }
    u32 total;
    u32 r = boff[blockIdx.x] + spx_block_scan(s, s_w, total);
    for (int k = 0; k < SPX_ITEMS; k++)
        if (v[k] != SENT)
            out[r++] = v[k];
}

__global__ void sparse_leave_kernel(DevState *st)
{
    if (st->layout != LAYOUT_SPARSE)
        return;
    u32 *t = st->tok[st->cur];
    st->cur = 0;
    st->tok[0] = st->start_of;
    st->tok[1] = t;
    st->start_of = nullptr;
    st->layout = st->layout_next = LAYOUT_DENSE;
}

// ---- the pass -----------------------------------------------------------------------------------------------------
__device__ __forceinline__ u32 sp_prev_tok(const u32 *tok, const u32 *so, u32 p) { return p ? tok[so[p - 1]] : SENT; }

// one warp-aggregated atomicAdd per distinct address
__device__ __forceinline__ u32 sp_bump(u32 *ctr)
{
    const unsigned m = __activemask();
    const int lane = threadIdx.x & 31;
    const unsigned peers = __match_any_sync(m, (unsigned long long)ctr);
    const int leader = __ffs(peers) - 1;
    u32 base = 0;
    if (lane == leader)
        base = atomicAdd(ctr, (u32)__popc(peers));
    base = __shfl_sync(peers, base, leader);
    return base + (u32)__popc(peers & ((1u << lane) - 1u));
}

// Where the occurrences of merge i of the pass are listed.  kind 0: frozen index (positions of a), kind 1: creation
// list of a, kind 2: creation list of b (positions of b).
__device__ __forceinline__ void sparse_plan(const DevState *st, u32 a, u32 b, const u32 *&src, u32 &len, u32 &kind)
{
    const u32 zsw = st->zsw;
    src = nullptr;
    len = 0;
    kind = 0;
    if (a < zsw && b < zsw)
    {
        const u64 slot = table_find(st->ikey, st->icap, (u64)a | ((u64)b << 32), murmur3_pair(a, b));
        if (slot != NO_SLOT)
        {
            src = st->ipos + st->ioff[slot];
            len = st->ioff[slot + 1] - st->ioff[slot];
        }
        return;
    }
    const bool ya = a >= zsw, yb = b >= zsw;
    const u32 ca = ya ? st->cl_cnt[a] : ~0u, cb = yb ? st->cl_cnt[b] : ~0u;
    kind = (ca <= cb) ? 1u : 2u;
    const u32 t = (kind == 1) ? a : b;
    src = st->pool + st->cl_off[t];
    len = st->cl_cnt[t];
}

// The first of a sparse pass's two launches (the second, the delta application, rewrites the stream: sparse_rewrite).
// Every block plans the pass's lists itself (nb probes, L2 hits after the first block), so no launch of its own is
// needed for that, whichever launch decided the pass.  The counters it adds to (sp_cnt) are zero on entry: finish_pass
// clears them.
__global__ void __launch_bounds__(SPX_THREADS) sparse_scan_kernel(DevState *st, int32_t *delta)
{
    pdl_wait();
    pdl_launch_dependents();
    if (st->stop != STOP_RUN || st->skip)
        return;
    __shared__ u32 s_a[BATCH_MAX], s_b[BATCH_MAX], s_la[BATCH_MAX], s_lb[BATCH_MAX], s_len[BATCH_MAX], s_kind[BATCH_MAX];
    __shared__ const u32 *s_src[BATCH_MAX];
    __shared__ u32 s_pre[BATCH_MAX + 1];
    __shared__ unsigned long long s_bytes;
    const u32 nb = st->nb, z = st->z, VS = z + nb;
    const u32 *tok = st->tok[st->cur], *so = st->start_of;
    u32 *slen = st->slen;
    int32_t *gdelta = delta + HDR_INTS;
    if (threadIdx.x < BATCH_MAX)
    {
        const u32 i = threadIdx.x;
        const u32 a = i < nb ? st->ba[i] : SENT, b = i < nb ? st->bb[i] : SENT;
        const u32 *src = nullptr;
        u32 len = 0, kind = 0;
        if (i < nb)
            sparse_plan(st, a, b, src, len, kind);
        s_a[i] = a;
        s_b[i] = b;
        s_la[i] = i < nb ? slen[a] : 0;
        s_lb[i] = i < nb ? slen[b] : 0;
        s_len[i] = len;
        s_kind[i] = kind;
        s_src[i] = src;
        if (blockIdx.x == 0 && i < nb)
            slen[z + i] = s_la[i] + s_lb[i]; // (ids below z only are read in this launch)
    }
    if (threadIdx.x == 0)
        s_bytes = 0;
    __syncthreads();
    if (threadIdx.x == 0)
    {
        u32 r = 0;
        for (u32 i = 0; i < BATCH_MAX; i++)
        {
            s_pre[i] = r;
            r += s_len[i];
        }
        s_pre[BATCH_MAX] = r;
        if (blockIdx.x == 0)
        {
            for (u32 i = 0; i < nb; i++)
                st->sp_ent[i] = s_pre[i];
            st->sparse_entries += r;
            if (s_a[0] == s_b[0] && nb != 1)
                atomicOr(&st->err, ERR_PROBE); // a == a passes carry one merge
        }
    }
    __syncthreads();
    const u32 total = s_pre[BATCH_MAX];
    const bool same = (s_a[0] == s_b[0]);
    u32 my_bytes = 0;
    for (u32 e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x)
    {
        u32 i = 0;
        while (e >= s_pre[i + 1])
            i++;
        const u32 a = s_a[i], b = s_b[i], la = s_la[i], lb = s_lb[i];
        const u32 ent = s_src[i][e - s_pre[i]];
        my_bytes += 8;
        u32 p, q;
        if (s_kind[i] == 2)
        {
            q = ent;
            if (tok[q] != b || q == 0)
                continue;
            p = so[q - 1];
            my_bytes += 8;
            if (tok[p] != a)
                continue;
        }
        else
        {
            p = ent;
            if (tok[p] != a)
                continue;
            q = p + la;
            my_bytes += 4;
            if (tok[q] != b)
                continue;
        }
        const u64 off = (u64)i * 4 * VS;
        if (same)
        {
            // a == a: the run that holds p is paired from its left end (bpe.c:760-772), so only the entry at the
            // run's start walks it (SURVEY.md A.5, same_pair_range's delta rules)
            u32 x = sp_prev_tok(tok, so, p);
            my_bytes += 8;
            if (x == a)
                continue;
            u32 cur = p;
            bool first = true;
            for (;;)
            {
                const u32 q2 = cur + la;
                if (tok[q2] != a)
                    break;
                const u32 yp = q2 + la;
                const u32 y = tok[yp];
                const bool nm = (y == a) && (tok[yp + la] == a);
                const u32 xx = first ? x : a;
                if (xx != SENT)
                {
                    if (xx != a)
                        delta_add(st, gdelta, off + (u64)xx * 4 + 0, 1);
                    delta_add(st, gdelta, off + (u64)(first ? xx : z) * 4 + 2, 1);
                }
                if (y != SENT && !nm)
                {
                    if (y != a)
                        delta_add(st, gdelta, off + (u64)y * 4 + 1, 1);
                    delta_add(st, gdelta, off + (u64)y * 4 + 3, 1);
                }
                st->pass_buf[s_pre[0] + sp_bump(&st->sp_cnt[0])] = cur;
                my_bytes += 16 + 8 + 16;
                first = false;
                if (!nm)
                    break;
                cur = yp;
            }
            continue;
        }
        // a != b: the neighbours as replace_stream_kernel sees them (pm: a pair of the pass ends right in front,
        // nm: one starts right behind; the pass's 2*nb ids are all different)
        const u32 xp = p ? so[p - 1] : 0u;
        const u32 x = p ? tok[xp] : SENT;
        u32 xn = x;
        if (x != SENT && xp > 0)
            for (u32 j = 0; j < nb; j++)
                if (x == s_b[j])
                {
                    if (tok[so[xp - 1]] == s_a[j])
                        xn = z + j;
                    break;
                }
        const u32 yp = q + lb;
        const u32 y = tok[yp];
        bool nm = false;
        for (u32 j = 0; j < nb; j++)
            if (y == s_a[j])
            {
                nm = tok[yp + s_la[j]] == s_b[j];
                break;
            }
        if (x != SENT)
        {
            delta_add(st, gdelta, off + (u64)x * 4 + 0, 1);
            delta_add(st, gdelta, off + (u64)xn * 4 + 2, 1);
        }
        if (y != SENT && !nm)
        {
            delta_add(st, gdelta, off + (u64)y * 4 + 1, 1);
            delta_add(st, gdelta, off + (u64)y * 4 + 3, 1);
        }
        st->pass_buf[s_pre[i] + sp_bump(&st->sp_cnt[i])] = p;
        my_bytes += 24 + 8 + 16;
    }
    if (my_bytes)
        atomicAdd(&s_bytes, (unsigned long long)my_bytes);
    __syncthreads();
    // (a block that checked no entry adds nothing: a pass of a few thousand entries costs a few dozen global atomics)
    if (threadIdx.x == 0 && s_bytes)
        atomicAdd(&st->sparse_bytes, s_bytes);
}

} // namespace bpe
