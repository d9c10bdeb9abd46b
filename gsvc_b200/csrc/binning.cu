// Kernel group (2): tile/depth key duplication, in-house radix sort, tile ranges
// (SURVEY.md Appendix A.2; upstream stages duplicateWithKeys / SortPairs / identifyTileRanges).
//
// The reference order is "stable ascending sort of key = (tile << 32) | depth_key over instances
// emitted in Gaussian-index order".  Instead of a 6-pass global LSD sort (144 B of HBM traffic per
// instance) the sort is done MSD-first, shaped to the key:
//   digit 0 = the whole tile field.  A counting sort on it needs only the per-tile histogram
//             (atomics in the preprocess kernel), one exclusive scan over T tiles — which IS
//             identifyTileRanges — and one scatter pass (8 B written per instance);
//   digit 1 = the 32-bit depth key, sorted per tile bucket inside shared memory.
// Bit-exactness: each Gaussian emits at most one instance per tile, so "emission order within a
// tile" is "ascending Gaussian id"; sorting each bucket by the 64-bit composite
// (depth_key << 32 | id) therefore reproduces the stable order exactly, whatever order the scatter
// atomics land in.
#include "common.cuh"

namespace gsvc {

// ---- exclusive scan over tiles: offsets, ranges, num_rendered; resets the scatter cursors ----------
// Multi-CTA single-pass scan: CTA b scans its 1024 tiles (one tile per thread, coalesced), publishes
// its aggregate (flag bit 63) and adds up the aggregates of all predecessors (decoupled look-back on
// aggregates only: nothing depends on a predecessor's look-back, so there is no serial chain).
// b is NOT blockIdx.x but a ticket drawn on entry: whoever holds ticket b knows that tickets 0..b-1 were drawn by
// CTAs that are already running, so spinning on their aggregates cannot deadlock however the hardware orders or
// limits the residency of the grid (a 16-view 4K batch is 507 CTAs of 1024 threads, more than fit at once).
// The partials array sits right behind tile_count and is zeroed by the same memset.  The last CTA
// also writes num_rendered, tagged with the caller's ticket, straight into mapped pinned host memory
// so the host learns R as soon as the scan ends — long before the blend kernel finishes.
constexpr int SCAN_THREADS = 1024;
constexpr unsigned long long SCAN_FLAG = 1ull << 63;

__global__ void __launch_bounds__(SCAN_THREADS) tile_scan_kernel(int T, ImageView im, unsigned long long* host_slot,
                                                                 unsigned int ticket)
{
    __shared__ unsigned long long warp_sums[SCAN_THREADS / 32];
    __shared__ unsigned long long s_prefix;
    __shared__ int s_ticket;
    pdl_prologue();
    const int nb = (int)gridDim.x;
    if (threadIdx.x == 0) s_ticket = (int)atomicAdd(im.scan_partials + nb, 1ull);   // the word behind the aggregates
    __syncthreads();
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, b = s_ticket;
    const int t = b * SCAN_THREADS + tid;
    const unsigned int c = t < T ? im.tile_count[t] : 0u;
    unsigned long long v = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long o = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v += o;
    }
    if (lane == 31) warp_sums[wid] = v;
    __syncthreads();
    if (wid == 0) {
        unsigned long long w = warp_sums[lane];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned long long o = __shfl_up_sync(0xffffffffu, w, d);
            if (lane >= d) w += o;
        }
        warp_sums[lane] = w;  // inclusive over warps
        const unsigned long long total = __shfl_sync(0xffffffffu, w, 31);
        volatile unsigned long long* partials = im.scan_partials;
        if (lane == 0) partials[b] = SCAN_FLAG | total;
        unsigned long long prefix = 0ull;
        for (int base = b - 1; base >= 0; base -= 32) {
            const int idx = base - lane;
            unsigned long long a = 0ull;
            if (idx >= 0) {
                do { a = partials[idx]; } while (!(a & SCAN_FLAG));
                a &= ~SCAN_FLAG;
            }
#pragma unroll
            for (int d = 16; d >= 1; d >>= 1) a += __shfl_xor_sync(0xffffffffu, a, d);
            prefix += a;
        }
        if (lane == 0) {
            s_prefix = prefix;
            if (b == nb - 1) {
                const unsigned long long R = prefix + total;
                im.hdr->num_rendered = R;
                im.hdr->overflow = 0u;
                im.hdr->n_heavy = 0u;
                if (host_slot) *host_slot = ((unsigned long long)ticket << 40) | (R < (1ull << 40) ? R : (1ull << 40) - 1);
            }
        }
    }
    __syncthreads();
    if (t < T) {
        const unsigned long long incl = s_prefix + (wid ? warp_sums[wid - 1] : 0ull) + v;
        const unsigned long long excl = incl - c;
        im.tile_offset[t] = (unsigned int)excl;
        im.tile_cursor[t] = 0u;
        im.ranges[t] = c ? make_uint2((unsigned int)excl, (unsigned int)incl) : make_uint2(0u, 0u);
    }
}

cudaError_t launch_tile_scan(const DevSettings& s, ImageView im, unsigned long long* host_slot, unsigned int ticket,
                             cudaStream_t st)
{
    const int T = s.gx * s.gy * s.n_views;
    count_launch();
    return launch_pdl(tile_scan_kernel, dim3((T + SCAN_THREADS - 1) / SCAN_THREADS), dim3(SCAN_THREADS), st, T, im,
                      host_slot, ticket);
}

// ---- scatter: one instance (depth_key << 32 | id) per (Gaussian, tile in rect) into its tile bucket ----
// Slot = tile_offset + atomicAdd(cursor).  The atomic's round trip is the cost, so the warp walks the
// flattened list of all its (Gaussian, tile) pairs (common.cuh) and issues SCATTER_ILP full-width atomics
// before it consumes the first result: a warp needs ~(pairs / 128) round trips, whatever the rectangle sizes.
constexpr int SCATTER_ILP = 4;

// Sticky, process-wide count of scatter launches that ran out of instance capacity (their frames are invalid: the
// sort and blend kernels skip overflowed tiles).  The eager call notices an overflow from num_rendered and re-runs
// with a larger buffer; a CUDA-graph replay has nobody to do that, so its owner polls this counter after a
// synchronisation (gsvc_rast_overflow_events).
__device__ unsigned int g_overflow_events = 0u;

cudaError_t read_overflow_events(unsigned int* host_value, bool reset, cudaStream_t st)
{
    cudaError_t e = cudaMemcpyFromSymbolAsync(host_value, g_overflow_events, sizeof(unsigned int), 0,
                                              cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && reset) {
        static const unsigned int zero = 0u;
        e = cudaMemcpyToSymbolAsync(g_overflow_events, &zero, sizeof(unsigned int), 0, cudaMemcpyHostToDevice, st);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    return e;
}

// RAGGED: view v's Gaussians are rows rows.off[v] .. rows.off[v+1]-1 (virtual Gaussian = row); the grid is
// (ceil(max_v P_v / 256), n_views) and a CTA wholly past its view's rows leaves at once
template <bool RAGGED>
__global__ void __launch_bounds__(256) scatter_kernel(int P, int gx, int Tv, GeomView geo, ImageView im, BinView bin,
                                                      unsigned long long cap, int count_events, ViewRows rows)
{
    pdl_prologue();
    const int v = blockIdx.y;                       // view of the batch: virtual Gaussian v*P + g, tiles v*Tv + t
    const int Pv = RAGGED ? rows.off[v + 1] - rows.off[v] : P;
    if (RAGGED && (int)(blockIdx.x * blockDim.x) >= Pv) return;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const size_t gv = RAGGED ? (size_t)rows.off[v] + g : (size_t)v * P + g;
    const int tbase = v * Tv;
    ushort4 r = make_ushort4(0, 0, 0, 0);
    if (g < Pv) r = geo.rect[gv];
    const int w = (int)r.z - (int)r.x, h = (int)r.w - (int)r.y;
    const int area = (w > 0 && h > 0) ? w * h : 0;
    unsigned long long item = 0ull;
    if (area > 0) item = ((unsigned long long)ordered_u32(geo.feat2[gv].w) << 32) | (unsigned int)gv;

    const WarpTiles wt = warp_tiles_begin(area, r.x, r.y, w > 0 ? w : 1);
    for (int base = 0; base < wt.total; base += 32 * SCATTER_ILP) {
        int tile[SCATTER_ILP];
        unsigned int slot[SCATTER_ILP];
        unsigned long long it[SCATTER_ILP];
#pragma unroll
        for (int u = 0; u < SCATTER_ILP; u++) {
            int owner;
            tile[u] = warp_tiles_get(wt, base + 32 * u + lane, gx, owner);
            if (tile[u] >= 0) tile[u] += tbase;
            it[u] = __shfl_sync(0xffffffffu, item, owner);
            slot[u] = 0u;
            if (tile[u] >= 0) slot[u] = atomicAdd(im.tile_cursor + tile[u], 1u);
        }
#pragma unroll
        for (int u = 0; u < SCATTER_ILP; u++) {
            if (tile[u] >= 0) {
                const unsigned long long sl = (unsigned long long)im.tile_offset[tile[u]] + slot[u];
                if (sl < cap) {
                    bin.inst[sl] = it[u];
                } else if (atomicExch(&im.hdr->overflow, 1u) == 0u && count_events) {
                    atomicAdd(&g_overflow_events, 1u);     // once per overflowed launch
                }
            }
        }
    }
}

cudaError_t launch_scatter(const DevSettings& s, int P, GeomView g, ImageView im, BinView b, long long cap,
                           bool count_overflow_events, cudaStream_t st)
{
    const int Pmax = max_view_rows(s, P);
    if (Pmax <= 0) return cudaSuccess;
    count_launch();
    return launch_pdl(s.ragged ? scatter_kernel<true> : scatter_kernel<false>, dim3((Pmax + 255) / 256, s.n_views),
                      dim3(256), st, P, s.gx, s.gx * s.gy, g, im, b, (unsigned long long)cap,
                      count_overflow_events ? 1 : 0, s.rows);
}

// ---- per-tile sort of the 64-bit composites -----------------------------------------------------
// Normalised bitonic network (every compare-exchange moves the minimum to the lower index; slots past
// the bucket's end hold +inf, so any length works).  Typical buckets hold 50..150 instances: one WARP
// sorts one bucket entirely IN REGISTERS — element e = lane*R + r lives in register r of its lane, a
// compare-exchange at distance < R is a register pair of the same lane, at distance >= R a 64-bit warp
// shuffle.  (The earlier shared-memory version of the same network was bound by shared-memory
// wavefronts — ncu: 390 per bucket, l1tex 53 %, issue 37 % — not by instructions; the shuffle version
// moves 8 B per element per stage through that pipe instead of up to 32.)  Buckets above
// SORT_WARP_ITEMS are sorted by the whole CTA afterwards (shared memory up to SORT_SMEM_ITEMS, in place
// in global memory beyond).
constexpr int SORT_THREADS = 256;
constexpr int SORT_WARPS = SORT_THREADS / 32;
constexpr int SORT_WARP_ITEMS = 256;   // 8 registers of 64 bits per lane (the kernel tuned for typical buckets)
constexpr int SORT_WARP_ITEMS_BIG = 512;  // 16 registers per lane (the kernel tuned for dense scenes: more registers, fewer warps)
constexpr int SORT_SMEM_ITEMS = 2048;  // 16 KB

template <bool BLOCK, typename Ptr>
__device__ __forceinline__ void bitonic_sort(Ptr a, int n, int tid, int nthreads)
{
    int lg = 0;
    while ((1 << lg) < n) lg++;
    const int half = (1 << lg) >> 1;
    for (int p = 1; p <= lg; p++) {          // merge size k = 2^p
        const int k = 1 << p, hk = k >> 1;
        for (int i = tid; i < half; i += nthreads) {
            const int blk = i >> (p - 1), pos = i & (hk - 1);
            const int lo = blk * k + pos, hi = blk * k + k - 1 - pos;
            if (hi < n) {
                const unsigned long long x = a[lo], y = a[hi];
                if (x > y) { a[lo] = y; a[hi] = x; }
            }
        }
        if (BLOCK) __syncthreads(); else __syncwarp();
        for (int q = p - 2; q >= 0; q--) {   // half-cleaners, distance j = 2^q
            const int j = 1 << q;
            for (int i = tid; i < half; i += nthreads) {
                const int lo = ((i >> q) << (q + 1)) + (i & (j - 1)), hi = lo + j;
                if (hi < n) {
                    const unsigned long long x = a[lo], y = a[hi];
                    if (x > y) { a[lo] = y; a[hi] = x; }
                }
            }
            if (BLOCK) __syncthreads(); else __syncwarp();
        }
    }
}

// One step of the network on R = 2^LR registers per lane, BLOCKED layout: element e = lane*R + r.  Element e is
// compared with element e ^ M and keeps the minimum iff bit DB of e is clear (DB = the highest set bit of M).
// The low LR bits of M pick the partner's register, the rest its lane: a step with M < R (13 of the 28 steps of
// a 128-element sort) never leaves the lane, every other one is one 64-bit shuffle per element.
template <int R, int M, int DB>
__device__ __forceinline__ void bitonic_step(unsigned long long (&v)[R], int lane)
{
    constexpr int LR = R == 1 ? 0 : R == 2 ? 1 : R == 4 ? 2 : R == 8 ? 3 : 4;
    constexpr int mr = M & (R - 1), ml = M >> LR;
    unsigned long long nv[R];
#pragma unroll
    for (int r = 0; r < R; r++) {
        const unsigned long long o = v[r ^ mr];
        const unsigned long long pv = ml ? __shfl_xor_sync(0xffffffffu, o, ml) : o;
        const bool keep_min = DB < LR ? ((r >> (DB < LR ? DB : 0)) & 1) == 0 : ((lane >> (DB >= LR ? DB - LR : 0)) & 1) == 0;
        nv[r] = ((v[r] < pv) == keep_min) ? v[r] : pv;
    }
#pragma unroll
    for (int r = 0; r < R; r++) v[r] = nv[r];
}

template <int R, int P, int Q>
struct BitonicHalfCleaners {   // distances 2^Q, 2^(Q-1), ..., 1
    static __device__ __forceinline__ void run(unsigned long long (&v)[R], int lane)
    {
        bitonic_step<R, (1 << Q), Q>(v, lane);
        BitonicHalfCleaners<R, P, Q - 1>::run(v, lane);
    }
};
template <int R, int P>
struct BitonicHalfCleaners<R, P, -1> {
    static __device__ __forceinline__ void run(unsigned long long (&)[R], int) {}
};
template <int R, int P, int LG>
struct BitonicMerges {          // merge sizes 2^P .. 2^LG
    static __device__ __forceinline__ void run(unsigned long long (&v)[R], int lane)
    {
        bitonic_step<R, (1 << P) - 1, P - 1>(v, lane);          // mirrored compare inside each 2^P block
        BitonicHalfCleaners<R, P, P - 2>::run(v, lane);
        BitonicMerges<R, P + 1, LG>::run(v, lane);
    }
};
template <int R, int LG>
struct BitonicMerges<R, LG + 1, LG> {
    static __device__ __forceinline__ void run(unsigned long long (&)[R], int) {}
};

// Sort one bucket of n <= 32*R composites by one warp, registers only; writes the sorted ids / depth keys.
template <int R, int LG>
__device__ __forceinline__ void sort_bucket_regs(const unsigned long long* __restrict__ src, int n, int lane,
                                                 unsigned int* __restrict__ ids, unsigned int* __restrict__ keys)
{
    unsigned long long v[R];
#pragma unroll
    for (int r = 0; r < R; r++) {
        const int e = lane * R + r;
        v[r] = e < n ? src[e] : ~0ull;
    }
    BitonicMerges<R, 1, LG>::run(v, lane);
#pragma unroll
    for (int r = 0; r < R; r++) {
        const int e = lane * R + r;
        if (e < n) {
            ids[e] = (unsigned int)v[r];
            keys[e] = (unsigned int)(v[r] >> 32);
        }
    }
}

// The same, reading and writing the bucket IN PLACE as (depth key, id) pairs split over two arrays: what the range
// split of a heavy bucket leaves behind (below).
template <int R, int LG>
__device__ __forceinline__ void sort_bucket_regs_soa(unsigned int* __restrict__ ids, unsigned int* __restrict__ keys,
                                                     int n, int lane)
{
    unsigned long long v[R];
#pragma unroll
    for (int r = 0; r < R; r++) {
        const int e = lane * R + r;
        v[r] = e < n ? (((unsigned long long)keys[e] << 32) | ids[e]) : ~0ull;
    }
    __syncwarp();
    BitonicMerges<R, 1, LG>::run(v, lane);
#pragma unroll
    for (int r = 0; r < R; r++) {
        const int e = lane * R + r;
        if (e < n) {
            ids[e] = (unsigned int)v[r];
            keys[e] = (unsigned int)(v[r] >> 32);
        }
    }
}

template <bool BIG>
__device__ __forceinline__ void sort_sub_bucket_warp(unsigned int* ids, unsigned int* keys, int n, int lane)
{
    if (n <= 32) sort_bucket_regs_soa<1, 5>(ids, keys, n, lane);
    else if (n <= 64) sort_bucket_regs_soa<2, 6>(ids, keys, n, lane);
    else if (n <= 128) sort_bucket_regs_soa<4, 7>(ids, keys, n, lane);
    else if (!BIG || n <= 256) sort_bucket_regs_soa<8, 8>(ids, keys, n, lane);
    else sort_bucket_regs_soa<16, 9>(ids, keys, n, lane);
}

// Heavy buckets (more entries than the CTA's shared-memory sort holds: thousands of instances on one tile).  One more
// MSD step, shaped to the data again: the depth keys of a tile are spread over its slab, so the bucket is split by a
// MONOTONE map of the depth key onto SPLIT_BINS ranges (counting sort inside the CTA: shared-memory histogram, scan,
// scatter into the output arrays used as scratch), and the ranges — a few hundred entries each — are sorted by the
// warps in registers like ordinary buckets.  A range that is still too large for a warp (thousands of equal depths)
// goes through the CTA's shared-memory network, and only a range beyond THAT falls back to the in-place global
// network the whole bucket used to take (O(n log^2 n) global-memory passes with a block barrier each: a 50k-entry
// tile serialised the chain for milliseconds).
constexpr int SPLIT_BINS = 1024;

template <bool BIG>
__device__ __forceinline__ void sort_heavy_bucket(unsigned long long* __restrict__ src, unsigned int* __restrict__ ids,
                                  unsigned int* __restrict__ keys, int nb, unsigned long long* s_items, int tid)
{
    constexpr int WARP_ITEMS = BIG ? SORT_WARP_ITEMS_BIG : SORT_WARP_ITEMS;
    unsigned int* s_off = reinterpret_cast<unsigned int*>(s_items);          // [SPLIT_BINS + 1] range starts
    unsigned int* s_cur = s_off + SPLIT_BINS + 1;                             // [SPLIT_BINS] counters, then cursors
    // (one word of padding: s_off holds an odd number of words, and with s_red starting on an odd word the compiler
    //  fetched s_red[0] together with s_cur[SPLIT_BINS - 1] in one 8-byte load — harmless, the extra word is dropped, but
    //  it reads a counter another thread is writing: racecheck's one finding on this library)
    unsigned int* s_red = s_cur + SPLIT_BINS + 1;                             // [2 * SORT_WARPS] min / max, then a list
    const int lane = tid & 31, warp = tid >> 5;
    // 1. depth-key range of the bucket
    unsigned int kmin = 0xffffffffu, kmax = 0u;
    for (int i = tid; i < nb; i += SORT_THREADS) {
        const unsigned int k = (unsigned int)(src[i] >> 32);
        kmin = min(kmin, k); kmax = max(kmax, k);
    }
    kmin = __reduce_min_sync(0xffffffffu, kmin); kmax = __reduce_max_sync(0xffffffffu, kmax);
    if (lane == 0) { s_red[warp] = kmin; s_red[SORT_WARPS + warp] = kmax; }
    for (int i = tid; i < SPLIT_BINS; i += SORT_THREADS) s_cur[i] = 0u;
    __syncthreads();
#pragma unroll
    for (int w = 0; w < SORT_WARPS; w++) { kmin = min(kmin, s_red[w]); kmax = max(kmax, s_red[SORT_WARPS + w]); }
    // ranges of ~128 entries on average (a warp sorts one in registers in ~2 us; thousands of 30-entry ranges would
    // be bound by their load -> sort -> store latency instead)
    int nbins = 64;
    while (nbins < SPLIT_BINS && nbins * 128 < nb) nbins <<= 1;
    // monotone (non-decreasing) in k: conversions, a product with a positive constant and a truncation all are
    const float scale = (float)nbins / ((float)(kmax - kmin) + 1.0f);
    auto bin_of = [&](unsigned int k) { return min(nbins - 1, (int)((float)(k - kmin) * scale)); };
    // 2. histogram, exclusive scan
    for (int i = tid; i < nb; i += SORT_THREADS) atomicAdd(&s_cur[bin_of((unsigned int)(src[i] >> 32))], 1u);
    __syncthreads();
    {
        // SPLIT_BINS / SORT_THREADS consecutive bins per thread, warp scan of the thread sums, then across warps
        constexpr int PER = SPLIT_BINS / SORT_THREADS;
        unsigned int c[PER], sum = 0u;
#pragma unroll
        for (int j = 0; j < PER; j++) { c[j] = s_cur[tid * PER + j]; sum += c[j]; }
        unsigned int incl = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned int o = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += o;
        }
        __syncthreads();                       // everyone has read its counters and s_red
        if (lane == 31) s_red[warp] = incl;
        __syncthreads();
        unsigned int before = incl - sum;
#pragma unroll
        for (int w = 0; w < SORT_WARPS; w++)
            if (w < warp) before += s_red[w];
#pragma unroll
        for (int j = 0; j < PER; j++) { s_off[tid * PER + j] = before; s_cur[tid * PER + j] = before; before += c[j]; }
        if (tid == SORT_THREADS - 1) s_off[SPLIT_BINS] = before;
    }
    __syncthreads();
    // 3. scatter into the output arrays (in range order; unordered inside a range)
    for (int i = tid; i < nb; i += SORT_THREADS) {
        const unsigned long long v = src[i];
        const unsigned int pos = atomicAdd(&s_cur[bin_of((unsigned int)(v >> 32))], 1u);
        ids[pos] = (unsigned int)v;
        keys[pos] = (unsigned int)(v >> 32);
    }
    __syncthreads();
    // 4. ranges a warp can hold: in registers, 8 ranges at a time; larger ones are noted for the CTA
    int n_large = 0;
    for (int b = warp; b < nbins; b += SORT_WARPS) {
        const int o = (int)s_off[b], n = (int)s_off[b + 1] - o;
        if (n > 1 && n <= WARP_ITEMS) sort_sub_bucket_warp<BIG>(ids + o, keys + o, n, lane);
    }
    __syncthreads();
    for (int b = 0; b < nbins; b++) {                         // block-uniform scan for the (rare) large ranges
        const int o = (int)s_off[b], n = (int)s_off[b + 1] - o;
        if (n <= WARP_ITEMS) continue;
        n_large++;
        // the split tables live in s_items: a large range borrows the bucket's own (now free) source area instead
        unsigned long long* tmp = src + o;
        for (int i = tid; i < n; i += SORT_THREADS) tmp[i] = ((unsigned long long)keys[o + i] << 32) | ids[o + i];
        __syncthreads();
        bitonic_sort<true>(tmp, n, tid, SORT_THREADS);        // global memory, block barriers: ranges of equal depths only
        for (int i = tid; i < n; i += SORT_THREADS) {
            const unsigned long long v = tmp[i];
            ids[o + i] = (unsigned int)v;
            keys[o + i] = (unsigned int)(v >> 32);
        }
        __syncthreads();
    }
    (void)n_large;
}

// BIG = false: buckets up to 256 entries in registers (32 registers per thread, 8 CTAs per SM) — the common case.
// BIG = true: up to 512 (dense scenes, e.g. 1 M Gaussians at 1080p = ~360 per tile); chosen by the launcher from
// the expected bucket size.  Either kernel sorts any bucket correctly (CTA-wide fallbacks beyond its register path).
template <bool BIG>
__global__ void __launch_bounds__(SORT_THREADS, 4) sort_tiles_kernel(int T, ImageView im, BinView bin,
                                                                  unsigned long long cap)
{
    constexpr int WARP_ITEMS = BIG ? SORT_WARP_ITEMS_BIG : SORT_WARP_ITEMS;
    __shared__ unsigned long long s_items[SORT_SMEM_ITEMS];
    __shared__ int s_big[SORT_WARPS];
    pdl_prologue();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int t = blockIdx.x * SORT_WARPS + warp;
    uint2 rg = make_uint2(0u, 0u);
    int n = 0;
    if (t < T) {
        rg = im.ranges[t];
        n = (unsigned long long)rg.y > cap ? 0 : (int)(rg.y - rg.x);
    }
    const bool big = n > WARP_ITEMS;
    if (lane == 0) s_big[warp] = big ? t : -1;
    if (!big && n > 0) {
        const unsigned long long* src = bin.inst + rg.x;
        unsigned int* ids = bin.point_list + rg.x;
        unsigned int* keys = bin.depth_keys + rg.x;
        if (n <= 32) sort_bucket_regs<1, 5>(src, n, lane, ids, keys);
        else if (n <= 64) sort_bucket_regs<2, 6>(src, n, lane, ids, keys);
        else if (n <= 128) sort_bucket_regs<4, 7>(src, n, lane, ids, keys);
        else if (!BIG || n <= 256) sort_bucket_regs<8, 8>(src, n, lane, ids, keys);
        else sort_bucket_regs<16, 9>(src, n, lane, ids, keys);
    }
    __syncthreads();
    for (int w = 0; w < SORT_WARPS; w++) {
        const int tb = s_big[w];
        if (tb < 0) continue;  // block-uniform
        const uint2 rb = im.ranges[tb];
        const int nb = (int)(rb.y - rb.x);
        unsigned long long* src = bin.inst + rb.x;
        if (nb <= SORT_SMEM_ITEMS) {
            for (int i = tid; i < nb; i += SORT_THREADS) s_items[i] = src[i];
            __syncthreads();
            bitonic_sort<true>(s_items, nb, tid, SORT_THREADS);
            for (int i = tid; i < nb; i += SORT_THREADS) {
                const unsigned long long v = s_items[i];
                bin.point_list[rb.x + i] = (unsigned int)v;
                bin.depth_keys[rb.x + i] = (unsigned int)(v >> 32);
            }
        } else if (tid == 0) {
            // thousands of instances on one tile: left to sort_heavy_kernel (its own launch, so that its registers and
            // its run time are not this kernel's)
            im.heavy_tiles[atomicAdd(&im.hdr->n_heavy, 1u)] = (unsigned int)tb;
        }
        __syncthreads();
    }
}

// The tiles the sort kernel left: a small persistent grid walks the list (empty for ordinary frames: every CTA reads
// one word and leaves), one CTA per heavy tile at a time.
constexpr int HEAVY_CTAS = 148;
__global__ void __launch_bounds__(SORT_THREADS) sort_heavy_kernel(ImageView im, BinView bin, unsigned long long cap)
{
    __shared__ unsigned long long s_items[SORT_SMEM_ITEMS];
    pdl_prologue();
    const unsigned int n_heavy = im.hdr->n_heavy;
    for (unsigned int i = blockIdx.x; i < n_heavy; i += gridDim.x) {
        const unsigned int t = im.heavy_tiles[i];
        const uint2 rb = im.ranges[t];
        if ((unsigned long long)rb.y > cap) continue;
        __syncthreads();
        sort_heavy_bucket<true>(bin.inst + rb.x, bin.point_list + rb.x, bin.depth_keys + rb.x, (int)(rb.y - rb.x), s_items,
                                (int)threadIdx.x);
    }
}

cudaError_t launch_sort_tiles(const DevSettings& s, ImageView im, BinView b, long long cap, cudaStream_t st)
{
    const int T = s.gx * s.gy * s.n_views;
    if (T <= 0) return cudaSuccess;
    count_launch(2);
    // expected bucket size from the instance capacity (1.25 x the last num_rendered seen for this shape)
    const bool dense = cap / T > 160;
    cudaError_t e = launch_pdl(dense ? sort_tiles_kernel<true> : sort_tiles_kernel<false>,
                               dim3((T + SORT_WARPS - 1) / SORT_WARPS), dim3(SORT_THREADS), st, T, im, b,
                               (unsigned long long)cap);
    if (e != cudaSuccess) return e;
    return launch_pdl(sort_heavy_kernel, dim3(HEAVY_CTAS), dim3(SORT_THREADS), st, im, b, (unsigned long long)cap);
}

// ---- export for the bit-exact stage tests --------------------------------------------------------
__global__ void export_keys_kernel(int T, ImageView im, BinView bin, unsigned long long* sorted_keys,
                                   unsigned int* point_list, unsigned int* ranges)
{
    const int t = blockIdx.x;
    if (t >= T) return;
    const uint2 rg = im.ranges[t];
    if (ranges && threadIdx.x == 0) { ranges[2 * t] = rg.x; ranges[2 * t + 1] = rg.y; }
    for (unsigned int i = rg.x + threadIdx.x; i < rg.y; i += blockDim.x) {
        if (sorted_keys) sorted_keys[i] = ((unsigned long long)t << 32) | bin.depth_keys[i];
        if (point_list) point_list[i] = bin.point_list[i];
    }
}

cudaError_t launch_export_keys(const DevSettings& s, ImageView im, BinView b, long long R,
                               unsigned long long* sorted_keys, unsigned int* point_list, unsigned int* ranges,
                               cudaStream_t st)
{
    (void)R;
    const int T = s.gx * s.gy * s.n_views;   // virtual tiles: keys carry v*Tv + t, point_list v*P + g
    export_keys_kernel<<<T, 128, 0, st>>>(T, im, b, sorted_keys, point_list, ranges);
    count_launch();
    return cudaGetLastError();
}

__global__ void export_geom_kernel(int P, GeomView geo, float* depth, float* xy, float* conic_opacity, float* rgb,
                                   int32_t* rect)
{
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= P) return;
    const ushort4 r = geo.rect[g];
    const bool vis = r.z > r.x && r.w > r.y;
    float4 f0 = make_float4(0, 0, 0, 0), f1 = f0, f2 = f0;
    if (vis) { f0 = geo.feat0[g]; f1 = geo.feat1[g]; f2 = geo.feat2[g]; }
    if (depth) depth[g] = f2.w;
    if (xy) { xy[2 * g] = f0.x; xy[2 * g + 1] = f0.y; }
    if (conic_opacity) reinterpret_cast<float4*>(conic_opacity)[g] = f1;
    if (rgb) { rgb[3 * g] = f2.x; rgb[3 * g + 1] = f2.y; rgb[3 * g + 2] = f2.z; }
    if (rect) { rect[4 * g] = r.x; rect[4 * g + 1] = r.y; rect[4 * g + 2] = r.z; rect[4 * g + 3] = r.w; }
}

cudaError_t launch_export_geom(int P, GeomView g, float* depth, float* xy, float* conic_opacity, float* rgb,
                               int32_t* rect, cudaStream_t st)
{
    if (P <= 0) return cudaSuccess;
    export_geom_kernel<<<(P + 255) / 256, 256, 0, st>>>(P, g, depth, xy, conic_opacity, rgb, rect);
    count_launch();
    return cudaGetLastError();
}

}  // namespace gsvc
