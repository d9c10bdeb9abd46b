// extern "C" boundary of libgsvc_rast.so (see include/gsvc_rast.h for the contract and the
// reference call sites each entry point replaces).  No torch types, no allocation: raw device
// pointers, sizes and a cudaStream_t.
#include <atomic>
#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <cstring>

#include "common.cuh"

namespace gsvc {

static thread_local char g_err[512] = "";
// process-wide (the backward runs on PyTorch's autograd thread, not on the caller's)
static std::atomic<long long> g_launches{0};
// set by the caller around launches it is capturing into a CUDA graph: only those feed the sticky overflow counter
// (an eager launch that outgrows its capacity is re-run by its caller and must not look like a lost frame)
static thread_local bool g_count_overflows = false;

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// ---- optional per-stage device timing (CUDA events on the launching stream) ----------------------
enum Stage { ST_PREPROCESS = 0, ST_TILE_SCAN, ST_SCATTER, ST_SORT, ST_RENDER_FWD, ST_RENDER_BWD, ST_PREPROCESS_BWD,
             ST_VISIBLE_FILTER, ST_COUNT };
static std::atomic<bool> g_timing{false};
constexpr int EV_RING = 256;                       // per-stage samples kept between two queries
static cudaEvent_t g_ev[ST_COUNT][EV_RING][2];
static bool g_ev_made = false;
static std::atomic<unsigned int> g_ev_n[ST_COUNT];  // samples recorded since the last query

struct StageScope {
    int id; cudaStream_t s; unsigned int slot;
    StageScope(int id_, cudaStream_t s_) : id(id_), s(s_), slot(0)
    {
        if (g_timing) { slot = g_ev_n[id].load() % EV_RING; cudaEventRecord(g_ev[id][slot][0], s); }
    }
    ~StageScope()
    {
        if (g_timing) { cudaEventRecord(g_ev[id][slot][1], s); g_ev_n[id].fetch_add(1); }
    }
};

// (also the error channel of loss.cu)
int fail(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CK(expr, what)                                                                                       \
    do {                                                                                                     \
        cudaError_t e__ = (expr);                                                                            \
        if (e__ != cudaSuccess) return fail(GSVC_RAST_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e__));    \
        if (dbg) {                                                                                           \
            e__ = cudaStreamSynchronize(stream);                                                             \
            if (e__ != cudaSuccess)                                                                          \
                return fail(GSVC_RAST_ERR_CUDA, "%s (debug sync): %s", what, cudaGetErrorString(e__));       \
        }                                                                                                    \
    } while (0)

static int make_settings_views(const gsvc_rast_settings* st, int n_views, const gsvc_rast_view* views, int n_out,
                               int sh_M, DevSettings& d)
{
    if (!st) return fail(GSVC_RAST_ERR_INVALID, "settings is NULL");
    if (st->image_width <= 0 || st->image_height <= 0) return fail(GSVC_RAST_ERR_INVALID, "image size must be positive");
    if (n_views < 1 || n_views > MAX_VIEWS)
        return fail(GSVC_RAST_ERR_INVALID, "n_views must be in 1..%d, got %d", MAX_VIEWS, n_views);
    if (!views) return fail(GSVC_RAST_ERR_INVALID, "views is NULL");
    if (n_out < 1 || n_out > n_views) return fail(GSVC_RAST_ERR_INVALID, "n_out must be in 1..n_views");
    d.W = st->image_width; d.H = st->image_height;
    d.gx = (d.W + TILE - 1) / TILE; d.gy = (d.H + TILE - 1) / TILE;
    if (d.gx > 65535 || d.gy > 65535) return fail(GSVC_RAST_ERR_INVALID, "image too large for 16-bit tile coordinates");
    if ((long long)d.gx * d.gy * n_views > 0x7fffffffll) return fail(GSVC_RAST_ERR_INVALID, "too many tiles");
    if ((long long)d.gx * d.gy > (1ll << 24))   // warp_tiles_get divides tile counts in fp32 (exact below 2^24)
        return fail(GSVC_RAST_ERR_INVALID, "image has more than 2^24 tiles");
    d.x_min = st->x_min; d.y_min = st->y_min; d.scale = st->scale; d.threshold = st->threshold;
    d.scale_modifier = st->scale_modifier;
    d.bg = st->bg;
    d.sh_degree = st->sh_degree; d.sh_M = sh_M;
    d.n_views = n_views;
    d.ragged = 0;
    memset(&d.rows, 0, sizeof(d.rows));
    int used[MAX_VIEWS] = {0};
    d.accumulate = 0;
    memset(&d.vt, 0, sizeof(d.vt));
    for (int v = 0; v < n_views; v++) {
        if (!views[v].viewmatrix) return fail(GSVC_RAST_ERR_INVALID, "viewmatrix of view %d is NULL", v);
        if (views[v].out_image < 0 || views[v].out_image >= n_out)
            return fail(GSVC_RAST_ERR_INVALID, "out_image of view %d is %d, expected 0..%d", v, views[v].out_image, n_out - 1);
        d.vt.V[v] = views[v].viewmatrix; d.vt.vs_r[v] = views[v].vm_stride_r; d.vt.vs_c[v] = views[v].vm_stride_c;
        for (int k = 0; k < 3; k++) d.vt.campos[v][k] = views[v].campos[k];
        d.vt.out_image[v] = views[v].out_image; d.vt.flip_x[v] = views[v].flip_x != 0; d.vt.weight[v] = views[v].weight;
        if (used[views[v].out_image]++) d.accumulate = 1;
    }
    for (int o = 0; o < n_out; o++)
        if (!used[o]) return fail(GSVC_RAST_ERR_INVALID, "output image %d has no view", o);
    return 0;
}

// A ragged batch: the view map as above, then the views' own counts (n_views entries), summed into P.
static int make_settings_ragged(const gsvc_rast_settings* st, int n_views, const gsvc_rast_view* views, int n_out,
                                const int32_t* counts_host, int sh_M, DevSettings& d, int32_t& P)
{
    int rc = make_settings_views(st, n_views, views, n_out, sh_M, d);
    if (rc) return rc;
    if (!counts_host) return fail(GSVC_RAST_ERR_INVALID, "counts_host is NULL");
    long long total = 0;
    for (int v = 0; v < n_views; v++) {
        if (counts_host[v] < 0) return fail(GSVC_RAST_ERR_INVALID, "count of view %d is %d, expected >= 0", v, counts_host[v]);
        total += counts_host[v];
        if (total > 0x7fffffffll) return fail(GSVC_RAST_ERR_INVALID, "the views' counts sum to more than 2^31 - 1 rows");
        d.rows.off[v + 1] = (int)total;
    }
    d.ragged = 1;
    P = (int32_t)total;
    return 0;
}

static int make_settings(const gsvc_rast_settings* st, int sh_M, DevSettings& d)
{
    if (!st) return fail(GSVC_RAST_ERR_INVALID, "settings is NULL");
    if (!st->viewmatrix) return fail(GSVC_RAST_ERR_INVALID, "viewmatrix is NULL");
    gsvc_rast_view one;
    one.viewmatrix = st->viewmatrix; one.vm_stride_r = st->vm_stride_r; one.vm_stride_c = st->vm_stride_c;
    one.campos[0] = st->campos[0]; one.campos[1] = st->campos[1]; one.campos[2] = st->campos[2];
    one.out_image = 0; one.flip_x = 0; one.weight = 1.0f;
    return make_settings_views(st, 1, &one, 1, sh_M, d);
}

static int check_inputs(int P, int sh_M, int sh_degree, const float* means3D, const float* shs,
                        const float* colors_precomp, const float* opacities, const float* scales,
                        const float* rotations, const float* cov3D_precomp, bool need_color)
{
    if (P < 0) return fail(GSVC_RAST_ERR_INVALID, "P must be >= 0");
    if (P == 0) return 0;  // empty inputs carry NULL pointers
    if (P > 0 && !means3D) return fail(GSVC_RAST_ERR_INVALID, "means3D is NULL");
    const bool sr = scales && rotations;
    if ((scales == nullptr) != (rotations == nullptr) || (sr == (cov3D_precomp != nullptr)))
        return fail(GSVC_RAST_ERR_INVALID, "Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!");
    if (need_color) {
        if ((shs != nullptr) == (colors_precomp != nullptr))
            return fail(GSVC_RAST_ERR_INVALID, "Please provide excatly one of either SHs or precomputed colors!");
        if (P > 0 && !opacities) return fail(GSVC_RAST_ERR_INVALID, "opacities is NULL");
        if (shs) {
            if (sh_degree < 0 || sh_degree > 3) return fail(GSVC_RAST_ERR_INVALID, "sh_degree must be in 0..3");
            if (sh_M < (sh_degree + 1) * (sh_degree + 1))
                return fail(GSVC_RAST_ERR_INVALID, "shs has %d coefficients, sh_degree %d needs %d", sh_M, sh_degree,
                            (sh_degree + 1) * (sh_degree + 1));
        }
    }
    return 0;
}

static int render_stages(const DevSettings& d, int P, GeomView g, ImageView im, void* binning, long long cap,
                         float* out_color, cudaStream_t stream, bool dbg)
{
    BinView b = bin_view(binning, cap);
    { StageScope t(ST_SCATTER, stream); CK(launch_scatter(d, P, g, im, b, cap, g_count_overflows, stream), "scatter"); }
    { StageScope t(ST_SORT, stream); CK(launch_sort_tiles(d, im, b, cap, stream), "sort_tiles"); }
    { StageScope t(ST_RENDER_FWD, stream); CK(launch_render_forward(d, g, im, b, cap, out_color, stream), "render_forward"); }
    return 0;
}

}  // namespace gsvc

using namespace gsvc;

extern "C" {

int gsvc_rast_abi_version(void) { return GSVC_RAST_ABI_VERSION; }
const char* gsvc_rast_last_error(void) { return g_err; }
size_t gsvc_rast_geom_bytes(int32_t P, int32_t sh_M) { return geom_bytes(P < 1 ? 1 : P, sh_M); }
size_t gsvc_rast_image_bytes(int32_t W, int32_t H) { return image_bytes(W < 1 ? 1 : W, H < 1 ? 1 : H); }
size_t gsvc_rast_image_bytes_views(int32_t W, int32_t H, int32_t n_views)
{
    return image_bytes(W < 1 ? 1 : W, H < 1 ? 1 : H, n_views < 1 ? 1 : n_views);
}
size_t gsvc_rast_binning_bytes(int64_t cap) { return bin_bytes(cap < 1 ? 1 : cap); }
size_t gsvc_rast_backward_scratch_bytes(int32_t P) { return bwd_scratch_bytes(P < 1 ? 1 : P); }
int64_t gsvc_rast_launch_count(int32_t reset)
{
    return reset ? g_launches.exchange(0) : g_launches.load();
}

int gsvc_rast_densify_stats(int32_t n_views, int32_t P, const float* dL_dmeans2D, const int32_t* radii, float* stats,
                            int64_t stride, int32_t accumulate, void* stream_)
{
    if (n_views < 1) return fail(GSVC_RAST_ERR_INVALID, "n_views must be >= 1");
    if (P < 0) return fail(GSVC_RAST_ERR_INVALID, "P must be >= 0");
    if ((long long)P * n_views > 0x7fffffffll) return fail(GSVC_RAST_ERR_INVALID, "P * n_views exceeds 31 bits");
    if (stride < 2) return fail(GSVC_RAST_ERR_INVALID, "stride must be >= 2 floats");
    if (P > 0 && (!dL_dmeans2D || !radii || !stats))
        return fail(GSVC_RAST_ERR_INVALID, "dL_dmeans2D/radii/stats must be non-NULL");
    cudaError_t e = launch_densify_stats(n_views, P, dL_dmeans2D, radii, stats, (long long)stride, accumulate != 0,
                                         static_cast<cudaStream_t>(stream_));
    if (e != cudaSuccess) return fail(GSVC_RAST_ERR_CUDA, "densify_stats: %s", cudaGetErrorString(e));
    return GSVC_RAST_OK;
}

int gsvc_rast_switch_allreduce(void* multicast, void* buffers, void* signal_pads, void* state, int32_t rank,
                               int32_t world, int64_t numel, int32_t n_ctas, void* stream_)
{
    if (world < 1 || rank < 0 || rank >= world) return fail(GSVC_RAST_ERR_INVALID, "rank %d outside world %d", rank, world);
    if (numel < 0 || (numel & 3)) return fail(GSVC_RAST_ERR_INVALID, "numel must be a non-negative multiple of 4");
    if (n_ctas < 1 || n_ctas > 592) return fail(GSVC_RAST_ERR_INVALID, "n_ctas must be in 1..592 (co-resident CTAs)");
    if (!signal_pads || !state) return fail(GSVC_RAST_ERR_INVALID, "signal_pads / state must be non-NULL");
    if (!multicast && !buffers) return fail(GSVC_RAST_ERR_INVALID, "one of multicast / buffers must be non-NULL");
    if (!multicast && world != 1 && world != 2 && world != 4 && world != 8)
        return fail(GSVC_RAST_ERR_INVALID, "the peer-load path is built for 1, 2, 4 or 8 ranks, got %d", world);
    if (reinterpret_cast<uintptr_t>(multicast) & 15) return fail(GSVC_RAST_ERR_INVALID, "multicast address must be 16-byte aligned");
    cudaError_t e = launch_switch_allreduce(static_cast<float*>(multicast), static_cast<void* const*>(buffers),
                                            static_cast<unsigned int* const*>(signal_pads), static_cast<unsigned int*>(state),
                                            rank, world, (long long)numel, n_ctas, static_cast<cudaStream_t>(stream_));
    if (e != cudaSuccess) return fail(GSVC_RAST_ERR_CUDA, "switch_allreduce: %s", cudaGetErrorString(e));
    return GSVC_RAST_OK;
}

int gsvc_rast_count_overflows(int32_t enable)
{
    g_count_overflows = enable != 0;
    return 0;
}

int64_t gsvc_rast_overflow_events(int32_t reset, void* stream_)
{
    unsigned int v = 0u;
    cudaError_t e = read_overflow_events(&v, reset != 0, static_cast<cudaStream_t>(stream_));
    if (e != cudaSuccess) return fail(GSVC_RAST_ERR_CUDA, "overflow_events: %s", cudaGetErrorString(e));
    return (int64_t)v;
}

int gsvc_rast_stage_timing(int32_t enable)
{
    if (enable && !g_ev_made) {
        for (int i = 0; i < ST_COUNT; i++)
            for (int k = 0; k < EV_RING; k++)
                for (int j = 0; j < 2; j++)
                    if (cudaEventCreate(&g_ev[i][k][j]) != cudaSuccess)
                        return fail(GSVC_RAST_ERR_CUDA, "cudaEventCreate failed");
        g_ev_made = true;
    }
    g_timing = enable != 0;
    for (int i = 0; i < ST_COUNT; i++) g_ev_n[i] = 0;
    return 0;
}

int gsvc_rast_stage_times(float* ms_host)
{
    if (!ms_host) return fail(GSVC_RAST_ERR_INVALID, "ms_host is NULL");
    for (int i = 0; i < ST_COUNT; i++) {
        ms_host[i] = -1.f;
        const unsigned int n = g_ev_made ? g_ev_n[i].exchange(0) : 0;
        if (n == 0) continue;
        const unsigned int cnt = n < (unsigned)EV_RING ? n : (unsigned)EV_RING;
        double sum = 0.0;
        for (unsigned int k = 0; k < cnt; k++) {
            if (cudaEventSynchronize(g_ev[i][k][1]) != cudaSuccess)
                return fail(GSVC_RAST_ERR_CUDA, "cudaEventSynchronize failed");
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, g_ev[i][k][0], g_ev[i][k][1]) != cudaSuccess)
                return fail(GSVC_RAST_ERR_CUDA, "cudaEventElapsedTime failed");
            sum += ms;
        }
        ms_host[i] = (float)(sum / cnt);
    }
    return ST_COUNT;
}

static int check_range(int32_t P, int32_t& lo, int32_t& hi)
{
    if (lo == 0 && hi == 0) hi = P;    // (0, 0) = no range given: everything
    if (lo < 0 || hi > P || lo > hi) return fail(GSVC_RAST_ERR_INVALID, "index range [%d, %d) is not inside [0, %d)", lo, hi, P);
    return 0;
}

int gsvc_rast_visible_filter(const gsvc_rast_settings* st, int32_t P, const float* means3D, const float* scales,
                             const float* rotations, const float* cov3D_precomp, int32_t* radii, int32_t range_lo,
                             int32_t range_hi, void* stream_)
{
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    DevSettings d;
    int rc = make_settings(st, 0, d);
    if (rc) return rc;
    rc = check_inputs(P, 0, 0, means3D, nullptr, nullptr, nullptr, scales, rotations, cov3D_precomp, false);
    if (rc) return rc;
    if (P > 0 && !radii) return fail(GSVC_RAST_ERR_INVALID, "radii is NULL");
    rc = check_range(P, range_lo, range_hi);
    if (rc) return rc;
    const bool dbg = st->debug != 0;
    PreInputs in{P, means3D, nullptr, nullptr, nullptr, scales, rotations, cov3D_precomp, range_lo, range_hi};
    { StageScope t(ST_VISIBLE_FILTER, stream); CK(launch_visible_filter(d, in, radii, stream), "visible_filter"); }
    return 0;
}

static int forward_launch_core(const gsvc_rast_settings* st, const DevSettings& d, int n_out, int32_t P, int32_t sh_M,
                               const float* means3D, const float* shs, const float* colors_precomp,
                               const float* opacities, const float* scales, const float* rotations,
                               const float* cov3D_precomp, void* geom, void* image, void* binning, int64_t capacity,
                               void* bwd_scratch, float* out_color, int32_t* radii, uint64_t* count_slot_host,
                               uint32_t ticket, cudaStream_t stream)
{
    int rc = check_inputs(P, sh_M, st->sh_degree, means3D, shs, colors_precomp, opacities, scales, rotations, cov3D_precomp, true);
    if (rc) return rc;
    if (!st->bg) return fail(GSVC_RAST_ERR_INVALID, "bg is NULL");
    if (!geom || !image || !out_color || (P > 0 && !radii))
        return fail(GSVC_RAST_ERR_INVALID, "geom/image/out_color/radii must be non-NULL");
    if (capacity > 0 && !binning) return fail(GSVC_RAST_ERR_INVALID, "binning is NULL");
    if (!d.ragged && (long long)P * d.n_views > 0x7fffffffll)
        return fail(GSVC_RAST_ERR_INVALID, "P * n_views exceeds 31 bits");
    const bool dbg = st->debug != 0;
    GeomView g = geom_view(geom, state_rows(d, P < 1 ? 1 : P), d.sh_M);
    ImageView im = image_view(image, d.W, d.H, d.n_views);
    PreInputs in{P, means3D, shs, colors_precomp, opacities, scales, rotations, cov3D_precomp, 0, P};
    if (d.accumulate)   // views that share an output image add into it
        CK(cudaMemsetAsync(out_color, 0, (size_t)n_out * 3 * d.W * d.H * sizeof(float), stream), "zero out_color");
    { StageScope t(ST_PREPROCESS, stream); CK(launch_preprocess(d, in, radii, g, im, static_cast<float4*>(bwd_scratch), stream), "preprocess"); }
    {
        StageScope t(ST_TILE_SCAN, stream);
        CK(launch_tile_scan(d, im, reinterpret_cast<unsigned long long*>(count_slot_host), ticket & 0xFFFFFFu, stream),
           "tile_scan");
    }
    if (capacity > 0) {
        rc = render_stages(d, P, g, im, binning, capacity, out_color, stream, dbg);
        if (rc) return rc;
    }
    return 0;
}

size_t gsvc_rast_compact_scratch_bytes(int32_t P) { return compact_scratch_bytes(P); }

int gsvc_rast_visible_filter_compact(const gsvc_rast_settings* st, int32_t P, const float* means3D, const float* scales,
                                     const float* rotations, const float* cov3D_precomp, int32_t* radii,
                                     int32_t* visible_indices, void* scratch, uint64_t* count_slot_host,
                                     uint32_t ticket, int32_t range_lo, int32_t range_hi, void* stream_)
{
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    DevSettings d;
    int rc = make_settings(st, 0, d);
    if (rc) return rc;
    rc = check_inputs(P, 0, 0, means3D, nullptr, nullptr, nullptr, scales, rotations, cov3D_precomp, false);
    if (rc) return rc;
    if (!scratch || (P > 0 && !visible_indices))
        return fail(GSVC_RAST_ERR_INVALID, "visible_indices/scratch must be non-NULL");
    rc = check_range(P, range_lo, range_hi);
    if (rc) return rc;
    const bool dbg = st->debug != 0;
    PreInputs in{P, means3D, nullptr, nullptr, nullptr, scales, rotations, cov3D_precomp, range_lo, range_hi};
    {
        StageScope t(ST_VISIBLE_FILTER, stream);
        CK(launch_visible_filter_compact(d, in, radii, visible_indices, scratch,
                                         reinterpret_cast<unsigned long long*>(count_slot_host), ticket & 0xFFFFFFu,
                                         stream),
           "visible_filter_compact");
    }
    return 0;
}

int gsvc_rast_forward_launch(const gsvc_rast_settings* st, int32_t P, int32_t sh_M, const float* means3D,
                             const float* shs, const float* colors_precomp, const float* opacities,
                             const float* scales, const float* rotations, const float* cov3D_precomp, void* geom,
                             void* image, void* binning, int64_t capacity, void* bwd_scratch, float* out_color,
                             int32_t* radii, uint64_t* count_slot_host, uint32_t ticket, void* stream_)
{
    DevSettings d;
    int rc = make_settings(st, shs ? sh_M : 0, d);
    if (rc) return rc;
    return forward_launch_core(st, d, 1, P, sh_M, means3D, shs, colors_precomp, opacities, scales, rotations,
                               cov3D_precomp, geom, image, binning, capacity, bwd_scratch, out_color, radii,
                               count_slot_host, ticket, static_cast<cudaStream_t>(stream_));
}

int gsvc_rast_forward_views_launch(const gsvc_rast_settings* st, int32_t n_views, const gsvc_rast_view* views_host,
                                   int32_t n_out, int32_t P, int32_t sh_M, const float* means3D, const float* shs,
                                   const float* colors_precomp, const float* opacities, const float* scales,
                                   const float* rotations, const float* cov3D_precomp, void* geom, void* image,
                                   void* binning, int64_t capacity, void* bwd_scratch, float* out_color,
                                   int32_t* radii, uint64_t* count_slot_host, uint32_t ticket, void* stream_)
{
    DevSettings d;
    int rc = make_settings_views(st, n_views, views_host, n_out, shs ? sh_M : 0, d);
    if (rc) return rc;
    return forward_launch_core(st, d, n_out, P, sh_M, means3D, shs, colors_precomp, opacities, scales, rotations,
                               cov3D_precomp, geom, image, binning, capacity, bwd_scratch, out_color, radii,
                               count_slot_host, ticket, static_cast<cudaStream_t>(stream_));
}

int64_t gsvc_rast_wait_count(const uint64_t* count_slot_host, uint32_t ticket, void* stream_)
{
    if (!count_slot_host) return fail(GSVC_RAST_ERR_INVALID, "count_slot_host is NULL");
    const volatile uint64_t* slot = count_slot_host;
    const uint64_t want = (uint64_t)(ticket & 0xFFFFFFu);
    // The scan runs a few tens of microseconds after launch: spin briefly, then fall back to a stream
    // synchronise (which also surfaces asynchronous launch errors).
    for (long long spin = 0; spin < 20000000ll; spin++) {
        const uint64_t v = *slot;
        if ((v >> 40) == want) return (int64_t)(v & ((1ull << 40) - 1));
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
    }
    cudaError_t e = cudaStreamSynchronize(static_cast<cudaStream_t>(stream_));
    if (e != cudaSuccess) return fail(GSVC_RAST_ERR_CUDA, "wait_count: %s", cudaGetErrorString(e));
    const uint64_t v = *slot;
    if ((v >> 40) == want) return (int64_t)(v & ((1ull << 40) - 1));
    return fail(GSVC_RAST_ERR_CUDA, "wait_count: the tile scan never published ticket %u", (unsigned)want);
}

static int forward_render_core(const gsvc_rast_settings* st, const DevSettings& d, int n_out, int32_t P,
                               const void* geom, void* image, void* binning, int64_t capacity, float* out_color,
                               cudaStream_t stream)
{
    if (!geom || !image || !binning || !out_color || capacity <= 0)
        return fail(GSVC_RAST_ERR_INVALID, "geom/image/binning/out_color must be non-NULL and capacity > 0");
    const bool dbg = st->debug != 0;
    // sh_M only affects the tail of the geom layout (clamp flags), which these stages never touch
    GeomView g = geom_view(const_cast<void*>(geom), state_rows(d, P < 1 ? 1 : P), 0);
    ImageView im = image_view(image, d.W, d.H, d.n_views);
    // the scatter cursors were consumed by a previous attempt: reset them
    CK(cudaMemsetAsync(im.tile_cursor, 0, (size_t)d.gx * d.gy * d.n_views * sizeof(unsigned int), stream), "cursor reset");
    // ... and so were the overflow flag of that attempt (the blend backward refuses to replay an overflowed frame) and
    // its list of heavy tiles: the sort of the first attempt may already have queued some, and a tile queued twice is
    // sorted by two CTAs of sort_heavy_kernel at once (found by the randomised sweep: a 2 231-instance tile rendered
    // after an overflowed first attempt came out with pixels off by 0.26)
    static_assert(offsetof(ImageHeader, n_heavy) == offsetof(ImageHeader, overflow) + sizeof(unsigned int),
                  "overflow and n_heavy are reset with one memset");
    CK(cudaMemsetAsync(&im.hdr->overflow, 0, 2 * sizeof(unsigned int), stream), "overflow flag / heavy list reset");
    if (d.accumulate)
        CK(cudaMemsetAsync(out_color, 0, (size_t)n_out * 3 * d.W * d.H * sizeof(float), stream), "zero out_color");
    return render_stages(d, P, g, im, binning, capacity, out_color, stream, dbg);
}

int gsvc_rast_forward_render(const gsvc_rast_settings* st, int32_t P, const void* geom, void* image, void* binning,
                             int64_t capacity, float* out_color, void* stream_)
{
    DevSettings d;
    int rc = make_settings(st, 0, d);
    if (rc) return rc;
    return forward_render_core(st, d, 1, P, geom, image, binning, capacity, out_color, static_cast<cudaStream_t>(stream_));
}

int gsvc_rast_forward_views_render(const gsvc_rast_settings* st, int32_t n_views, const gsvc_rast_view* views_host,
                                   int32_t n_out, int32_t P, const void* geom, void* image, void* binning,
                                   int64_t capacity, float* out_color, void* stream_)
{
    DevSettings d;
    int rc = make_settings_views(st, n_views, views_host, n_out, 0, d);
    if (rc) return rc;
    return forward_render_core(st, d, n_out, P, geom, image, binning, capacity, out_color,
                               static_cast<cudaStream_t>(stream_));
}

int64_t gsvc_rast_forward(const gsvc_rast_settings* st, int32_t P, int32_t sh_M, const float* means3D,
                          const float* shs, const float* colors_precomp, const float* opacities, const float* scales,
                          const float* rotations, const float* cov3D_precomp, gsvc_rast_alloc_fn alloc, void* user,
                          float* out_color, int32_t* radii, void* stream_)
{
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (!alloc) return fail(GSVC_RAST_ERR_INVALID, "alloc callback is NULL");
    if (!st) return fail(GSVC_RAST_ERR_INVALID, "settings is NULL");
    void* geom = alloc(user, 0, gsvc_rast_geom_bytes(P, shs ? sh_M : 0));
    void* image = alloc(user, 2, gsvc_rast_image_bytes(st->image_width, st->image_height));
    if (!geom || !image) return fail(GSVC_RAST_ERR_INVALID, "alloc callback returned NULL");
    // phase A: preprocess + tile scan; the exact instance count sizes the binning buffer
    int rc = gsvc_rast_forward_launch(st, P, sh_M, means3D, shs, colors_precomp, opacities, scales, rotations,
                                      cov3D_precomp, geom, image, nullptr, 0, nullptr, out_color, radii, nullptr, 0,
                                      stream_);
    if (rc) return rc;
    ImageView im = image_view(image, st->image_width, st->image_height);
    unsigned long long R = 0;
    cudaError_t e = cudaMemcpyAsync(&R, &im.hdr->num_rendered, sizeof(R), cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) return fail(GSVC_RAST_ERR_CUDA, "num_rendered readback: %s", cudaGetErrorString(e));
    if (R > 0xFFFFFFFFull) return fail(GSVC_RAST_ERR_OVERFLOW, "num_rendered %llu exceeds 32-bit tile ranges", R);
    const int64_t cap = R > 0 ? (int64_t)R : 1;
    void* binning = alloc(user, 1, gsvc_rast_binning_bytes(cap));
    if (!binning) return fail(GSVC_RAST_ERR_INVALID, "alloc callback returned NULL");
    rc = gsvc_rast_forward_render(st, P, geom, image, binning, cap, out_color, stream_);
    if (rc) return rc;
    return (int64_t)R;
}

static int backward_core(const gsvc_rast_settings* st, const DevSettings& d, int32_t P, int32_t sh_M, int64_t capacity,
                         const float* means3D, const float* shs, const float* colors_precomp, const float* scales,
                         const float* rotations, const float* cov3D_precomp, const int32_t* radii, const void* geom,
                         const void* image, const void* binning, void* scratch, int32_t scratch_is_zero,
                         const float* dL_dout, BwdOutputs out, cudaStream_t stream, ExchangeArgs ex = ExchangeArgs{})
{
    int rc = check_inputs(P, sh_M, st->sh_degree, means3D, shs, colors_precomp, reinterpret_cast<const float*>(1), scales,
                          rotations, cov3D_precomp, true);
    if (rc) return rc;
    if (!st->bg) return fail(GSVC_RAST_ERR_INVALID, "bg is NULL");
    if (!geom || !image || !scratch || !dL_dout || (P > 0 && !radii))
        return fail(GSVC_RAST_ERR_INVALID, "geom/image/scratch/dL_dout/radii must be non-NULL");
    if (capacity <= 0 || !binning) return fail(GSVC_RAST_ERR_INVALID, "binning is NULL or capacity <= 0");
    if (out.packed && (shs || cov3D_precomp))
        return fail(GSVC_RAST_ERR_INVALID, "dL_packed needs colors_precomp and the scale/rotation pair");
    const bool dbg = st->debug != 0;
    GeomView g = geom_view(const_cast<void*>(geom), state_rows(d, P < 1 ? 1 : P), d.sh_M);
    ImageView im = image_view(const_cast<void*>(image), d.W, d.H, d.n_views);
    BinView b = bin_view(const_cast<void*>(binning), capacity);
    float4* acc = static_cast<float4*>(scratch);
    PreInputs in{P, means3D, shs, colors_precomp, nullptr, scales, rotations, cov3D_precomp, 0, P};
    { StageScope t(ST_RENDER_BWD, stream); CK(launch_render_backward(d, state_rows(d, P), g, im, b, capacity, dL_dout, acc, scratch_is_zero != 0, stream), "render_backward"); }
    { StageScope t(ST_PREPROCESS_BWD, stream); CK(launch_preprocess_backward(d, in, radii, g, acc, out, ex, stream), "preprocess_backward"); }
    return 0;
}

int gsvc_rast_backward(const gsvc_rast_settings* st, int32_t P, int32_t sh_M, int64_t capacity,
                       const float* means3D, const float* shs, const float* colors_precomp, const float* scales,
                       const float* rotations, const float* cov3D_precomp, const int32_t* radii, const void* geom,
                       const void* image, const void* binning, void* scratch, int32_t scratch_is_zero,
                       const float* dL_dout,
                       float* dL_dmeans3D, float* dL_dmeans2D, float* dL_dcolors, float* dL_dopacities,
                       float* dL_dscales, float* dL_drotations, float* dL_dcov3D, float* dL_dshs, float* dL_packed,
                       void* stream_)
{
    DevSettings d;
    int rc = make_settings(st, shs ? sh_M : 0, d);
    if (rc) return rc;
    BwdOutputs out{dL_dmeans3D, dL_dmeans2D, dL_dcolors, dL_dopacities, dL_dscales, dL_drotations, dL_dcov3D, dL_dshs,
                   dL_packed};
    return backward_core(st, d, P, sh_M, capacity, means3D, shs, colors_precomp, scales, rotations, cov3D_precomp, radii,
                         geom, image, binning, scratch, scratch_is_zero, dL_dout, out, static_cast<cudaStream_t>(stream_));
}

int gsvc_rast_backward_views(const gsvc_rast_settings* st, int32_t n_views, const gsvc_rast_view* views_host,
                             int32_t n_out, int32_t P, int32_t sh_M, int64_t capacity, const float* means3D,
                             const float* shs, const float* colors_precomp, const float* scales,
                             const float* rotations, const float* cov3D_precomp, const int32_t* radii,
                             const void* geom, const void* image, const void* binning, void* scratch,
                             int32_t scratch_is_zero, const float* dL_dout, float* dL_dmeans3D, float* dL_dmeans2D,
                             float* dL_dcolors, float* dL_dopacities, float* dL_dscales, float* dL_drotations,
                             float* dL_dcov3D, float* dL_dshs, float* dL_packed, void* stream_)
{
    DevSettings d;
    int rc = make_settings_views(st, n_views, views_host, n_out, shs ? sh_M : 0, d);
    if (rc) return rc;
    BwdOutputs out{dL_dmeans3D, dL_dmeans2D, dL_dcolors, dL_dopacities, dL_dscales, dL_drotations, dL_dcov3D, dL_dshs,
                   dL_packed};
    return backward_core(st, d, P, sh_M, capacity, means3D, shs, colors_precomp, scales, rotations, cov3D_precomp, radii,
                         geom, image, binning, scratch, scratch_is_zero, dL_dout, out, static_cast<cudaStream_t>(stream_));
}

int gsvc_rast_backward_views_exchange(const gsvc_rast_settings* st, int32_t n_views, const gsvc_rast_view* views_host,
                                      int32_t n_out, int32_t P, int32_t sh_M, int64_t capacity, const float* means3D,
                                      const float* shs, const float* colors_precomp, const float* scales,
                                      const float* rotations, const float* cov3D_precomp, const int32_t* radii,
                                      const void* geom, const void* image, const void* binning, void* scratch,
                                      int32_t scratch_is_zero, const float* dL_dout, float* dL_dmeans2D,
                                      float* dL_packed, const gsvc_rast_exchange* x, void* stream_)
{
    if (!x) return fail(GSVC_RAST_ERR_INVALID, "exchange is NULL");
    if (!dL_packed) return fail(GSVC_RAST_ERR_INVALID, "the exchange sums the packed [P,14] rows: dL_packed is NULL");
    if (x->world < 1 || x->rank < 0 || x->rank >= x->world)
        return fail(GSVC_RAST_ERR_INVALID, "rank %d outside world %d", x->rank, x->world);
    if (P < 2 || (P & 1)) return fail(GSVC_RAST_ERR_INVALID, "the exchange moves 16-byte words: P must be even and > 0");
    if (!x->signal_pads || !x->state || (!x->multicast && !x->buffers))
        return fail(GSVC_RAST_ERR_INVALID, "signal_pads / state and one of multicast / buffers must be non-NULL");
    if (!x->multicast && x->world > 8) return fail(GSVC_RAST_ERR_INVALID, "the peer-load path holds up to 8 ranks");
    if ((reinterpret_cast<uintptr_t>(x->multicast) | reinterpret_cast<uintptr_t>(dL_packed)) & 15)
        return fail(GSVC_RAST_ERR_INVALID, "dL_packed (and its multicast address) must be 16-byte aligned");
    const int n_compute = (P + 127) / 128;
    int chunk_rows = x->chunk_rows > 0 ? x->chunk_rows : ((P / 4 + 127) / 128) * 128;
    if (chunk_rows % 128) return fail(GSVC_RAST_ERR_INVALID, "chunk_rows must be a multiple of 128");
    if (chunk_rows < 128) chunk_rows = 128;
    int chunk_ctas = chunk_rows / 128;
    int n_chunks = (n_compute + chunk_ctas - 1) / chunk_ctas;
    if (n_chunks > GSVC_RAST_EXCHANGE_MAX_CHUNKS) {               // fewer, larger chunks
        chunk_ctas = (n_compute + GSVC_RAST_EXCHANGE_MAX_CHUNKS - 1) / GSVC_RAST_EXCHANGE_MAX_CHUNKS;
        n_chunks = (n_compute + chunk_ctas - 1) / chunk_ctas;
    }
    const int n_ex = x->n_ctas > 0 ? x->n_ctas : 65;                 // one coordinator + 64 movers
    if (n_ex < 2) return fail(GSVC_RAST_ERR_INVALID, "the exchange role needs a coordinator and at least one mover: n_ctas >= 2");
    if (n_ex > 296) return fail(GSVC_RAST_ERR_INVALID, "n_ctas must be <= 296 (the exchange CTAs must stay co-resident)");
    ExchangeArgs ex{};
    ex.mc = static_cast<float4*>(x->multicast);
    ex.bufs = static_cast<float4* const*>(x->buffers);
    ex.pads = static_cast<unsigned int* const*>(x->signal_pads);
    ex.state = static_cast<unsigned int*>(x->state);
    ex.rank = x->rank; ex.world = x->world; ex.n_ex = n_ex;
    ex.chunk_ctas = chunk_ctas; ex.n_chunks = n_chunks; ex.n_compute = n_compute;
    ex.chunk_f4 = (long long)chunk_ctas * 128 * 14 / 4;
    ex.total_f4 = (long long)P * 14 / 4;
    DevSettings d;
    int rc = make_settings_views(st, n_views, views_host, n_out, shs ? sh_M : 0, d);
    if (rc) return rc;
    BwdOutputs out{nullptr, dL_dmeans2D, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, dL_packed};
    return backward_core(st, d, P, sh_M, capacity, means3D, shs, colors_precomp, scales, rotations, cov3D_precomp, radii,
                         geom, image, binning, scratch, scratch_is_zero, dL_dout, out, static_cast<cudaStream_t>(stream_),
                         ex);
}

int gsvc_rast_forward_ragged_launch(const gsvc_rast_settings* st, int32_t n_views, const gsvc_rast_view* views_host,
                                    int32_t n_out, const int32_t* counts_host, int32_t sh_M, const float* means3D,
                                    const float* shs, const float* colors_precomp, const float* opacities,
                                    const float* scales, const float* rotations, const float* cov3D_precomp, void* geom,
                                    void* image, void* binning, int64_t capacity, void* bwd_scratch, float* out_color,
                                    int32_t* radii, uint64_t* count_slot_host, uint32_t ticket, void* stream_)
{
    DevSettings d;
    int32_t P = 0;
    int rc = make_settings_ragged(st, n_views, views_host, n_out, counts_host, shs ? sh_M : 0, d, P);
    if (rc) return rc;
    return forward_launch_core(st, d, n_out, P, sh_M, means3D, shs, colors_precomp, opacities, scales, rotations,
                               cov3D_precomp, geom, image, binning, capacity, bwd_scratch, out_color, radii,
                               count_slot_host, ticket, static_cast<cudaStream_t>(stream_));
}

int gsvc_rast_forward_ragged_render(const gsvc_rast_settings* st, int32_t n_views, const gsvc_rast_view* views_host,
                                    int32_t n_out, const int32_t* counts_host, const void* geom, void* image,
                                    void* binning, int64_t capacity, float* out_color, void* stream_)
{
    DevSettings d;
    int32_t P = 0;
    int rc = make_settings_ragged(st, n_views, views_host, n_out, counts_host, 0, d, P);
    if (rc) return rc;
    return forward_render_core(st, d, n_out, P, geom, image, binning, capacity, out_color,
                               static_cast<cudaStream_t>(stream_));
}

int gsvc_rast_backward_ragged(const gsvc_rast_settings* st, int32_t n_views, const gsvc_rast_view* views_host,
                              int32_t n_out, const int32_t* counts_host, int32_t sh_M, int64_t capacity,
                              const float* means3D, const float* shs, const float* colors_precomp, const float* scales,
                              const float* rotations, const float* cov3D_precomp, const int32_t* radii,
                              const void* geom, const void* image, const void* binning, void* scratch,
                              int32_t scratch_is_zero, const float* dL_dout, float* dL_dmeans3D, float* dL_dmeans2D,
                              float* dL_dcolors, float* dL_dopacities, float* dL_dscales, float* dL_drotations,
                              float* dL_dcov3D, float* dL_dshs, void* stream_)
{
    DevSettings d;
    int32_t P = 0;
    int rc = make_settings_ragged(st, n_views, views_host, n_out, counts_host, shs ? sh_M : 0, d, P);
    if (rc) return rc;
    BwdOutputs out{dL_dmeans3D, dL_dmeans2D, dL_dcolors, dL_dopacities, dL_dscales, dL_drotations, dL_dcov3D, dL_dshs,
                   nullptr};
    return backward_core(st, d, P, sh_M, capacity, means3D, shs, colors_precomp, scales, rotations, cov3D_precomp, radii,
                         geom, image, binning, scratch, scratch_is_zero, dL_dout, out, static_cast<cudaStream_t>(stream_));
}

int gsvc_rast_export_keys(const gsvc_rast_settings* st, int32_t n_views, int64_t capacity, const void* image,
                          const void* binning, uint64_t* sorted_keys, uint32_t* point_list, uint32_t* ranges,
                          void* stream_)
{
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    DevSettings d;
    int rc = make_settings(st, 0, d);
    if (rc) return rc;
    if (n_views < 1 || n_views > MAX_VIEWS) return fail(GSVC_RAST_ERR_INVALID, "n_views out of range");
    d.n_views = n_views;
    if (!image || !binning) return fail(GSVC_RAST_ERR_INVALID, "image/binning is NULL");
    const bool dbg = st->debug != 0;
    ImageView im = image_view(const_cast<void*>(image), d.W, d.H, n_views);
    BinView b = bin_view(const_cast<void*>(binning), capacity > 0 ? capacity : 1);
    CK(launch_export_keys(d, im, b, capacity, reinterpret_cast<unsigned long long*>(sorted_keys), point_list,
                          ranges, stream),
       "export_keys");
    return 0;
}

int gsvc_rast_export_geom(int32_t P, int32_t sh_M, const void* geom, float* depth, float* xy, float* conic_opacity,
                          float* rgb, int32_t* rect, void* stream_)
{
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (!geom) return fail(GSVC_RAST_ERR_INVALID, "geom is NULL");
    const bool dbg = false;
    GeomView g = geom_view(const_cast<void*>(geom), P < 1 ? 1 : P, sh_M);
    CK(launch_export_geom(P, g, depth, xy, conic_opacity, rgb, rect, stream), "export_geom");
    return 0;
}

int gsvc_rast_export_image(const gsvc_rast_settings* st, int32_t n_views, const void* image, float* final_T,
                           uint32_t* n_contrib, void* stream_)
{
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    DevSettings d;
    int rc = make_settings(st, 0, d);
    if (rc) return rc;
    if (n_views < 1 || n_views > MAX_VIEWS) return fail(GSVC_RAST_ERR_INVALID, "n_views out of range");
    if (!image) return fail(GSVC_RAST_ERR_INVALID, "image is NULL");
    const bool dbg = false;
    ImageView im = image_view(const_cast<void*>(image), d.W, d.H, n_views);
    const size_t N = (size_t)d.W * d.H * n_views;
    if (final_T) CK(cudaMemcpyAsync(final_T, im.final_T, N * 4, cudaMemcpyDeviceToDevice, stream), "export final_T");
    if (n_contrib) CK(cudaMemcpyAsync(n_contrib, im.n_contrib, N * 4, cudaMemcpyDeviceToDevice, stream), "export n_contrib");
    return 0;
}

}  // extern "C"
