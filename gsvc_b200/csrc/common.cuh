// Shared device/host definitions for libgsvc_rast.so (sm_100a).
// Layout of the three scratch buffers, the by-value kernel parameter block, and small helpers.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#include "../../include/gsvc_rast.h"

namespace gsvc {

constexpr int TILE = GSVC_RAST_TILE;          // 16x16 pixel tiles (SURVEY.md §8, Appendix A.2)
constexpr int TILE_PIX = TILE * TILE;
constexpr float ALPHA_MIN = 1.0f / 255.0f;    // Appendix A.3
constexpr float ALPHA_MAX = 0.99f;
constexpr float T_STOP = 0.0001f;
constexpr float LOWPASS = 0.3f;               // U5

// A batch of views of one Gaussian set (the TSW window: front/back views of one or more frames) is
// rasterized as ONE virtual problem: virtual Gaussian v*P + g, virtual tile v*Tv + t, virtual pixel
// v*N + pix.  Every kernel of the chain then runs once for the whole batch.  The drop-in calls are the
// batch of one view.
constexpr int MAX_VIEWS = GSVC_RAST_MAX_VIEWS;
struct ViewTable {
    const float* V[MAX_VIEWS];           // logical V[r][c] at V[r*vs_r + c*vs_c] (renderer.py:77 passes a permuted view)
    long long vs_r[MAX_VIEWS], vs_c[MAX_VIEWS];
    float campos[MAX_VIEWS][3];
    int out_image[MAX_VIEWS];            // which output image the view is blended into
    int flip_x[MAX_VIEWS];               // write / read that image mirrored in x (the back view of a frame)
    float weight[MAX_VIEWS];             // out[out_image] += weight * view  (1 for a plain view, 0.5 for a toast half)
};

// A per-view-set ("ragged") batch: every view has Gaussians of its own, concatenated in view order.  View v owns rows
// off[v] .. off[v+1]-1 of the inputs, and the virtual Gaussian is the row itself (tiles stay v*Tv + t).  By value in the
// launch parameters (68 bytes), so a ragged chain needs no device table.
struct ViewRows {
    int off[MAX_VIEWS + 1];
};

// Settings as the kernels see them (passed by value in the launch parameters).
struct DevSettings {
    int W, H, gx, gy;
    float x_min, y_min, scale, threshold, scale_modifier;
    const float* bg;
    int sh_degree, sh_M;
    int n_views, accumulate;   // accumulate: several views share an output image (atomic adds onto a zeroed image)
    ViewTable vt;
    int ragged;                // 0: one Gaussian set shared by every view (virtual Gaussian v*P + g); 1: `rows`
    ViewRows rows;
};

// Rows of the per-Gaussian state (geom, accumulators, radii) of a call with P input Gaussians (the total of the views'
// counts when ragged), and the most rows any one view has (the x extent of the per-view kernel grids).
inline int state_rows(const DevSettings& d, int P) { return d.ragged ? P : P * d.n_views; }
inline int max_view_rows(const DevSettings& d, int P)
{
    if (!d.ragged) return P;
    int m = 0;
    for (int v = 0; v < d.n_views; v++) m = d.rows.off[v + 1] - d.rows.off[v] > m ? d.rows.off[v + 1] - d.rows.off[v] : m;
    return m;
}

// ---- per-Gaussian state ("geom") -------------------------------------------------------------
//  feat0 = (pix.x, pix.y, rho_hi, B/C)   rho = B/A as rho_hi + rho_lo (fp64 quotient split into two floats); the two
//          ratios also steer the blend kernels' exact sub-tile culling
//  feat1 = (conic.A, conic.B, conic.C, opacity)      feat2 = (r, g, b, view depth)
//  feat3 = (l11, rho_lo, l22, opacity): Cholesky factor L = (l11 0; l11 rho, l22) of the conic times log2(e)/2 —
//          what the blend kernels evaluate: alpha = opacity * 2^-((l11 (dx + rho dy))^2 + (l22 dy)^2)
//  rect  = tile rectangle (minx, miny, maxx, maxy), max exclusive; all-zero when culled
struct GeomView {
    float4* feat0;
    float4* feat1;
    float4* feat2;
    float4* feat3;
    ushort4* rect;
    uint8_t* clamped;  // [P,3], SH clamp flags (only when shs are given)
};

// ---- per-tile / per-pixel state ("image") -----------------------------------------------------
struct ImageHeader {
    unsigned long long num_rendered;  // R = sum of tile counts
    unsigned int overflow;            // set by the scatter kernel when capacity was exceeded
    unsigned int n_heavy;             // tiles whose bucket the sort kernel left to sort_heavy_kernel (reset by the scan)
    unsigned int pad[28];
};
struct ImageView {
    ImageHeader* hdr;
    // T below = n_views * tiles per view, H*W = n_views * pixels per view (virtual tiles / pixels)
    unsigned int* tile_count;   // [T] instances per tile (atomics in preprocess)
    unsigned long long* scan_partials;  // [T/1024 + 1] per-CTA aggregates of the tile scan, then ONE ticket word
                                        // (the scan's dynamic CTA order); all zeroed with tile_count
    unsigned int* tile_offset;  // [T] exclusive scan of tile_count
    unsigned int* tile_cursor;  // [T] scatter cursors
    uint2* ranges;              // [T] (start,end) — (0,0) for untouched tiles, as identifyTileRanges leaves them
    unsigned int* heavy_tiles;  // [T] tiles with more instances than the sort kernel's shared-memory path holds
    float* final_T;             // [H*W]
    unsigned int* n_contrib;    // [H*W]
};

// ---- per-instance state ("binning") -----------------------------------------------------------
struct BinView {
    unsigned long long* inst;   // [cap] unsorted (depth_key << 32 | gaussian id), grouped by tile
    unsigned int* point_list;   // [cap] sorted Gaussian ids
    unsigned int* depth_keys;   // [cap] sorted depth keys (for export_keys)
};

__host__ __device__ inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

template <typename T>
__host__ __device__ inline T* carve(char*& p, size_t count)
{
    T* r = reinterpret_cast<T*>(p);
    p += align_up(count * sizeof(T), 256);
    return r;
}

inline GeomView geom_view(void* buf, int P, int sh_M)
{
    char* p = static_cast<char*>(buf);
    GeomView g;
    g.feat0 = carve<float4>(p, P);
    g.feat1 = carve<float4>(p, P);
    g.feat2 = carve<float4>(p, P);
    g.feat3 = carve<float4>(p, P);
    g.rect = carve<ushort4>(p, P);
    g.clamped = sh_M > 0 ? carve<uint8_t>(p, (size_t)P * 3) : nullptr;
    return g;
}
inline size_t geom_bytes(int P, int sh_M)
{
    char* p = nullptr;
    carve<float4>(p, P); carve<float4>(p, P); carve<float4>(p, P); carve<float4>(p, P); carve<ushort4>(p, P);
    if (sh_M > 0) carve<uint8_t>(p, (size_t)P * 3);
    return (size_t)p + 256;
}
inline ImageView image_view(void* buf, int W, int H, int n_views = 1)
{
    char* p = static_cast<char*>(buf);
    size_t T = (size_t)((W + TILE - 1) / TILE) * ((H + TILE - 1) / TILE) * n_views;
    size_t N = (size_t)W * H * n_views;
    ImageView v;
    v.hdr = carve<ImageHeader>(p, 1);
    v.tile_count = carve<unsigned int>(p, T);
    v.scan_partials = carve<unsigned long long>(p, T / 1024 + 2);
    v.tile_offset = carve<unsigned int>(p, T);
    v.tile_cursor = carve<unsigned int>(p, T);
    v.ranges = carve<uint2>(p, T);
    v.heavy_tiles = carve<unsigned int>(p, T);
    v.final_T = carve<float>(p, N);
    v.n_contrib = carve<unsigned int>(p, N);
    return v;
}
inline size_t image_bytes(int W, int H, int n_views = 1)
{
    char* p = nullptr;
    size_t T = (size_t)((W + TILE - 1) / TILE) * ((H + TILE - 1) / TILE) * n_views;
    size_t N = (size_t)W * H * n_views;
    carve<ImageHeader>(p, 1); carve<unsigned int>(p, T); carve<unsigned long long>(p, T / 1024 + 2);
    carve<unsigned int>(p, T); carve<unsigned int>(p, T); carve<uint2>(p, T); carve<unsigned int>(p, T); carve<float>(p, N);
    carve<unsigned int>(p, N);
    return (size_t)p + 256;
}
inline BinView bin_view(void* buf, long long cap)
{
    char* p = static_cast<char*>(buf);
    BinView b;
    b.inst = carve<unsigned long long>(p, (size_t)cap);
    b.point_list = carve<unsigned int>(p, (size_t)cap);
    b.depth_keys = carve<unsigned int>(p, (size_t)cap);
    return b;
}
inline size_t bin_bytes(long long cap)
{
    char* p = nullptr;
    carve<unsigned long long>(p, (size_t)cap); carve<unsigned int>(p, (size_t)cap); carve<unsigned int>(p, (size_t)cap);
    return (size_t)p + 256;
}

// Per-Gaussian gradient accumulators written by the blend backward (3 float4 per Gaussian):
//  acc0 = (S w u, S w v, S w u^2, S w u v)  acc1 = (S w v^2, S w, dL/dr, dL/dg)  acc2 = (dL/db,0,0,0)
//  with w = Gs * dL/dGs summed over the Gaussian's pixels and (u, v) = L^T (xy - pixel) the offset whitened by the
//  Cholesky factor in feat3; preprocess_backward turns the moments into dL/dpix, dL/dcov2D (a congruence with L)
inline size_t bwd_scratch_bytes(int P) { return align_up((size_t)P * 48, 256) + 256; }

// U2: order-preserving float -> uint32 (ascending key == ascending view depth, negatives included)
__host__ __device__ inline unsigned int ordered_u32(float z)
{
#ifdef __CUDA_ARCH__
    unsigned int u = __float_as_uint(z);
#else
    unsigned int u; memcpy(&u, &z, 4);
#endif
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// [P,4] float rows (quaternions and their gradients) move as ONE 16-byte access when the base pointer allows it and as
// four scalars otherwise: the C-ABI promises nothing beyond float alignment, and a torch slice of a flat parameter
// buffer at float offset 10*P (hostpipe / graphed layouts) is only 8-byte aligned when P is odd.
__device__ __forceinline__ float4 ld_row4(const float* __restrict__ base, size_t row)
{
    if ((reinterpret_cast<uintptr_t>(base) & 15u) == 0u) return __ldg(reinterpret_cast<const float4*>(base) + row);
    const float* p = base + 4 * row;
    return make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3));
}
__device__ __forceinline__ void st_row4(float* __restrict__ base, size_t row, float4 v)
{
    if ((reinterpret_cast<uintptr_t>(base) & 15u) == 0u) { reinterpret_cast<float4*>(base)[row] = v; return; }
    float* p = base + 4 * row;
    p[0] = v.x; p[1] = v.y; p[2] = v.z; p[3] = v.w;
}

// ---- the forward's covariance arithmetic, contraction-proof ---------------------------------------------------------
// Sigma = (R S)(R S)^T and cov2D = scale^2 (W Sigma W^T)[0:2,0:2] + 0.3 I in fp32 with every product and sum rounded
// separately, in this order (explicit _rn intrinsics: never fused, whatever -fmad says).  The preprocess kernel
// builds radii / rectangles / the conic from these numbers, bit-reproducibly against the scalar CPU oracle; the
// per-Gaussian backward evaluates d(conic)/d(cov2D) at THE SAME fp32 (a, b, c) — for an elongated Gaussian the
// inverse is so ill-conditioned (det = a c - b^2 cancels by the squared axis ratio) that "the same to 1e-7" would
// already be a different Gaussian along the long axis.
#define GSVC_MUL(a, b) __fmul_rn((a), (b))
#define GSVC_ADD(a, b) __fadd_rn((a), (b))
#define GSVC_SUB(a, b) __fsub_rn((a), (b))

// Quaternion (r,x,y,z) -> rotation, convention of /root/reference/utils/general_utils.py:98-119, used as given
// (callers normalise: guassian.py:287).
__device__ __forceinline__ void quat_to_rot(const float4 q, float R[9])
{
    const float r = q.x, x = q.y, y = q.z, z = q.w;
    R[0] = GSVC_SUB(1.f, GSVC_MUL(2.f, GSVC_ADD(GSVC_MUL(y, y), GSVC_MUL(z, z))));
    R[1] = GSVC_MUL(2.f, GSVC_SUB(GSVC_MUL(x, y), GSVC_MUL(r, z)));
    R[2] = GSVC_MUL(2.f, GSVC_ADD(GSVC_MUL(x, z), GSVC_MUL(r, y)));
    R[3] = GSVC_MUL(2.f, GSVC_ADD(GSVC_MUL(x, y), GSVC_MUL(r, z)));
    R[4] = GSVC_SUB(1.f, GSVC_MUL(2.f, GSVC_ADD(GSVC_MUL(x, x), GSVC_MUL(z, z))));
    R[5] = GSVC_MUL(2.f, GSVC_SUB(GSVC_MUL(y, z), GSVC_MUL(r, x)));
    R[6] = GSVC_MUL(2.f, GSVC_SUB(GSVC_MUL(x, z), GSVC_MUL(r, y)));
    R[7] = GSVC_MUL(2.f, GSVC_ADD(GSVC_MUL(y, z), GSVC_MUL(r, x)));
    R[8] = GSVC_SUB(1.f, GSVC_MUL(2.f, GSVC_ADD(GSVC_MUL(x, x), GSVC_MUL(y, y))));
}

__device__ __forceinline__ float dot3_rn(float a0, float b0, float a1, float b1, float a2, float b2)
{
    return GSVC_ADD(GSVC_ADD(GSVC_MUL(a0, b0), GSVC_MUL(a1, b1)), GSVC_MUL(a2, b2));
}

__device__ __forceinline__ void cov3d_from_scale_rot(const float* s3, float mod, const float4 q, float cov[6])
{
    float R[9], M[9];
    quat_to_rot(q, R);
    const float sx = GSVC_MUL(mod, s3[0]), sy = GSVC_MUL(mod, s3[1]), sz = GSVC_MUL(mod, s3[2]);
#pragma unroll
    for (int i = 0; i < 3; i++) {
        M[3 * i + 0] = GSVC_MUL(R[3 * i + 0], sx);
        M[3 * i + 1] = GSVC_MUL(R[3 * i + 1], sy);
        M[3 * i + 2] = GSVC_MUL(R[3 * i + 2], sz);
    }
    cov[0] = dot3_rn(M[0], M[0], M[1], M[1], M[2], M[2]);
    cov[1] = dot3_rn(M[0], M[3], M[1], M[4], M[2], M[5]);
    cov[2] = dot3_rn(M[0], M[6], M[1], M[7], M[2], M[8]);
    cov[3] = dot3_rn(M[3], M[3], M[4], M[4], M[5], M[5]);
    cov[4] = dot3_rn(M[3], M[6], M[4], M[7], M[5], M[8]);
    cov[5] = dot3_rn(M[6], M[6], M[7], M[7], M[8], M[8]);
}

// cov2D = scale^2 (W Sigma W^T)[0:2,0:2] + 0.3 I  — the orthographic Jacobian is scale*[I2|0] (no perspective term)
__device__ __forceinline__ void cov2d_ortho(const float cov[6], const float w0[3], const float w1[3], float scale,
                                            float& a, float& b, float& c)
{
    const float u00 = dot3_rn(cov[0], w0[0], cov[1], w0[1], cov[2], w0[2]);
    const float u01 = dot3_rn(cov[1], w0[0], cov[3], w0[1], cov[4], w0[2]);
    const float u02 = dot3_rn(cov[2], w0[0], cov[4], w0[1], cov[5], w0[2]);
    const float u10 = dot3_rn(cov[0], w1[0], cov[1], w1[1], cov[2], w1[2]);
    const float u11 = dot3_rn(cov[1], w1[0], cov[3], w1[1], cov[4], w1[2]);
    const float u12 = dot3_rn(cov[2], w1[0], cov[4], w1[1], cov[5], w1[2]);
    const float s2 = GSVC_MUL(scale, scale);
    a = GSVC_ADD(GSVC_MUL(s2, dot3_rn(w0[0], u00, w0[1], u01, w0[2], u02)), LOWPASS);
    b = GSVC_MUL(s2, dot3_rn(w0[0], u10, w0[1], u11, w0[2], u12));
    c = GSVC_ADD(GSVC_MUL(s2, dot3_rn(w1[0], u10, w1[1], u11, w1[2], u12)), LOWPASS);
}

// ---- programmatic dependent launch (sm_90+): every kernel of a forward / backward chain is launched with
// programmaticStreamSerializationAllowed, signals launch_dependents on entry and waits for its predecessor's
// memory before touching any data, so launch latency and prologue of kernel N+1 overlap the tail of kernel N.
__device__ __forceinline__ void pdl_prologue()
{
#if defined(__CUDA_ARCH__)
    asm volatile("griddepcontrol.launch_dependents;");
    asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, cudaStream_t st, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ---- warp-flattened enumeration of (Gaussian, tile) pairs ---------------------------------------------
// Every lane owns one Gaussian with a tile rectangle of `area` tiles (0 = none).  Instead of each lane
// looping over its own rectangle (a divergent loop whose length is the largest rectangle of the warp, up to
// hundreds of tiles), the warp enumerates the concatenation of all its rectangles 32 pairs at a time:
// pair index -> owner lane by a 5-step binary search over the inclusive scan of the areas.
struct WarpTiles {
    int incl, excl, total;  // inclusive / exclusive scan of area over the warp, and its total
    int rx, ry, rw;         // this lane's rectangle origin and width
};

__device__ __forceinline__ WarpTiles warp_tiles_begin(int area, int rx, int ry, int rw)
{
    const int lane = threadIdx.x & 31;
    int v = area;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v += o;
    }
    WarpTiles w;
    w.incl = v; w.excl = v - area; w.total = __shfl_sync(0xffffffffu, v, 31);
    w.rx = rx; w.ry = ry; w.rw = rw;
    return w;
}

// Pair `idx` of the warp (all 32 lanes must call): returns its tile id (or -1 if idx >= total) and the owner lane.
__device__ __forceinline__ int warp_tiles_get(const WarpTiles& w, int idx, int gx, int& owner)
{
    int o = 0;
#pragma unroll
    for (int step = 16; step >= 1; step >>= 1) {
        const int v = __shfl_sync(0xffffffffu, w.incl, o + step - 1);
        if (v <= idx) o += step;
    }
    o = min(o, 31);
    const int local = idx - __shfl_sync(0xffffffffu, w.excl, o);
    const int rw = __shfl_sync(0xffffffffu, w.rw, o);
    const int rx = __shfl_sync(0xffffffffu, w.rx, o), ry = __shfl_sync(0xffffffffu, w.ry, o);
    owner = o;
    if (idx >= w.total) return -1;
    // row = local / rw without the ~30-instruction signed integer division: approximate quotient in fp32
    // (local < 2^24, rw < 2^16 for any image this library accepts), then one exact correction step
    int row = __float2int_rz(__fdividef(__int2float_rz(local), __int2float_rz(rw)));
    int rem = local - row * rw;
    if (rem < 0) { row--; rem += rw; }
    else if (rem >= rw) { row++; rem -= rw; }
    return (ry + row) * gx + rx + rem;
}

// ---- launch stages implemented in the .cu files ------------------------------------------------
struct PreInputs {
    int P;                     // Gaussians of the shared set, or rows of a ragged batch (all views)
    const float* means3D;
    const float* shs;
    const float* colors_precomp;
    const float* opacities;
    const float* scales;
    const float* rotations;
    const float* cov3D_precomp;
    // visible_filter only: anchors outside [range_lo, range_hi) are declared culled WITHOUT being read
    // (slab-ordered anchors: the caller knows which index range can intersect the TSW slab); 0, P = everything
    int range_lo, range_hi;
};

cudaError_t launch_visible_filter(const DevSettings& s, const PreInputs& in, int32_t* radii, cudaStream_t st);
// scratch of the filter + compaction: [count | visible count per 256-anchor CTA | CTA offsets | one ballot word per warp]
inline size_t compact_scratch_bytes(int P)
{
    const size_t n = ((size_t)(P < 1 ? 1 : P) + 255) / 256;
    return 256 + 2 * align_up(n * 4, 256) + align_up(n * 32, 256) + 256;
}
cudaError_t launch_visible_filter_compact(const DevSettings& s, const PreInputs& in, int32_t* radii, int32_t* indices,
                                          void* scratch, unsigned long long* host_slot, unsigned int ticket,
                                          cudaStream_t st);
cudaError_t launch_preprocess(const DevSettings& s, const PreInputs& in, int32_t* radii, GeomView g, ImageView im,
                              float4* acc_to_zero, cudaStream_t st);
cudaError_t launch_tile_scan(const DevSettings& s, ImageView im, unsigned long long* host_slot, unsigned int ticket,
                             cudaStream_t st);
cudaError_t launch_scatter(const DevSettings& s, int P, GeomView g, ImageView im, BinView b, long long cap,
                           bool count_overflow_events, cudaStream_t st);
cudaError_t launch_sort_tiles(const DevSettings& s, ImageView im, BinView b, long long cap, cudaStream_t st);
cudaError_t launch_render_forward(const DevSettings& s, GeomView g, ImageView im, BinView b, long long cap,
                                  float* out_color, cudaStream_t st);
cudaError_t launch_render_backward(const DevSettings& s, int rows, GeomView g, ImageView im, BinView b, long long cap,
                                   const float* dL_dout, float4* acc, bool acc_is_zero, cudaStream_t st);
struct BwdOutputs {
    float* dL_dmeans3D; float* dL_dmeans2D; float* dL_dcolors; float* dL_dopacities;   // dL_dmeans2D is [n_views,P,3]
    float* dL_dscales; float* dL_drotations; float* dL_dcov3D; float* dL_dshs;
    float* packed;  // optional [P,14] (means3D, colours, opacity, scales, rotation) replacing the five dense arrays
};
// the exchange a per-Gaussian backward launch may carry (collective.cuh: exchange_role)
struct ExchangeArgs {
    float4* mc;                        // the buffer through the multicast mapping (nullptr: peer loads / stores)
    float4* const* bufs;               // [world] the ranks' buffers as mapped here
    unsigned int* const* pads;         // [world] the ranks' signal pads as mapped here
    unsigned int* state;               // [2 + n_chunks] zeroed words of local memory: go, done, chunk counters
    int rank, world;
    int n_ex;                          // CTAs of the exchange role (0: the launch carries no exchange)
    int chunk_ctas, n_chunks;          // compute CTAs per chunk; chunks of the buffer
    int n_compute;                     // compute CTAs of the launch
    long long chunk_f4, total_f4;      // 16-byte words per chunk / in the buffer
};
cudaError_t launch_preprocess_backward(const DevSettings& s, const PreInputs& in, const int32_t* radii, GeomView g,
                                       const float4* acc, BwdOutputs out, ExchangeArgs ex, cudaStream_t st);
cudaError_t launch_export_keys(const DevSettings& s, ImageView im, BinView b, long long R,
                               unsigned long long* sorted_keys, unsigned int* point_list, unsigned int* ranges,
                               cudaStream_t st);
cudaError_t launch_export_geom(int P, GeomView g, float* depth, float* xy, float* conic_opacity, float* rgb,
                               int32_t* rect, cudaStream_t st);

cudaError_t read_overflow_events(unsigned int* host_value, bool reset, cudaStream_t st);
cudaError_t launch_densify_stats(int n_views, int P, const float* dm2d, const int32_t* radii, float* stats,
                                 long long stride, bool accumulate, cudaStream_t st);

cudaError_t launch_switch_allreduce(float* multicast, void* const* buffers, unsigned int* const* pads, unsigned int* state,
                                    int rank, int world, long long numel, int n_ctas, cudaStream_t st);
void count_launch(int n = 1);

}  // namespace gsvc
