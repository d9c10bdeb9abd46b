// Frame quality metrics (SPEC "Evaluation metrics", decision U10): PSNR, SSIM and MS-SSIM of each rendered image
// against its target, on the device, in one pass over the full-size images.
//
// Level 0 (the images themselves): one CTA per 32x32 tile of one channel plane stages the tile and its 5-pixel halo
// (x clamped to [0, 1] on read, zero outside the image), runs the window of ssim.cuh and leaves four partial sums:
// sum (x - y)^2 and sum S over its pixels (PSNR, SSIM), sum S and sum cs over its interior pixels (>= 5 px from
// every border, where the zero-padded window equals the valid one: level 0 of MS-SSIM).  From the same stage it
// writes its share of the 2x2-pooled images of level 1: the halo holds the straddling pool window of an odd side's
// front padding, so the pooling costs no extra read of the full-size images.  Levels 1-4 (a third of a pair's pixels
// together) run the same tile kernel on the pooled images: interior sums plus the next pooled level.  One reduce
// kernel then sums each plane's partials in a fixed order in double and forms (PSNR, SSIM, MS-SSIM) per image.
// No atomics: the results are bit-reproducible, and an image's result does not depend on its batch.
#include "ssim.cuh"

#include <math.h>

#include <type_traits>

namespace gsvc {

namespace quality {

using namespace ssim;

constexpr int LEVELS = 5;
constexpr int MS_MIN_SIDE = 161;            // MS-SSIM needs min(H, W) > (11 - 1) * 2^4 (pytorch_msssim's assertion)
constexpr int PT = T / 2;                   // pooled outputs per CTA edge

// Scratch: per level the CTA partials (double4 each), then the pooled x / y images of levels 1..4.
struct Layout {
    int h[LEVELS], w[LEVELS], gx[LEVELS], gy[LEVELS];
    size_t part[LEVELS], img_x[LEVELS], img_y[LEVELS];
    size_t bytes;
};

static Layout layout(int n, int H, int W)
{
    Layout L;
    const size_t planes = (size_t)n * 3;
    size_t o = 0;
    for (int l = 0; l < LEVELS; l++) {
        L.h[l] = l == 0 ? H : (L.h[l - 1] + 1) / 2;
        L.w[l] = l == 0 ? W : (L.w[l - 1] + 1) / 2;
        L.gx[l] = (L.w[l] + T - 1) / T;
        L.gy[l] = (L.h[l] + T - 1) / T;
        L.part[l] = o;
        o += align_up(planes * L.gx[l] * L.gy[l] * sizeof(double4), 256);
    }
    L.img_x[0] = L.img_y[0] = 0;
    for (int l = 1; l < LEVELS; l++) {
        const size_t b = align_up(planes * L.h[l] * L.w[l] * sizeof(float), 256);
        L.img_x[l] = o;
        L.img_y[l] = o + b;
        o += 2 * b;
    }
    L.bytes = o + 256;
    return L;
}

// One 32x32 tile of one plane of an h x w level.  L0: x is clamped on read and the all-pixel sums are formed.
// partials[cta] = (sum (x - y)^2, sum S, interior sum S, interior sum cs); xo / yo (nullptr after the last level):
// the ceil(h/2) x ceil(w/2) pooled images, avg_pool2d(2, 2, padding = (h % 2, w % 2), count_include_pad).
// Tgt: PlanarTarget, or Rgb8Target at level 0 (ssim.cuh).  A CTA whose target frame is out of range leaves NaN
// partials and NaN pooled values, so every level of its image is NaN.
template <bool L0, class Tgt>
__global__ void __launch_bounds__(THREADS) quality_level_kernel(int h, int w, const float* __restrict__ xi, Tgt yi,
                                                                  double4* __restrict__ partials,
                                                                  float* __restrict__ xo, float* __restrict__ yo)
{
    __shared__ float s_x[F_SW * F_SW], s_y[F_SW * F_SW];
    __shared__ float s_h[5 * F_HR * T];
    __shared__ float s_red[4][THREADS / 32];
    pdl_prologue();
    const int tx = blockIdx.x, ty = blockIdx.y, plane = blockIdx.z;      // plane = n * 3 + c
    const size_t off = (size_t)plane * h * w;
    const int r0 = ty * T - R, c0 = tx * T - R;                          // image coordinates of stage (0, 0)
    typename Tgt::Plane y;
    if (!yi.plane(plane, h, w, y)) {
        if (xo) {
            const int ho = (h + 1) / 2, wo = (w + 1) / 2;
            const int oi = ty * PT + threadIdx.x / PT, oj = tx * PT + threadIdx.x % PT;
            if (oi < ho && oj < wo) {
                const size_t o = (size_t)plane * ho * wo + (size_t)oi * wo + oj;
                xo[o] = NAN;
                yo[o] = NAN;
            }
        }
        if (threadIdx.x == 0) partials[((size_t)plane * gridDim.y + ty) * gridDim.x + tx] = make_double4(NAN, NAN, NAN, NAN);
        return;
    }
    stage<L0>(xi + off, y, h, w, r0, c0, F_SW, F_SW, s_x, s_y);
    __syncthreads();
    hpass_moments(s_x, s_y, F_HR, T, F_SW, s_h);
    if (xo) {                                   // pooled level: one output per thread from the stage
        const int ho = (h + 1) / 2, wo = (w + 1) / 2;
        const int oi = ty * PT + threadIdx.x / PT, oj = tx * PT + threadIdx.x % PT;
        if (oi < ho && oj < wo) {
            const int r = 2 * oi - (h & 1) - r0, c = 2 * oj - (w & 1) - c0;
            const int q = r * F_SW + c;
            const size_t o = (size_t)plane * ho * wo + (size_t)oi * wo + oj;
            xo[o] = 0.25f * ((s_x[q] + s_x[q + 1]) + (s_x[q + F_SW] + s_x[q + F_SW + 1]));
            yo[o] = 0.25f * ((s_y[q] + s_y[q + 1]) + (s_y[q + F_SW] + s_y[q + F_SW + 1]));
        }
    }
    __syncthreads();
    const int j = threadIdx.x % T, i0 = (threadIdx.x / T) * RUN;
    float mo[5][RUN];
    vpass_moments(s_h, F_HR, T, i0, j, mo);
    float sum_sq = 0.0f, sum_s = 0.0f, in_s = 0.0f, in_cs = 0.0f;
    const int gc = tx * T + j;
    if (gc < w) {
        const bool col_in = gc >= R && gc < w - R;
#pragma unroll
        for (int u = 0; u < RUN; u++) {
            const int gr = ty * T + i0 + u;
            if (gr >= h) break;
            // every product and sum rounded on its own: x == y gives a1 == b1 and a2 == b2, so S == cs == 1 exactly
            const float mux = mo[0][u], muy = mo[1][u];
            const float a1 = __fadd_rn(__fmul_rn(2.0f, __fmul_rn(mux, muy)), C1);
            const float b1 = __fadd_rn(__fadd_rn(__fmul_rn(mux, mux), __fmul_rn(muy, muy)), C1);
            const float a2 = __fadd_rn(__fmul_rn(2.0f, mo[4][u]), C2);
            const float b2 = __fadd_rn(__fadd_rn(mo[2][u], mo[3][u]), C2);
            const float s = __fdiv_rn(__fmul_rn(a1, a2), __fmul_rn(b1, b2));
            if (L0) {
                const int q = (i0 + u + R) * F_SW + j + R;
                const float d = s_x[q] - s_y[q];
                sum_sq = fmaf(d, d, sum_sq);
                sum_s += s;
            }
            if (col_in && gr >= R && gr < h - R) {
                in_s += s;
                in_cs += __fdiv_rn(a2, b2);
            }
        }
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        if (L0) {
            sum_sq += __shfl_xor_sync(0xffffffffu, sum_sq, d);
            sum_s += __shfl_xor_sync(0xffffffffu, sum_s, d);
        }
        in_s += __shfl_xor_sync(0xffffffffu, in_s, d);
        in_cs += __shfl_xor_sync(0xffffffffu, in_cs, d);
    }
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        s_red[0][warp] = sum_sq; s_red[1][warp] = sum_s; s_red[2][warp] = in_s; s_red[3][warp] = in_cs;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double4 a = make_double4(0.0, 0.0, 0.0, 0.0);
#pragma unroll
        for (int k = 0; k < THREADS / 32; k++) {
            a.x += s_red[0][k]; a.y += s_red[1][k]; a.z += s_red[2][k]; a.w += s_red[3][k];
        }
        partials[((size_t)plane * gridDim.y + ty) * gridDim.x + tx] = a;
    }
}

struct ReduceArgs {
    const double4* part[LEVELS];
    long long ctas[LEVELS];                 // CTAs per plane of each level
    double valid[LEVELS];                   // (h - 10)(w - 10) of each level
    double count;                           // 3 H W
    int levels;                             // 1 (no MS-SSIM) or LEVELS
};

// One CTA per image: every (channel, level) sum in a fixed order (strided per thread, butterfly per warp, warps in
// index order), then PSNR, SSIM and MS-SSIM in double.  NAN_ROWS (8-bit targets, whose values are finite): a NaN
// level-0 sum marks an out-of-range frame, and the whole row is NaN (MS-SSIM's clamp at 0 would otherwise hide it).
template <bool NAN_ROWS>
__global__ void __launch_bounds__(THREADS) quality_reduce_kernel(ReduceArgs a, float* __restrict__ quality)
{
    __shared__ double s_w[4][THREADS / 32];
    __shared__ double s_tot[3][LEVELS][4];
    pdl_prologue();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int c = 0; c < 3; c++) {
        for (int l = 0; l < a.levels; l++) {
            const double4* p = a.part[l] + ((long long)blockIdx.x * 3 + c) * a.ctas[l];
            double v[4] = {0.0, 0.0, 0.0, 0.0};
            for (long long i = threadIdx.x; i < a.ctas[l]; i += THREADS) {
                const double4 q = p[i];
                v[0] += q.x; v[1] += q.y; v[2] += q.z; v[3] += q.w;
            }
#pragma unroll
            for (int k = 0; k < 4; k++) {
#pragma unroll
                for (int d = 16; d >= 1; d >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], d);
                if (lane == 0) s_w[k][warp] = v[k];
            }
            __syncthreads();
            if (threadIdx.x < 4) {
                double t = 0.0;
                for (int k = 0; k < THREADS / 32; k++) t += s_w[threadIdx.x][k];
                s_tot[c][l][threadIdx.x] = t;
            }
            __syncthreads();
        }
    }
    if (threadIdx.x != 0) return;
    const double sq = s_tot[0][0][0] + s_tot[1][0][0] + s_tot[2][0][0];
    const double ss = s_tot[0][0][1] + s_tot[1][0][1] + s_tot[2][0][1];
    const double psnr = sq == 0.0 ? (double)INFINITY : -10.0 * log10(sq / a.count);
    double ms = (double)NAN;
    if (a.levels == LEVELS) {
        const double wt[LEVELS] = {0.0448, 0.2856, 0.3001, 0.2363, 0.1333};
        ms = 0.0;
        for (int c = 0; c < 3; c++) {
            double prod = 1.0;
            for (int l = 0; l < LEVELS; l++) {
                const double m = s_tot[c][l][l == LEVELS - 1 ? 2 : 3] / a.valid[l];   // cs of levels 0-3, ssim of 4
                prod *= pow(fmax(m, 0.0), wt[l]);
            }
            ms += prod;
        }
        ms /= 3.0;
    }
    if (NAN_ROWS && isnan(ss)) ms = (double)NAN;
    float* out = quality + (size_t)blockIdx.x * 3;
    out[0] = (float)psnr;
    out[1] = (float)(ss / a.count);
    out[2] = (float)ms;
}

}  // namespace quality

int fail(int code, const char* fmt, ...);

int rgb8_target_check(int32_t n, int32_t H, int32_t W, int32_t n_frames, const int32_t* frame_index);   // loss.cu

static int quality_check(int32_t n, int32_t H, int32_t W, const float* image, const void* target, const float* out,
                         const void* scratch)
{
    if (!image || !target) return fail(GSVC_RAST_ERR_INVALID, "image / target is NULL");
    if (!out || !scratch) return fail(GSVC_RAST_ERR_INVALID, "quality / scratch is NULL");
    if (n < 1 || H < 1 || W < 1) return fail(GSVC_RAST_ERR_INVALID, "n_images, H and W must be >= 1, got %d, %d, %d", n, H, W);
    if ((long long)n * 3 > 65535 || (H + quality::T - 1) / quality::T > 65535)
        return fail(GSVC_RAST_ERR_INVALID, "size too large: n_images * 3 and ceil(H / 32) must be <= 65535");
    if ((double)n * 3.0 * (double)H * (double)W >= 9.0e18)
        return fail(GSVC_RAST_ERR_INVALID, "size too large: n_images * 3 * H * W overflows a 64-bit index");
    return GSVC_RAST_OK;
}

template <class Tgt>
static int quality_run(int32_t n_images, int32_t H, int32_t W, const float* image, Tgt target, float* quality,
                       void* scratch, cudaStream_t st)
{
    using namespace quality;
    constexpr bool rgb8 = !std::is_same<Tgt, PlanarTarget>::value;
    const Layout L = layout(n_images, H, W);
    char* base = static_cast<char*>(scratch);
    const int levels = (H < MS_MIN_SIDE || W < MS_MIN_SIDE) ? 1 : LEVELS;   // no pyramid without MS-SSIM
    ReduceArgs ra;
    for (int l = 0; l < LEVELS; l++) {
        ra.part[l] = reinterpret_cast<const double4*>(base + L.part[l]);
        ra.ctas[l] = (long long)L.gx[l] * L.gy[l];
        ra.valid[l] = (double)(L.h[l] - 2 * R) * (double)(L.w[l] - 2 * R);
    }
    ra.count = 3.0 * (double)H * (double)W;
    ra.levels = levels;
    cudaError_t e = cudaSuccess;
    for (int l = 0; l < levels && e == cudaSuccess; l++) {
        const dim3 grid(L.gx[l], L.gy[l], n_images * 3);
        double4* part = reinterpret_cast<double4*>(base + L.part[l]);
        float* xo = l + 1 < levels ? reinterpret_cast<float*>(base + L.img_x[l + 1]) : nullptr;
        float* yo = l + 1 < levels ? reinterpret_cast<float*>(base + L.img_y[l + 1]) : nullptr;
        if (l == 0)
            e = launch_pdl(quality_level_kernel<true, Tgt>, grid, dim3(THREADS), st, H, W, image, target, part, xo, yo);
        else
            e = launch_pdl(quality_level_kernel<false, PlanarTarget>, grid, dim3(THREADS), st, L.h[l], L.w[l],
                           reinterpret_cast<const float*>(base + L.img_x[l]),
                           PlanarTarget{reinterpret_cast<const float*>(base + L.img_y[l])}, part, xo, yo);
    }
    if (e == cudaSuccess) e = launch_pdl(quality_reduce_kernel<rgb8>, dim3(n_images), dim3(THREADS), st, ra, quality);
    count_launch(levels + 1);
    if (e == cudaSuccess) e = cudaGetLastError();
    return e == cudaSuccess ? GSVC_RAST_OK : fail(GSVC_RAST_ERR_CUDA, "quality: %s", cudaGetErrorString(e));
}

}  // namespace gsvc

using namespace gsvc;

extern "C" {

size_t gsvc_rast_quality_scratch_bytes(int32_t n_images, int32_t H, int32_t W)
{
    return quality::layout(n_images < 1 ? 1 : n_images, H < 1 ? 1 : H, W < 1 ? 1 : W).bytes;
}

int gsvc_rast_quality(int32_t n_images, int32_t H, int32_t W, const float* image, const float* target, float* quality,
                      void* scratch, void* stream_)
{
    int rc = quality_check(n_images, H, W, image, target, quality, scratch);
    if (rc != GSVC_RAST_OK) return rc;
    return quality_run(n_images, H, W, image, ssim::PlanarTarget{target}, quality, scratch, static_cast<cudaStream_t>(stream_));
}

int gsvc_rast_quality_rgb8(int32_t n_images, int32_t H, int32_t W, const float* image, const uint8_t* frames,
                           int32_t n_frames, const int32_t* frame_index, float* quality, void* scratch, void* stream_)
{
    int rc = quality_check(n_images, H, W, image, frames, quality, scratch);
    if (rc == GSVC_RAST_OK) rc = rgb8_target_check(n_images, H, W, n_frames, frame_index);
    if (rc != GSVC_RAST_OK) return rc;
    return quality_run(n_images, H, W, image, ssim::Rgb8Target{frames, frame_index, n_frames}, quality, scratch,
                       static_cast<cudaStream_t>(stream_));
}

}  // extern "C"
