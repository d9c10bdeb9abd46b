// Fused L1 + D-SSIM photometric loss (SPEC "Photometric loss", decision U9) and its exact backward.
//
// The upstream 3DGS expression (utils/loss_utils.py:41-72, SURVEY.md row 17) evaluates SSIM as five depthwise 11x11
// Gaussian convolutions and ~20 element-wise ops over full-size fp32 tensors.  Here one CTA owns a 32x32 tile of one
// channel of one image: it stages the tile plus its halo of x and y in shared memory (zero outside the image, as
// F.conv2d's padding=5), runs the separable 11-tap window over the five signals x, y, x^2, y^2, xy, forms S and
// |x - y| per pixel and leaves one partial sum per CTA; a second small kernel sums the partials of each image in index
// order.  No atomics anywhere: loss and gradient are bit-reproducible.
//
// Precision: the moments are centred in each separable pass (ssim.cuh), never E[x^2] - mu^2.
//
// Backward (recompute, nothing stored by the forward): per pixel p of image n
//     dSbar/dx(p) = 1/(3HW) sum_q w(q-p) [dS/dmu_x(q) + 2 x(p) dS/dExx(q) + y(p) dS/dExy(q)]
// where dS/dmu_x contains -2 mu_x dS/dExx - mu_y dS/dExy: on flat patches the sum cancels like the variance.  The
// CTA therefore takes a shift k (x and y at its tile centre) and correlates the three maps
//     a(q) = dS/dmu_x|direct - 2 (mu_x(q) - kx) e(q) - (mu_y(q) - ky) f(q),   e = dS/dExx,   f = dS/dExy
// then dSbar/dx(p) = (A(p) + 2 (x(p) - kx) E(p) + (y(p) - ky) F(p)) / (3HW) with A, E, F the window sums of a, e, f.  The maps are recomputed over the tile plus a 5-pixel ring (moments from a
// 10-pixel halo of x and y): about 2.5x the forward's FMAs, but only x and y are read and dL/dx written once.
#include "ssim.cuh"

#include <atomic>
#include <cmath>

namespace gsvc {

namespace loss {

using namespace ssim;

// backward: maps on the (T+10)^2 ring region (padded to a multiple of RUN: 44), moments there from a 54^2 stage
constexpr int B_MW = 44;                    // map region rows / cols (42 used)
constexpr int B_SW = B_MW + 2 * R;          // 54: staged rows / cols
constexpr int B_SMEM_FLOATS = 2 * B_SW * B_SW + 5 * B_SW * B_MW;   // stage (later the maps) + horizontal sums
constexpr size_t B_SMEM_BYTES = (size_t)B_SMEM_FLOATS * 4;
static_assert(3 * B_MW * B_MW <= 2 * B_SW * B_SW, "maps alias the stage");
static_assert(3 * (T + 2 * R) * T <= 5 * B_SW * B_MW, "second horizontal pass aliases the first");

// Vertical 11-tap window sum of NS planes of `cols` columns: thread item = (column j, rows i0..i0+RUN-1);
// out[s][u] = sum_i g[i] * h[s][i0 + u + i][j].
template <int NS>
__device__ __forceinline__ void vpass(const float* h, int hrows, int cols, int i0, int j, float out[NS][RUN])
{
    const int plane = hrows * cols;
#pragma unroll
    for (int s = 0; s < NS; s++)
#pragma unroll
        for (int u = 0; u < RUN; u++) out[s][u] = 0.0f;
#pragma unroll
    for (int t = 0; t < RUN + 10; t++) {
        float v[NS];
#pragma unroll
        for (int s = 0; s < NS; s++) v[s] = h[s * plane + (i0 + t) * cols + j];
#pragma unroll
        for (int u = 0; u < RUN; u++) {
            const int i = t - u;
            if (i >= 0 && i < 11) {
#pragma unroll
                for (int s = 0; s < NS; s++) out[s][u] = fmaf(c_g[i], v[s], out[s][u]);
            }
        }
    }
}

// the shift of a CTA: x and y at its tile centre, clamped into the image
template <class Y>
__device__ __forceinline__ void tile_shift(const float* x, Y y, int H, int W, int ty, int tx, float& kx, float& ky)
{
    const int r = min(ty * T + T / 2, H - 1), c = min(tx * T + T / 2, W - 1);
    kx = __ldg(x + (size_t)r * W + c);
    ky = y((size_t)r * W + c);
}

// Tgt: PlanarTarget (fp32) or Rgb8Target (ssim.cuh); a CTA whose target frame is out of range leaves a NaN partial
template <class Tgt>
__global__ void __launch_bounds__(THREADS) loss_forward_kernel(int H, int W, const float* __restrict__ image,
                                                                 Tgt target, double2* __restrict__ partials)
{
    __shared__ float s_x[F_SW * F_SW], s_y[F_SW * F_SW];
    __shared__ float s_h[5 * F_HR * T];
    __shared__ float s_red[2][THREADS / 32];
    const int tx = blockIdx.x, ty = blockIdx.y, plane = blockIdx.z;      // plane = n * 3 + c
    const size_t off = (size_t)plane * H * W;
    const float* x = image + off;
    typename Tgt::Plane y;
    if (!target.plane(plane, H, W, y)) {
        if (threadIdx.x == 0) partials[((size_t)plane * gridDim.y + ty) * gridDim.x + tx] = make_double2(NAN, NAN);
        return;
    }
    stage(x, y, H, W, ty * T - R, tx * T - R, F_SW, F_SW, s_x, s_y);
    __syncthreads();
    hpass_moments(s_x, s_y, F_HR, T, F_SW, s_h);
    __syncthreads();
    // vertical pass + per-pixel terms: item = (column j, rows i0..i0+3): 32 x 8 items = one per thread
    const int j = threadIdx.x % T, i0 = (threadIdx.x / T) * RUN;
    float mo[5][RUN];
    vpass_moments(s_h, F_HR, T, i0, j, mo);
    float sum_s = 0.0f, sum_l1 = 0.0f;
    const int gc = tx * T + j;
    if (gc < W) {
#pragma unroll
        for (int u = 0; u < RUN; u++) {
            const int gr = ty * T + i0 + u;
            if (gr >= H) break;
            const float mux = mo[0][u], muy = mo[1][u];
            const float a1 = 2.0f * mux * muy + C1, a2 = 2.0f * mo[4][u] + C2;
            const float b1 = mux * mux + muy * muy + C1, b2 = mo[2][u] + mo[3][u] + C2;
            sum_s += (a1 * a2) / (b1 * b2);
            const size_t o = (size_t)gr * W + gc;
            sum_l1 += fabsf(__ldg(x + o) - y(o));
        }
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        sum_s += __shfl_xor_sync(0xffffffffu, sum_s, d);
        sum_l1 += __shfl_xor_sync(0xffffffffu, sum_l1, d);
    }
    if ((threadIdx.x & 31) == 0) { s_red[0][threadIdx.x >> 5] = sum_s; s_red[1][threadIdx.x >> 5] = sum_l1; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0;
#pragma unroll
        for (int w = 0; w < THREADS / 32; w++) { a += s_red[0][w]; b += s_red[1][w]; }
        partials[((size_t)plane * gridDim.y + ty) * gridDim.x + tx] = make_double2(a, b);
    }
}

// One CTA per image: the partials of its 3 * tiles CTAs summed in a fixed order (strided per thread, then a tree).
__global__ void __launch_bounds__(THREADS) loss_reduce_kernel(int per_image, double inv_count, float lambda,
                                                                const double2* __restrict__ partials,
                                                                float* __restrict__ loss)
{
    __shared__ double s_s[THREADS], s_l[THREADS];
    const double2* p = partials + (size_t)blockIdx.x * per_image;
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < per_image; i += THREADS) { a += p[i].x; b += p[i].y; }
    s_s[threadIdx.x] = a; s_l[threadIdx.x] = b;
    __syncthreads();
    for (int d = THREADS / 2; d >= 1; d >>= 1) {
        if (threadIdx.x < d) { s_s[threadIdx.x] += s_s[threadIdx.x + d]; s_l[threadIdx.x] += s_l[threadIdx.x + d]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double lam = lambda;
        loss[blockIdx.x] = (float)((1.0 - lam) * s_l[0] * inv_count + lam * (1.0 - s_s[0] * inv_count));
    }
}

// a CTA whose target frame is out of range writes zeros over its tile
template <class Tgt>
__global__ void __launch_bounds__(THREADS) loss_backward_kernel(int H, int W, const float* __restrict__ image,
                                                                  Tgt target, float lambda,
                                                                  const float* __restrict__ dL_dloss,
                                                                  float* __restrict__ dL_dimage)
{
    extern __shared__ float smem[];
    float* s_x = smem;                                   // stage [54][54] x2, later the maps a, e, f [44][44]
    float* s_y = smem + B_SW * B_SW;
    float* s_h = smem + 2 * B_SW * B_SW;                 // horizontal sums [5][54][44], later [3][42][32]
    const int tx = blockIdx.x, ty = blockIdx.y, plane = blockIdx.z;
    const size_t off = (size_t)plane * H * W;
    const float* x = image + off;
    typename Tgt::Plane y;
    if (!target.plane(plane, H, W, y)) {
        const int j = threadIdx.x % T, i0 = (threadIdx.x / T) * RUN, gc = tx * T + j;
        for (int u = 0; u < RUN && gc < W && ty * T + i0 + u < H; u++)
            dL_dimage[off + (size_t)(ty * T + i0 + u) * W + gc] = 0.0f;
        return;
    }
    float kx, ky;
    tile_shift(x, y, H, W, ty, tx, kx, ky);
    const int mr0 = ty * T - R, mc0 = tx * T - R;        // image coordinates of map element (0, 0)
    stage(x, y, H, W, mr0 - R, mc0 - R, B_SW, B_SW, s_x, s_y);
    __syncthreads();
    hpass_moments(s_x, s_y, B_SW, B_MW, B_SW, s_h);
    __syncthreads();
    // moments and maps on the 44 x 44 region: 44 columns x 11 row runs
    float* s_a = smem;
    float* s_e = smem + B_MW * B_MW;
    float* s_f = smem + 2 * B_MW * B_MW;
    for (int it = threadIdx.x; it < B_MW * (B_MW / RUN); it += THREADS) {
        const int j = it % B_MW, i0 = (it / B_MW) * RUN;
        float mo[5][RUN];
        vpass_moments(s_h, B_SW, B_MW, i0, j, mo);
        const int gc = mc0 + j;
        const bool col_in = gc >= 0 && gc < W;
#pragma unroll
        for (int u = 0; u < RUN; u++) {
            const int gr = mr0 + i0 + u;
            float a = 0.0f, e = 0.0f, f = 0.0f;
            if (col_in && gr >= 0 && gr < H) {                     // q outside the image is not a term of the mean
                const float mux = mo[0][u], muy = mo[1][u];
                const float a1 = 2.0f * mux * muy + C1, a2 = 2.0f * mo[4][u] + C2;
                const float b1 = mux * mux + muy * muy + C1, b2 = mo[2][u] + mo[3][u] + C2;
                const float r = 1.0f / (b1 * b2);
                const float s = a1 * a2 * r;                           // S
                e = -s / b2;                                           // dS/dExx = -A1 A2 / (B1 B2^2)
                f = 2.0f * a1 * r;                                     // dS/dExy = 2 A1 / (B1 B2)
                const float direct = 2.0f * muy * a2 * r - 2.0f * mux * s / b1;
                a = direct - 2.0f * (mux - kx) * e - (muy - ky) * f;
            }
            const int q = (i0 + u) * B_MW + j;
            s_a[q] = a; s_e[q] = e; s_f[q] = f;
        }
    }
    __syncthreads();
    // horizontal pass of the three maps: rows 0..41, 32 output columns
    {
        constexpr int HR = T + 2 * R, runs = T / RUN, pl = HR * T;
        for (int it = threadIdx.x; it < HR * runs; it += THREADS) {
            const int r = it / runs, j0 = (it - r * runs) * RUN;
            float acc[3][RUN];
#pragma unroll
            for (int s = 0; s < 3; s++)
#pragma unroll
                for (int u = 0; u < RUN; u++) acc[s][u] = 0.0f;
#pragma unroll
            for (int t = 0; t < RUN + 10; t++) {
                const int q = r * B_MW + j0 + t;
                const float va = s_a[q], ve = s_e[q], vf = s_f[q];
#pragma unroll
                for (int u = 0; u < RUN; u++) {
                    const int i = t - u;
                    if (i >= 0 && i < 11) {
                        acc[0][u] = fmaf(c_g[i], va, acc[0][u]);
                        acc[1][u] = fmaf(c_g[i], ve, acc[1][u]);
                        acc[2][u] = fmaf(c_g[i], vf, acc[2][u]);
                    }
                }
            }
#pragma unroll
            for (int s = 0; s < 3; s++)
#pragma unroll
                for (int u = 0; u < RUN; u++) s_h[s * pl + r * T + j0 + u] = acc[s][u];
        }
    }
    __syncthreads();
    const int j = threadIdx.x % T, i0 = (threadIdx.x / T) * RUN;
    float sm[3][RUN];
    vpass<3>(s_h, T + 2 * R, T, i0, j, sm);
    const int gc = tx * T + j;
    if (gc >= W) return;
    const float inv = 1.0f / (3.0f * (float)H * (float)W);
    const float g = __ldg(dL_dloss + plane / 3);
    const float wl1 = g * (1.0f - lambda) * inv, wss = g * lambda * inv;
#pragma unroll
    for (int u = 0; u < RUN; u++) {
        const int gr = ty * T + i0 + u;
        if (gr >= H) break;
        const size_t o = (size_t)gr * W + gc;
        const float vx = __ldg(x + o), vy = y(o);
        const float d = vx - vy;
        const float sgn = d > 0.0f ? 1.0f : (d < 0.0f ? -1.0f : 0.0f);   // torch.sign: 0 where x == y
        const float dss = sm[0][u] + 2.0f * (vx - kx) * sm[1][u] + (vy - ky) * sm[2][u];
        dL_dimage[off + o] = wl1 * sgn - wss * dss;
    }
}

// the backward's 71 KB of shared memory: opted into once per device and instantiation (an attribute, no stream work)
template <class Tgt>
static cudaError_t prepare_backward()
{
    static std::atomic<unsigned long long> done{0};          // bit per device
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const unsigned long long bit = 1ull << (dev & 63);
    if (done.load() & bit) return cudaSuccess;
    e = cudaFuncSetAttribute(loss_backward_kernel<Tgt>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B_SMEM_BYTES);
    if (e == cudaSuccess) done.fetch_or(bit);
    return e;
}

}  // namespace loss

int fail(int code, const char* fmt, ...);

static int loss_check(int32_t n, int32_t H, int32_t W, const float* image, const void* target, float lambda)
{
    if (!image || !target) return fail(GSVC_RAST_ERR_INVALID, "image / target is NULL");
    if (n < 1 || H < 1 || W < 1) return fail(GSVC_RAST_ERR_INVALID, "n_images, H and W must be >= 1, got %d, %d, %d", n, H, W);
    if (!std::isfinite(lambda) || lambda < 0.0f || lambda > 1.0f)
        return fail(GSVC_RAST_ERR_INVALID, "lambda_dssim must be a finite value in [0, 1], got %g", (double)lambda);
    if ((long long)n * 3 > 65535 || (H + loss::T - 1) / loss::T > 65535)
        return fail(GSVC_RAST_ERR_INVALID, "size too large: n_images * 3 and ceil(H / 32) must be <= 65535");
    if ((double)n * 3.0 * (double)H * (double)W >= 9.0e18)
        return fail(GSVC_RAST_ERR_INVALID, "size too large: n_images * 3 * H * W overflows a 64-bit index");
    return GSVC_RAST_OK;
}

// the frame cube of an 8-bit target (SPEC U12), after the size rules of the call it goes with
int rgb8_target_check(int32_t n, int32_t H, int32_t W, int32_t n_frames, const int32_t* frame_index)
{
    if (n_frames < 1) return fail(GSVC_RAST_ERR_INVALID, "n_frames must be >= 1, got %d", n_frames);
    if (!frame_index && n > n_frames)
        return fail(GSVC_RAST_ERR_INVALID, "frame_index is NULL (image n against frame n) but n_images %d > n_frames %d",
                    n, n_frames);
    if ((double)n_frames * 3.0 * (double)H * (double)W >= 9.0e18)
        return fail(GSVC_RAST_ERR_INVALID, "size too large: n_frames * H * W * 3 overflows a 64-bit index");
    return GSVC_RAST_OK;
}

template <class Tgt>
static int loss_forward(int32_t n_images, int32_t H, int32_t W, const float* image, Tgt target, float lambda_dssim,
                        float* loss, void* scratch, cudaStream_t st)
{
    const dim3 grid((W + loss::T - 1) / loss::T, (H + loss::T - 1) / loss::T, n_images * 3);
    double2* partials = static_cast<double2*>(scratch);
    count_launch(2);
    loss::loss_forward_kernel<<<grid, loss::THREADS, 0, st>>>(H, W, image, target, partials);
    loss::loss_reduce_kernel<<<n_images, loss::THREADS, 0, st>>>((int)(3 * grid.x * grid.y),
                                                                  1.0 / (3.0 * (double)H * (double)W), lambda_dssim,
                                                                  partials, loss);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? GSVC_RAST_OK : fail(GSVC_RAST_ERR_CUDA, "loss_forward: %s", cudaGetErrorString(e));
}

template <class Tgt>
static int loss_backward(int32_t n_images, int32_t H, int32_t W, const float* image, Tgt target, float lambda_dssim,
                         const float* dL_dloss, float* dL_dimage, cudaStream_t st)
{
    cudaError_t e = loss::prepare_backward<Tgt>();
    if (e != cudaSuccess) return fail(GSVC_RAST_ERR_CUDA, "loss_backward: %s", cudaGetErrorString(e));
    const dim3 grid((W + loss::T - 1) / loss::T, (H + loss::T - 1) / loss::T, n_images * 3);
    count_launch();
    loss::loss_backward_kernel<<<grid, loss::THREADS, loss::B_SMEM_BYTES, st>>>(H, W, image, target, lambda_dssim,
                                                                                 dL_dloss, dL_dimage);
    e = cudaGetLastError();
    return e == cudaSuccess ? GSVC_RAST_OK : fail(GSVC_RAST_ERR_CUDA, "loss_backward: %s", cudaGetErrorString(e));
}

}  // namespace gsvc

using namespace gsvc;

extern "C" {

size_t gsvc_rast_loss_scratch_bytes(int32_t n_images, int32_t H, int32_t W)
{
    const size_t n = (size_t)(n_images < 1 ? 1 : n_images);
    const size_t tiles = (size_t)((H < 1 ? 1 : H) + loss::T - 1) / loss::T * (size_t)(((W < 1 ? 1 : W) + loss::T - 1) / loss::T);
    return align_up(n * 3 * tiles * sizeof(double2), 256) + 256;
}

int gsvc_rast_loss_forward(int32_t n_images, int32_t H, int32_t W, const float* image, const float* target,
                           float lambda_dssim, float* loss, void* scratch, void* stream_)
{
    int rc = loss_check(n_images, H, W, image, target, lambda_dssim);
    if (rc != GSVC_RAST_OK) return rc;
    if (!loss || !scratch) return fail(GSVC_RAST_ERR_INVALID, "loss / scratch is NULL");
    return loss_forward(n_images, H, W, image, ssim::PlanarTarget{target}, lambda_dssim, loss, scratch,
                        static_cast<cudaStream_t>(stream_));
}

int gsvc_rast_loss_backward(int32_t n_images, int32_t H, int32_t W, const float* image, const float* target,
                            float lambda_dssim, const float* dL_dloss, float* dL_dimage, void* stream_)
{
    int rc = loss_check(n_images, H, W, image, target, lambda_dssim);
    if (rc != GSVC_RAST_OK) return rc;
    if (!dL_dloss || !dL_dimage) return fail(GSVC_RAST_ERR_INVALID, "dL_dloss / dL_dimage is NULL");
    return loss_backward(n_images, H, W, image, ssim::PlanarTarget{target}, lambda_dssim, dL_dloss, dL_dimage,
                         static_cast<cudaStream_t>(stream_));
}

int gsvc_rast_loss_forward_rgb8(int32_t n_images, int32_t H, int32_t W, const float* image, const uint8_t* frames,
                                int32_t n_frames, const int32_t* frame_index, float lambda_dssim, float* loss,
                                void* scratch, void* stream_)
{
    int rc = loss_check(n_images, H, W, image, frames, lambda_dssim);
    if (rc == GSVC_RAST_OK) rc = rgb8_target_check(n_images, H, W, n_frames, frame_index);
    if (rc != GSVC_RAST_OK) return rc;
    if (!loss || !scratch) return fail(GSVC_RAST_ERR_INVALID, "loss / scratch is NULL");
    return loss_forward(n_images, H, W, image, ssim::Rgb8Target{frames, frame_index, n_frames}, lambda_dssim, loss, scratch,
                        static_cast<cudaStream_t>(stream_));
}

int gsvc_rast_loss_backward_rgb8(int32_t n_images, int32_t H, int32_t W, const float* image, const uint8_t* frames,
                                 int32_t n_frames, const int32_t* frame_index, float lambda_dssim,
                                 const float* dL_dloss, float* dL_dimage, void* stream_)
{
    int rc = loss_check(n_images, H, W, image, frames, lambda_dssim);
    if (rc == GSVC_RAST_OK) rc = rgb8_target_check(n_images, H, W, n_frames, frame_index);
    if (rc != GSVC_RAST_OK) return rc;
    if (!dL_dloss || !dL_dimage) return fail(GSVC_RAST_ERR_INVALID, "dL_dloss / dL_dimage is NULL");
    return loss_backward(n_images, H, W, image, ssim::Rgb8Target{frames, frame_index, n_frames}, lambda_dssim, dL_dloss,
                         dL_dimage, static_cast<cudaStream_t>(stream_));
}

}  // extern "C"
