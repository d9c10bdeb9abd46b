// The SSIM window machinery shared by the photometric loss (loss.cu, SPEC U9) and the frame quality metrics
// (quality.cu, SPEC U10): the 11x11 Gaussian window (sigma 1.5) as two separable passes over a tile staged in shared
// memory, with centred moments in each pass.
//
// Precision.  sigma^2 = E[x^2] - mu^2 cancels on flat patches (sigma^2 << mu^2, and C2 = 9e-4 does not hide it), so
// the moments are never formed that way.  Each separable pass is a two-pass (centred) computation over its 11 taps,
// the weights of the zero-padded window summing to 1:
//     horizontal, per row r:  m(r) = sum_i g_i x_i                 v(r) = sum_i g_i (x_i - m(r))^2   (and y, xy)
//     vertical:               mu   = sum_r g_r m(r)                var  = sum_r g_r v(r) + sum_r g_r (m(r) - mu)^2
// (the law of total variance): every sum is of non-negative or centred terms, exact to fp32 rounding at any level of
// the image, flat regions included.
//
// Targets (SPEC U12).  A kernel reads its target through a reader type: PlanarTarget is the fp32 [N,3,H,W] tensor,
// Rgb8Target an 8-bit [F,H,W,3] frame cube with an optional device frame index (image n is compared with frame
// index[n], frame n without one).  Every thread of a CTA reads its plane's index word (one broadcast load per warp,
// no barrier before the staging can start); a CTA whose index is outside [0, F) reads no target byte, and its kernel
// writes NaN (forward, quality) or zero (backward) for it instead.  A byte q reads as fl(q / 255), the one correctly
// rounded division of torchvision's to_tensor.
//
// Every .cu file is compiled as its own whole-program module, so each includer gets its own copy of c_g.
#pragma once

#include "common.cuh"

namespace gsvc {

namespace ssim {

constexpr int T = 32;                       // output tile edge (pixels)
constexpr int R = 5;                        // window radius (11 taps)
constexpr int RUN = 4;                      // outputs per thread along the pass direction
constexpr int THREADS = 256;
constexpr float C1 = 0.01f * 0.01f;
constexpr float C2 = 0.03f * 0.03f;

// moments on the T x T tile from a (T+10)^2 stage
constexpr int F_SW = T + 2 * R;             // 42: staged rows / cols
constexpr int F_HR = T + 2 * R;             // 42: rows of the horizontal pass

// g[i] = exp(-(i-5)^2 / (2 * 1.5^2)) / sum_k (...), computed in double and rounded to fp32
__constant__ float c_g[11] = {0x1.0d956cp-10f, 0x1.f1fe02p-8f, 0x1.26eb18p-5f, 0x1.bff0fep-4f, 0x1.b43c40p-3f,
                              0x1.106560p-2f, 0x1.b43c40p-3f, 0x1.bff0fep-4f, 0x1.26eb18p-5f, 0x1.f1fe02p-8f,
                              0x1.0d956cp-10f};

// fp32 targets, planar like the images: the plane of CTA plane p starts at y + p * H * W
struct PlanarTarget {
    const float* y;
    struct Plane {
        const float* y;
        __device__ __forceinline__ float operator()(size_t o) const { return __ldg(y + o); }
    };
    __device__ __forceinline__ bool plane(int p, int H, int W, Plane& out) const
    {
        out.y = y + (size_t)p * H * W;
        return true;
    }
};

// 8-bit targets: frames [n_frames, H, W, 3] (RGB interleaved, any alignment), index [N] int32 or nullptr
struct Rgb8Target {
    const uint8_t* frames;
    const int32_t* index;
    int n_frames;
    struct Plane {
        const uint8_t* q;                       // channel c of the frame: pixel o at q[3 o]
        __device__ __forceinline__ float operator()(size_t o) const
        {
            return __fdiv_rn((float)__ldg(q + 3 * o), 255.0f);
        }
    };
    // false (for every thread of the CTA) when the frame of plane p's image is outside [0, n_frames)
    __device__ __forceinline__ bool plane(int p, int H, int W, Plane& out) const
    {
        const int n = p / 3;
        const int f = index ? __ldg(index + n) : n;
        if (f < 0 || f >= n_frames) return false;
        out.q = frames + (size_t)f * H * W * 3 + (p - n * 3);
        return true;
    }
};

// Stage rows [r0, r0+rows) x cols [c0, c0+cols) of x and y (0 outside the image: the zero padding) into sx / sy.
// CLAMP_X: x is read clamped to [0, 1] as torch.clamp does it: NaN stays NaN, +-Inf become 1 / 0.
// y: a target plane reader (PlanarTarget::Plane, Rgb8Target::Plane).
template <bool CLAMP_X = false, class Y>
__device__ __forceinline__ void stage(const float* __restrict__ x, Y y, int H, int W, int r0, int c0, int rows,
                                      int cols, float* sx, float* sy)
{
    for (int e = threadIdx.x; e < rows * cols; e += THREADS) {
        const int r = e / cols, c = e - r * cols;
        const int gr = r0 + r, gc = c0 + c;
        float vx = 0.0f, vy = 0.0f;
        if (gr >= 0 && gr < H && gc >= 0 && gc < W) {
            const size_t o = (size_t)gr * W + gc;
            vx = __ldg(x + o);
            vy = y(o);
            if (CLAMP_X) vx = vx < 0.0f ? 0.0f : (vx > 1.0f ? 1.0f : vx);
        }
        sx[e] = vx;
        sy[e] = vy;
    }
}

// Horizontal pass, two-pass per output: h = (m_x, m_y, v_x, v_y, c_xy)[r][j] over taps j..j+10 of row r, rows < rows,
// j < cols (a multiple of RUN); the stage is `scols` wide.  Each thread makes RUN adjacent outputs from RUN + 10 loads.
__device__ __forceinline__ void hpass_moments(const float* sx, const float* sy, int rows, int cols, int scols, float* h)
{
    const int runs = cols / RUN, plane = rows * cols;
    for (int e = threadIdx.x; e < rows * runs; e += THREADS) {
        const int r = e / runs, j0 = (e - r * runs) * RUN;
        float vx[RUN + 10], vy[RUN + 10];
#pragma unroll
        for (int t = 0; t < RUN + 10; t++) { vx[t] = sx[r * scols + j0 + t]; vy[t] = sy[r * scols + j0 + t]; }
#pragma unroll
        for (int u = 0; u < RUN; u++) {
            float mx = 0.0f, my = 0.0f;
#pragma unroll
            for (int i = 0; i < 11; i++) { mx = fmaf(c_g[i], vx[u + i], mx); my = fmaf(c_g[i], vy[u + i], my); }
            float sxx = 0.0f, syy = 0.0f, sxy = 0.0f;
#pragma unroll
            for (int i = 0; i < 11; i++) {
                const float dx = vx[u + i] - mx, dy = vy[u + i] - my;
                const float gx = c_g[i] * dx;
                sxx = fmaf(gx, dx, sxx);
                sxy = fmaf(gx, dy, sxy);
                syy = fmaf(c_g[i] * dy, dy, syy);
            }
            const int o = r * cols + j0 + u;
            h[o] = mx; h[plane + o] = my; h[2 * plane + o] = sxx; h[3 * plane + o] = syy; h[4 * plane + o] = sxy;
        }
    }
}

// Vertical pass of the horizontal moments: thread item = (column j, rows i0..i0+RUN-1); out = (mu_x, mu_y, var_x,
// var_y, cov_xy)[u].  The within-row parts are plain window sums (shared by the RUN outputs), the between-row parts
// are centred on each output's own mean.
__device__ __forceinline__ void vpass_moments(const float* h, int hrows, int cols, int i0, int j, float out[5][RUN])
{
    const int plane = hrows * cols;
    float m[RUN + 10], n[RUN + 10], lin[3][RUN];
#pragma unroll
    for (int s = 0; s < 3; s++)
#pragma unroll
        for (int u = 0; u < RUN; u++) lin[s][u] = 0.0f;
#pragma unroll
    for (int t = 0; t < RUN + 10; t++) {
        const int o = (i0 + t) * cols + j;
        m[t] = h[o];
        n[t] = h[plane + o];
        const float a = h[2 * plane + o], b = h[3 * plane + o], c = h[4 * plane + o];
#pragma unroll
        for (int u = 0; u < RUN; u++) {
            const int i = t - u;
            if (i >= 0 && i < 11) {
                lin[0][u] = fmaf(c_g[i], a, lin[0][u]);
                lin[1][u] = fmaf(c_g[i], b, lin[1][u]);
                lin[2][u] = fmaf(c_g[i], c, lin[2][u]);
            }
        }
    }
#pragma unroll
    for (int u = 0; u < RUN; u++) {
        float mu = 0.0f, nu = 0.0f;
#pragma unroll
        for (int i = 0; i < 11; i++) { mu = fmaf(c_g[i], m[u + i], mu); nu = fmaf(c_g[i], n[u + i], nu); }
        float sxx = lin[0][u], syy = lin[1][u], sxy = lin[2][u];
#pragma unroll
        for (int i = 0; i < 11; i++) {
            const float dx = m[u + i] - mu, dy = n[u + i] - nu;
            const float gx = c_g[i] * dx;
            sxx = fmaf(gx, dx, sxx);
            sxy = fmaf(gx, dy, sxy);
            syy = fmaf(c_g[i] * dy, dy, syy);
        }
        out[0][u] = mu; out[1][u] = nu; out[2][u] = sxx; out[3][u] = syy; out[4][u] = sxy;
    }
}

}  // namespace ssim

}  // namespace gsvc
