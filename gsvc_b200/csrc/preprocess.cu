// Kernel (1)/(1'): per-Gaussian preprocess for the orthographic TSW camera (SURVEY.md Appendix A.1;
// call sites /root/reference/ortho_gaussian_renderer/renderer.py:90-98 and preprocess.py:99-104).
//
// THIS TRANSLATION UNIT IS COMPILED WITH -fmad=false: every product and sum below rounds
// separately, in the written order, so radii / tile rectangles / depth keys — the integers the
// binning stage is built from — are reproducible bit-for-bit by a scalar fp32 CPU restatement.
// The kernel is a pure stream (56 B in, <= 60 B out per Gaussian): HBM-bound, FMA fusion buys nothing.
#include "common.cuh"

namespace gsvc {

__device__ __forceinline__ float ldV(const DevSettings& s, int v, int r, int c)
{
    return __ldg(s.vt.V[v] + r * s.vt.vs_r[v] + c * s.vt.vs_c[v]);
}

// /root/reference/utils/sh_utils.py:26-43
__device__ const float SH_C0 = 0.28209479177387814f;
__device__ const float SH_C1 = 0.4886025119029199f;
__device__ const float SH_C2[5] = {1.0925484305920792f, -1.0925484305920792f, 0.31539156525252005f,
                                   -1.0925484305920792f, 0.5462742152960396f};
__device__ const float SH_C3[7] = {-0.5900435899266435f, 2.890611442640554f, -0.4570457994644658f,
                                   0.3731763325901154f, -0.4570457994644658f, 1.445305721320277f,
                                   -0.5900435899266435f};

// quat_to_rot / cov3d_from_scale_rot / cov2d_ortho: common.cuh (shared, bit for bit, with the per-Gaussian backward)

__device__ __forceinline__ void sh_to_rgb(int deg, const float* sh, const float p[3], const float campos[3],
                                          float rgb[3], uint8_t clamped[3])
{
    const float dx = p[0] - campos[0], dy = p[1] - campos[1], dz = p[2] - campos[2];
    const float inv = 1.0f / sqrtf(dx * dx + dy * dy + dz * dz);
    const float x = dx * inv, y = dy * inv, z = dz * inv;
#pragma unroll
    for (int c = 0; c < 3; c++) {
        float r = SH_C0 * sh[0 * 3 + c];
        if (deg > 0) {
            r = r - SH_C1 * y * sh[1 * 3 + c] + SH_C1 * z * sh[2 * 3 + c] - SH_C1 * x * sh[3 * 3 + c];
            if (deg > 1) {
                const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
                r = r + SH_C2[0] * xy * sh[4 * 3 + c] + SH_C2[1] * yz * sh[5 * 3 + c] +
                    SH_C2[2] * (2.0f * zz - xx - yy) * sh[6 * 3 + c] + SH_C2[3] * xz * sh[7 * 3 + c] +
                    SH_C2[4] * (xx - yy) * sh[8 * 3 + c];
                if (deg > 2) {
                    r = r + SH_C3[0] * y * (3.0f * xx - yy) * sh[9 * 3 + c] + SH_C3[1] * xy * z * sh[10 * 3 + c] +
                        SH_C3[2] * y * (4.0f * zz - xx - yy) * sh[11 * 3 + c] +
                        SH_C3[3] * z * (2.0f * zz - 3.0f * xx - 3.0f * yy) * sh[12 * 3 + c] +
                        SH_C3[4] * x * (4.0f * zz - xx - yy) * sh[13 * 3 + c] +
                        SH_C3[5] * z * (xx - yy) * sh[14 * 3 + c] + SH_C3[6] * x * (xx - 3.0f * yy) * sh[15 * 3 + c];
                }
            }
        }
        r += 0.5f;
        clamped[c] = (r < 0.0f);
        rgb[c] = r < 0.0f ? 0.0f : r;
    }
}

// Stable stream compaction of the visible anchors (SURVEY.md §8f row f2: what `anchor[radii_pure > 0]` — a nonzero
// pass + a host synchronisation — does after prefilter_voxel, preprocess.py:99-108, guassian.py:147-153).
// Reduce-then-scan, no spinning: the filter kernel (MODE 2) also writes one ballot word per warp and one visible
// count per 256-anchor CTA; a single-CTA kernel scans the CTA counts and publishes the total; a write kernel turns
// ballots + CTA offsets into ascending indices.  (A single-pass decoupled look-back was built first and measured
// 2-3x slower than the filter itself: with one 256-anchor CTA per look-back word, ~1200 concurrently started CTAs
// spin on each other through L2 — profiles/r1_notes.md.)
struct CompactOut {
    unsigned int* ballots;            // [ceil(P/32)] visibility bits, one word per warp
    unsigned int* cta_count;          // [n_ctas] visible anchors per 256-anchor CTA
};

__global__ void __launch_bounds__(1024) compact_scan_kernel(int n_ctas, const unsigned int* __restrict__ cta_count,
                                                            unsigned int* __restrict__ cta_offset,
                                                            unsigned long long* count_dev,
                                                            unsigned long long* host_slot, unsigned int ticket)
{
    __shared__ unsigned int s_warp[32];
    __shared__ unsigned int s_carry;
    pdl_prologue();
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) s_carry = 0u;
    __syncthreads();
    for (int base = 0; base < n_ctas; base += 1024) {
        const int i = base + tid;
        const unsigned int c = i < n_ctas ? cta_count[i] : 0u;
        unsigned int v = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned int o = __shfl_up_sync(0xffffffffu, v, d);
            if (lane >= d) v += o;
        }
        if (lane == 31) s_warp[wid] = v;
        __syncthreads();
        if (wid == 0) {
            unsigned int w = s_warp[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned int o = __shfl_up_sync(0xffffffffu, w, d);
                if (lane >= d) w += o;
            }
            s_warp[lane] = w;   // inclusive over warps
        }
        __syncthreads();
        const unsigned int carry = s_carry;
        if (i < n_ctas) cta_offset[i] = carry + (wid ? s_warp[wid - 1] : 0u) + v - c;
        __syncthreads();
        if (tid == 0) s_carry = carry + s_warp[31];
        __syncthreads();
    }
    if (tid == 0) {
        const unsigned long long cnt = s_carry;
        if (count_dev) *count_dev = cnt;
        if (host_slot) *host_slot = ((unsigned long long)ticket << 40) | cnt;
    }
}

__global__ void __launch_bounds__(256) compact_write_kernel(int P, const unsigned int* __restrict__ ballots,
                                                            const unsigned int* __restrict__ cta_offset,
                                                            int32_t* __restrict__ indices)
{
    __shared__ unsigned int s_wsum[8];
    pdl_prologue();
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int g = blockIdx.x * 256 + tid;
    const int word = blockIdx.x * 8 + wid;
    const unsigned int bal = word * 32 < P ? ballots[word] : 0u;
    if (lane == 0) s_wsum[wid] = __popc(bal);
    __syncthreads();
    unsigned int before = cta_offset[blockIdx.x];
#pragma unroll
    for (int w = 0; w < 8; w++)
        if (w < wid) before += s_wsum[w];
    if ((bal >> lane) & 1u) indices[before + __popc(bal & ((1u << lane) - 1u))] = g;
}

// MODE 0: full preprocess + per-tile instance counting.  MODE 1: visible_filter (radii only).
// MODE 2: visible_filter + stable compaction of the visible indices.
// RAGGED (MODE 0 only): every view has its own rows (s.rows); the grid is (ceil(max_v P_v / 256), n_views).
template <int MODE, bool RAGGED = false>
__global__ void __launch_bounds__(256) preprocess_kernel(DevSettings s, PreInputs in, int32_t* __restrict__ radii,
                                                         GeomView geo, unsigned int* __restrict__ tile_count,
                                                         float4* __restrict__ acc_to_zero, CompactOut co)
{
    constexpr bool FILTER = MODE != 0;
    pdl_prologue();
    // Gaussians of this view: the shared set's P, or the view's own count (a CTA wholly past it has nothing to do)
    const int Pv = RAGGED ? s.rows.off[blockIdx.y + 1] - s.rows.off[blockIdx.y] : in.P;
    if (RAGGED && (int)(blockIdx.x * blockDim.x) >= Pv) return;
    // Lanes past the end stay in the warp (they redo the last Gaussian with all stores masked) so that the
    // warp-wide tile walk at the end (and the block-wide compaction) runs converged.
    const int g_raw = blockIdx.x * blockDim.x + threadIdx.x;
    bool valid = g_raw < Pv;
    if (FILTER) {
        // Slab-ordered anchors (SURVEY.md §8f row f4; the reference's stream codec keeps them z-sorted in 0.01
        // intervals, utils/encodings.py:827-862): only indices in [range_lo, range_hi) can be inside the TSW slab.
        // A CTA wholly outside writes its zeros and leaves before touching the inputs: the filter costs
        // O(slab) reads + 4 bytes per anchor.
        const int cta_lo = blockIdx.x * blockDim.x, cta_hi = cta_lo + blockDim.x;
        if (cta_hi <= in.range_lo || cta_lo >= in.range_hi) {
            if (valid && radii) radii[g_raw] = 0;
            if (MODE == 2) {
                if ((threadIdx.x & 31) == 0) co.ballots[g_raw >> 5] = 0u;
                if (threadIdx.x == 0) co.cta_count[blockIdx.x] = 0u;
            }
            return;
        }
    }
    const bool in_range = !FILTER || (g_raw >= in.range_lo && g_raw < in.range_hi);
    const int g = valid ? (in_range ? g_raw : min(max(g_raw, in.range_lo), in.range_hi - 1)) : Pv - 1;
    // view of the batch (grid.y)
    const int v = FILTER ? 0 : (int)blockIdx.y;
    // row of the inputs: g of the shared set, or the view's own row off_v + g.  Per-Gaussian state of view v lives
    // at virtual index v*P + g (shared) or at that row (ragged), its tiles at v*Tv + t
    const int gp = RAGGED ? s.rows.off[v] + g : g;
    const size_t gv = RAGGED ? (size_t)gp : (size_t)v * in.P + g;
    const float p[3] = {__ldg(in.means3D + 3 * gp), __ldg(in.means3D + 3 * gp + 1), __ldg(in.means3D + 3 * gp + 2)};
    // scales / quaternion are fetched together with the position (one memory round trip per Gaussian, at the
    // price of 28 wasted bytes for the third of the Gaussians the slab test culls)
    float sc[3] = {0.f, 0.f, 0.f};
    float4 q_pre = make_float4(1.f, 0.f, 0.f, 0.f);
    if (!in.cov3D_precomp) {
        sc[0] = __ldg(in.scales + 3 * gp); sc[1] = __ldg(in.scales + 3 * gp + 1); sc[2] = __ldg(in.scales + 3 * gp + 2);
        q_pre = ld_row4(in.rotations, (size_t)gp);
    }
    // The CTA's view matrix (strided device tensor: 12 loads + 64-bit stride arithmetic per thread otherwise) is
    // fetched once by 12 threads and broadcast through shared memory; the Gaussian's own loads above are already
    // in flight when the barrier is reached.
    __shared__ float s_V[12];
    if (threadIdx.x < 12) s_V[threadIdx.x] = ldV(s, v, threadIdx.x >> 2, threadIdx.x & 3);
    __syncthreads();
    const float w0[3] = {s_V[0], s_V[1], s_V[2]};
    const float w1[3] = {s_V[4], s_V[5], s_V[6]};
    const float vx = w0[0] * p[0] + w0[1] * p[1] + w0[2] * p[2] + s_V[3];
    const float vy = w1[0] * p[0] + w1[1] * p[1] + w1[2] * p[2] + s_V[7];
    const float vz = s_V[8] * p[0] + s_V[9] * p[1] + s_V[10] * p[2] + s_V[11];

    int radius = 0;
    int rminx = 0, rminy = 0, rmaxx = 0, rmaxy = 0;
    float a = 0.f, b = 0.f, c = 0.f, det = 0.f, px = 0.f, py = 0.f;
    // U6: TSW slab — keep |z_view| <= threshold (preprocess.py:109-116)
    bool ok = valid && in_range && !(fabsf(vz) > s.threshold);
    if (ok) {
        float cov[6];
        if (in.cov3D_precomp) {
#pragma unroll
            for (int k = 0; k < 6; k++) cov[k] = __ldg(in.cov3D_precomp + 6 * (size_t)gp + k);
        } else {
            cov3d_from_scale_rot(sc, s.scale_modifier, q_pre, cov);
        }
        cov2d_ortho(cov, w0, w1, s.scale, a, b, c);
        det = a * c - b * b;
        ok = (det != 0.0f);
    }
    if (ok) {
        const float mid = 0.5f * (a + c);
        const float lam = mid + sqrtf(fmaxf(0.1f, mid * mid - det));
        const float rad_f = ceilf(3.f * sqrtf(lam));
        radius = (int)rad_f;
        px = (vx - s.x_min) * s.scale - 0.5f;  // U1
        py = (vy - s.y_min) * s.scale - 0.5f;
        const float fgx = (float)s.gx, fgy = (float)s.gy, ft = (float)TILE;
        rminx = (int)fminf(fgx, fmaxf(0.f, truncf((px - rad_f) / ft)));
        rminy = (int)fminf(fgy, fmaxf(0.f, truncf((py - rad_f) / ft)));
        rmaxx = (int)fminf(fgx, fmaxf(0.f, truncf((px + rad_f + (float)(TILE - 1)) / ft)));
        rmaxy = (int)fminf(fgy, fmaxf(0.f, truncf((py + rad_f + (float)(TILE - 1)) / ft)));
        ok = (rmaxx - rminx) * (rmaxy - rminy) > 0;
    }
    if (valid && radii) radii[FILTER ? (size_t)g_raw : gv] = ok ? radius : 0;
    if (MODE == 2) {
        __shared__ unsigned int s_vis[8];
        const unsigned int bal = __ballot_sync(0xffffffffu, ok);
        if ((threadIdx.x & 31) == 0) {
            co.ballots[g_raw >> 5] = bal;
            s_vis[threadIdx.x >> 5] = __popc(bal);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned int tot = 0;
#pragma unroll
            for (int w = 0; w < 8; w++) tot += s_vis[w];
            co.cta_count[blockIdx.x] = tot;
        }
    }
    if (FILTER) return;

    if (ok) {
        const float det_inv = 1.f / det;
        const float cA = c * det_inv, cB = -b * det_inv, cC = a * det_inv;
        const float op = __ldg(in.opacities + gp);
        float rgb[3];
        if (in.colors_precomp) {
            rgb[0] = __ldg(in.colors_precomp + 3 * gp);
            rgb[1] = __ldg(in.colors_precomp + 3 * gp + 1);
            rgb[2] = __ldg(in.colors_precomp + 3 * gp + 2);
        } else {
            uint8_t cl[3];
            const float campos[3] = {s.vt.campos[v][0], s.vt.campos[v][1], s.vt.campos[v][2]};
            sh_to_rgb(s.sh_degree, in.shs + (size_t)gp * s.sh_M * 3, p, campos, rgb, cl);
            geo.clamped[3 * gv] = cl[0];
            geo.clamped[3 * gv + 1] = cl[1];
            geo.clamped[3 * gv + 2] = cl[2];
        }
        if (acc_to_zero) {
            // the blend backward accumulates into these 9 sums with atomics: zero them here (stores this kernel
            // hides) instead of a memset launch in the backward — visible Gaussians only, nobody reads the others
            const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
            acc_to_zero[3 * gv] = z; acc_to_zero[3 * gv + 1] = z; acc_to_zero[3 * gv + 2] = z;
        }
        // What the blend kernels evaluate: the STORED conic (A, B; B, C) times log2(e)/2 = K, factored as L L^T with
        // L = (l11 0; l11 rho, l22), rho = B / A:
        //   alpha = op * 2^-(u^2 + v^2),   u = l11 (dx + rho dy),   v = l22 dy
        // a sum of squares where A dx^2 + 2 B dx dy + C dy^2 cancels.  Two places need more than fp32 for an elongated,
        // rotated Gaussian (B^2 ~ A C):
        //  * the Schur complement C - B^2/A behind l22: from A C - B^2 with the products' rounding errors recovered by
        //    FMAs (two-product);
        //  * the shear rho.  dx + rho dy cancels along the needle (hundreds of pixels against a result of a few), so a
        //    1e-7 relative error of rho is 1e-4 px of lateral offset 1000 px out — 1e-4 relative in alpha for a needle
        //    half a pixel wide, and the same in every moment its gradients are made of (found by the referee checker:
        //    scale / rotation gradients of 256:1 needles off by 4e-4).  rho is therefore carried as an unevaluated
        //    sum rho_hi + rho_lo of two floats from the fp64 quotient, and the blend accumulates dx + rho_hi dy +
        //    rho_lo dy with FMAs (exact products, rounding at the small result).
        // l11 and l22 only scale u and v: their fp32 rounding is a 1e-7 relative error of the exponent, harmless.
        const float kL = 0.5f * 1.4426950408889634f;
        const float pac = cA * cC, pbb = cB * cB;
        const float det_c = (pac - pbb) + (fmaf(cA, cC, -pac) - fmaf(cB, cB, -pbb));
        const float aL = cA * kL;
        const float d22 = fmaxf(__fdividef(det_c, cA) * kL, 1e-30f);
        const double rho = (double)cB / (double)cA;            // A > 0: cov2D is positive definite (+0.3 on the diagonal)
        const float rho_hi = (float)rho, rho_lo = (float)(rho - (double)rho_hi);
        geo.feat0[gv] = make_float4(px, py, rho_hi, __fdividef(cB, cC));   // .z, .w also steer the blend's sub-tile culling
        geo.feat3[gv] = make_float4(aL * rsqrtf(aL), rho_lo, d22 * rsqrtf(d22), op);
        geo.feat1[gv] = make_float4(cA, cB, cC, op);
        geo.feat2[gv] = make_float4(rgb[0], rgb[1], rgb[2], vz);
        geo.rect[gv] = make_ushort4((unsigned short)rminx, (unsigned short)rminy, (unsigned short)rmaxx,
                                    (unsigned short)rmaxy);
    } else if (valid) {
        geo.rect[gv] = make_ushort4(0, 0, 0, 0);
    }
    // per-tile instance histogram (the counting sort's digit): the warp walks the flattened list of all its
    // (Gaussian, tile) pairs, 32 at a time, so every RED instruction is full width whatever the rectangle sizes
    const int rw = rmaxx - rminx;
    const WarpTiles wt = warp_tiles_begin(ok ? rw * (rmaxy - rminy) : 0, rminx, rminy, rw > 0 ? rw : 1);
    for (int base = 0; base < wt.total; base += 32) {
        int owner;
        const int t = warp_tiles_get(wt, base + (threadIdx.x & 31), s.gx, owner);
        if (t >= 0) atomicAdd(tile_count + (size_t)v * (s.gx * s.gy) + t, 1u);
    }
    // Measured and rejected (profiles/r1_notes.md): (a) taking each instance's rank inside its tile from this
    // atomic's return value and writing (composite, tile, rank) records so that the scatter needs no second atomic
    // pass; (b) running the tile scan in the last CTA of this kernel (threadfence + counter).  Both made the
    // 2-view step slower (+15 us): this kernel is instruction-bound, the fire-and-forget RED is free for it while
    // a returning ATOM or a serial single-CTA scan tail is not.

}

// the compaction scan on its own (the generator epilogue, epilogue.cu, compacts with the same three-kernel scheme)
cudaError_t launch_compact_scan(int n_ctas, const unsigned int* cta_count, unsigned int* cta_offset,
                                unsigned long long* count_dev, unsigned long long* host_slot, unsigned int ticket,
                                cudaStream_t st)
{
    return launch_pdl(compact_scan_kernel, dim3(1), dim3(1024), st, n_ctas, cta_count, cta_offset, count_dev, host_slot,
                      ticket);
}

cudaError_t launch_visible_filter(const DevSettings& s, const PreInputs& in, int32_t* radii, cudaStream_t st)
{
    if (in.P <= 0) return cudaSuccess;
    GeomView none{};
    count_launch();
    return launch_pdl(preprocess_kernel<1>, dim3((in.P + 255) / 256), dim3(256), st, s, in, radii, none,
                      (unsigned int*)nullptr, (float4*)nullptr, CompactOut{});
}

cudaError_t launch_visible_filter_compact(const DevSettings& s, const PreInputs& in, int32_t* radii, int32_t* indices,
                                          void* scratch, unsigned long long* host_slot, unsigned int ticket,
                                          cudaStream_t st)
{
    if (in.P <= 0) {
        if (host_slot) *host_slot = (unsigned long long)ticket << 40;   // pinned HOST memory: count 0, no launch
        return cudaSuccess;
    }
    // scratch: [count (8 B, 256-aligned) | CTA counts | CTA offsets | ballot words]
    const int n_ctas = (in.P + 255) / 256;
    char* p = static_cast<char*>(scratch);
    unsigned long long* count_dev = carve<unsigned long long>(p, 1);
    unsigned int* cta_count = carve<unsigned int>(p, n_ctas);
    unsigned int* cta_offset = carve<unsigned int>(p, n_ctas);
    unsigned int* ballots = carve<unsigned int>(p, (size_t)n_ctas * 8);
    CompactOut co{ballots, cta_count};
    GeomView none{};
    count_launch(3);
    cudaError_t e = launch_pdl(preprocess_kernel<2>, dim3(n_ctas), dim3(256), st, s, in, radii, none,
                               (unsigned int*)nullptr, (float4*)nullptr, co);
    if (e != cudaSuccess) return e;
    e = launch_pdl(compact_scan_kernel, dim3(1), dim3(1024), st, n_ctas, (const unsigned int*)cta_count, cta_offset,
                   count_dev, host_slot, ticket);
    if (e != cudaSuccess) return e;
    return launch_pdl(compact_write_kernel, dim3(n_ctas), dim3(256), st, in.P, (const unsigned int*)ballots,
                      (const unsigned int*)cta_offset, indices);
}

cudaError_t launch_preprocess(const DevSettings& s, const PreInputs& in, int32_t* radii, GeomView g, ImageView im,
                              float4* acc_to_zero, cudaStream_t st)
{
    // one memset clears the per-tile counters and the scan's per-CTA partials that sit right behind them
    const size_t T = (size_t)s.gx * s.gy * s.n_views;
    const size_t nbytes = reinterpret_cast<char*>(im.scan_partials + (T / 1024 + 2)) - reinterpret_cast<char*>(im.tile_count);
    cudaError_t e = cudaMemsetAsync(im.tile_count, 0, nbytes, st);
    if (e != cudaSuccess) return e;
    const int Pmax = max_view_rows(s, in.P);
    if (Pmax <= 0) return cudaSuccess;
    count_launch();
    return launch_pdl(s.ragged ? preprocess_kernel<0, true> : preprocess_kernel<0, false>,
                      dim3((Pmax + 255) / 256, s.n_views), dim3(256), st, s, in, radii, g, im.tile_count, acc_to_zero,
                      CompactOut{});
}

}  // namespace gsvc
