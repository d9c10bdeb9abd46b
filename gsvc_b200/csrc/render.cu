// Kernels (3) and (4): front-to-back alpha blend forward and its backward
// (SURVEY.md Appendix A.3 / A.4; the reference reaches them through
//  /root/reference/ortho_gaussian_renderer/renderer.py:90-98 and loss.backward(), pipeline/train.py:462).
//
// One CTA per 16x16 tile.  Forward: 128 threads, each of the 4 warps owns an 8x8-pixel block and every lane
// two pixels of it (rows r and r+4 of one column).  Backward: 64 threads, each HALF warp owns an 8x8 block and
// every lane four pixels of it (see there).  Gaussians of the tile's depth-sorted list are
// gathered with float4 loads into shared memory in batches of 256.  Both kernels are
// instruction-issue bound (ncu: ~85 % issue-active, < 5 % DRAM), so the design goal is to execute
// fewer and cheaper pixel-Gaussian evaluations, not to move fewer bytes:
//   * exact sub-tile culling — per chunk of 32 staged Gaussians every lane tests ONE Gaussian: can
//     its alpha >= 1/255 ellipse reach the warp's 8x8 block (closed-form maximum of the concave
//     exponent over the rectangle)?  A ballot gives the warp its private work list.  Only pairs the
//     reference would `continue` past (alpha < 1/255, no state change) are skipped, so results are
//     unchanged;
//   * two pixels per lane share the Gaussian fetch, the x terms of the exponent, the loop control and
//     — in the backward — the warp reduction, which is the single most expensive step;
//   * the conic is pre-scaled by -log2(e)/2 while staging, so a pair costs ~5 FP32 ops + one
//     ex2.approx (MUFU) up to the alpha test; staged records are 48 B interleaved so one address
//     serves all three LDS.128;
//   * warp-ballot early termination once all 64 pixels of a block are saturated (T < 1e-4 stop rule);
//   * backward: branch-free per-pair arithmetic on raw moments (the per-Gaussian kernel finishes
//     dL/dpix and dL/dconic), 9 sums reduced across a half warp with a transpose-butterfly (12 shuffles
//     instead of 36), two hits per loop iteration, and 9 lanes of each half issue the 9 atomics of its
//     Gaussian in a single instruction.
#include "common.cuh"

namespace gsvc {

constexpr int BLEND_THREADS = 128;  // 4 warps x (8x8 pixels), 2 pixels per lane
constexpr int BATCH = 256;          // Gaussians staged per round (2 per thread)
constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ float ex2_approx(float x)
{
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x)
{
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// ---- packed fp32 pairs (sm_100 FFMA2 / FMUL2 / FADD2) ---------------------------------------------
// Each lane blends two pixels (A = low half, B = high half) with identical instruction streams, and both
// blend kernels are bound by instruction issue, not by the FP32 pipes (ncu: ~85 % issue-active, fma pipe
// ~35 %).  One f32x2 instruction does the work of two scalar ones in a single issue slot (measured on
// B200: scripts/ubench/ffma2.cu); ptxas folds broadcast scalars, immediates and negations into its operands.
struct f2 { unsigned long long v; };
__device__ __forceinline__ f2 mk2(float lo, float hi)
{
    f2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r.v) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ f2 bc2(float s) { return mk2(s, s); }
__device__ __forceinline__ float lo(f2 a)
{
    float x;
    [[maybe_unused]] float y;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(a.v));
    return x;
}
__device__ __forceinline__ float hi(f2 a)
{
    [[maybe_unused]] float x;
    float y;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(a.v));
    return y;
}
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c)
{
    f2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r.v) : "l"(a.v), "l"(b.v), "l"(c.v));
    return r;
}
// c += a * b in place (ties the accumulator to one register pair across loop iterations)
__device__ __forceinline__ void fma2_acc(f2& c, f2 a, f2 b)
{
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(c.v) : "l"(a.v), "l"(b.v));
}
__device__ __forceinline__ f2 mul2(f2 a, f2 b)
{
    f2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
    return r;
}
__device__ __forceinline__ f2 add2(f2 a, f2 b)
{
    f2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
    return r;
}
__device__ __forceinline__ f2 sub2(f2 a, f2 b)
{
    f2 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
    return r;
}
__device__ __forceinline__ f2 neg2(f2 a) { return mk2(-lo(a), -hi(a)); }

// MINUS the log2 of the falloff of one staged Gaussian at this lane's two pixels, as a sum of squares:
//   -q = (l11 (dx + rho dy))^2 + (l22 dy)^2,   L = (l11 0; l11 rho, l22) = Cholesky factor of the conic scaled by log2(e)/2
// (dx is shared: same column).  Unlike A dx^2 + B dx dy + C dy^2 nothing cancels — for a needle-like Gaussian far
// from its centre those three terms are ~1e2 each and sum to ~1, which costs ~1e-5 of absolute accuracy in fp32 —
// and -q >= 0 holds by construction, so the reference's `power > 0 -> continue` (only ever taken through rounding)
// needs no test.
// rho = B/A comes as rho_hi + rho_lo (see preprocess.cu): dx + rho dy cancels along an elongated Gaussian, so the
// shear is accumulated with two FMAs (exact products, rounding at the small result) before the scale by l11.
__device__ __forceinline__ f2 neg_falloff_log2(float rho_hi, const float4 f1, float dx, f2 dy2, f2& u2, f2& v2)
{
    const f2 t2 = fma2(bc2(f1.y), dy2, fma2(bc2(rho_hi), dy2, bc2(dx)));
    u2 = mul2(bc2(f1.x), t2);
    v2 = mul2(bc2(f1.z), dy2);
    return fma2(u2, u2, mul2(v2, v2));
}
__device__ __forceinline__ f2 neg_falloff_log2(float rho_hi, const float4 f1, float dx, f2 dy2)
{
    f2 u2, v2;
    return neg_falloff_log2(rho_hi, f1, dx, dy2, u2, v2);
}

struct BlockGeom {
    int px, py;                    // this lane's first pixel; the second one is (px, py + 4)
    float xmin, xmax, ymin, ymax;  // pixel-centre bounds of the warp's 8x8 block
};

__device__ __forceinline__ BlockGeom block_geom(int tile, int gx, int tid)
{
    const int tx = tile % gx, ty = tile / gx;
    const int warp = tid >> 5, lane = tid & 31;
    const int bx0 = tx * TILE + (warp & 1) * 8, by0 = ty * TILE + (warp >> 1) * 8;
    BlockGeom b;
    b.px = bx0 + (lane & 7);
    b.py = by0 + (lane >> 3);
    b.xmin = (float)bx0; b.xmax = (float)(bx0 + 7);
    b.ymin = (float)by0; b.ymax = (float)(by0 + 7);
    return b;
}

// Staged record k = s_feat[3k .. 3k+2]:
//   [0] = (pix.x, pix.y, rho_hi, B/C)        rho = B/A = rho_hi + rho_lo
//   [1] = (l11, rho_lo, l22, opacity): Cholesky factor (l11 0; l11 rho, l22) of (A, B; B, C) * log2(e)/2, so that
//         alpha = opacity * 2^q(d),  -q(d) = (l11 (dx + rho dy))^2 + (l22 dy)^2
//   [2] = (r, g, b, Gaussian id as bits)
constexpr float CULL_MARGIN = 1e-3f;  // in log2 units (7e-4 relative in alpha) >> fp32 rounding of q

__device__ __forceinline__ void stage(float4* s_feat, int slot, const GeomView& geo, unsigned int id)
{
    // everything was prepared per Gaussian by the preprocess kernel: three 16-byte gathers, no arithmetic
    const float4 f0 = __ldg(geo.feat0 + id);
    const float4 f1 = __ldg(geo.feat3 + id);
    float4 f2 = __ldg(geo.feat2 + id);
    f2.w = __uint_as_float(id);   // rides along with the colour: the backward's atomics need it per hit
    s_feat[3 * slot] = f0;
    s_feat[3 * slot + 1] = f1;
    s_feat[3 * slot + 2] = f2;
}

// Exact sub-tile culling: can the staged Gaussian reach alpha >= 1/255 anywhere in the block
// [xmin,xmax] x [ymin,ymax]?  q is concave with its maximum (0) at the centre, so its maximum over
// the rectangle is attained at the centre if that lies inside, else on an edge facing the centre:
// on the vertical line x = clamp(cx) the maximiser is y = cy - (B/C)(x - cx), on the horizontal
// line y = clamp(cy) it is x = cx - (B/A)(y - cy), each clamped to the edge.  Both candidates are
// points of the rectangle, so max(q1, q2) never over-estimates, and it equals the true maximum.
__device__ __forceinline__ bool block_hit(const BlockGeom& b, const float4* e)
{
    const float4 f0 = e[0];
    const float4 f1 = e[1];
    const float thr = -__log2f(255.0f * f1.w) - CULL_MARGIN;   // alpha >= 1/255  <=>  q >= thr (+margin)
    const float ex = fminf(fmaxf(f0.x, b.xmin), b.xmax), ey = fminf(fmaxf(f0.y, b.ymin), b.ymax);
    const float dxe = ex - f0.x, dye = ey - f0.y;
    const float dy1 = fminf(fmaxf(fmaf(-f0.w, dxe, f0.y), b.ymin), b.ymax) - f0.y;
    const float dx2 = fminf(fmaxf(fmaf(-f0.z, dye, f0.x), b.xmin), b.xmax) - f0.x;
    const float u1 = f1.x * fmaf(f0.z, dy1, dxe), v1 = f1.z * dy1;     // (rho_lo is far below the culling margin)
    const float u2 = f1.x * fmaf(f0.z, dye, dx2), v2 = f1.z * dye;
    const float nq1 = fmaf(u1, u1, v1 * v1), nq2 = fmaf(u2, u2, v2 * v2);   // -q at the two candidates
    return -fminf(nq1, nq2) >= thr;
}

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(BLEND_THREADS)
render_forward_kernel(DevSettings s, GeomView geo, ImageView im, BinView bin, unsigned long long cap,
                      float* __restrict__ out_color)
{
    __shared__ float4 s_feat[3 * BATCH];

    pdl_prologue();
    // virtual tile blockIdx.x = view * Tv + tile (a batch of views is one launch; the drop-in call has one view)
    const int Tv = s.gx * s.gy;
    const int view = (int)blockIdx.x / Tv;
    const int tile = (int)blockIdx.x - view * Tv;
    const int tid = threadIdx.x, lane = tid & 31;
    const BlockGeom bg = block_geom(tile, s.gx, tid);
    const bool inA = bg.px < s.W && bg.py < s.H, inB = bg.px < s.W && bg.py + 4 < s.H;
    const float pxf = (float)bg.px, pyf = (float)bg.py;

    const uint2 rg = im.ranges[blockIdx.x];
    if ((unsigned long long)rg.y > cap) return;  // capacity overflow: host re-runs with a larger buffer
    const int n = (int)(rg.y - rg.x);

    // pixel A = (px, py) in the low halves, pixel B = (px, py + 4) in the high halves
    float TA = 1.f, A0 = 0.f, A1 = 0.f, A2 = 0.f;
    float TB = 1.f, B0 = 0.f, B1 = 0.f, B2 = 0.f;
    const f2 npy2 = mk2(-pyf, -(pyf + 4.f));
    unsigned int lastA = 0, lastB = 0;
    // A pixel that is finished (outside the image, or stopped by the T < 1e-4 rule) is represented by an
    // unreachable alpha floor, so "still live" costs no instruction in the pair loop: the reference's
    // alpha >= 1/255 test is made against this per-pixel register.
    constexpr float DONE = 2.f;   // alpha <= 0.99 < DONE
    float minA = inA ? ALPHA_MIN : DONE, minB = inB ? ALPHA_MIN : DONE;

    for (int base = 0; base < n; base += BATCH) {
        // block-wide vote doubles as the barrier that protects the staging buffer
        if (__syncthreads_count(minA > 1.f && minB > 1.f) == BLEND_THREADS) break;
#pragma unroll
        for (int r = 0; r < BATCH / BLEND_THREADS; r++) {
            const int slot = tid + r * BLEND_THREADS;
            if (base + slot < n) stage(s_feat, slot, geo, bin.point_list[rg.x + base + slot]);
        }
        __syncthreads();
        const int cnt = min(BATCH, n - base);
        for (int c = 0; c < cnt; c += 32) {
            // warp-ballot early termination: all 64 pixels of the block saturated
            if (__ballot_sync(FULL, !(minA > 1.f && minB > 1.f)) == 0u) break;
            bool hit = false;
            if (c + lane < cnt) hit = block_hit(bg, s_feat + 3 * (c + lane));
            unsigned int m = __ballot_sync(FULL, hit);
            const float4* chunk = s_feat + 3 * c;
            const unsigned int pos1 = (unsigned int)(base + c + 1);
            while (m) {
                const int k = __ffs(m) - 1;
                m &= m - 1;
                const float4* e = chunk + 3 * k;
                const float4 f0 = e[0];
                const float4 f1 = e[1];
                const float4 f2v = e[2];
                const f2 nq2 = neg_falloff_log2(f0.z, f1, f0.x - pxf, add2(bc2(f0.y), npy2));
                const f2 a2 = mul2(bc2(f1.w), mk2(ex2_approx(-lo(nq2)), ex2_approx(-hi(nq2))));
                const float aA = fminf(ALPHA_MAX, lo(a2)), aB = fminf(ALPHA_MAX, hi(a2));
                // the reference `continue`s on alpha < 1/255 (power > 0 cannot happen here; a finished pixel's
                // floor is unreachable)
                const bool okA = !(aA < minA);
                const bool okB = !(aB < minB);
                const unsigned int pos = pos1 + (unsigned int)k;
                const f2 ac = mk2(aA, aB), T2 = mk2(TA, TB);
                const f2 tT2 = mul2(T2, sub2(bc2(1.f), ac));
                const f2 w2 = mul2(ac, T2);
                const float tTA = lo(tT2), tTB = hi(tT2);
                // T' < 1e-4: the pixel stops and this Gaussian is NOT added
                if (okA && tTA < T_STOP) minA = DONE;
                if (okB && tTB < T_STOP) minB = DONE;
                const bool addA = okA && !(tTA < T_STOP), addB = okB && !(tTB < T_STOP);
                const f2 wz = mk2(addA ? lo(w2) : 0.f, addB ? hi(w2) : 0.f);   // adding 0 leaves the colour bit-identical
                { const f2 c = fma2(bc2(f2v.x), wz, mk2(A0, B0)); A0 = lo(c); B0 = hi(c); }
                { const f2 c = fma2(bc2(f2v.y), wz, mk2(A1, B1)); A1 = lo(c); B1 = hi(c); }
                { const f2 c = fma2(bc2(f2v.z), wz, mk2(A2, B2)); A2 = lo(c); B2 = hi(c); }
                if (addA) { TA = tTA; lastA = pos; }
                if (addB) { TB = tTB; lastB = pos; }
            }
        }
    }
    const size_t N = (size_t)s.W * s.H;
    const float bg0 = __ldg(s.bg + 0), bg1 = __ldg(s.bg + 1), bg2 = __ldg(s.bg + 2);
    // the view's own per-pixel state (unflipped), and its target: image out_image, optionally mirrored in x,
    // scaled by weight; views that share an image (toast halves) accumulate with atomics onto a zeroed image
    float* const fT = im.final_T + (size_t)view * N;
    unsigned int* const nc = im.n_contrib + (size_t)view * N;
    float* const out = out_color + (size_t)s.vt.out_image[view] * 3 * N;
    const float wgt = s.vt.weight[view];
    const int ox = s.vt.flip_x[view] ? s.W - 1 - bg.px : bg.px;
    if (inA) {
        const size_t pix = (size_t)bg.py * s.W + bg.px, opix = (size_t)bg.py * s.W + ox;
        const float c0 = wgt * (A0 + TA * bg0), c1 = wgt * (A1 + TA * bg1), c2 = wgt * (A2 + TA * bg2);
        if (s.accumulate) {
            atomicAdd(out + opix, c0); atomicAdd(out + N + opix, c1); atomicAdd(out + 2 * N + opix, c2);
        } else {
            out[opix] = c0; out[N + opix] = c1; out[2 * N + opix] = c2;
        }
        fT[pix] = TA;
        nc[pix] = lastA;
    }
    if (inB) {
        const size_t pix = (size_t)(bg.py + 4) * s.W + bg.px, opix = (size_t)(bg.py + 4) * s.W + ox;
        const float c0 = wgt * (B0 + TB * bg0), c1 = wgt * (B1 + TB * bg1), c2 = wgt * (B2 + TB * bg2);
        if (s.accumulate) {
            atomicAdd(out + opix, c0); atomicAdd(out + N + opix, c1); atomicAdd(out + 2 * N + opix, c2);
        } else {
            out[opix] = c0; out[N + opix] = c1; out[2 * N + opix] = c2;
        }
        fT[pix] = TB;
        nc[pix] = lastB;
    }
}

cudaError_t launch_render_forward(const DevSettings& s, GeomView g, ImageView im, BinView b, long long cap,
                                  float* out_color, cudaStream_t st)
{
    const int T = s.gx * s.gy * s.n_views;
    if (T <= 0) return cudaSuccess;
    count_launch();
    return launch_pdl(render_forward_kernel, dim3(T), dim3(BLEND_THREADS), st, s, g, im, b, (unsigned long long)cap,
                      out_color);
}

// ------------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------------
// One CTA of 64 threads per 16x16 tile.  A warp owns TWO 8x8 blocks side by side (lanes 0-15 the left one, lanes
// 16-31 the right one) and a lane four pixels of one column of its block (two packed pairs).  Each half warp has its
// OWN list of the staged Gaussians that reach its block (the exact test of the forward); the two halves walk their
// lists in lockstep, so one loop iteration replays two (block, Gaussian) hits.  What this buys over one block per
// warp (the layout of the forward, and of this kernel until round 2): the 9 sums every hit ends in are reduced over
// 16 lanes instead of 32 — one butterfly level less — and the reduction's instructions are issued once per
// ITERATION, i.e. half of them per hit; fetching the record and the atomics are shared by the pair as well.  ncu: 169 M
// warp instructions per launch instead of 209 M.  The hit lists are built per BATCH of staged Gaussians, not per chunk
// of 32 candidates, so the halves only wait for each other at the end of a batch (measured: 11 % more iterations than
// hits / 2 with per-chunk lists).
constexpr int BWD_THREADS = 64;                   // 2 warps x (2 blocks of 8x8) = one 16x16 tile
constexpr int BWD_STAGE = BATCH / BWD_THREADS;    // Gaussians staged per thread and batch

// Per-lane replay state: the four pixels of a lane are column px, rows py0 + {0, 2, 4, 6}, packed as (0, 2) and (4, 6).
//   T   running transmittance (T_i before the current Gaussian)
//   Sg  g . (colour composited behind the current Gaussian, incl. T_final * bg):
//         Sg_i = sum_{j>i} (c_j . g) alpha_j T_j + T_final (bg . g)
//   g*  dL/dC of the pixel
// With dC/dalpha_i = c_i T_i - (sum_{j>i} c_j alpha_j T_j + T_final bg) / (1 - alpha_i) contracted with
// g = dL/dC up front, the behind-colour recursion is ONE scalar per pixel (Sg) instead of three channels.
struct QuadBwd {
    f2 T01, T23, Sg01, Sg23;
    f2 g0_01, g0_23, g1_01, g1_23, g2_01, g2_23;
    unsigned int last0, last1, last2, last3;   // n_contrib
};

// Sum 8 values over the 16 lanes of a half warp with 8 shuffles (all of them stay inside the half: xor 8, 4, 2, 1):
// three exchange-and-halve steps leave every lane with one partial, one butterfly step finishes it.  Lane l of the
// half ends up with value index ((l >> 3) & 1) * 4 + ((l >> 2) & 1) * 2 + ((l >> 1) & 1).
__device__ __forceinline__ float half_reduce8(float v[8], int lane)
{
    bool hi = lane & 8;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const float send = hi ? v[i] : v[i + 4];
        const float keep = hi ? v[i + 4] : v[i];
        v[i] = keep + __shfl_xor_sync(FULL, send, 8);
    }
    hi = lane & 4;
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const float send = hi ? v[i] : v[i + 2];
        const float keep = hi ? v[i + 2] : v[i];
        v[i] = keep + __shfl_xor_sync(FULL, send, 4);
    }
    hi = lane & 2;
    {
        const float send = hi ? v[0] : v[1];
        const float keep = hi ? v[1] : v[0];
        v[0] = keep + __shfl_xor_sync(FULL, send, 2);
    }
    v[0] += __shfl_xor_sync(FULL, v[0], 1);
    return v[0];
}

__device__ __forceinline__ float half_sum(float v)
{
#pragma unroll
    for (int d = 8; d >= 1; d >>= 1) v += __shfl_xor_sync(FULL, v, d);
    return v;
}

// DET = false: the 9 sums of every (block, Gaussian) hit are added into the Gaussian's row of `acc` ([P][12]) with
// atomics, in whatever order the hits land.  DET = true (docs/SPEC.md U14): `acc` is the partials buffer of
// det_partials(), and each hit's 9 sums are STORED into the slot of its (instance, block), whose hit flag is set;
// det_reduce_kernel then adds every row's slots in a fixed order.  Slots of hits that are never replayed keep their
// zeroed flag and are not read.
template <bool DET>
__global__ void __launch_bounds__(BWD_THREADS, 12)
render_backward_kernel(DevSettings s, GeomView geo, ImageView im, BinView bin, unsigned long long cap,
                       const float* __restrict__ dL_dout, float* __restrict__ acc /* [P][12] */)
{
    __shared__ float4 s_feat[3 * BATCH];
    __shared__ unsigned char s_list[2][2][BATCH];   // [warp][half]: staged slots that reach the half's block
    __shared__ unsigned int s_max[2];

    pdl_prologue();
    const int Tv = s.gx * s.gy;
    const int view = (int)blockIdx.x / Tv;          // virtual tile = view * Tv + tile
    const int tile = (int)blockIdx.x - view * Tv;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, half = lane >> 4, l16 = lane & 15;
    const unsigned int lt_mask = (1u << lane) - 1u;
    const int tx = tile % s.gx, ty = tile / s.gx;
    const int by0 = ty * TILE + warp * 8;
    const int bx0 = tx * TILE + half * 8;           // this half's block
    const int px = bx0 + (l16 & 7), py0 = by0 + (l16 >> 3);
    // both blocks of the warp: every lane tests ITS candidate Gaussian against the left and the right one
    BlockGeom gA, gB;
    gA.px = gB.px = 0; gA.py = gB.py = 0;
    gA.xmin = (float)(tx * TILE); gA.xmax = gA.xmin + 7.f; gB.xmin = gA.xmin + 8.f; gB.xmax = gB.xmin + 7.f;
    gA.ymin = gB.ymin = (float)by0; gA.ymax = gB.ymax = (float)(by0 + 7);
    const size_t N = (size_t)s.W * s.H;
    // dL/d(view image) = weight * dL/d(output image), read mirrored in x for a flipped view
    const float wgt = s.vt.weight[view];
    const float* const dL = dL_dout + (size_t)s.vt.out_image[view] * 3 * N;
    const float* const fT = im.final_T + (size_t)view * N;
    const unsigned int* const nc = im.n_contrib + (size_t)view * N;
    const int ox = s.vt.flip_x[view] ? s.W - 1 - px : px;

    const uint2 rg = im.ranges[blockIdx.x];
    const int n = (int)(rg.y - rg.x);
    if (n <= 0) return;
    // Capacity overflow (only a CUDA-graph replay can get here with one: the eager caller re-runs the forward on a
    // larger buffer first): the forward skipped the overflowed tiles, so their final_T / n_contrib are stale and the
    // point list beyond `cap` does not exist.  The whole launch is void — the frame is invalid and its owner is told
    // so by capacity_ok() — hence every tile leaves before it reads a list entry.
    if ((unsigned long long)rg.y > cap || im.hdr->overflow != 0u) return;

    // The tile's start-up is a chain of dependent memory round trips: ranges -> n_contrib (-> deepest contributor) ->
    // point list -> per-Gaussian records -> shared memory.  Where the replay starts depends on n_contrib, but for most
    // tiles it starts at the end of the list (nothing saturated): the ids of the last BATCH entries are fetched
    // speculatively right away, in parallel with the pixel state, which takes one round trip out of the chain.
    unsigned int spec_id[BWD_STAGE];
#pragma unroll
    for (int r = 0; r < BWD_STAGE; r++) {
        const int kp = n - 1 - (tid + r * BWD_THREADS);
        spec_id[r] = kp >= 0 ? __ldg(bin.point_list + rg.x + kp) : 0u;
    }

    const float bg0 = __ldg(s.bg), bg1 = __ldg(s.bg + 1), bg2 = __ldg(s.bg + 2);
    QuadBwd S;
    {
        float T[4], Sg[4], g0[4], g1[4], g2[4];
        unsigned int last[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int py = py0 + 2 * i;
            T[i] = 0.f; Sg[i] = 0.f; g0[i] = g1[i] = g2[i] = 0.f; last[i] = 0u;
            if (px < s.W && py < s.H) {
                const size_t pix = (size_t)py * s.W + px, opix = (size_t)py * s.W + ox;
                T[i] = fT[pix]; last[i] = nc[pix];
                g0[i] = wgt * dL[opix]; g1[i] = wgt * dL[N + opix]; g2[i] = wgt * dL[2 * N + opix];
                Sg[i] = T[i] * (bg0 * g0[i] + bg1 * g1[i] + bg2 * g2[i]);
            }
        }
        S.T01 = mk2(T[0], T[1]); S.T23 = mk2(T[2], T[3]); S.Sg01 = mk2(Sg[0], Sg[1]); S.Sg23 = mk2(Sg[2], Sg[3]);
        S.g0_01 = mk2(g0[0], g0[1]); S.g0_23 = mk2(g0[2], g0[3]); S.g1_01 = mk2(g1[0], g1[1]); S.g1_23 = mk2(g1[2], g1[3]);
        S.g2_01 = mk2(g2[0], g2[1]); S.g2_23 = mk2(g2[2], g2[3]);
        S.last0 = last[0]; S.last1 = last[1]; S.last2 = last[2]; S.last3 = last[3];
    }
    const float pxf = (float)px, pyf = (float)py0;
    const f2 npy01 = mk2(-pyf, -(pyf + 2.f)), npy23 = mk2(-(pyf + 4.f), -(pyf + 6.f));

    // nothing behind the deepest contributor matters: of a block for its hit list, of the tile for where staging starts
    const unsigned int lmax = max(max(S.last0, S.last1), max(S.last2, S.last3));
    const unsigned int hmaxA = __reduce_max_sync(FULL, half == 0 ? lmax : 0u);
    const unsigned int hmaxB = __reduce_max_sync(FULL, half == 1 ? lmax : 0u);
    if (lane == 0) s_max[warp] = max(hmaxA, hmaxB);
    __syncthreads();
    const int m_len = min((int)max(s_max[0], s_max[1]), n);  // list entries [0, m_len) are replayed, back to front

    // the lanes of a half with bit 0 clear own its 8 reduced sums, lane 1 of the half the ninth: one atomic instruction
    const int red_lane = ((l16 & 1) == 0 || l16 == 1) ? 1 : 0;
    const int red_off = l16 == 1 ? 8 : (((l16 >> 3) & 1) * 4 + ((l16 >> 2) & 1) * 2 + ((l16 >> 1) & 1));

    for (int base = 0; base < m_len; base += BATCH) {
        __syncthreads();
#pragma unroll
        for (int r = 0; r < BWD_STAGE; r++) {
            const int slot = tid + r * BWD_THREADS;
            const int kpos = m_len - 1 - (base + slot);  // list position staged in this slot
            if (kpos >= 0) {
                const unsigned int id = (base == 0 && m_len == n) ? spec_id[r] : bin.point_list[rg.x + kpos];
                stage(s_feat, slot, geo, id);
            }
        }
        __syncthreads();
        const int cnt = min(BATCH, m_len - base);
        const int posb = m_len - 1 - base;               // list position of staged slot 0 (slot j holds posb - j)
        // hit lists of the two halves over the whole batch, in slot order (= back to front)
        int nA = 0, nB = 0;
        for (int c = 0; c < cnt; c += 32) {
            const int pos = posb - c - lane;
            bool hitA = false, hitB = false;
            if (c + lane < cnt) {
                const float4* e = s_feat + 3 * (c + lane);
                if ((unsigned int)pos < hmaxA) hitA = block_hit(gA, e);
                if ((unsigned int)pos < hmaxB) hitB = block_hit(gB, e);
            }
            const unsigned int mA = __ballot_sync(FULL, hitA), mB = __ballot_sync(FULL, hitB);
            if (hitA) s_list[warp][0][nA + __popc(mA & lt_mask)] = (unsigned char)(c + lane);
            if (hitB) s_list[warp][1][nB + __popc(mB & lt_mask)] = (unsigned char)(c + lane);
            nA += __popc(mA); nB += __popc(mB);
        }
        __syncwarp();
        const int nh = half ? nB : nA;
        const int iters = max(nA, nB);
        const unsigned char* const list = s_list[warp][half];
        for (int it = 0; it < iters; it++) {
            // A half whose list has run out replays slot 0 with every pixel masked off: like a pair that does not
            // contribute it leaves T, Sg and the sums unchanged, and its atomics are predicated off.
            const bool valid = it < nh;
            const int k = valid ? (int)list[it] : 0;
            const float4* e = s_feat + 3 * k;
            const float4 f0 = e[0];
            const float4 f1 = e[1];
            const float4 f2v = e[2];
            const float dx = f0.x - pxf;
            const f2 dy01 = add2(bc2(f0.y), npy01), dy23 = add2(bc2(f0.y), npy23);
            f2 u01, v01, u23, v23;                                    // (u, v) = L^T d: the whitened offset
            const f2 nq01 = neg_falloff_log2(f0.z, f1, dx, dy01, u01, v01);
            const f2 nq23 = neg_falloff_log2(f0.z, f1, dx, dy23, u23, v23);
            // opacity * Gs, before the 0.99 cap
            const f2 a01 = mul2(bc2(f1.w), mk2(ex2_approx(-lo(nq01)), ex2_approx(-hi(nq01))));
            const f2 a23 = mul2(bc2(f1.w), mk2(ex2_approx(-lo(nq23)), ex2_approx(-hi(nq23))));
            const unsigned int pos = (unsigned int)(posb - k);
            // min(0.99, a) < 1/255  <=>  a < 1/255: the floor is tested on the uncapped value
            const bool u0 = valid && (pos < S.last0) && !(lo(a01) < ALPHA_MIN);
            const bool u1 = valid && (pos < S.last1) && !(hi(a01) < ALPHA_MIN);
            const bool u2 = valid && (pos < S.last2) && !(lo(a23) < ALPHA_MIN);
            const bool u3 = valid && (pos < S.last3) && !(hi(a23) < ALPHA_MIN);
            // Branch-free: a pair that does not contribute is blended with alpha = 0, which leaves T, the
            // behind-colour sum and every gradient sum unchanged (bit-identically).
            // The masked UNCAPPED value am does double duty: capped it is the blended alpha, and times
            // dL/dalpha it is w = opacity * Gs * dL/dalpha (U4: straight through the cap), already zero for a
            // pair that does not contribute — no separate masking of dL/dalpha.
            const f2 am01 = mk2(u0 ? lo(a01) : 0.f, u1 ? hi(a01) : 0.f);
            const f2 am23 = mk2(u2 ? lo(a23) : 0.f, u3 ? hi(a23) : 0.f);
            const f2 ae01 = mk2(fminf(ALPHA_MAX, lo(am01)), fminf(ALPHA_MAX, hi(am01)));
            const f2 ae23 = mk2(fminf(ALPHA_MAX, lo(am23)), fminf(ALPHA_MAX, hi(am23)));
            const f2 om01 = sub2(bc2(1.f), ae01), om23 = sub2(bc2(1.f), ae23);
            const f2 ra01 = mk2(rcp_approx(lo(om01)), rcp_approx(hi(om01)));
            const f2 ra23 = mk2(rcp_approx(lo(om23)), rcp_approx(hi(om23)));
            S.T01 = mul2(S.T01, ra01); S.T23 = mul2(S.T23, ra23);     // T_i = T_{i+1} / (1 - alpha_i)
            const f2 cg01 = fma2(bc2(f2v.x), S.g0_01, fma2(bc2(f2v.y), S.g1_01, mul2(bc2(f2v.z), S.g2_01)));
            const f2 cg23 = fma2(bc2(f2v.x), S.g0_23, fma2(bc2(f2v.y), S.g1_23, mul2(bc2(f2v.z), S.g2_23)));
            const f2 dla01 = fma2(S.T01, cg01, neg2(mul2(ra01, S.Sg01)));   // dL/dalpha
            const f2 dla23 = fma2(S.T23, cg23, neg2(mul2(ra23, S.Sg23)));
            const f2 dch01 = mul2(ae01, S.T01), dch23 = mul2(ae23, S.T23);
            S.Sg01 = fma2(dch01, cg01, S.Sg01); S.Sg23 = fma2(dch23, cg23, S.Sg23);
            const f2 w01 = mul2(am01, dla01), w23 = mul2(am23, dla23);      // w = opacity * Gs * dL/dalpha
            // Per-pair sums are raw moments of w = Gs * dL/dGs in the WHITENED offset (u, v) = L^T d, which the
            // exponent above has already formed (q = -(u^2 + v^2)):
            //   v = (S w u, S w v, S w u^2, S w u v, S w v^2, S w, dL/dr, dL/dg), d_b = dL/db
            // The per-Gaussian kernel turns them into dL/dpix = -(1/K) L (S w [u v]) and
            // dL/dcov2D = (1/2K^2) L (S w [u v][u v]^T) L^T, a congruence with the factor L it already holds.
            // Moments in pixel axes (S w dx^2, ...) say the same in exact arithmetic, but the way from them to
            // the covariance gradient divides by det^2 and subtracts terms that cancel for an elongated
            // Gaussian: at 256:1 axes the fp32 rounding of the accumulated moments came back 1e3 times larger
            // (scale / rotation gradients off by 4e-4, found by the referee checker).  |u|, |v| <= ~3.4 where
            // alpha >= 1/255, whatever the shape, so these sums are well scaled by construction.
            // (S w = opacity * S Gs dL/dalpha: the per-Gaussian kernel divides by the opacity for dL/dopacity)
            const f2 wu01 = mul2(w01, u01), wu23 = mul2(w23, u23), wv01 = mul2(w01, v01), wv23 = mul2(w23, v23);
            // the lane's four pixels first: the two pairs (packed), then the two halves of the pair
            const f2 s_wu = add2(wu01, wu23), s_wv = add2(wv01, wv23);
            const f2 s_wuu = fma2(wu01, u01, mul2(wu23, u23)), s_wuv = fma2(wu01, v01, mul2(wu23, v23));
            const f2 s_wvv = fma2(wv01, v01, mul2(wv23, v23)), s_w = add2(w01, w23);
            const f2 s_r = fma2(dch01, S.g0_01, mul2(dch23, S.g0_23)), s_g = fma2(dch01, S.g1_01, mul2(dch23, S.g1_23));
            const f2 s_b = fma2(dch01, S.g2_01, mul2(dch23, S.g2_23));
            float v[8];
            v[0] = lo(s_wu) + hi(s_wu);
            v[1] = lo(s_wv) + hi(s_wv);
            v[2] = lo(s_wuu) + hi(s_wuu);
            v[3] = lo(s_wuv) + hi(s_wuv);
            v[4] = lo(s_wvv) + hi(s_wvv);
            v[5] = lo(s_w) + hi(s_w);
            v[6] = lo(s_r) + hi(s_r);
            v[7] = lo(s_g) + hi(s_g);
            float d_b = lo(s_b) + hi(s_b);
            const float sum8 = half_reduce8(v, lane);
            d_b = half_sum(d_b);
            if constexpr (DET) {
                if (valid) {
                    // instance rg.x + list position, block (warp, half) of the tile in row-major order
                    const size_t slot = ((size_t)rg.x + (unsigned int)(posb - k)) * 4 + warp * 2 + half;
                    const DetPartials dp = det_partials(acc, cap);
                    if (red_lane) dp.val[slot * 9 + red_off] = l16 == 1 ? d_b : sum8;
                    if (l16 == 0) dp.hit[slot] = 1;
                }
            } else {
                if (red_lane && valid) atomicAdd(acc + (size_t)__float_as_uint(f2v.w) * 12 + red_off, l16 == 1 ? d_b : sum8);
            }
        }
    }
}


cudaError_t launch_render_backward(const DevSettings& s, int rows, GeomView g, ImageView im, BinView b, long long cap,
                                   const float* dL_dout, float4* acc, bool acc_is_zero, cudaStream_t st)
{
    if (!acc_is_zero) {
        cudaError_t e = cudaMemsetAsync(acc, 0, (size_t)rows * 48, st);
        if (e != cudaSuccess) return e;
    }
    const int T = s.gx * s.gy * s.n_views;
    if (T <= 0 || rows <= 0) return cudaSuccess;
    count_launch();
    return launch_pdl(render_backward_kernel<false>, dim3(T), dim3(BWD_THREADS), st, s, g, im, b,
                      (unsigned long long)cap, dL_dout, reinterpret_cast<float*>(acc));
}

// ---- fixed-order reduction of the deterministic backward (docs/SPEC.md U14) ------------------------------------
// One thread per row.  Its rectangle's tiles are visited in row-major order; in each tile the row's instance is found
// by a binary search of the tile's sorted (depth key, id) pairs for the row's own pair (the sort's order, ties broken
// by the id; a Gaussian occurs at most once per tile), and the flagged slots of its four blocks are added in block
// order.  The sum is kept in double and rounded once into the fp32 accumulator row, which is fully written (zeros for
// a culled row, and for every row of a void launch, as the atomic path leaves them).
constexpr int REDUCE_THREADS = 128;

__global__ void __launch_bounds__(REDUCE_THREADS)
det_reduce_kernel(DevSettings s, int P, int rows, GeomView geo, ImageView im, BinView bin, unsigned long long cap,
                  const float* __restrict__ partials, float4* __restrict__ acc)
{
    pdl_prologue();
    const int r = blockIdx.x * REDUCE_THREADS + threadIdx.x;
    if (r >= rows) return;
    double sum[9];
#pragma unroll
    for (int i = 0; i < 9; i++) sum[i] = 0.0;
    const ushort4 rc = geo.rect[r];
    if (im.hdr->overflow == 0u && rc.z > rc.x && rc.w > rc.y) {
        int v = 0;
        if (s.ragged) {
            while (v + 1 < s.n_views && r >= s.rows.off[v + 1]) v++;
        } else {
            v = r / P;
        }
        const DetPartials dp = det_partials(partials, cap);
        const unsigned int key = ordered_u32(geo.feat2[r].w);
        const unsigned int* const hit4 = reinterpret_cast<const unsigned int*>(dp.hit);
        const unsigned int* const ids = bin.point_list;
        const unsigned int* const keys = bin.depth_keys;
        const int tbase = v * s.gx * s.gy;
        for (int ty = rc.y; ty < rc.w; ty++) {
            for (int tx = rc.x; tx < rc.z; tx++) {
                const uint2 rg = im.ranges[tbase + ty * s.gx + tx];
                if ((unsigned long long)rg.y > cap) continue;
                // first position whose (key, id) is not below the row's
                unsigned int lo = rg.x, hi = rg.y;
                while (lo < hi) {
                    const unsigned int mid = lo + ((hi - lo) >> 1);
                    const unsigned int km = __ldg(keys + mid), im_ = __ldg(ids + mid);
                    if (km < key || (km == key && im_ < (unsigned int)r)) lo = mid + 1;
                    else hi = mid;
                }
                if (lo >= rg.y || __ldg(ids + lo) != (unsigned int)r) continue;
                const unsigned int f = hit4[lo];
                const float* const pv = dp.val + (size_t)lo * 36;
#pragma unroll
                for (int b = 0; b < 4; b++) {
                    if ((f >> (8 * b)) & 0xffu) {
#pragma unroll
                        for (int i = 0; i < 9; i++) sum[i] += (double)pv[9 * b + i];
                    }
                }
            }
        }
    }
    acc[3 * (size_t)r] = make_float4((float)sum[0], (float)sum[1], (float)sum[2], (float)sum[3]);
    acc[3 * (size_t)r + 1] = make_float4((float)sum[4], (float)sum[5], (float)sum[6], (float)sum[7]);
    acc[3 * (size_t)r + 2] = make_float4((float)sum[8], 0.f, 0.f, 0.f);
}

cudaError_t launch_render_backward_det(const DevSettings& s, int P, int rows, GeomView g, ImageView im, BinView b,
                                       long long cap, const float* dL_dout, float4* acc, void* partials,
                                       cudaStream_t st)
{
    const DetPartials dp = det_partials(static_cast<float*>(partials), (unsigned long long)cap);
    cudaError_t e = cudaMemsetAsync(dp.hit, 0, (size_t)cap * 4, st);
    if (e != cudaSuccess) return e;
    const int T = s.gx * s.gy * s.n_views;
    if (rows <= 0) return cudaSuccess;
    if (T > 0) {
        count_launch();
        e = launch_pdl(render_backward_kernel<true>, dim3(T), dim3(BWD_THREADS), st, s, g, im, b,
                       (unsigned long long)cap, dL_dout, static_cast<float*>(partials));
        if (e != cudaSuccess) return e;
    }
    count_launch();
    return launch_pdl(det_reduce_kernel, dim3((rows + REDUCE_THREADS - 1) / REDUCE_THREADS), dim3(REDUCE_THREADS), st,
                      s, P, rows, g, im, b, (unsigned long long)cap, static_cast<const float*>(partials), acc);
}

}  // namespace gsvc
