// Fused epilogue of the neural-Gaussian generator (SURVEY.md §8f row f2, second half).
//
// What /root/reference/ortho_gaussian_renderer/guassian.py does between the four per-anchor MLPs and the rasterizer
// call (lines 147-153 and 251-287): gather anchor / offsets / scaling / mask rows of the visible anchors with a
// boolean mask, mask the opacities, select the Gaussians with opacity > 0 through a [N_vis*K, 22] concatenation
// (repeat + three cats + a boolean-mask index + split), then scaling = s[3:6] * sigmoid(.), rot = normalize(.),
// xyz = clamp(anchor + (offset + neural_offset) * s[0:3]).  About twenty full passes over [N_vis*K, ...] tensors and
// two host synchronisations (boolean-mask indexing = nonzero).
// Here: ONE marking pass (opacity * mask, selection bits, per-CTA counts), the compaction scan of the filter
// (preprocess.cu, count published through the pinned slot), and ONE writing pass that gathers by the visible-anchor
// index, computes the activations and writes the rasterizer's five input arrays compacted, in the reference's order.
// The backward is one pass per visible anchor (deterministic: no atomics).
#include "common.cuh"

namespace gsvc {

struct EpiIn {
    int n_vis, K;
    const int32_t* vis;          // [n_vis] ascending anchor indices (visible_filter_compact) or NULL: inputs are gathered
    const float* anchor;         // [N,3]
    const float* grid_offsets;   // [N,K,3]
    const float* grid_scaling;   // [N,6]
    const float* masks;          // [N,K]
    const float* neural_opacity; // [n_vis,K]      MLP outputs, per visible anchor
    const float* color;          // [n_vis,K*3]
    const float* scale_rot;      // [n_vis,K*7]
    const float* neural_offset;  // [n_vis,K*3]
    const float* bound_min;      // [3]
    const float* bound_max;      // [3]
};

__global__ void __launch_bounds__(256) epi_mark_kernel(EpiIn in, float* __restrict__ nop_full,
                                                       uint8_t* __restrict__ selection, unsigned int* __restrict__ ballots,
                                                       unsigned int* __restrict__ cta_count)
{
    __shared__ unsigned int s_cnt[8];
    pdl_prologue();
    const long long total = (long long)in.n_vis * in.K;
    const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
    bool sel = false;
    if (e < total) {
        const int n = (int)(e / in.K), k = (int)(e - (long long)n * in.K);
        const long long row = in.vis ? (long long)__ldg(in.vis + n) : n;
        const float op = __ldg(in.neural_opacity + e) * __ldg(in.masks + row * in.K + k);
        nop_full[e] = op;
        sel = op > 0.0f;
        selection[e] = sel ? 1 : 0;
    }
    const unsigned int bal = __ballot_sync(0xffffffffu, sel);
    if ((threadIdx.x & 31) == 0) {
        ballots[e >> 5] = bal;
        s_cnt[threadIdx.x >> 5] = __popc(bal);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int t = 0;
#pragma unroll
        for (int w = 0; w < 8; w++) t += s_cnt[w];
        cta_count[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(256) epi_write_kernel(EpiIn in, const unsigned int* __restrict__ ballots,
                                                        const unsigned int* __restrict__ cta_offset,
                                                        int32_t* __restrict__ rank, float* __restrict__ xyz,
                                                        float* __restrict__ color_out, float* __restrict__ opacity_out,
                                                        float* __restrict__ scaling_out, float* __restrict__ rot_out,
                                                        const float* __restrict__ nop_full)
{
    __shared__ unsigned int s_cnt[8];
    pdl_prologue();
    const long long total = (long long)in.n_vis * in.K;
    const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const unsigned int bal = ballots[e >> 5];     // (the mark kernel wrote a word for every warp of the grid)
    if (lane == 0) s_cnt[wid] = __popc(bal);
    __syncthreads();
    if (e >= total) return;
    if (!((bal >> lane) & 1u)) { rank[e] = -1; return; }
    unsigned int j = cta_offset[blockIdx.x] + __popc(bal & ((1u << lane) - 1u));
#pragma unroll
    for (int w = 0; w < 8; w++)
        if (w < wid) j += s_cnt[w];
    rank[e] = (int32_t)j;
    const int n = (int)(e / in.K), k = (int)(e - (long long)n * in.K);
    const long long row = in.vis ? (long long)__ldg(in.vis + n) : n;
    const float* gs = in.grid_scaling + row * 6;
    const float* an = in.anchor + row * 3;
    const float* go = in.grid_offsets + (row * in.K + k) * 3;
    const float* no = in.neural_offset + e * 3;
    const float* sr = in.scale_rot + e * 7;
    opacity_out[j] = nop_full[e];
#pragma unroll
    for (int c = 0; c < 3; c++) {
        color_out[3 * (size_t)j + c] = __ldg(in.color + e * 3 + c);
        const float sg = 1.0f / (1.0f + expf(-__ldg(sr + c)));                 // torch.sigmoid
        scaling_out[3 * (size_t)j + c] = __ldg(gs + 3 + c) * sg;
        const float off = (__ldg(go + c) + __ldg(no + c)) * __ldg(gs + c);
        const float v = __ldg(an + c) + off;
        xyz[3 * (size_t)j + c] = fminf(fmaxf(v, __ldg(in.bound_min + c)), __ldg(in.bound_max + c));   // torch.clamp
    }
    const float q0 = __ldg(sr + 3), q1 = __ldg(sr + 4), q2 = __ldg(sr + 5), q3 = __ldg(sr + 6);
    const float nrm = fmaxf(sqrtf(q0 * q0 + q1 * q1 + q2 * q2 + q3 * q3), 1e-12f);       // F.normalize, eps 1e-12
    rot_out[4 * (size_t)j] = q0 / nrm; rot_out[4 * (size_t)j + 1] = q1 / nrm;
    rot_out[4 * (size_t)j + 2] = q2 / nrm; rot_out[4 * (size_t)j + 3] = q3 / nrm;
}

struct EpiGrads {
    const float* dxyz; const float* dcolor; const float* dopacity; const float* dscaling; const float* drot;   // [M,...]
    const float* dnop_full;      // [n_vis*K] or NULL: gradient arriving through the un-selected opacity output
    float* d_neural_opacity; float* d_color; float* d_scale_rot; float* d_neural_offset;    // per visible anchor, dense
    float* d_anchor; float* d_grid_offsets; float* d_grid_scaling; float* d_masks;
};

// One thread per visible anchor, its K offsets in a loop: the per-anchor sums (anchor, grid scaling) need no atomics.
__global__ void __launch_bounds__(128) epi_backward_kernel(EpiIn in, const int32_t* __restrict__ rank, EpiGrads g)
{
    pdl_prologue();
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= in.n_vis) return;
    const int K = in.K;
    const long long row = in.vis ? (long long)__ldg(in.vis + n) : n;
    float gs[6];
#pragma unroll
    for (int c = 0; c < 6; c++) gs[c] = __ldg(in.grid_scaling + row * 6 + c);
    float an[3], lo[3], hi[3];
#pragma unroll
    for (int c = 0; c < 3; c++) { an[c] = __ldg(in.anchor + row * 3 + c); lo[c] = __ldg(in.bound_min + c); hi[c] = __ldg(in.bound_max + c); }
    float d_an[3] = {0.f, 0.f, 0.f}, d_gs[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int k = 0; k < K; k++) {
        const long long e = (long long)n * K + k;
        const int32_t j = rank[e];
        const float m = __ldg(in.masks + row * K + k), nop = __ldg(in.neural_opacity + e);
        float d_op = g.dnop_full ? __ldg(g.dnop_full + e) : 0.f;        // d/d(neural_opacity * mask)
        float d_col[3] = {0.f, 0.f, 0.f}, d_sr[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, d_no[3] = {0.f, 0.f, 0.f};
        if (j >= 0) {
            d_op += __ldg(g.dopacity + j);
            const float* sr = in.scale_rot + e * 7;
#pragma unroll
            for (int c = 0; c < 3; c++) {
                d_col[c] = __ldg(g.dcolor + 3 * (size_t)j + c);
                const float sg = 1.0f / (1.0f + expf(-__ldg(sr + c)));
                const float ds = __ldg(g.dscaling + 3 * (size_t)j + c);
                d_sr[c] = ds * gs[3 + c] * sg * (1.0f - sg);
                d_gs[3 + c] += ds * sg;
                const float osum = __ldg(in.grid_offsets + (row * K + k) * 3 + c) + __ldg(in.neural_offset + e * 3 + c);
                const float v = an[c] + osum * gs[c];
                const float gx = (v >= lo[c] && v <= hi[c]) ? __ldg(g.dxyz + 3 * (size_t)j + c) : 0.f;   // clamp passes inside
                d_an[c] += gx;
                d_no[c] = gx * gs[c];
                d_gs[c] += gx * osum;
            }
            const float q[4] = {__ldg(sr + 3), __ldg(sr + 4), __ldg(sr + 5), __ldg(sr + 6)};
            const float nrm = fmaxf(sqrtf(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]), 1e-12f);
            float dr[4], dot = 0.f;
#pragma unroll
            for (int c = 0; c < 4; c++) { dr[c] = __ldg(g.drot + 4 * (size_t)j + c); dot += dr[c] * (q[c] / nrm); }
#pragma unroll
            for (int c = 0; c < 4; c++) d_sr[3 + c] = (dr[c] - (q[c] / nrm) * dot) / nrm;
        }
        g.d_neural_opacity[e] = d_op * m;
        g.d_masks[e] = d_op * nop;
#pragma unroll
        for (int c = 0; c < 3; c++) {
            g.d_color[e * 3 + c] = d_col[c];
            g.d_neural_offset[e * 3 + c] = d_no[c];
            g.d_grid_offsets[e * 3 + c] = d_no[c];       // offsets = grid_offsets + neural_offset
        }
#pragma unroll
        for (int c = 0; c < 7; c++) g.d_scale_rot[e * 7 + c] = d_sr[c];
    }
#pragma unroll
    for (int c = 0; c < 3; c++) g.d_anchor[(size_t)n * 3 + c] = d_an[c];
#pragma unroll
    for (int c = 0; c < 6; c++) g.d_grid_scaling[(size_t)n * 6 + c] = d_gs[c];
}

int fail(int code, const char* fmt, ...);   // api.cu: the last_error channel

cudaError_t launch_compact_scan(int n_ctas, const unsigned int* cta_count, unsigned int* cta_offset,
                                unsigned long long* count_dev, unsigned long long* host_slot, unsigned int ticket,
                                cudaStream_t st);

}  // namespace gsvc

using namespace gsvc;

extern "C" {

size_t gsvc_gen_epilogue_scratch_bytes(int32_t n_vis, int32_t K)
{
    const size_t total = (size_t)(n_vis < 1 ? 1 : n_vis) * (size_t)(K < 1 ? 1 : K);
    const size_t n_ctas = (total + 255) / 256;
    return 256 + 2 * align_up(n_ctas * 4, 256) + align_up(n_ctas * 32, 256) + 256;
}

int gsvc_gen_epilogue_forward(int32_t n_vis, int32_t K, const int32_t* visible_indices, const float* anchor,
                              const float* grid_offsets, const float* grid_scaling, const float* masks,
                              const float* neural_opacity, const float* color, const float* scale_rot,
                              const float* neural_offset, const float* bound_min, const float* bound_max, float* xyz,
                              float* color_out, float* opacity_out, float* scaling_out, float* rot_out,
                              float* neural_opacity_full, uint8_t* selection_mask, int32_t* rank, void* scratch,
                              uint64_t* count_slot_host, uint32_t ticket, void* stream_)
{
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (n_vis < 0 || K < 1)
        return fail(GSVC_RAST_ERR_INVALID, "epilogue_forward: n_vis must be >= 0 and K >= 1, got %d, %d", n_vis, K);
    if (n_vis == 0) {
        if (count_slot_host) *count_slot_host = (uint64_t)(ticket & 0xFFFFFFu) << 40;
        return GSVC_RAST_OK;
    }
    if (!anchor || !grid_offsets || !grid_scaling || !masks || !neural_opacity || !color || !scale_rot || !neural_offset ||
        !bound_min || !bound_max || !xyz || !color_out || !opacity_out || !scaling_out || !rot_out || !neural_opacity_full ||
        !selection_mask || !rank || !scratch)
        return fail(GSVC_RAST_ERR_INVALID, "epilogue_forward: an input, output or scratch pointer is NULL");
    const long long total = (long long)n_vis * K;
    if (total > 0x7fffffffll)
        return fail(GSVC_RAST_ERR_INVALID, "epilogue_forward: n_vis * K = %lld exceeds 2^31 - 1", total);
    const int n_ctas = (int)((total + 255) / 256);
    char* p = static_cast<char*>(scratch);
    unsigned long long* count_dev = carve<unsigned long long>(p, 1);
    unsigned int* cta_count = carve<unsigned int>(p, n_ctas);
    unsigned int* cta_offset = carve<unsigned int>(p, n_ctas);
    unsigned int* ballots = carve<unsigned int>(p, (size_t)n_ctas * 8);
    EpiIn in{n_vis, K, visible_indices, anchor, grid_offsets, grid_scaling, masks, neural_opacity, color, scale_rot,
             neural_offset, bound_min, bound_max};
    count_launch(3);
    cudaError_t e = launch_pdl(epi_mark_kernel, dim3(n_ctas), dim3(256), st, in, neural_opacity_full, selection_mask,
                               ballots, cta_count);
    if (e == cudaSuccess)
        e = launch_compact_scan(n_ctas, cta_count, cta_offset, count_dev,
                                reinterpret_cast<unsigned long long*>(count_slot_host), ticket & 0xFFFFFFu, st);
    if (e == cudaSuccess)
        e = launch_pdl(epi_write_kernel, dim3(n_ctas), dim3(256), st, in, (const unsigned int*)ballots,
                       (const unsigned int*)cta_offset, rank, xyz, color_out, opacity_out, scaling_out, rot_out,
                       (const float*)neural_opacity_full);
    return e == cudaSuccess ? GSVC_RAST_OK : fail(GSVC_RAST_ERR_CUDA, "epilogue_forward: %s", cudaGetErrorString(e));
}

int gsvc_gen_epilogue_backward(int32_t n_vis, int32_t K, const int32_t* visible_indices, const float* anchor,
                               const float* grid_offsets, const float* grid_scaling, const float* masks,
                               const float* neural_opacity, const float* scale_rot, const float* neural_offset,
                               const float* bound_min, const float* bound_max, const int32_t* rank, const float* dL_dxyz,
                               const float* dL_dcolor, const float* dL_dopacity, const float* dL_dscaling,
                               const float* dL_drot, const float* dL_dnop_full, float* d_neural_opacity, float* d_color,
                               float* d_scale_rot, float* d_neural_offset, float* d_anchor, float* d_grid_offsets,
                               float* d_grid_scaling, float* d_masks, void* stream_)
{
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    if (n_vis < 0 || K < 1)
        return fail(GSVC_RAST_ERR_INVALID, "epilogue_backward: n_vis must be >= 0 and K >= 1, got %d, %d", n_vis, K);
    if (n_vis == 0) return GSVC_RAST_OK;
    if (!anchor || !grid_offsets || !grid_scaling || !masks || !neural_opacity || !scale_rot || !neural_offset || !rank ||
        !bound_min || !bound_max || !dL_dxyz || !dL_dcolor || !dL_dopacity || !dL_dscaling || !dL_drot ||
        !d_neural_opacity || !d_color || !d_scale_rot || !d_neural_offset || !d_anchor || !d_grid_offsets ||
        !d_grid_scaling || !d_masks)
        return fail(GSVC_RAST_ERR_INVALID, "epilogue_backward: an input, gradient or output pointer is NULL");
    EpiIn in{n_vis, K, visible_indices, anchor, grid_offsets, grid_scaling, masks, neural_opacity, nullptr, scale_rot,
             neural_offset, bound_min, bound_max};
    EpiGrads g{dL_dxyz, dL_dcolor, dL_dopacity, dL_dscaling, dL_drot, dL_dnop_full, d_neural_opacity, d_color,
               d_scale_rot, d_neural_offset, d_anchor, d_grid_offsets, d_grid_scaling, d_masks};
    count_launch();
    cudaError_t e = launch_pdl(epi_backward_kernel, dim3((n_vis + 127) / 128), dim3(128), st, in, rank, g);
    return e == cudaSuccess ? GSVC_RAST_OK : fail(GSVC_RAST_ERR_CUDA, "epilogue_backward: %s", cudaGetErrorString(e));
}

}  // extern "C"
