// 8-bit frame export (SPEC "8-bit frame export", decision U11): composed fp32 frames [n,3,H,W] in, RGB-interleaved
// bytes [n,H,W,3] out, in one pass.  Per value q = uint8(min(max(fl(fl(x * 255) + 0.5), 0), 255)), truncated: the
// product and the sum are rounded separately (__fmul_rn / __fadd_rn cannot be contracted into an FMA, which changes
// the byte of some inputs next to (k - 0.5) / 255), fmaxf(NaN, 0) = 0 gives NaN -> 0, and +-inf saturate.
//
// One thread converts 4 consecutive pixels of one image.  Vector path (H*W % 4 == 0, image 16-byte and out 4-byte
// aligned): one float4 load from each of the R, G and B planes and three 32-bit stores of the 12 interleaved bytes;
// a plane then holds a whole number of quads, so nothing is read or written past its end.  Otherwise the scalar path
// converts the same 4 pixels with bounds checks and byte stores.  No shared memory, no atomics.
#include "common.cuh"

namespace gsvc {

namespace rgb8 {

constexpr int THREADS = 256;
constexpr unsigned MAX_GRID_X = 1u << 20;            // larger quad counts loop (grid-stride)
constexpr unsigned MAX_GRID_Y = 65535;               // more images loop

__device__ __forceinline__ uint32_t q8(float x)
{
    const float v = __fadd_rn(__fmul_rn(x, 255.0f), 0.5f);
    return __float2uint_rz(fminf(fmaxf(v, 0.0f), 255.0f));
}

template <bool VEC>
__global__ void __launch_bounds__(THREADS) frames_rgb8_kernel(int n, long long hw, const float* __restrict__ image,
                                                               uint8_t* __restrict__ out)
{
    pdl_prologue();
    const long long quads = (hw + 3) / 4;
    for (long long img = blockIdx.y; img < n; img += gridDim.y) {
        const float* r = image + img * 3 * hw;
        const float* g = r + hw;
        const float* b = g + hw;
        uint8_t* o = out + img * 3 * hw;
        for (long long q = (long long)blockIdx.x * THREADS + threadIdx.x; q < quads;
             q += (long long)gridDim.x * THREADS) {
            const long long p = 4 * q;
            if (VEC) {
                const float4 R = __ldg(reinterpret_cast<const float4*>(r + p));
                const float4 G = __ldg(reinterpret_cast<const float4*>(g + p));
                const float4 B = __ldg(reinterpret_cast<const float4*>(b + p));
                uint32_t* w = reinterpret_cast<uint32_t*>(o + 3 * p);
                w[0] = q8(R.x) | q8(G.x) << 8 | q8(B.x) << 16 | q8(R.y) << 24;
                w[1] = q8(G.y) | q8(B.y) << 8 | q8(R.z) << 16 | q8(G.z) << 24;
                w[2] = q8(B.z) | q8(R.w) << 8 | q8(G.w) << 16 | q8(B.w) << 24;
            } else {
                for (long long i = p; i < p + 4 && i < hw; i++) {
                    o[3 * i + 0] = (uint8_t)q8(__ldg(r + i));
                    o[3 * i + 1] = (uint8_t)q8(__ldg(g + i));
                    o[3 * i + 2] = (uint8_t)q8(__ldg(b + i));
                }
            }
        }
    }
}

}  // namespace rgb8

int fail(int code, const char* fmt, ...);

}  // namespace gsvc

using namespace gsvc;

extern "C" {

int gsvc_rast_frames_rgb8(int32_t n_images, int32_t H, int32_t W, const float* image, uint8_t* out, void* stream_)
{
    if (!image) return fail(GSVC_RAST_ERR_INVALID, "frames_rgb8: image is NULL");
    if (!out) return fail(GSVC_RAST_ERR_INVALID, "frames_rgb8: out is NULL");
    if (n_images < 1 || H < 1 || W < 1)
        return fail(GSVC_RAST_ERR_INVALID, "frames_rgb8: n_images, H and W must be >= 1, got %d, %d, %d", n_images, H, W);
    if ((double)n_images * (double)H * (double)W * 3.0 >= 9.0e18)
        return fail(GSVC_RAST_ERR_INVALID, "frames_rgb8: size too large: n_images * H * W * 3 overflows a 64-bit index");
    using namespace rgb8;
    cudaStream_t st = static_cast<cudaStream_t>(stream_);
    const long long hw = (long long)H * W;
    const long long blocks = ((hw + 3) / 4 + THREADS - 1) / THREADS;
    const dim3 grid((unsigned)(blocks < MAX_GRID_X ? blocks : MAX_GRID_X),
                    (unsigned)n_images < MAX_GRID_Y ? (unsigned)n_images : MAX_GRID_Y);
    const bool vec = hw % 4 == 0 && reinterpret_cast<uintptr_t>(image) % 16 == 0 &&
                     reinterpret_cast<uintptr_t>(out) % 4 == 0;
    count_launch();
    cudaError_t e = vec ? launch_pdl(frames_rgb8_kernel<true>, grid, dim3(THREADS), st, n_images, hw, image, out)
                        : launch_pdl(frames_rgb8_kernel<false>, grid, dim3(THREADS), st, n_images, hw, image, out);
    if (e == cudaSuccess) e = cudaGetLastError();
    return e == cudaSuccess ? GSVC_RAST_OK : fail(GSVC_RAST_ERR_CUDA, "frames_rgb8: %s", cudaGetErrorString(e));
}

}  // extern "C"
