// Raw sensor frame -> the engine's C8 lenslet views in ONE pass: the crop + normalisation of extract_views_kernel
// (elementwise.cu) fused with the fp32 -> C8 conversion (nchw_to_c8, conv_tc.cu), so the fp32 views never exist in HBM.
// Output [B][Cp/8][SH][SW][8] half, bitwise equal to to_c8(extract_views(image.float())): the same window rule, the same
// IEEE (r - mean) / std, the same round-to-nearest pack2, and the lenslet slots L..Cp-1 are 0 (not the normalised zero), as
// the converter pads them.
#include <limits.h>
#include "common.cuh"
#include "tc_common.cuh"

namespace cwfa {

// blockIdx.y = (sample, 8-lenslet chunk): the 8 windows' geometry is computed once per block into shared memory; blockIdx.x
// strides over view rows, threads over view columns.  One thread writes one 16-byte chunk (one view pixel x 8 lenslets):
// each of its 8 sensor reads is coalesced across the warp (neighbouring threads, neighbouring columns) and the stores are
// contiguous.  No per-element division or modulo except the normalisation itself.
template <typename TIn, bool BF16>
__global__ void __launch_bounds__(256) extract_views_c8_kernel(const TIn* __restrict__ img, const int32_t* __restrict__ coords,
                                                               uint4* __restrict__ out, int Hi, int Wi, int L, int chunks,
                                                               int SH, int SW, float mean, float stdv, int normalise) {
    // volatile: re-read (a broadcast) on every pixel instead of being hoisted into ~40 loop-invariant registers, which would
    // halve the resident warps of this latency-bound gather (35-38 registers instead of 78-80, no spills)
    __shared__ volatile int64_t s_base[8];   // image offset of view pixel (0, 0): pixel (i, j) of the window is s_base + i * Wi + j
    __shared__ volatile int s_i0[8], s_j0[8];  // first view row / column inside the window (INT_MAX: the view has no window)
    __shared__ volatile float s_fill[8];     // value outside the window: the normalised zero, or 0 in a padding slot
    const int b = blockIdx.y / chunks, ch = blockIdx.y - b * chunks;
    if (threadIdx.x < 8) {
        const int c = ch * 8 + threadIdx.x;
        int i0 = INT_MAX, j0 = INT_MAX;
        int64_t base = 0;
        float fill = 0.f;
        if (c < L) {
            const int cy = __ldg(coords + 2 * c), cx = __ldg(coords + 2 * c + 1);
            const int ly = max(cy - SH / 2, 0), lx = max(cx - SW / 2, 0);
            const int uy = min(cy + SH / 2, Hi), ux = min(cx + SW / 2, Wi);
            const int ph = max(uy - ly, 0), pw = max(ux - lx, 0);
            if (ph > 0 && pw > 0) {                       // bottom/right aligned patch (reference quirk)
                i0 = SH - ph;
                j0 = SW - pw;
                base = (int64_t)(ly - i0) * Wi + (lx - j0);
            }
            fill = normalise ? (0.f - mean) / stdv : 0.f;
        }
        s_base[threadIdx.x] = base;
        s_i0[threadIdx.x] = i0;
        s_j0[threadIdx.x] = j0;
        s_fill[threadIdx.x] = fill;
    }
    __syncthreads();
    const TIn* ib = img + (int64_t)b * Hi * Wi;
    uint4* ob = out + (int64_t)blockIdx.y * SH * SW;
    for (int i = blockIdx.x; i < SH; i += gridDim.x) {
        const int64_t row = (int64_t)i * Wi;
        for (int j = threadIdx.x; j < SW; j += blockDim.x) {
            // all eight (predicated) reads first, then the arithmetic: eight independent requests in flight per thread
            float r[8];
            bool in[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                in[k] = i >= s_i0[k] && j >= s_j0[k];
                r[k] = in[k] ? (float)ib[s_base[k] + row + j] : 0.f;
            }
            float v[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) v[k] = in[k] ? (normalise ? (r[k] - mean) / stdv : r[k]) : s_fill[k];
            uint4 o;
            o.x = tcx::pack2<BF16>(v[0], v[1]); o.y = tcx::pack2<BF16>(v[2], v[3]);
            o.z = tcx::pack2<BF16>(v[4], v[5]); o.w = tcx::pack2<BF16>(v[6], v[7]);
            ob[(int64_t)i * SW + j] = o;
        }
    }
}

template <typename TIn>
static void launch_extract_views_c8(const void* image, const int32_t* coords, void* out, int B, int Hi, int Wi, int L,
                                    int chunks, int SH, int SW, float mean, float stdv, int normalise, int out_is_bf16,
                                    cudaStream_t st) {
    int gx = ceil_div(kNumSMs * 8, (int64_t)B * chunks);
    if (gx > SH) gx = SH;
    if (gx < 1) gx = 1;
    const int threads = SW >= 256 ? 256 : (SW >= 128 ? 128 : 64);
    const dim3 grid(gx, B * chunks);
    if (out_is_bf16)
        extract_views_c8_kernel<TIn, true><<<grid, threads, 0, st>>>((const TIn*)image, coords, (uint4*)out, Hi, Wi, L, chunks, SH,
                                                                     SW, mean, stdv, normalise);
    else
        extract_views_c8_kernel<TIn, false><<<grid, threads, 0, st>>>((const TIn*)image, coords, (uint4*)out, Hi, Wi, L, chunks, SH,
                                                                      SW, mean, stdv, normalise);
}

}  // namespace cwfa

using namespace cwfa;

extern "C" int cwfa_extract_views_c8(const void* image, int image_dtype, const int32_t* coords, void* out, int B, int Hi, int Wi,
                                     int L, int Cp, int SH, int SW, float mean, float stdv, int normalise, int out_is_bf16,
                                     void* stream) {
    if (B <= 0 || Hi <= 0 || Wi <= 0 || L <= 0 || SH <= 0 || SW <= 0 || Cp < L || (Cp % 8) || (normalise && stdv == 0.f) ||
        (int64_t)B * (Cp / 8) > 65535 || image_dtype < 0 || image_dtype > 2 || !image || !coords || !out) {
        set_error("extract_views_c8: bad arguments");
        return CWFA_EINVAL;
    }
    if (!aligned16(out)) { set_error("extract_views_c8: out must be 16-byte aligned"); return CWFA_EINVAL; }
    const cudaStream_t st = (cudaStream_t)stream;
    const int chunks = Cp / 8;
    if (image_dtype == 2)
        launch_extract_views_c8<uint16_t>(image, coords, out, B, Hi, Wi, L, chunks, SH, SW, mean, stdv, normalise, out_is_bf16, st);
    else if (image_dtype == 1)
        launch_extract_views_c8<__half>(image, coords, out, B, Hi, Wi, L, chunks, SH, SW, mean, stdv, normalise, out_is_bf16, st);
    else
        launch_extract_views_c8<float>(image, coords, out, B, Hi, Wi, L, chunks, SH, SW, mean, stdv, normalise, out_is_bf16, st);
    return check_launch("extract_views_c8");
}
