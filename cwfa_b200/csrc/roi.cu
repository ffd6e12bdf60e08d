// Posterior mean and exact standard deviation of region readouts (ROIs) of the reconstructed volume.
//
// On CAT-only levels level n's detail half is affine in its latent, hi_n[e] = beta_n[e] + alpha_n[e] z_n[pi_n(e)]; alpha_n is
// the F8 scale tensor that cwfa_coupling_f8_scale carries along the level's chain.  The levels are independent and the Haar
// merges are orthonormal, so a readout r = sum_v w_v V_v has, exactly,
//     E[r] = sum_v w_v V(z = 0)_v,        Var[r] = sigma^2 sum_n sum_e (alpha_n[e] w~_n[e])^2,
// with w~_n level n's detail coefficients of the forward depth Haar analysis of w (RoiSet / data.roi_tables build them).
//
// One warp per (batch item, ROI): a lane-strided walk over the ROI's table entries, fp64 products and accumulators, then a
// fixed xor-butterfly over the 32 lanes.  No atomics: the result is the same bits on every run.  fp64 keeps the readout within
// a few fp32 ulps of the float64 sum whatever the ROI's size; the walk is bound by the gathers, not by the arithmetic.
#include <math.h>
#include "common.cuh"

namespace cwfa {

constexpr int kRoiMaxLevels = 8;
constexpr int kRoiThreads = 256;

struct RoiLevels {
    const float* scale[kRoiMaxLevels];      // level n's F8 scale tensor, (B, ceil(ch_n / 8), H, W, 8)
    int64_t stride[kRoiMaxLevels];          //   floats per batch item
};

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__global__ void __launch_bounds__(kRoiThreads) roi_readout_f8_kernel(const float* __restrict__ vol, int64_t vol_stride,
                                                                     const RoiLevels lv, int L, const int64_t* __restrict__ mean_ptr,
                                                                     const int32_t* __restrict__ mean_idx,
                                                                     const float* __restrict__ mean_w,
                                                                     const int64_t* __restrict__ coef_ptr,
                                                                     const int32_t* __restrict__ coef_idx,
                                                                     const float* __restrict__ coef_val, int B, int R, float sigma,
                                                                     float* __restrict__ mean, float* __restrict__ std_out) {
    const int64_t warp = ((int64_t)blockIdx.x * kRoiThreads + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= (int64_t)B * R) return;                     // whole warps only: B * R warps, kRoiThreads a multiple of 32
    const int b = (int)(warp / R), r = (int)(warp - (int64_t)b * R);
    const float* v = vol + (int64_t)b * vol_stride;
    double m = 0.0;
    for (int64_t e = __ldg(mean_ptr + r) + lane, end = __ldg(mean_ptr + r + 1); e < end; e += 32)
        m = fma((double)__ldg(mean_w + e), (double)__ldg(v + __ldg(mean_idx + e)), m);
    double q = 0.0;
#pragma unroll
    for (int n = 0; n < kRoiMaxLevels; ++n) {               // static indices into lv: a dynamic one copies it to the stack
        if (n >= L) break;
        const float* s = lv.scale[n] + (int64_t)b * lv.stride[n];
        const int64_t* p = coef_ptr + (int64_t)n * (R + 1) + r;
        for (int64_t e = __ldg(p) + lane, end = __ldg(p + 1); e < end; e += 32) {
            const double t = (double)__ldg(coef_val + e) * (double)__ldg(s + __ldg(coef_idx + e));
            q = fma(t, t, q);
        }
    }
    m = warp_sum_f64(m);
    q = warp_sum_f64(q);
    if (lane == 0) {
        mean[warp] = (float)m;
        std_out[warp] = (float)((double)sigma * sqrt(q));
    }
}

}  // namespace cwfa

using namespace cwfa;

extern "C" int cwfa_roi_readout_f8(const float* vol, int64_t vol_stride, const float* const* scale_f8, const int64_t* scale_stride, int L,
                                   const int64_t* mean_ptr, const int32_t* mean_idx, const float* mean_w, const int64_t* coef_ptr,
                                   const int32_t* coef_idx, const float* coef_val, int B, int R, float sigma, float* mean,
                                   float* std_out, void* stream) {
    if (L < 1 || L > kRoiMaxLevels) {
        set_error("roi_readout_f8: L must be in 1..%d, got %d", kRoiMaxLevels, L);
        return CWFA_EINVAL;
    }
    if (!(sigma >= 0.f && sigma <= 3.402823466e38f)) {      // also rejects NaN and +inf
        set_error("roi_readout_f8: sigma must be finite and >= 0");
        return CWFA_EINVAL;
    }
    if (R < 1 || B < 1 || vol_stride < 1) {
        set_error("roi_readout_f8: needs R >= 1, B >= 1 and vol_stride >= 1");
        return CWFA_EINVAL;
    }
    if (!vol || !scale_f8 || !scale_stride || !mean_ptr || !mean_idx || !mean_w || !coef_ptr || !coef_idx || !coef_val || !mean ||
        !std_out) {
        set_error("roi_readout_f8: vol, scale_f8, scale_stride, the tables, mean and std must not be NULL");
        return CWFA_EINVAL;
    }
    RoiLevels lv = {};
    for (int n = 0; n < L; ++n) {                           // host arrays: copied into the launch's parameters
        if (!scale_f8[n] || scale_stride[n] < 1) {
            set_error("roi_readout_f8: level %d has a NULL scale tensor or a stride < 1", n);
            return CWFA_EINVAL;
        }
        lv.scale[n] = scale_f8[n];
        lv.stride[n] = scale_stride[n];
    }
    const int64_t blocks = ((int64_t)B * R * 32 + kRoiThreads - 1) / kRoiThreads;
    if (blocks > 0x7fffffff) {
        set_error("roi_readout_f8: B * R too large for one grid");
        return CWFA_EINVAL;
    }
    roi_readout_f8_kernel<<<(unsigned)blocks, kRoiThreads, 0, (cudaStream_t)stream>>>(vol, vol_stride, lv, L, mean_ptr, mean_idx, mean_w,
                                                                                     coef_ptr, coef_idx, coef_val, B, R, sigma, mean,
                                                                                     std_out);
    return check_launch("roi_readout_f8");
}
