// Memory-bound kernels of the CWFA path: Haar DWT/IDWT (1-D depth-wise and FrEIA 2-D),
// permutations, affine coupling with fused per-sample log-det, normalisation helpers.
// All are single-pass, 128-bit vectorised where alignment allows, grid sized in multiples
// of the SM count.  Reference arithmetic cited per function in include/cwfa_b200.h.
#include <stdarg.h>
#include <algorithm>
#include "common.cuh"

namespace cwfa {
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return CWFA_ECUDA;
    }
    return CWFA_OK;
}
}  // namespace cwfa
using namespace cwfa;

extern "C" const char* cwfa_version(void) { return "cwfa_b200 0.1 (sm_100a)"; }
extern "C" const char* cwfa_last_error(void) { return cwfa::g_err; }
extern "C" int cwfa_device_check(void) {
    int dev = 0, major = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { set_error("no CUDA device"); return CWFA_ECUDA; }
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    if (major != 10) { set_error("device is sm_%d0, need sm_100", major); return CWFA_ENOTSUP; }
    return CWFA_OK;
}

#define INV_SQRT2 0.70710678118654752440f

// ------------------------------------------------------------------------------------------
// K1: depth-wise Haar
// ------------------------------------------------------------------------------------------
template <int VEC, bool INV>
__global__ void __launch_bounds__(256) haar1d_kernel(const float* __restrict__ a, const float* __restrict__ b2,
                                                     float* __restrict__ o1, float* __restrict__ o2,
                                                     int B, int h, int64_t P, int64_t ld_lo, int64_t ld_hi) {
    // fwd: a = x (B,2h,P), o1 = lo, o2 = hi.   inv: a = lo, b2 = hi, o1 = x.
    const int64_t Pv = P / VEC;
    const int64_t total = (int64_t)B * h * Pv;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t p = (idx % Pv) * VEC;
        const int64_t r = idx / Pv;
        const int i = (int)(r % h);
        const int b = (int)(r / h);
        const int64_t xo = ((int64_t)b * 2 * h + 2 * i) * P + p;
        const int64_t lo_o = (int64_t)b * ld_lo + (int64_t)i * P + p;
        const int64_t hi_o = (int64_t)b * ld_hi + (int64_t)i * P + p;
        if constexpr (VEC == 4) {
            if constexpr (!INV) {
                const float4 e = __ldg(reinterpret_cast<const float4*>(a + xo));
                const float4 o = __ldg(reinterpret_cast<const float4*>(a + xo + P));
                float4 l, hh;
                l.x = (e.x + o.x) * INV_SQRT2; hh.x = (e.x - o.x) * INV_SQRT2;
                l.y = (e.y + o.y) * INV_SQRT2; hh.y = (e.y - o.y) * INV_SQRT2;
                l.z = (e.z + o.z) * INV_SQRT2; hh.z = (e.z - o.z) * INV_SQRT2;
                l.w = (e.w + o.w) * INV_SQRT2; hh.w = (e.w - o.w) * INV_SQRT2;
                *reinterpret_cast<float4*>(o1 + lo_o) = l;
                *reinterpret_cast<float4*>(o2 + hi_o) = hh;
            } else {
                const float4 l = __ldg(reinterpret_cast<const float4*>(a + lo_o));
                const float4 hh = __ldg(reinterpret_cast<const float4*>(b2 + hi_o));
                float4 e, o;
                e.x = (l.x + hh.x) * INV_SQRT2; o.x = (l.x - hh.x) * INV_SQRT2;
                e.y = (l.y + hh.y) * INV_SQRT2; o.y = (l.y - hh.y) * INV_SQRT2;
                e.z = (l.z + hh.z) * INV_SQRT2; o.z = (l.z - hh.z) * INV_SQRT2;
                e.w = (l.w + hh.w) * INV_SQRT2; o.w = (l.w - hh.w) * INV_SQRT2;
                *reinterpret_cast<float4*>(o1 + xo) = e;
                *reinterpret_cast<float4*>(o1 + xo + P) = o;
            }
        } else {
            if constexpr (!INV) {
                const float e = a[xo], o = a[xo + P];
                o1[lo_o] = (e + o) * INV_SQRT2;
                o2[hi_o] = (e - o) * INV_SQRT2;
            } else {
                const float l = a[lo_o], hh = b2[hi_o];
                o1[xo] = (l + hh) * INV_SQRT2;
                o1[xo + P] = (l - hh) * INV_SQRT2;
            }
        }
    }
}

static int haar1d_launch(bool inv, const float* x_or_lo, const float* hi_in, float* o1, float* o2, int B, int C,
                         int64_t P, int64_t ld_lo, int64_t ld_hi, cudaStream_t st) {
    if (B <= 0 || C <= 0 || (C & 1) || P <= 0) { set_error("haar1d: bad shape B=%d C=%d", B, C); return CWFA_EINVAL; }
    const int h = C / 2;
    const bool vec = (P % 4 == 0) && (ld_lo % 4 == 0) && (ld_hi % 4 == 0) && aligned16(x_or_lo) && aligned16(o1) &&
                     (inv ? aligned16(hi_in) : aligned16(o2));
    const int64_t total = (int64_t)B * h * (vec ? P / 4 : P);
    int blocks = (int)((total + 255) / 256);
    const int maxb = kNumSMs * 16;
    if (blocks > maxb) blocks = maxb;
    if (blocks < 1) blocks = 1;
    if (vec) {
        if (inv) haar1d_kernel<4, true><<<blocks, 256, 0, st>>>(x_or_lo, hi_in, o1, o2, B, h, P, ld_lo, ld_hi);
        else haar1d_kernel<4, false><<<blocks, 256, 0, st>>>(x_or_lo, hi_in, o1, o2, B, h, P, ld_lo, ld_hi);
    } else {
        if (inv) haar1d_kernel<1, true><<<blocks, 256, 0, st>>>(x_or_lo, hi_in, o1, o2, B, h, P, ld_lo, ld_hi);
        else haar1d_kernel<1, false><<<blocks, 256, 0, st>>>(x_or_lo, hi_in, o1, o2, B, h, P, ld_lo, ld_hi);
    }
    return check_launch("haar1d");
}

extern "C" int cwfa_haar1d_fwd(const float* x, float* lo, float* hi, int B, int C, int64_t P, int64_t ld_lo,
                               int64_t ld_hi, void* stream) {
    return haar1d_launch(false, x, nullptr, lo, hi, B, C, P, ld_lo, ld_hi, (cudaStream_t)stream);
}
extern "C" int cwfa_haar1d_inv(const float* lo, const float* hi, float* x, int B, int C, int64_t P, int64_t ld_lo,
                               int64_t ld_hi, void* stream) {
    return haar1d_launch(true, lo, hi, x, nullptr, B, C, P, ld_lo, ld_hi, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------
// K1b: FrEIA 2-D Haar.  One thread per 2x2 input block (one output pixel of 4 wavelets).
// ------------------------------------------------------------------------------------------
template <bool UP>
__global__ void __launch_bounds__(256) haar2d_kernel(const float* __restrict__ src, float* __restrict__ dst, int C, int H2,
                                                     int W2, int by_wavelet, float fac) {
    // Fine grid is (B,C,2*H2,2*W2); coarse grid is (B,4C,H2,W2).  blockIdx.y = (sample, channel) plane of the fine
    // tensor, blockIdx.x strides over coarse rows, threads over coarse columns: no index divisions.
    const int c = blockIdx.y % C;
    const int64_t b4c = (int64_t)(blockIdx.y - c) * 4;            // b * 4C
    const int64_t cplane = (int64_t)H2 * W2;
    const int W = 2 * W2;
    const float* fsrc = src + (int64_t)blockIdx.y * 4 * cplane;   // fine plane (UP: unused)
    float* fdst = dst + (int64_t)blockIdx.y * 4 * cplane;
    int64_t cbase[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) cbase[k] = (b4c + (by_wavelet ? k * C + c : 4 * c + k)) * cplane;
    for (int h2 = blockIdx.x; h2 < H2; h2 += gridDim.x) {
        const int64_t frow = (int64_t)(2 * h2) * W;
        const int64_t crow = (int64_t)h2 * W2;
        for (int w2 = threadIdx.x; w2 < W2; w2 += blockDim.x) {
            if constexpr (!UP) {
                const float2 r0 = __ldg(reinterpret_cast<const float2*>(fsrc + frow + 2 * w2));
                const float2 r1 = __ldg(reinterpret_cast<const float2*>(fsrc + frow + W + 2 * w2));
                const float a = r0.x, bb = r0.y, cc = r1.x, d = r1.y;
                dst[cbase[0] + crow + w2] = fac * (a + bb + cc + d);
                dst[cbase[1] + crow + w2] = fac * (a - bb + cc - d);
                dst[cbase[2] + crow + w2] = fac * (a + bb - cc - d);
                dst[cbase[3] + crow + w2] = fac * (a - bb - cc + d);
            } else {
                const float y0 = fac * __ldg(src + cbase[0] + crow + w2), y1 = fac * __ldg(src + cbase[1] + crow + w2);
                const float y2 = fac * __ldg(src + cbase[2] + crow + w2), y3 = fac * __ldg(src + cbase[3] + crow + w2);
                float2 r0, r1;
                r0.x = y0 + y1 + y2 + y3;
                r0.y = y0 - y1 + y2 - y3;
                r1.x = y0 + y1 - y2 - y3;
                r1.y = y0 - y1 - y2 + y3;
                *reinterpret_cast<float2*>(fdst + frow + 2 * w2) = r0;
                *reinterpret_cast<float2*>(fdst + frow + W + 2 * w2) = r1;
            }
        }
    }
}

static int haar2d_launch(bool up, const float* src, float* dst, int B, int C, int H, int W, int obw, float fac,
                         cudaStream_t st) {
    // (C,H,W) always describe the FINE tensor.
    if (B <= 0 || C <= 0 || H <= 0 || W <= 0 || (H & 1) || (W & 1) || (int64_t)B * C > 65535) {
        set_error("haar2d: H and W must be even (got %dx%d)", H, W);
        return CWFA_EINVAL;
    }
    const int planes = B * C, H2 = H / 2, W2 = W / 2;
    int gx = ceil_div(kNumSMs * 8, planes);
    if (gx > H2) gx = H2;
    if (gx < 1) gx = 1;
    const int threads = W2 >= 256 ? 256 : (W2 >= 128 ? 128 : 64);
    dim3 grid(gx, planes);
    if (up) haar2d_kernel<true><<<grid, threads, 0, st>>>(src, dst, C, H2, W2, obw, fac);
    else haar2d_kernel<false><<<grid, threads, 0, st>>>(src, dst, C, H2, W2, obw, fac);
    return check_launch("haar2d");
}
extern "C" int cwfa_haar2d_down(const float* x, float* y, int B, int C, int H, int W, int obw, float fac,
                                void* stream) {
    return haar2d_launch(false, x, y, B, C, H, W, obw, fac, (cudaStream_t)stream);
}
extern "C" int cwfa_haar2d_up(const float* y, float* x, int B, int C, int H, int W, int obw, float fac,
                              void* stream) {
    return haar2d_launch(true, y, x, B, C, H, W, obw, fac, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------
// K4: permutations (gather along one axis)
// ------------------------------------------------------------------------------------------
// blockIdx.y = (sample, channel) plane, blockIdx.x strides over rows, threads over (vectors of) columns: no index
// divisions.  AXIS 1 / 2 copy whole rows from the permuted plane / row with 16-byte accesses; AXIS 3 stages the source
// row in shared memory (coalesced read) and gathers from there (coalesced write).
template <int AXIS, int VEC>
__global__ void __launch_bounds__(256) permute_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                      const int32_t* __restrict__ perm, int C, int H, int W) {
    extern __shared__ __align__(16) float s_row[];   // AXIS 3: W floats (source row) per warp + W ints (perm)
    const int c = blockIdx.y % C;
    const int64_t plane = (int64_t)H * W;
    const int64_t splane = (AXIS == 1) ? ((int64_t)(blockIdx.y - c) + __ldg(perm + c)) * plane : (int64_t)blockIdx.y * plane;
    const float* xp = x + splane;
    float* yp = y + (int64_t)blockIdx.y * plane;
    if constexpr (AXIS == 3) {
        // one row per warp (private shared-memory slice, warp-level syncs only); perm table shared by the block
        const int nw = blockDim.x >> 5, wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
        int* s_perm = reinterpret_cast<int*>(s_row + (size_t)nw * W);
        for (int w = threadIdx.x; w < W; w += blockDim.x) s_perm[w] = __ldg(perm + w);
        __syncthreads();
        float* row = s_row + (size_t)wid * W;
        if constexpr (VEC == 4) {
            // 16-byte global accesses on both sides: the row lands in shared memory as float4, four gathered columns leave as one float4
            const int W4 = W >> 2;
            const int4* s_perm4 = reinterpret_cast<const int4*>(s_perm);
            for (int h = blockIdx.x * nw + wid; h < H; h += gridDim.x * nw) {
                const float4* xr = reinterpret_cast<const float4*>(xp + (int64_t)h * W);
                for (int w = lane; w < W4; w += 32) reinterpret_cast<float4*>(row)[w] = __ldg(xr + w);
                __syncwarp();
                float4* yr = reinterpret_cast<float4*>(yp + (int64_t)h * W);
                for (int w = lane; w < W4; w += 32) {
                    const int4 pp = s_perm4[w];
                    yr[w] = make_float4(row[pp.x], row[pp.y], row[pp.z], row[pp.w]);
                }
                __syncwarp();
            }
        } else {
            for (int h = blockIdx.x * nw + wid; h < H; h += gridDim.x * nw) {
                for (int w = lane; w < W; w += 32) row[w] = __ldg(xp + (int64_t)h * W + w);
                __syncwarp();
                for (int w = lane; w < W; w += 32) yp[(int64_t)h * W + w] = row[s_perm[w]];
                __syncwarp();
            }
        }
    } else {
        const int Wv = W / VEC;
        for (int h = blockIdx.x; h < H; h += gridDim.x) {
            const int sh = (AXIS == 2) ? __ldg(perm + h) : h;
            const float* xr = xp + (int64_t)sh * W;
            float* yr = yp + (int64_t)h * W;
            for (int w = threadIdx.x; w < Wv; w += blockDim.x) {
                if constexpr (VEC == 4) reinterpret_cast<float4*>(yr)[w] = __ldg(reinterpret_cast<const float4*>(xr) + w);
                else yr[w] = __ldg(xr + w);
            }
        }
    }
}

extern "C" int cwfa_permute(const float* x, float* y, const int32_t* perm, int axis, int B, int C, int H, int W,
                            void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (axis < 1 || axis > 3 || B <= 0 || C <= 0 || H <= 0 || W <= 0 || (int64_t)B * C > 65535 || W > 8192) {
        set_error("permute: bad args");
        return CWFA_EINVAL;
    }
    const bool vec = axis != 3 && (W % 4 == 0) && aligned16(x) && aligned16(y);
    const int planes = B * C;
    int gx = ceil_div(kNumSMs * 8, planes);
    if (gx > H) gx = H;
    if (gx < 1) gx = 1;
    const int cols = vec ? W / 4 : W;
    const int threads = cols >= 256 ? 256 : (cols >= 128 ? 128 : 64);
    dim3 grid(gx, planes);
    if (axis == 1) {
        if (vec) permute_kernel<1, 4><<<grid, threads, 0, st>>>(x, y, perm, C, H, W);
        else permute_kernel<1, 1><<<grid, threads, 0, st>>>(x, y, perm, C, H, W);
    } else if (axis == 2) {
        if (vec) permute_kernel<2, 4><<<grid, threads, 0, st>>>(x, y, perm, C, H, W);
        else permute_kernel<2, 1><<<grid, threads, 0, st>>>(x, y, perm, C, H, W);
    } else {
        int g3 = ceil_div(H, 8);                   // 8 rows (one per warp) per block pass; ~8 resident blocks per SM overall
        if (g3 > gx) g3 = gx;
        dim3 grid3(g3 > 0 ? g3 : 1, planes);
        if ((W % 4 == 0) && aligned16(x) && aligned16(y)) permute_kernel<3, 4><<<grid3, 256, (size_t)W * 4 * 9, st>>>(x, y, perm, C, H, W);
        else permute_kernel<3, 1><<<grid3, 256, (size_t)W * 4 * 9, st>>>(x, y, perm, C, H, W);
    }
    return check_launch("permute");
}

// ------------------------------------------------------------------------------------------
// K3: affine coupling + per-sample log-det (+ sum of squares).  Deterministic two-stage sum.
// ------------------------------------------------------------------------------------------
constexpr int kAffineBlocks = kNumSMs * 2;   // blocks per sample

template <int VEC, bool INV>
__global__ void __launch_bounds__(256) affine_kernel(const float* __restrict__ x, const float* __restrict__ a_s,
                                                     const float* __restrict__ a_t, float* __restrict__ y,
                                                     float* __restrict__ ws, int ch, int64_t P, int64_t ld_s,
                                                     int64_t ld_t, float kk, float t_scale, int raw, float k_in) {
    const int b = blockIdx.y;
    const int64_t n = (int64_t)ch * P;           // elements of this sample
    const float* xs = x ? x + (int64_t)b * n : nullptr;
    const float* ss = a_s + (int64_t)b * ld_s;
    const float* ts = a_t + (int64_t)b * ld_t;
    float* ys = y + (int64_t)b * n;
    float sum_s = 0.f, sum_q = 0.f;
    for (int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) * VEC; i < n;
         i += (int64_t)gridDim.x * blockDim.x * VEC) {
        float xv[VEC], sv[VEC], tv[VEC], yv[VEC];
        if constexpr (VEC == 4) {
            const float4 s4 = __ldg(reinterpret_cast<const float4*>(ss + i));
            const float4 t4 = __ldg(reinterpret_cast<const float4*>(ts + i));
            sv[0] = s4.x; sv[1] = s4.y; sv[2] = s4.z; sv[3] = s4.w;
            tv[0] = t4.x; tv[1] = t4.y; tv[2] = t4.z; tv[3] = t4.w;
            if (xs) {
                const float4 x4 = __ldg(reinterpret_cast<const float4*>(xs + i));
                xv[0] = x4.x; xv[1] = x4.y; xv[2] = x4.z; xv[3] = x4.w;
            } else {
                xv[0] = xv[1] = xv[2] = xv[3] = 0.f;
            }
        } else {
            sv[0] = ss[i]; tv[0] = ts[i]; xv[0] = xs ? xs[i] : 0.f;
        }
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
            const float s = raw == 1 ? sv[k] : (raw == 2 ? kk * tanhf(k_in * sv[k]) : kk * atanf(sv[k]));
            const float t = t_scale * tv[k];
            sum_s += s;
            yv[k] = INV ? (xv[k] - t) * expf(-s) : expf(s) * xv[k] + t;
            sum_q += yv[k] * yv[k];
        }
        if constexpr (VEC == 4) {
            *reinterpret_cast<float4*>(ys + i) = make_float4(yv[0], yv[1], yv[2], yv[3]);
        } else {
            ys[i] = yv[0];
        }
    }
    block_sum2(sum_s, sum_q);
    if (threadIdx.x == 0) {
        ws[((int64_t)b * gridDim.x + blockIdx.x) * 2 + 0] = INV ? -sum_s : sum_s;
        ws[((int64_t)b * gridDim.x + blockIdx.x) * 2 + 1] = sum_q;
    }
}

__global__ void affine_finalize_kernel(const float* __restrict__ ws, float* __restrict__ logdet,
                                       float* __restrict__ sumsq, int nblocks) {
    // one warp per sample; fixed summation order -> bit-reproducible
    const int b = blockIdx.x;
    double s = 0.0, q = 0.0;
    for (int i = threadIdx.x; i < nblocks; i += 32) {
        s += (double)ws[((int64_t)b * nblocks + i) * 2 + 0];
        q += (double)ws[((int64_t)b * nblocks + i) * 2 + 1];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        q += __shfl_xor_sync(0xffffffffu, q, o);
    }
    if (threadIdx.x == 0) {
        logdet[b] = (float)s;
        if (sumsq) sumsq[b] = (float)q;
    }
}

extern "C" int cwfa_affine_workspace_blocks(void) { return kAffineBlocks; }

extern "C" int cwfa_affine(const float* x, const float* a_s, const float* a_t, float* y, float* logdet, float* sumsq,
                           float* workspace, int B, int ch, int64_t P, int64_t ld_s, int64_t ld_t, float clamp,
                           float k_atan, float t_scale, int flags, void* stream) {
    const int inverse = flags & 1, raw = (flags & 4) ? 2 : ((flags >> 1) & 1);
    cudaStream_t st = (cudaStream_t)stream;
    if (B <= 0 || ch <= 0 || P <= 0 || !a_s || !a_t || !y || !logdet || !workspace) {
        set_error("affine: bad args");
        return CWFA_EINVAL;
    }
    if (!x && !inverse) { set_error("affine: x may be NULL only in inverse mode"); return CWFA_EINVAL; }
    const int64_t n = (int64_t)ch * P;
    const bool vec = (n % 4 == 0) && (ld_s % 4 == 0) && (ld_t % 4 == 0) && aligned16(a_s) && aligned16(a_t) &&
                     aligned16(y) && (!x || aligned16(x));
    dim3 grid(kAffineBlocks, B);
    const float kk = raw == 2 ? clamp : clamp * k_atan;      // TANH mode: s = clamp * tanh(k_atan * a)
    if (vec) {
        if (inverse) affine_kernel<4, true><<<grid, 256, 0, st>>>(x, a_s, a_t, y, workspace, ch, P, ld_s, ld_t, kk, t_scale, raw, k_atan);
        else affine_kernel<4, false><<<grid, 256, 0, st>>>(x, a_s, a_t, y, workspace, ch, P, ld_s, ld_t, kk, t_scale, raw, k_atan);
    } else {
        if (inverse) affine_kernel<1, true><<<grid, 256, 0, st>>>(x, a_s, a_t, y, workspace, ch, P, ld_s, ld_t, kk, t_scale, raw, k_atan);
        else affine_kernel<1, false><<<grid, 256, 0, st>>>(x, a_s, a_t, y, workspace, ch, P, ld_s, ld_t, kk, t_scale, raw, k_atan);
    }
    int rc = check_launch("affine");
    if (rc) return rc;
    affine_finalize_kernel<<<B, 32, 0, st>>>(workspace, logdet, sumsq, kAffineBlocks);
    return check_launch("affine_finalize");
}

// ------------------------------------------------------------------------------------------
// Normalisation / pooling helpers (LRNN)
// ------------------------------------------------------------------------------------------
constexpr int kStatsBlocks = 32;   // blocks per channel

__global__ void __launch_bounds__(256) channel_stats_kernel(const float* __restrict__ x, float* __restrict__ ws, int N,
                                                            int C, int64_t P) {
    const int c = blockIdx.y;
    float s = 0.f, q = 0.f;
    for (int n = 0; n < N; ++n) {
        const float* xp = x + ((int64_t)n * C + c) * P;
        for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < P; p += (int64_t)gridDim.x * blockDim.x) {
            const float v = __ldg(xp + p);
            s += v;
            q += v * v;
        }
    }
    block_sum2(s, q);
    if (threadIdx.x == 0) {
        ws[((int64_t)c * gridDim.x + blockIdx.x) * 2 + 0] = s;
        ws[((int64_t)c * gridDim.x + blockIdx.x) * 2 + 1] = q;
    }
}
__global__ void stats_finalize_kernel(const float* __restrict__ ws, float* __restrict__ stats, int C, int nblocks) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double s = 0.0, q = 0.0;
    for (int i = 0; i < nblocks; ++i) {
        s += (double)ws[((int64_t)c * nblocks + i) * 2 + 0];
        q += (double)ws[((int64_t)c * nblocks + i) * 2 + 1];
    }
    stats[c] = (float)s;
    stats[C + c] = (float)q;
}
extern "C" int cwfa_stats_workspace_blocks(void) { return kStatsBlocks; }
extern "C" int cwfa_channel_stats_f32(const float* x, float* stats, float* workspace, int N, int C, int64_t P,
                                      void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (N <= 0 || C <= 0 || P <= 0) { set_error("channel_stats: bad shape"); return CWFA_EINVAL; }
    channel_stats_kernel<<<dim3(kStatsBlocks, C), 256, 0, st>>>(x, workspace, N, C, P);
    int rc = check_launch("channel_stats");
    if (rc) return rc;
    stats_finalize_kernel<<<ceil_div(C, 128), 128, 0, st>>>(workspace, stats, C, kStatsBlocks);
    return check_launch("stats_finalize");
}

__global__ void bn_finalize_kernel(const float* __restrict__ stats, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float* __restrict__ scale, float* __restrict__ shift,
                                   int C, double count, float eps) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const double mean = (double)stats[c] / count;
    double var = (double)stats[C + c] / count - mean * mean;   // biased, as BatchNorm normalises with
    if (var < 0.0) var = 0.0;
    const double sc = (double)gamma[c] / sqrt(var + (double)eps);
    scale[c] = (float)sc;
    shift[c] = (float)((double)beta[c] - mean * sc);
}
extern "C" int cwfa_bn_finalize_f32(const float* stats, const float* gamma, const float* beta, float* scale,
                                    float* shift, int C, double count, float eps, void* stream) {
    bn_finalize_kernel<<<ceil_div(C, 128), 128, 0, (cudaStream_t)stream>>>(stats, gamma, beta, scale, shift, C, count, eps);
    return check_launch("bn_finalize");
}

template <int VEC>
__global__ void __launch_bounds__(256) scale_shift_kernel(const float* __restrict__ x, const float* __restrict__ scale,
                                                          const float* __restrict__ shift, float* __restrict__ y,
                                                          int64_t NC, int C, int64_t P) {
    const int64_t Pv = P / VEC;
    const int64_t total = NC * Pv;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t nc = idx / Pv;
        const int c = (int)(nc % C);
        const float sc = __ldg(scale + c), sh = __ldg(shift + c);
        const int64_t o = nc * P + (idx % Pv) * VEC;
        if constexpr (VEC == 4) {
            float4 v = __ldg(reinterpret_cast<const float4*>(x + o));
            v.x = v.x * sc + sh; v.y = v.y * sc + sh; v.z = v.z * sc + sh; v.w = v.w * sc + sh;
            *reinterpret_cast<float4*>(y + o) = v;
        } else {
            y[o] = x[o] * sc + sh;
        }
    }
}
extern "C" int cwfa_scale_shift_f32(const float* x, const float* scale, const float* shift, float* y, int N, int C,
                                    int64_t P, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    const bool vec = (P % 4 == 0) && aligned16(x) && aligned16(y);
    const int64_t total = (int64_t)N * C * (vec ? P / 4 : P);
    int blocks = (int)((total + 255) / 256);
    if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
    if (vec) scale_shift_kernel<4><<<blocks, 256, 0, st>>>(x, scale, shift, y, (int64_t)N * C, C, P);
    else scale_shift_kernel<1><<<blocks, 256, 0, st>>>(x, scale, shift, y, (int64_t)N * C, C, P);
    return check_launch("scale_shift");
}

__global__ void __launch_bounds__(256) maxpool2_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                       int64_t NC, int H2, int W2) {
    const int64_t total = NC * H2 * W2;
    const int W = 2 * W2;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int w2 = (int)(idx % W2);
        const int h2 = (int)((idx / W2) % H2);
        const int64_t nc = idx / ((int64_t)W2 * H2);
        const float* p = x + (nc * (2 * H2) + 2 * h2) * W + 2 * w2;
        const float2 a = __ldg(reinterpret_cast<const float2*>(p));
        const float2 b = __ldg(reinterpret_cast<const float2*>(p + W));
        y[idx] = fmaxf(fmaxf(a.x, a.y), fmaxf(b.x, b.y));
    }
}
extern "C" int cwfa_maxpool2_f32(const float* x, float* y, int N, int C, int H, int W, void* stream) {
    if ((H & 1) || (W & 1)) { set_error("maxpool2: odd size"); return CWFA_EINVAL; }
    const int64_t total = (int64_t)N * C * (H / 2) * (W / 2);
    int blocks = (int)((total + 255) / 256);
    if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
    maxpool2_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(x, y, (int64_t)N * C, H / 2, W / 2);
    return check_launch("maxpool2");
}

// LayerNorm over (C,H,W): stage 1 partial sums, stage 2 normalise with element-wise affine.
constexpr int kLNBlocks = kNumSMs * 2;
__global__ void __launch_bounds__(256) ln_stats_kernel(const float* __restrict__ x, float* __restrict__ ws, int64_t n) {
    const int b = blockIdx.y;
    const float* xs = x + (int64_t)b * n;
    float s = 0.f, q = 0.f;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float v = __ldg(xs + i);
        s += v;
        q += v * v;
    }
    block_sum2(s, q);
    if (threadIdx.x == 0) {
        ws[((int64_t)b * gridDim.x + blockIdx.x) * 2 + 0] = s;
        ws[((int64_t)b * gridDim.x + blockIdx.x) * 2 + 1] = q;
    }
}
__global__ void __launch_bounds__(256) ln_apply_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                       const float* __restrict__ beta, float* __restrict__ y,
                                                       const float* __restrict__ ws, int64_t n, float eps) {
    const int b = blockIdx.y;
    __shared__ float s_mean, s_rstd;
    if (threadIdx.x == 0) {
        double s = 0.0, q = 0.0;
        for (int i = 0; i < kLNBlocks; ++i) {
            s += (double)ws[((int64_t)b * kLNBlocks + i) * 2 + 0];
            q += (double)ws[((int64_t)b * kLNBlocks + i) * 2 + 1];
        }
        const double mean = s / (double)n;
        double var = q / (double)n - mean * mean;
        if (var < 0.0) var = 0.0;
        s_mean = (float)mean;
        s_rstd = (float)(1.0 / sqrt(var + (double)eps));
    }
    __syncthreads();
    const float mean = s_mean, rstd = s_rstd;
    const float* xs = x + (int64_t)b * n;
    float* ys = y + (int64_t)b * n;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        ys[i] = (__ldg(xs + i) - mean) * rstd * __ldg(gamma + i) + __ldg(beta + i);
}
extern "C" int cwfa_layernorm_chw_f32(const float* x, const float* gamma, const float* beta, float* y,
                                      float* workspace, int N, int64_t CHW, float eps, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (N <= 0 || CHW <= 0) { set_error("layernorm: bad shape"); return CWFA_EINVAL; }
    ln_stats_kernel<<<dim3(kLNBlocks, N), 256, 0, st>>>(x, workspace, CHW);
    int rc = check_launch("ln_stats");
    if (rc) return rc;
    ln_apply_kernel<<<dim3(kLNBlocks, N), 256, 0, st>>>(x, gamma, beta, y, workspace, CHW, eps);
    return check_launch("ln_apply");
}

__global__ void __launch_bounds__(256) gate_add_kernel(float* __restrict__ x, const float* __restrict__ m,
                                                       const float* __restrict__ g, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        x[i] += m[i] * 2.f * (g[i] - 0.5f);
}
// fp32 -> fp16 narrowing of a finished volume (optional half-size device->host transfer; the reference's own GPU output is
// fp16 under autocast, CWFA.py:845): 8 elements per thread, 2 x 16-byte loads, one 16-byte store, grid = multiple of the SM count.
__global__ void __launch_bounds__(256) cast_f32_f16_kernel(const float4* __restrict__ x, uint4* __restrict__ y, int64_t n8,
                                                           const float* __restrict__ xt, __half* __restrict__ yt, int64_t tail0, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 a = __ldg(x + 2 * i), b = __ldg(x + 2 * i + 1);
        __half2 h0 = __floats2half2_rn(a.x, a.y), h1 = __floats2half2_rn(a.z, a.w), h2 = __floats2half2_rn(b.x, b.y), h3 = __floats2half2_rn(b.z, b.w);
        uint4 o;
        o.x = *reinterpret_cast<uint32_t*>(&h0); o.y = *reinterpret_cast<uint32_t*>(&h1);
        o.z = *reinterpret_cast<uint32_t*>(&h2); o.w = *reinterpret_cast<uint32_t*>(&h3);
        y[i] = o;
    }
    if (blockIdx.x == 0)
        for (int64_t i = tail0 + threadIdx.x; i < n; i += blockDim.x) yt[i] = __float2half_rn(xt[i]);
}
extern "C" int cwfa_cast_f32_f16(const float* x, void* y, int64_t n, void* stream) {
    if (!x || !y || n < 0 || !aligned16(x) || !aligned16(y)) { set_error("cast_f32_f16: bad arguments (16-byte aligned pointers required)"); return CWFA_EINVAL; }
    if (n == 0) return CWFA_OK;
    const int64_t n8 = n / 8;
    const int blocks = (int)std::min<int64_t>((n8 + 255) / 256 + 1, (int64_t)kNumSMs * 8);
    cast_f32_f16_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(x), reinterpret_cast<uint4*>(y), n8, x,
                                                                  reinterpret_cast<__half*>(y), n8 * 8, n);
    return check_launch("cast_f32_f16");
}

extern "C" int cwfa_gate_add_f32(float* x, const float* m, const float* g, int64_t n, void* stream) {
    int blocks = (int)((n + 255) / 256);
    if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
    gate_add_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(x, m, g, n);
    return check_launch("gate_add");
}
extern "C" int cwfa_layernorm_workspace_blocks(void) { return kLNBlocks; }

// ------------------------------------------------------------------------------------------
// GlobalAttention gate of the LRNN (networks.py:244-262, :554), fused:
//   g = sigmoid(W2 * relu(W1 (*) v + b1) + b2)  with v = mean volume flattened over H*W (Conv1d k=3, zero pad),
//   x += m * 2 * (g - 0.5)
// One thread per sequence position; C <= 16 channels live in registers.
// ------------------------------------------------------------------------------------------
constexpr int kAttMaxC = 16;
// CT = compile-time channel count (exact loops, no predication: the LRNN uses 6); CT = 0 is the run-time fallback (C <= 16).
template <int CT>
__global__ void __launch_bounds__(256) attention_gate_kernel(float* __restrict__ x, const float* __restrict__ m,
                                                             const float* __restrict__ v, const float* __restrict__ w1,
                                                             const float* __restrict__ b1, const float* __restrict__ w2,
                                                             const float* __restrict__ b2, int C, int64_t L) {
    constexpr int NC = CT ? CT : kAttMaxC;
    const int Cc = CT ? CT : C;                      // compile-time stride of the weight tables when CT is set
    __shared__ float sw1[kAttMaxC * kAttMaxC * 3], sw2[kAttMaxC * kAttMaxC], sb1[kAttMaxC], sb2[kAttMaxC];
    for (int i = threadIdx.x; i < C * C * 3; i += blockDim.x) sw1[i] = __ldg(w1 + i);
    for (int i = threadIdx.x; i < C * C; i += blockDim.x) sw2[i] = __ldg(w2 + i);
    for (int i = threadIdx.x; i < C; i += blockDim.x) { sb1[i] = __ldg(b1 + i); sb2[i] = __ldg(b2 + i); }
    __syncthreads();
    const int b = blockIdx.y;
    const float* vb = v + (int64_t)b * C * L;
    for (int64_t l = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; l < L; l += (int64_t)gridDim.x * blockDim.x) {
        float h[NC];
#pragma unroll
        for (int o = 0; o < NC; ++o) h[o] = (CT || o < C) ? sb1[o] : 0.f;
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            if (CT || c < C) {
                const float vm = l > 0 ? __ldg(vb + (int64_t)c * L + l - 1) : 0.f;
                const float v0 = __ldg(vb + (int64_t)c * L + l);
                const float vp = l + 1 < L ? __ldg(vb + (int64_t)c * L + l + 1) : 0.f;
#pragma unroll
                for (int o = 0; o < NC; ++o)
                    if (CT || o < C) h[o] = fmaf(sw1[(o * Cc + c) * 3 + 2], vp, fmaf(sw1[(o * Cc + c) * 3 + 1], v0, fmaf(sw1[(o * Cc + c) * 3], vm, h[o])));
            }
        }
#pragma unroll
        for (int o = 0; o < NC; ++o) h[o] = fmaxf(h[o], 0.f);
#pragma unroll
        for (int o = 0; o < NC; ++o) {
            if (CT || o < C) {
                float a = sb2[o];
#pragma unroll
                for (int c = 0; c < NC; ++c)
                    if (CT || c < C) a = fmaf(sw2[o * Cc + c], h[c], a);
                const float g = 1.f / (1.f + expf(-a));
                const int64_t idx = ((int64_t)b * C + o) * L + l;
                x[idx] += m[idx] * 2.f * (g - 0.5f);
            }
        }
    }
}
extern "C" int cwfa_attention_gate_f32(float* x, const float* m, const float* v, const float* w1, const float* b1,
                                       const float* w2, const float* b2, int B, int C, int64_t L, void* stream) {
    if (B <= 0 || C <= 0 || C > kAttMaxC || L <= 0 || B > 65535) { set_error("attention_gate: unsupported shape (C <= 16)"); return CWFA_EINVAL; }
    int blocks = (int)((L + 255) / 256);
    if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
    dim3 grid(blocks, B);
    cudaStream_t st = (cudaStream_t)stream;
    switch (C) {        // (with CT = C the shared-memory weight indices are compile-time immediates)
        case 6: attention_gate_kernel<6><<<grid, 256, 0, st>>>(x, m, v, w1, b1, w2, b2, C, L); break;
        case 4: attention_gate_kernel<4><<<grid, 256, 0, st>>>(x, m, v, w1, b1, w2, b2, C, L); break;
        case 12: attention_gate_kernel<12><<<grid, 256, 0, st>>>(x, m, v, w1, b1, w2, b2, C, L); break;
        default: attention_gate_kernel<0><<<grid, 256, 0, st>>>(x, m, v, w1, b1, w2, b2, C, L); break;
    }
    return check_launch("attention_gate");
}

// ------------------------------------------------------------------------------------------
// Lenslet crop + normalisation (the step right before the path; SURVEY.md 8f-1):
// XLFMDataset.extract_views (XLFMDataset.py:212-242) followed by (x - mean) / std (CWFA.py:797), one gather pass.
// For lenslet n with centre (cy,cx): lower = max(c - S/2, 0), upper = min(c + S/2, image size); the patch is written
// bottom/right aligned into the S x S view (reference quirk), the rest of the view is zero (then normalised too).
// ------------------------------------------------------------------------------------------
// blockIdx.y = (sample, lenslet): the window geometry is computed once per block; blockIdx.x strides over view rows,
// threads over view columns (coalesced 4-byte reads of the window row, coalesced writes) -- no index divisions.
template <typename TIn>
__global__ void __launch_bounds__(256) extract_views_kernel(const TIn* __restrict__ img, const int32_t* __restrict__ coords,
                                                            float* __restrict__ out, int Hi, int Wi, int L, int SH, int SW,
                                                            float mean, float stdv, int normalise) {
    const int n = blockIdx.y % L, b = blockIdx.y / L;
    const int cy = __ldg(coords + 2 * n), cx = __ldg(coords + 2 * n + 1);
    const int ly = max(cy - SH / 2, 0), lx = max(cx - SW / 2, 0);
    const int uy = min(cy + SH / 2, Hi), ux = min(cx + SW / 2, Wi);
    const int ph = max(uy - ly, 0), pw = max(ux - lx, 0);
    const bool any = ph > 0 && pw > 0;
    const float zero_v = normalise ? (0.f - mean) / stdv : 0.f;
    const TIn* ib = img + (int64_t)b * Hi * Wi;
    float* ob = out + (int64_t)blockIdx.y * SH * SW;
    // 4 output columns per thread (one 16-byte store; the window start is arbitrary, so the reads stay 4-byte but cover the
    // same 16 contiguous bytes) and two view rows in flight per thread: ~8x the bytes in flight of the one-element form, which
    // is what this latency-bound gather was missing (0.30 -> of the HBM peak).
    const bool vec = (SW & 3) == 0;
    const int jw = vec ? SW >> 2 : SW;
    auto load_row = [&](int i, int j, float (&v)[4]) {
        const int ii = i - (SH - ph);
        const TIn* irow = ib + (int64_t)(ly + ii) * Wi + lx - (SW - pw);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int jj = vec ? 4 * j + k : j;
            v[k] = zero_v;
            if ((vec || k == 0) && any && ii >= 0 && jj >= SW - pw) {
                const float r = (float)irow[jj];
                v[k] = normalise ? (r - mean) / stdv : r;
            }
        }
    };
    auto store_row = [&](int i, int j, const float (&v)[4]) {
        float* orow = ob + (int64_t)i * SW;
        if (vec) *reinterpret_cast<float4*>(orow + 4 * j) = make_float4(v[0], v[1], v[2], v[3]);
        else orow[j] = v[0];
    };
    const int gstep = gridDim.x;
    for (int i = blockIdx.x; i < SH; i += 2 * gstep) {
        const bool two = i + gstep < SH;
        for (int j = threadIdx.x; j < jw; j += blockDim.x) {
            float a[4], b2[4];
            load_row(i, j, a);
            if (two) load_row(i + gstep, j, b2);
            store_row(i, j, a);
            if (two) store_row(i + gstep, j, b2);
        }
    }
}
extern "C" int cwfa_extract_views(const void* image, int image_dtype, const int32_t* coords, float* out, int B, int Hi,
                                  int Wi, int L, int SH, int SW, float mean, float stdv, int normalise, void* stream) {
    if (B <= 0 || Hi <= 0 || Wi <= 0 || L <= 0 || SH <= 0 || SW <= 0 || (normalise && stdv == 0.f) || (int64_t)B * L > 65535 ||
        image_dtype < 0 || image_dtype > 2) {
        set_error("extract_views: bad arguments");
        return CWFA_EINVAL;
    }
    int gx = ceil_div(kNumSMs * 8, B * L);
    if (gx > SH) gx = SH;
    if (gx < 1) gx = 1;
    const int work = (SW & 3) == 0 ? SW / 4 : SW;              // items per view row (4 columns each when SW % 4 == 0)
    const int threads = work >= 256 ? 256 : (work >= 128 ? 128 : 64);
    if ((SW & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 15)) { set_error("extract_views: out must be 16-byte aligned"); return CWFA_EINVAL; }
    dim3 grid(gx, B * L);
    if (image_dtype == 2)
        extract_views_kernel<uint16_t><<<grid, threads, 0, (cudaStream_t)stream>>>((const uint16_t*)image, coords, out, Hi, Wi, L, SH, SW, mean, stdv, normalise);
    else if (image_dtype == 1)
        extract_views_kernel<__half><<<grid, threads, 0, (cudaStream_t)stream>>>((const __half*)image, coords, out, Hi, Wi, L, SH, SW, mean, stdv, normalise);
    else
        extract_views_kernel<float><<<grid, threads, 0, (cudaStream_t)stream>>>((const float*)image, coords, out, Hi, Wi, L, SH, SW, mean, stdv, normalise);
    return check_launch("extract_views");
}
