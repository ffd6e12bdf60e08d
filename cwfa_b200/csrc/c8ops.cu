// Memory-bound helpers on C8 half-precision tensors for the LRNN U-Net (unet.py:72-113):
// per-channel batch statistics, BatchNorm apply fused with the 2x2 max-pool, both single pass,
// 128-bit accesses (one 16-byte chunk = 8 channels of one pixel).
#include "common.cuh"
using namespace cwfa;

namespace {
template <bool BF16>
__device__ __forceinline__ void unpack8(const uint4& u, float (&v)[8]) {
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float2 f;
        if constexpr (BF16) f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[i]));
        else f = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
        v[2 * i] = f.x;
        v[2 * i + 1] = f.y;
    }
}
template <bool BF16>
__device__ __forceinline__ uint4 pack8(const float (&v)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        if constexpr (BF16) {
            __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
            w[i] = *reinterpret_cast<uint32_t*>(&h);
        } else {
            __half2 h = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
            w[i] = *reinterpret_cast<uint32_t*>(&h);
        }
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

constexpr int kC8StatBlocks = 32;    // blocks per chunk
constexpr int kC8StatBlocksMax = 256;  // the activation adjoints use up to this many blocks per chunk (few-channel tensors)

template <bool BF16>
__global__ void __launch_bounds__(256) c8_stats_kernel(const uint4* __restrict__ x, float* __restrict__ ws, int N,
                                                       int chunks, int64_t P) {
    const int ch = blockIdx.y;
    float s[8], q[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j] = q[j] = 0.f;
    auto acc = [&](const uint4& u) {
        float v[8];
        unpack8<BF16>(u, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) { s[j] += v[j]; q[j] = fmaf(v[j], v[j], q[j]); }
    };
    // plane-by-plane walk (no per-element index division); 4 independent 16-byte loads in flight per thread
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int n = 0; n < N; ++n) {
        const uint4* xp = x + ((int64_t)n * chunks + ch) * P;
        int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
        for (; i + 3 * stride < P; i += 4 * stride) {
            const uint4 u0 = __ldg(xp + i), u1 = __ldg(xp + i + stride), u2 = __ldg(xp + i + 2 * stride),
                        u3 = __ldg(xp + i + 3 * stride);
            acc(u0); acc(u1); acc(u2); acc(u3);
        }
        for (; i < P; i += stride) acc(__ldg(xp + i));
    }
    __shared__ float red[8][16];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        s[j] = warp_sum(s[j]);
        q[j] = warp_sum(q[j]);
    }
    if (lane == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) { red[w][j] = s[j]; red[w][8 + j] = q[j]; }
    }
    __syncthreads();
    if (threadIdx.x < 16) {
        float t = 0.f;
        for (int k = 0; k < 8; ++k) t += red[k][threadIdx.x];
        ws[((int64_t)ch * gridDim.x + blockIdx.x) * 16 + threadIdx.x] = t;
    }
}
__global__ void c8_stats_finalize_kernel(const float* __restrict__ ws, float* __restrict__ stats, int Cp, int nblocks) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= Cp) return;
    const int ch = c >> 3, j = c & 7;
    double s = 0.0, q = 0.0;
    for (int i = 0; i < nblocks; ++i) {
        s += (double)ws[((int64_t)ch * nblocks + i) * 16 + j];
        q += (double)ws[((int64_t)ch * nblocks + i) * 16 + 8 + j];
    }
    stats[c] = (float)s;
    stats[Cp + c] = (float)q;
}

// y = x*scale[c] + shift[c]; optionally also the 2x2 max-pooled tensor.  blockIdx.y = (sample, chunk): the 8 scales
// and shifts live in registers; blockIdx.x strides over (pooled) rows, threads over (pooled) columns -- no index
// divisions.  POOL: one thread per 2x2 pixel block.
template <bool BF16, bool POOL>
__global__ void __launch_bounds__(256) c8_bn_apply_kernel(const uint4* __restrict__ x, const float* __restrict__ scale,
                                                          const float* __restrict__ shift, uint4* __restrict__ y,
                                                          uint4* __restrict__ ypool, int chunks, int H, int W) {
    const int H2 = POOL ? H / 2 : H, W2 = POOL ? W / 2 : W;
    const int ch = blockIdx.y % chunks;
    float sc[8], sh[8];
    {
        const float4 a0 = __ldg(reinterpret_cast<const float4*>(scale + ch * 8)), a1 = __ldg(reinterpret_cast<const float4*>(scale + ch * 8 + 4));
        const float4 b0 = __ldg(reinterpret_cast<const float4*>(shift + ch * 8)), b1 = __ldg(reinterpret_cast<const float4*>(shift + ch * 8 + 4));
        sc[0] = a0.x; sc[1] = a0.y; sc[2] = a0.z; sc[3] = a0.w; sc[4] = a1.x; sc[5] = a1.y; sc[6] = a1.z; sc[7] = a1.w;
        sh[0] = b0.x; sh[1] = b0.y; sh[2] = b0.z; sh[3] = b0.w; sh[4] = b1.x; sh[5] = b1.y; sh[6] = b1.z; sh[7] = b1.w;
    }
    const int64_t base = (int64_t)blockIdx.y * H * W;             // blockIdx.y = n * chunks + ch
    const uint4* xp = x + base;
    uint4* yp = y + base;
    for (int h2 = blockIdx.x; h2 < H2; h2 += gridDim.x) {
        for (int w2 = threadIdx.x; w2 < W2; w2 += blockDim.x) {
            if constexpr (POOL) {
                const int o00 = (2 * h2) * W + 2 * w2;
                const uint4 u[4] = {__ldg(xp + o00), __ldg(xp + o00 + 1), __ldg(xp + o00 + W), __ldg(xp + o00 + W + 1)};
                float mx[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) mx[j] = -INFINITY;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    float v[8];
                    unpack8<BF16>(u[k], v);
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = fmaf(v[j], sc[j], sh[j]);
                    const uint4 pk = pack8<BF16>(v);
                    yp[o00 + (k >> 1) * W + (k & 1)] = pk;
                    float r[8];
                    unpack8<BF16>(pk, r);      // pool the ROUNDED values so pooled == max of what is stored
#pragma unroll
                    for (int j = 0; j < 8; ++j) mx[j] = fmaxf(mx[j], r[j]);
                }
                ypool[(int64_t)blockIdx.y * H2 * W2 + (int64_t)h2 * W2 + w2] = pack8<BF16>(mx);
            } else {
                const int o = h2 * W + w2;
                float v[8];
                unpack8<BF16>(__ldg(xp + o), v);
#pragma unroll
                for (int j = 0; j < 8; ++j) v[j] = fmaf(v[j], sc[j], sh[j]);
                yp[o] = pack8<BF16>(v);
            }
        }
    }
}
// out[n, d, y, x] = bias[d] + sum_{ky,kx} g[n, (d/8)*72 + (ky*3+kx)*8 + d%8, y+ky-1, x+kx-1]   (zero outside the image).
// A 3x3 convolution whose per-tap partial products were produced by ONE 1x1 tensor-core convolution (9x fewer
// shared-memory operand reads than the tap-by-tap form when Cout is tiny and Cin huge): this kernel is the col2im.
// blockIdx.y = (sample, depth chunk); blockIdx.x strides over rows; threads over columns; 9 x 16-byte loads per output.
template <bool BF16>
__global__ void __launch_bounds__(256) c8_col2im3x3_kernel(const uint4* __restrict__ g, const float* __restrict__ bias,
                                                           uint4* __restrict__ out, int dchunks, int gchunks, int gvalid, int H, int W) {
    const int dc = blockIdx.y % dchunks, n = blockIdx.y / dchunks;
    if (dc >= gvalid) {                              // channel-padding chunk of the output: zeros
        uint4* oz = out + (int64_t)blockIdx.y * H * W;
        for (int h = blockIdx.x; h < H; h += gridDim.x)
            for (int w = threadIdx.x; w < W; w += blockDim.x) oz[(int64_t)h * W + w] = make_uint4(0, 0, 0, 0);
        return;
    }
    float b[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) b[j] = bias ? __ldg(bias + dc * 8 + j) : 0.f;
    const int64_t plane = (int64_t)H * W;
    const uint4* gp = g + ((int64_t)n * gchunks + (int64_t)dc * 9) * plane;
    uint4* op = out + (int64_t)blockIdx.y * plane;
    for (int h = blockIdx.x; h < H; h += gridDim.x) {
        for (int w = threadIdx.x; w < W; w += blockDim.x) {
            float acc[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[j] = b[j];
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
                const int hh = h + ky - 1;
                if (hh < 0 || hh >= H) continue;
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) {
                    const int ww = w + kx - 1;
                    if (ww < 0 || ww >= W) continue;
                    float v[8];
                    unpack8<BF16>(__ldg(gp + (int64_t)(ky * 3 + kx) * plane + (int64_t)hh * W + ww), v);
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[j] += v[j];
                }
            }
            op[(int64_t)h * W + w] = pack8<BF16>(acc);
        }
    }
}
// LayerNorm([C,H,W]) on a C8 tensor (ConvNeXt of the LRNN, networks.py:486-503): statistics over all C*H*W elements of a
// sample (channel padding is zero and is not counted), then y = (x - mean) * rstd * w + b with the element-wise affine
// parameters pre-converted to the same C8 half layout (half the parameter traffic of the fp32 NCHW form).
constexpr int kC8LnBlocks = 296;
template <bool BF16>
__global__ void __launch_bounds__(256) c8_ln_stats_kernel(const uint4* __restrict__ x, float* __restrict__ ws, int64_t n16) {
    const uint4* xs = x + (int64_t)blockIdx.y * n16;
    float s = 0.f, q = 0.f;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n16; i += (int64_t)gridDim.x * blockDim.x) {
        float v[8];
        unpack8<BF16>(__ldg(xs + i), v);
#pragma unroll
        for (int j = 0; j < 8; ++j) { s += v[j]; q = fmaf(v[j], v[j], q); }
    }
    s = warp_sum(s);
    q = warp_sum(q);
    __shared__ float red[8][2];
    if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5][0] = s; red[threadIdx.x >> 5][1] = q; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float a = 0.f, b = 0.f;
        for (int k = 0; k < 8; ++k) { a += red[k][0]; b += red[k][1]; }
        ws[((int64_t)blockIdx.y * gridDim.x + blockIdx.x) * 2] = a;
        ws[((int64_t)blockIdx.y * gridDim.x + blockIdx.x) * 2 + 1] = b;
    }
}
template <bool BF16>
__global__ void __launch_bounds__(256) c8_ln_apply_kernel(const uint4* __restrict__ x, const uint4* __restrict__ gamma,
                                                          const uint4* __restrict__ beta, uint4* __restrict__ y,
                                                          const float* __restrict__ ws, int64_t n16, double count, float eps) {
    __shared__ float s_mean, s_rstd;
    if (threadIdx.x == 0) {
        double s = 0.0, q = 0.0;
        for (int i = 0; i < kC8LnBlocks; ++i) {                  // fixed order
            s += (double)ws[((int64_t)blockIdx.y * kC8LnBlocks + i) * 2];
            q += (double)ws[((int64_t)blockIdx.y * kC8LnBlocks + i) * 2 + 1];
        }
        const double mean = s / count;
        double var = q / count - mean * mean;
        if (var < 0.0) var = 0.0;
        s_mean = (float)mean;
        s_rstd = (float)(1.0 / sqrt(var + (double)eps));
    }
    __syncthreads();
    const float mean = s_mean, rstd = s_rstd;
    const uint4* xs = x + (int64_t)blockIdx.y * n16;
    uint4* ys = y + (int64_t)blockIdx.y * n16;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n16; i += (int64_t)gridDim.x * blockDim.x) {
        float v[8], g[8], b[8];
        unpack8<BF16>(__ldg(xs + i), v);
        unpack8<BF16>(__ldg(gamma + i), g);
        unpack8<BF16>(__ldg(beta + i), b);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = fmaf((v[j] - mean) * rstd, g[j], b[j]);     // padded channels: g = b = 0 -> 0
        ys[i] = pack8<BF16>(v);
    }
}
}  // namespace

extern "C" int cwfa_c8_layernorm_workspace_floats(int N) { return 2 * N * kC8LnBlocks; }

// x, y: C8 (N, Cp, H, W); gamma, beta: C8 (1, Cp, H, W) element-wise affine parameters (zero in the channel padding);
// C = true channel count (statistics are over C*H*W elements).  workspace >= cwfa_c8_layernorm_workspace_floats(N).
extern "C" int cwfa_c8_layernorm(const void* x, const void* gamma, const void* beta, void* y, float* workspace, int N, int C,
                                 int Cp, int64_t P, float eps, int is_bf16, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (N <= 0 || C <= 0 || Cp < C || (Cp % 8) || P <= 0 || !workspace) { set_error("c8_layernorm: bad shape"); return CWFA_EINVAL; }
    const int64_t n16 = (int64_t)(Cp / 8) * P;
    dim3 grid(kC8LnBlocks, N);
    const double count = (double)C * (double)P;
    if (is_bf16) {
        c8_ln_stats_kernel<true><<<grid, 256, 0, st>>>((const uint4*)x, workspace, n16);
        c8_ln_apply_kernel<true><<<grid, 256, 0, st>>>((const uint4*)x, (const uint4*)gamma, (const uint4*)beta, (uint4*)y, workspace, n16, count, eps);
    } else {
        c8_ln_stats_kernel<false><<<grid, 256, 0, st>>>((const uint4*)x, workspace, n16);
        c8_ln_apply_kernel<false><<<grid, 256, 0, st>>>((const uint4*)x, (const uint4*)gamma, (const uint4*)beta, (uint4*)y, workspace, n16, count, eps);
    }
    return check_launch("c8_layernorm");
}

extern "C" int cwfa_c8_col2im3x3(const void* g, const float* bias, void* out, int N, int Dp, int Gp, int H, int W,
                                 int is_bf16, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (N <= 0 || Dp <= 0 || (Dp % 8) || (Gp % 8) || Gp < 72 || H <= 0 || W <= 0 || (int64_t)N * (Dp / 8) > 65535) {
        set_error("c8_col2im3x3: bad shape (needs Gp >= 72, Dp %% 8 == 0)");
        return CWFA_EINVAL;
    }
    const int gvalid = Gp / 72 < Dp / 8 ? Gp / 72 : Dp / 8;      // depth chunks that have partial products; the rest is channel padding
    const int planes = N * (Dp / 8);
    int gx = ceil_div(kNumSMs * 8, planes);
    if (gx > H) gx = H;
    const int threads = W >= 256 ? 256 : (W >= 128 ? 128 : 64);
    dim3 grid(gx, planes);
    if (is_bf16) c8_col2im3x3_kernel<true><<<grid, threads, 0, st>>>((const uint4*)g, bias, (uint4*)out, Dp / 8, Gp / 8, gvalid, H, W);
    else c8_col2im3x3_kernel<false><<<grid, threads, 0, st>>>((const uint4*)g, bias, (uint4*)out, Dp / 8, Gp / 8, gvalid, H, W);
    return check_launch("c8_col2im3x3");
}

// PReLU on a C8 tensor and its adjoint (training path of the conditioning net's banded depth stencil: the 32 D-channel hidden
// tensor stays in the C8 half layout between the two tensor-core convolutions instead of making fp32 NCHW round trips).
template <bool BF16>
__global__ void __launch_bounds__(256) c8_prelu_kernel(const uint4* __restrict__ x, const float* __restrict__ slope,
                                                       uint4* __restrict__ y, int64_t n16) {
    const float a = __ldg(slope);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n16; i += stride) {
        float v[8];
        unpack8<BF16>(__ldg(x + i), v);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = v[j] >= 0.f ? v[j] : a * v[j];
        y[i] = pack8<BF16>(v);
    }
}
// g = dy * PReLU'(pre); per-channel sums s[c] = sum g (bias gradient of the producing conv), q[c] = sum dy * min(pre, 0)
// (slope gradient), in the workspace layout of c8_stats_kernel (finalised by c8_stats_finalize_kernel)
template <bool BF16, int MODE>
__global__ void __launch_bounds__(256) c8_prelu_bwd_kernel(const uint4* __restrict__ dy, const uint4* __restrict__ pre,
                                                           const float* __restrict__ slope, uint4* __restrict__ g,
                                                           float* __restrict__ ws, int N, int chunks, int64_t P) {
    const int ch = blockIdx.y;
    const float a = MODE == 0 ? __ldg(slope) : 0.f;
    float s[8], q[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j] = q[j] = 0.f;
    // MODE 0: PReLU'(pre) = pre > 0 ? 1 : a (torch's PReLU adjoint convention at pre = 0), q += dy * min(pre, 0).
    // MODE 1: ELU' from the OUTPUT y: y > 0 ? 1 : y + 1.
    auto adj = [&](float (&dv)[8], const float (&pv)[8]) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if constexpr (MODE == 0) {
                q[j] = fmaf(dv[j], pv[j] < 0.f ? pv[j] : 0.f, q[j]);
                dv[j] = pv[j] > 0.f ? dv[j] : a * dv[j];
            } else {
                dv[j] *= pv[j] > 0.f ? 1.f : pv[j] + 1.f;
            }
            s[j] += dv[j];
        }
    };
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int n = 0; n < N; ++n) {
        const int64_t base = ((int64_t)n * chunks + ch) * P;
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < P; i += 2 * stride) {
            const bool two = i + stride < P;
            const uint4 d0 = __ldg(dy + base + i), p0 = __ldg(pre + base + i);
            const uint4 d1 = two ? __ldg(dy + base + i + stride) : make_uint4(0, 0, 0, 0);
            const uint4 p1 = two ? __ldg(pre + base + i + stride) : make_uint4(0, 0, 0, 0);
            float dv[8], pv[8];
            unpack8<BF16>(d0, dv);
            unpack8<BF16>(p0, pv);
            adj(dv, pv);
            g[base + i] = pack8<BF16>(dv);
            if (two) {
                unpack8<BF16>(d1, dv);
                unpack8<BF16>(p1, pv);
                adj(dv, pv);
                g[base + i + stride] = pack8<BF16>(dv);
            }
        }
    }
    __shared__ float red[8][16];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        s[j] = warp_sum(s[j]);
        q[j] = warp_sum(q[j]);
    }
    if (lane == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) { red[w][j] = s[j]; red[w][8 + j] = q[j]; }
    }
    __syncthreads();
    if (threadIdx.x < 16) {
        float t = 0.f;
        for (int k = 0; k < 8; ++k) t += red[k][threadIdx.x];
        ws[((int64_t)ch * gridDim.x + blockIdx.x) * 16 + threadIdx.x] = t;
    }
}

extern "C" int cwfa_c8_prelu(const void* x, const float* slope, void* y, int N, int Cp, int64_t P, int is_bf16, void* stream) {
    if (!x || !slope || !y || N <= 0 || Cp <= 0 || (Cp % 8) || P <= 0) { set_error("c8_prelu: bad arguments"); return CWFA_EINVAL; }
    const int64_t n16 = (int64_t)N * (Cp / 8) * P;
    int blocks = (int)((n16 + 255) / 256);
    if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
    if (is_bf16) c8_prelu_kernel<true><<<blocks, 256, 0, (cudaStream_t)stream>>>((const uint4*)x, slope, (uint4*)y, n16);
    else c8_prelu_kernel<false><<<blocks, 256, 0, (cudaStream_t)stream>>>((const uint4*)x, slope, (uint4*)y, n16);
    return check_launch("c8_prelu");
}

static int c8_act_bwd(const void* dy, const void* v, const float* slope, void* g, float* stats, float* workspace, int N, int Cp,
                      int64_t P, int is_bf16, int elu, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (!dy || !v || (!elu && !slope) || !g || !stats || !workspace || N <= 0 || Cp <= 0 || (Cp % 8) || P <= 0 || Cp / 8 > 65535) {
        set_error("c8 activation adjoint: bad arguments");
        return CWFA_EINVAL;
    }
    // enough blocks for the whole GPU also at 8 chunks (64 channels: 32 blocks per chunk left 40 % of the SMs idle, 39 us per pass)
    int nblk = ceil_div(kNumSMs * 8, Cp / 8);
    nblk = nblk < kC8StatBlocks ? kC8StatBlocks : (nblk > kC8StatBlocksMax ? kC8StatBlocksMax : nblk);
    dim3 grid(nblk, Cp / 8);
    const uint4 *d4 = (const uint4*)dy, *v4 = (const uint4*)v;
    if (elu) {
        if (is_bf16) c8_prelu_bwd_kernel<true, 1><<<grid, 256, 0, st>>>(d4, v4, slope, (uint4*)g, workspace, N, Cp / 8, P);
        else c8_prelu_bwd_kernel<false, 1><<<grid, 256, 0, st>>>(d4, v4, slope, (uint4*)g, workspace, N, Cp / 8, P);
    } else {
        if (is_bf16) c8_prelu_bwd_kernel<true, 0><<<grid, 256, 0, st>>>(d4, v4, slope, (uint4*)g, workspace, N, Cp / 8, P);
        else c8_prelu_bwd_kernel<false, 0><<<grid, 256, 0, st>>>(d4, v4, slope, (uint4*)g, workspace, N, Cp / 8, P);
    }
    int rc = check_launch("c8_act_bwd");
    if (rc) return rc;
    c8_stats_finalize_kernel<<<ceil_div(Cp, 128), 128, 0, st>>>(workspace, stats, Cp, nblk);
    return check_launch("c8_act_bwd_finalize");
}
extern "C" int cwfa_c8_prelu_bwd(const void* dy, const void* pre, const float* slope, void* g, float* stats, float* workspace,
                                 int N, int Cp, int64_t P, int is_bf16, void* stream) {
    return c8_act_bwd(dy, pre, slope, g, stats, workspace, N, Cp, P, is_bf16, 0, stream);
}
extern "C" int cwfa_c8_elu_bwd(const void* dy, const void* y, void* g, float* stats, float* workspace, int N, int Cp, int64_t P,
                               int is_bf16, void* stream) {
    return c8_act_bwd(dy, y, nullptr, g, stats, workspace, N, Cp, P, is_bf16, 1, stream);
}

extern "C" int cwfa_c8_stats_workspace_floats(int Cp) { return (Cp / 8) * kC8StatBlocksMax * 16; }

extern "C" int cwfa_c8_channel_stats(const void* x, float* stats, float* workspace, int N, int Cp, int64_t P,
                                     int is_bf16, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (N <= 0 || Cp <= 0 || (Cp % 8) || P <= 0) { set_error("c8_channel_stats: bad shape"); return CWFA_EINVAL; }
    dim3 grid(kC8StatBlocks, Cp / 8);
    if (is_bf16) c8_stats_kernel<true><<<grid, 256, 0, st>>>((const uint4*)x, workspace, N, Cp / 8, P);
    else c8_stats_kernel<false><<<grid, 256, 0, st>>>((const uint4*)x, workspace, N, Cp / 8, P);
    int rc = check_launch("c8_stats");
    if (rc) return rc;
    c8_stats_finalize_kernel<<<ceil_div(Cp, 128), 128, 0, st>>>(workspace, stats, Cp, kC8StatBlocks);
    return check_launch("c8_stats_finalize");
}

// Batch statistics straight to the BatchNorm scale / shift: the fixed-order sum of the block partials and
// scale = gamma / sqrt(var + eps), shift = beta - mean * scale in ONE finalize launch (unet.py:100-107 in batch-statistics mode).
__global__ void c8_stats_bn_finalize_kernel(const float* __restrict__ ws, const float* __restrict__ gamma,
                                            const float* __restrict__ beta, float* __restrict__ scale,
                                            float* __restrict__ shift, int Cp, int nblocks, double count, float eps) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= Cp) return;
    const int ch = c >> 3, j = c & 7;
    double s = 0.0, q = 0.0;
    for (int i = 0; i < nblocks; ++i) {
        s += (double)ws[((int64_t)ch * nblocks + i) * 16 + j];
        q += (double)ws[((int64_t)ch * nblocks + i) * 16 + 8 + j];
    }
    s = (double)(float)s;                       // the same roundings as c8_stats_finalize_kernel + bn_finalize_kernel
    q = (double)(float)q;
    const double mean = s / count;
    double var = q / count - mean * mean;
    if (var < 0.0) var = 0.0;
    const double sc = (double)gamma[c] / sqrt(var + (double)eps);
    scale[c] = (float)sc;
    shift[c] = (float)((double)beta[c] - mean * sc);
}

extern "C" int cwfa_c8_bn_batch_scale_shift(const void* x, const float* gamma, const float* beta, float eps, float* scale,
                                            float* shift, float* workspace, int N, int Cp, int64_t P, int is_bf16,
                                            void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (N <= 0 || Cp <= 0 || (Cp % 8) || P <= 0 || !gamma || !beta || !scale || !shift || !workspace) {
        set_error("c8_bn_batch_scale_shift: bad arguments");
        return CWFA_EINVAL;
    }
    dim3 grid(kC8StatBlocks, Cp / 8);
    if (is_bf16) c8_stats_kernel<true><<<grid, 256, 0, st>>>((const uint4*)x, workspace, N, Cp / 8, P);
    else c8_stats_kernel<false><<<grid, 256, 0, st>>>((const uint4*)x, workspace, N, Cp / 8, P);
    int rc = check_launch("c8_stats");
    if (rc) return rc;
    c8_stats_bn_finalize_kernel<<<ceil_div(Cp, 128), 128, 0, st>>>(workspace, gamma, beta, scale, shift, Cp, kC8StatBlocks,
                                                                 (double)N * (double)P, eps);
    return check_launch("c8_stats_bn_finalize");
}

extern "C" int cwfa_c8_bn_apply(const void* x, const float* scale, const float* shift, void* y, void* ypool, int N,
                                int Cp, int H, int W, int is_bf16, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (N <= 0 || Cp <= 0 || (Cp % 8) || H <= 0 || W <= 0) { set_error("c8_bn_apply: bad shape"); return CWFA_EINVAL; }
    const bool pool = ypool != nullptr;
    if (pool && ((H & 1) || (W & 1))) { set_error("c8_bn_apply: pooling needs even H, W"); return CWFA_EINVAL; }
    if ((int64_t)H * W >= (1ll << 31) || (int64_t)N * (Cp / 8) > 65535) { set_error("c8_bn_apply: shape too large"); return CWFA_EINVAL; }
    if ((reinterpret_cast<uintptr_t>(scale) & 15) || (reinterpret_cast<uintptr_t>(shift) & 15)) { set_error("c8_bn_apply: scale/shift must be 16-byte aligned"); return CWFA_EINVAL; }
    const int planes = N * (Cp / 8);
    const int H2 = pool ? H / 2 : H, W2 = pool ? W / 2 : W;
    int gx = ceil_div(kNumSMs * 8, planes);                      // ~8 resident blocks per SM overall
    if (gx > H2) gx = H2;
    if (gx < 1) gx = 1;
    const int threads = W2 >= 256 ? 256 : (W2 >= 128 ? 128 : 64);
    dim3 grid(gx, planes);
    const uint4* xi = (const uint4*)x;
    uint4 *yo = (uint4*)y, *yp = (uint4*)ypool;
    if (is_bf16) {
        if (pool) c8_bn_apply_kernel<true, true><<<grid, threads, 0, st>>>(xi, scale, shift, yo, yp, Cp / 8, H, W);
        else c8_bn_apply_kernel<true, false><<<grid, threads, 0, st>>>(xi, scale, shift, yo, yp, Cp / 8, H, W);
    } else {
        if (pool) c8_bn_apply_kernel<false, true><<<grid, threads, 0, st>>>(xi, scale, shift, yo, yp, Cp / 8, H, W);
        else c8_bn_apply_kernel<false, false><<<grid, threads, 0, st>>>(xi, scale, shift, yo, yp, Cp / 8, H, W);
    }
    return check_launch("c8_bn_apply");
}
