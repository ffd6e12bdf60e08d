// Engine-side coupling path on the "F8" layout of the detail half: [N][ceil(ch/8)][H][W][8] fp32 (one pixel's 8-channel group
// = 32 contiguous bytes = two 128-bit accesses; channels beyond ch are zero padding).
//
//  * coupling_f8_kernel: the LAST 3x3 conv of a coupling sub-network (64 hidden channels -> [s | t], networks.py:635-638) on
//    tcgen05 with the affine coupling (FrEIA/modules/coupling_layers.py:490-500), the log-det / sum-of-squares partial sums
//    and a preceding ROW / COLUMN permutation (INN_utils.py:73-81, as a gather on x) in its epilogue.  Same persistent
//    structure as coupling_tc.cu (weights resident in shared memory, halo tiles through a TMA ring, accumulators double
//    buffered in TMEM, 16 epilogue warps, last-CTA finalize), but the epilogue is lean: its instruction count per (s, t) pair
//    was 60 in coupling_tc (27 of them integer / predicate / branch work of the per-channel NCHW gathers) and is ~27 here:
//      - x / y / external shift move as 128-bit vectors, one address computation per 8 channels, no per-channel predicates
//        (padding channels carry zero weights and bias: s = t = 0, y = x = 0);
//      - CHANNEL permutations never touch data: the engine keeps the detail half in the order it entered the flow and
//        permutes the OUTPUT CHANNELS of each packed conv instead (engine.py), so s, t arrive in storage order;
//      - the bias enters the accumulator through one extra K = 16 MMA (ones tile x [hi | lo] split of the fp32 bias);
//      - exp(+-s) = ex2(c * atan(a)) with the clamp constant, the sign and log2(e) folded into c; the log-det accumulates
//        atan values and is scaled once per tile.
//  * haar1d_f8 kernels: depth-wise Haar DWT / IDWT (INN_utils.py:142-161) + Split / Split^-1 (graph_topology.py:73-80) with the
//    detail half in F8: every access 128-bit, fully coalesced (4 pixels x 8 channel pairs per thread).
//  * nchw <-> F8 converters with an optional channel map (the flow's accumulated channel permutation, applied once at the
//    boundary: latent z in / out).
#include "tc_common.cuh"
using namespace cwfa;
using namespace cwfa::tcx;

namespace {
constexpr float INV_SQRT2 = 0.70710678118654752440f;
constexpr int kChunks = 8;                                   // 64 hidden channels = 8 chunks
constexpr int kTH = 16, kTW = 16, kBH = 18, kBW = 18;
constexpr uint32_t kA1Bytes = kChunks * kBH * kBW * 16;      // 41472
constexpr int kMaxBN = 96;
constexpr uint32_t kOffOnes = 2048;                          // A tile of the bias MMA: [2 chunks][128 rows][8], e0 = e1 = 1
constexpr uint32_t kOnesBytes = 2 * 128 * 16;
constexpr uint32_t kOffBias = kOffOnes + kOnesBytes;         // B tile of the bias MMA: [2 chunks][BN][8], e0 = hi, e1 = lo
constexpr uint32_t kBiasBytes = 2 * kMaxBN * 16;
constexpr uint32_t kOffW = kOffBias + kBiasBytes;            // weights (9*8*BN*16 bytes), then the A ring
constexpr int kMaxAStages = 4;
constexpr int kThreads = 576, kEpiThreads = 512;
constexpr int kMaxG = 3;                                     // 8-channel groups per epilogue thread (chp8 <= 48, 2 M-blocks, 4-way split)
constexpr int kSampleBatch = 4;                              // K-sample epilogue: samples whose x loads are issued together

struct F8Params {
    int N, H, W, tiles_x, tiles_y, num_tiles;
    int BN, chp8, axis, a_stages, in_chunk_off;
    uint32_t off_a;
    const uint8_t* w;            // packed [9][8][BN][8]
    const float* bias;           // BN floats or NULL
    const float* x;              // F8 or NULL (zeros, inverse only)
    float* y;                    // F8
    const float* t_ext;          // F8 external shift or NULL
    const int* perm;             // row (axis 2) / column (axis 3) gather indices or NULL
    float* ws;                   // [num_tiles][16][2]
    float kk, c2, tscale;        // kk = clamp * k_atan (log-det scale, signed per direction); c2 = +-kk * log2(e)
    float* logdet;
    float* sumsq;
    int* ticket;
    int accumulate;
    int samples;                 // MS kernels: latent samples per condition image (x / y row n * samples + k)
    float* map;                  // MAP kernels: F8 per-element NLL map, indexed by the element's coordinate at the level's input
    const int* map_row;          //   R_b: input row of the element this block writes at output row h (NULL = identity)
    const int* map_col;          //   C_b: the same for columns
    int map_mode;                //   kMapFirst: write without reading; kMapLast: add 0.5 y^2 (both: a level of one block)
};
constexpr int kMapFirst = 1, kMapLast = 2;

__device__ __forceinline__ float4 ldg128(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// MS: the K-sample inverse variant (engine posterior statistics): one tile's accumulator, i.e. one evaluation of s and t,
// serves the p.samples latent samples of its condition image.  MS = false is the frame path, unchanged.
// MAP: the forward frame path that also accumulates each element's NLL term into p.map (see cwfa_coupling_f8_map); y, the
// log-det and sum-of-squares partials are the MAP = false kernel's, instruction for instruction.
template <bool BF16, bool INV, bool EXT, bool MS = false, bool MAP = false>
__global__ void __launch_bounds__(kThreads, 1) coupling_f8_kernel(const __grid_constant__ CUtensorMap tmap, const F8Params p) {
    static_assert(!MAP || (!INV && !MS), "the NLL map is forward-only, one sample per condition image");
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const uint32_t s0 = smem_u32(smem);
    const uint32_t w_full = s0;
    auto a_full = [&](int b) { return s0 + 8u * (1 + b); };
    auto a_empty = [&](int b) { return s0 + 8u * (5 + b); };
    auto acc_full = [&](int b) { return s0 + 8u * (9 + b); };
    auto acc_empty = [&](int b) { return s0 + 8u * (11 + b); };
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 128);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        mbar_init(w_full, 1);
        for (int b = 0; b < kMaxAStages; ++b) {
            mbar_init(a_full(b), 1);
            mbar_init(a_empty(b), 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(acc_full(b), 1);
            mbar_init(acc_empty(b), kEpiThreads);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // ones tile + [hi | lo] bias tile of the bias MMA (generic-proxy writes, made visible to the tensor core below)
    for (int i = threadIdx.x; i < (int)(kOnesBytes + kBiasBytes) / 16; i += kThreads) {
        uint4 v = make_uint4(0, 0, 0, 0);
        const int ones_units = kOnesBytes / 16;
        if (i < 128) {
            v.x = pack2<BF16>(1.f, 1.f);                                  // chunk 0 of the ones tile: e0 = e1 = 1
        } else if (i >= ones_units && i < ones_units + p.BN) {            // chunk 0 of the bias tile, row n
            const int nn = i - ones_units;
            const float bv = p.bias ? __ldg(p.bias + nn) : 0.f;
            float hi;
            if constexpr (BF16) hi = __bfloat162float(__float2bfloat16_rn(bv));
            else hi = __half2float(__float2half_rn(bv));
            v.x = pack2<BF16>(hi, bv - hi);
        }
        *reinterpret_cast<uint4*>(smem + kOffOnes + (size_t)i * 16) = v;
    }
    fence_proxy_async();
    if (warp == 1) tmem_alloc(smem_u32(tmem_slot), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const int my_tiles = (p.num_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int tiles_per_img = p.tiles_x * p.tiles_y;
    const uint32_t plane = (uint32_t)p.H * (uint32_t)p.W;

    if (warp == 0) {
        if (lane == 0) {
            const uint32_t wbytes = 9u * kChunks * p.BN * 16u;
            mbar_expect_tx(w_full, wbytes);
            bulk_load(s0 + kOffW, p.w, wbytes, w_full);
            int sa = 0;
            uint32_t pa = 0;
            for (int i = 0; i < my_tiles; ++i) {
                const int t = blockIdx.x + i * gridDim.x;
                const int n = t / tiles_per_img, r = t % tiles_per_img;
                const int h0 = (r / p.tiles_x) * kTH, w0 = (r % p.tiles_x) * kTW;
                mbar_wait(a_empty(sa), pa ^ 1);
                mbar_expect_tx(a_full(sa), kA1Bytes);
                tma_load_4d(s0 + p.off_a + sa * kA1Bytes, &tmap, a_full(sa), (w0 - 1) * 8, h0 - 1, p.in_chunk_off, n);
                if (++sa == p.a_stages) { sa = 0; pa ^= 1; }
            }
        }
    } else if (warp == 1) {
        const uint32_t idesc = idesc_f16(p.BN, BF16 ? 1 : 0);
        constexpr uint32_t a_lbo = kBH * kBW * 16, a_sbo = kBW * 16;
        const uint32_t w_lbo = p.BN * 16, tap_units = (kChunks * p.BN * 16) >> 4;
        const uint32_t a_hi = desc_hi(a_sbo), w_hi = desc_hi(128);
        const uint32_t w_lo0 = desc_lo(s0 + kOffW, w_lbo);
        const uint32_t ones_lo = desc_lo(s0 + kOffOnes, 128 * 16), ones_hi = desc_hi(128);
        const uint32_t bias_lo = desc_lo(s0 + kOffBias, kMaxBN * 16);     // the bias tile is laid out with the fixed pitch kMaxBN
        const uint32_t leader = elect_one();
        mbar_wait(w_full, 0);
        int sa = 0;
        uint32_t pa = 0;
        for (int i = 0; i < my_tiles; ++i) {
            const int b = i & 1, ph = (i >> 1) & 1;
            mbar_wait(a_full(sa), pa);
            mbar_wait(acc_empty(b), ph ^ 1);
            tc_fence_after();
            if (leader) {
                const uint32_t a_base = s0 + p.off_a + sa * kA1Bytes;
#pragma unroll
                for (int mb = 0; mb < 2; ++mb)                                                // acc = bias
                    tc_mma_f16_split(tmem + b * 256 + mb * p.BN, ones_lo, ones_hi, bias_lo, w_hi, idesc, 0u);
#pragma unroll 1
                for (int tap = 0; tap < 9; ++tap) {
                    const int kh = tap / 3, kw = tap - kh * 3;
                    const uint32_t w_lo = w_lo0 + tap * tap_units;
                    const uint32_t a_lo0 = desc_lo(a_base + (uint32_t)((kh * kBW + kw) * 16), a_lbo);
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
                        for (int mb = 0; mb < 2; ++mb)
                            tc_mma_f16_split(tmem + b * 256 + mb * p.BN, a_lo0 + mb * 8 + kk * ((2 * a_lbo) >> 4), a_hi,
                                             w_lo + kk * ((2 * w_lbo) >> 4), w_hi, idesc, 1u);
                    }
                }
                tc_commit(a_empty(sa));
                tc_commit(acc_full(b));
            }
            __syncwarp();
            if (++sa == p.a_stages) { sa = 0; pa ^= 1; }
        }
    } else if constexpr (MS) {
        // ====================== K-sample epilogue (inverse): 16 warps, same lane / group map as below ======================
        // s, t (or the external shift) of each of the thread's groups are read once per tile; atan / ex2 run once; then every sample
        // k of the condition image gets y = (x_k - t) * e with the single-sample kernel's instruction sequence per element, so
        // sample k is bitwise what a single-sample launch on x_k gives.  One group at a time, x and the external shift loaded after
        // the accumulator wait: e, t of all three groups plus a sample batch's x do not fit 576 threads' registers unspilled.
        static_assert(INV, "the K-sample coupling is inverse-only");
        const int q = warp & 3;
        const int sub = (warp - 2) >> 2;
        const int m = q * 32 + lane;
        const int gpc = p.chp8 >> 3;
        const int ngroups = 2 * gpc;
        const uint32_t sstride = (uint32_t)gpc * plane * 8u;         // floats per sample (the launcher checks samples * sstride < 2^31)
        for (int i = 0; i < my_tiles; ++i) {
            const int b = i & 1, ph = (i >> 1) & 1;
            const int t = blockIdx.x + i * gridDim.x;
            const int n = t / tiles_per_img, rr = t % tiles_per_img;
            const int h0 = (rr / p.tiles_x) * kTH, w0 = (rr % p.tiles_x) * kTW;
            const int orow = h0 + (m >> 3);
            const bool row_ok = orow < p.H;
            const size_t ibase = (size_t)n * sstride;                   // condition image n (external shift)
            const size_t xbase = (size_t)n * p.samples * sstride;       // its sample 0
            uint32_t ooff[kMaxG], soff[kMaxG];
            bool okg[kMaxG];
#pragma unroll
            for (int k = 0; k < kMaxG; ++k) {
                const int g = sub + 4 * k;
                const int mb = g >= gpc ? 1 : 0, cg = g - (mb ? gpc : 0);
                const int ocol = w0 + mb * 8 + (m & 7);
                const bool ok = g < ngroups && row_ok && ocol < p.W;
                okg[k] = ok;
                int srow = orow, scol = ocol;
                if (ok && p.perm && p.axis == 2) srow = __ldg(p.perm + orow);
                if (ok && p.perm && p.axis == 3) scol = __ldg(p.perm + ocol);
                const uint32_t gbase = (uint32_t)cg * plane;
                ooff[k] = (gbase + (uint32_t)orow * (uint32_t)p.W + (uint32_t)ocol) * 8u;
                soff[k] = (gbase + (uint32_t)srow * (uint32_t)p.W + (uint32_t)scol) * 8u;
            }
            mbar_wait(acc_full(b), ph);
            tc_fence_after();
            float sum_a = 0.f;
#pragma unroll
            for (int k = 0; k < kMaxG; ++k) {
                const int g = sub + 4 * k;
                if (g < ngroups) {                          // warp-uniform
                    const int mb = g >= gpc ? 1 : 0, cg = g - (mb ? gpc : 0);
                    uint32_t rs[8], rt[8];
                    __syncwarp();
                    const uint32_t ta = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(b * 256 + mb * p.BN + (cg << 3));
                    tmem_ld8_nowait(ta, rs);
                    if constexpr (!EXT) tmem_ld8_nowait(ta + p.chp8, rt);
                    tmem_ld_wait();
                    float av[8], ev[8], tv[8];              // EXT: tv = the raw external shift (scaled in the fma below)
#pragma unroll
                    for (int j = 0; j < 8; ++j) av[j] = atan_fast(__uint_as_float(rs[j]));
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ev[j]) : "f"(p.c2 * av[j]));
                        if constexpr (!EXT) tv[j] = __uint_as_float(rt[j]);
                    }
                    if constexpr (EXT) {
                        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
                        const float4 t0 = okg[k] ? ldg128(p.t_ext + ibase + ooff[k]) : z4;
                        const float4 t1 = okg[k] ? ldg128(p.t_ext + ibase + ooff[k] + 4) : z4;
                        tv[0] = t0.x; tv[1] = t0.y; tv[2] = t0.z; tv[3] = t0.w;
                        tv[4] = t1.x; tv[5] = t1.y; tv[6] = t1.z; tv[7] = t1.w;
                    }
                    float ga = 0.f;
#pragma unroll
                    for (int j = 0; j < 8; ++j) ga += av[j];
                    if (okg[k]) {
                        sum_a += ga;
                        // the samples in batches of kSampleBatch: their x loads are in flight together
#pragma unroll 1
                        for (int s0 = 0; s0 < p.samples; s0 += kSampleBatch) {
                            float4 xv[kSampleBatch][2];
#pragma unroll
                            for (int u = 0; u < kSampleBatch; ++u) {
                                if (s0 + u < p.samples) {
                                    const float* xp = p.x + xbase + (size_t)(s0 + u) * sstride + soff[k];
                                    xv[u][0] = ldg128(xp);
                                    xv[u][1] = ldg128(xp + 4);
                                }
                            }
#pragma unroll
                            for (int u = 0; u < kSampleBatch; ++u) {
                                if (s0 + u < p.samples) {
                                    const float xs[8] = {xv[u][0].x, xv[u][0].y, xv[u][0].z, xv[u][0].w,
                                                         xv[u][1].x, xv[u][1].y, xv[u][1].z, xv[u][1].w};
                                    float yv[8];
#pragma unroll
                                    for (int j = 0; j < 8; ++j) {
                                        // as the single-sample kernel: (x - tscale * t_ext) is one FFMA there, (x - t) one FADD
                                        const float d = EXT ? __fmaf_rn(-p.tscale, tv[j], xs[j]) : xs[j] - tv[j];
                                        yv[j] = d * ev[j];
                                    }
                                    float* yp = p.y + xbase + (size_t)(s0 + u) * sstride + ooff[k];
                                    *reinterpret_cast<float4*>(yp) = make_float4(yv[0], yv[1], yv[2], yv[3]);
                                    *reinterpret_cast<float4*>(yp + 4) = make_float4(yv[4], yv[5], yv[6], yv[7]);
                                }
                            }
                        }
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(acc_empty(b));
            sum_a = warp_sum(sum_a);
            if (lane == 0) {
                float* w = p.ws + ((size_t)t * 16 + (warp - 2)) * 2;
                w[0] = p.kk * sum_a;
                w[1] = 0.f;                          // no sum of squares: the inverse direction does not use it
            }
        }
        if (p.ticket) __threadfence();
    } else {
        // ============================ epilogue: 16 warps ============================
        const int q = warp & 3;
        const int sub = (warp - 2) >> 2;             // 0..3
        const int m = q * 32 + lane;
        const int gpc = p.chp8 >> 3;                 // 8-channel groups of the detail half
        const int ngroups = 2 * gpc;                 // x 2 M-blocks
        const bool has_x = p.x != nullptr;
        for (int i = 0; i < my_tiles; ++i) {
            const int b = i & 1, ph = (i >> 1) & 1;
            const int t = blockIdx.x + i * gridDim.x;
            const int n = t / tiles_per_img, rr = t % tiles_per_img;
            const int h0 = (rr / p.tiles_x) * kTH, w0 = (rr % p.tiles_x) * kTW;
            const int orow = h0 + (m >> 3);
            const bool row_ok = orow < p.H;
            const size_t nbase = (size_t)n * gpc * plane * 8;            // first float of sample n (F8)
            // coupling inputs of all of this thread's groups BEFORE the accumulator is ready (128-bit loads)
            float4 xv[kMaxG][2], tx[kMaxG][2];
            uint32_t ooff[kMaxG];                    // in-sample float offset of the output group
            uint32_t moff[kMaxG];                    // MAP: in-sample float offset of the group's map entry (input coordinates)
            bool okg[kMaxG];
            int mrow = orow;
            if constexpr (MAP) {
                if (row_ok && p.map_row) mrow = __ldg(p.map_row + orow);
            }
#pragma unroll
            for (int k = 0; k < kMaxG; ++k) {
                const int g = sub + 4 * k;
                const int mb = g >= gpc ? 1 : 0, cg = g - (mb ? gpc : 0);
                const int ocol = w0 + mb * 8 + (m & 7);
                const bool ok = g < ngroups && row_ok && ocol < p.W;
                okg[k] = ok;
                int srow = orow, scol = ocol;
                if (ok && p.perm && p.axis == 2) srow = __ldg(p.perm + orow);
                if (ok && p.perm && p.axis == 3) scol = __ldg(p.perm + ocol);
                const uint32_t gbase = (uint32_t)cg * plane;
                ooff[k] = (gbase + (uint32_t)orow * (uint32_t)p.W + (uint32_t)ocol) * 8u;
                const uint32_t soff = (gbase + (uint32_t)srow * (uint32_t)p.W + (uint32_t)scol) * 8u;
                if constexpr (MAP) {
                    const int mcol = (ok && p.map_col) ? __ldg(p.map_col + ocol) : ocol;
                    moff[k] = (gbase + (uint32_t)mrow * (uint32_t)p.W + (uint32_t)mcol) * 8u;
                }
                const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (ok && has_x) {
                    xv[k][0] = ldg128(p.x + nbase + soff);
                    xv[k][1] = ldg128(p.x + nbase + soff + 4);
                } else {
                    xv[k][0] = z4; xv[k][1] = z4;
                }
                if constexpr (EXT) {
                    if (ok) {
                        tx[k][0] = ldg128(p.t_ext + nbase + ooff[k]);
                        tx[k][1] = ldg128(p.t_ext + nbase + ooff[k] + 4);
                    } else {
                        tx[k][0] = z4; tx[k][1] = z4;
                    }
                }
            }
            // MAP: the running sums, one group ahead (those of all groups at once would not fit the register budget): group 0's
            // before the accumulator wait, group k + 1's when group k starts.  EXT loads each group's when it starts: one group
            // ahead spills there, and its block (the one with the external shift) is a level's first, which reads nothing.
            float4 mnext[2];
            auto map_load = [&](int k, float4* dst) {
                const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
                const bool rd = okg[k] && !(p.map_mode & kMapFirst);
                dst[0] = rd ? ldg128(p.map + nbase + moff[k]) : z4;
                dst[1] = rd ? ldg128(p.map + nbase + moff[k] + 4) : z4;
            };
            if constexpr (MAP && !EXT) map_load(0, mnext);
            mbar_wait(acc_full(b), ph);
            tc_fence_after();
            float sum_a = 0.f, sum_q = 0.f;
#pragma unroll
            for (int k = 0; k < kMaxG; ++k) {
                const int g = sub + 4 * k;
                if (g < ngroups) {                          // warp-uniform
                    const int mb = g >= gpc ? 1 : 0, cg = g - (mb ? gpc : 0);
                    float4 m4[2];
                    if constexpr (MAP && EXT) {
                        map_load(k, m4);
                    } else if constexpr (MAP) {
                        m4[0] = mnext[0];
                        m4[1] = mnext[1];
                        if (k + 1 < kMaxG && g + 4 < ngroups) map_load(k + 1, mnext);
                    }
                    uint32_t rs[8], rt[8];
                    __syncwarp();
                    const uint32_t ta = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(b * 256 + mb * p.BN + (cg << 3));
                    tmem_ld8_nowait(ta, rs);
                    if constexpr (!EXT) tmem_ld8_nowait(ta + p.chp8, rt);
                    tmem_ld_wait();
                    const float xs[8] = {xv[k][0].x, xv[k][0].y, xv[k][0].z, xv[k][0].w, xv[k][1].x, xv[k][1].y, xv[k][1].z, xv[k][1].w};
                    float te[8];
                    if constexpr (EXT) {
                        te[0] = tx[k][0].x; te[1] = tx[k][0].y; te[2] = tx[k][0].z; te[3] = tx[k][0].w;
                        te[4] = tx[k][1].x; te[5] = tx[k][1].y; te[6] = tx[k][1].z; te[7] = tx[k][1].w;
                    }
                    float yv[8], av[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) av[j] = atan_fast(__uint_as_float(rs[j]));
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        float tv;
                        if constexpr (EXT) {
                            tv = p.tscale * te[j];
                        } else {
                            tv = __uint_as_float(rt[j]);
                        }
                        float e;
                        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(p.c2 * av[j]));
                        if constexpr (INV) yv[j] = (xs[j] - tv) * e;
                        else yv[j] = fmaf(e, xs[j], tv);
                    }
                    float ga = 0.f, gq = 0.f;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        ga += av[j];
                        gq = fmaf(yv[j], yv[j], gq);
                    }
                    if (okg[k]) {
                        float* yp = p.y + nbase + ooff[k];
                        *reinterpret_cast<float4*>(yp) = make_float4(yv[0], yv[1], yv[2], yv[3]);
                        *reinterpret_cast<float4*>(yp + 4) = make_float4(yv[4], yv[5], yv[6], yv[7]);
                        sum_a += ga;
                        sum_q += gq;
                        if constexpr (MAP) {
                            // this block's term -s = -kk * atan(a_s) (the log-det's av, kk); the last block adds 0.5 y^2
                            float mv[8] = {m4[0].x, m4[0].y, m4[0].z, m4[0].w, m4[1].x, m4[1].y, m4[1].z, m4[1].w};
#pragma unroll
                            for (int j = 0; j < 8; ++j) mv[j] = fmaf(-p.kk, av[j], mv[j]);
                            if (p.map_mode & kMapLast) {
#pragma unroll
                                for (int j = 0; j < 8; ++j) mv[j] = fmaf(0.5f * yv[j], yv[j], mv[j]);
                            }
                            float* mp = p.map + nbase + moff[k];
                            *reinterpret_cast<float4*>(mp) = make_float4(mv[0], mv[1], mv[2], mv[3]);
                            *reinterpret_cast<float4*>(mp + 4) = make_float4(mv[4], mv[5], mv[6], mv[7]);
                        }
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(acc_empty(b));
            sum_a = warp_sum(sum_a);
            sum_q = warp_sum(sum_q);
            if (lane == 0) {
                float* w = p.ws + ((size_t)t * 16 + (warp - 2)) * 2;
                w[0] = p.kk * sum_a;                 // kk carries the direction's sign
                w[1] = sum_q;
            }
        }
        if (p.ticket) __threadfence();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem, 512);
    }
    if (p.ticket == nullptr) return;
    // ---- in-kernel finalize (as in coupling_tc.cu): the last CTA sums all partials of every sample in a fixed order
    volatile int* s_last = reinterpret_cast<volatile int*>(smem + 132);
    double* s_red = reinterpret_cast<double*>(smem + 256);          // [16 warps][2]
    if (threadIdx.x == 0) *s_last = (atomicAdd(p.ticket, 1) == (int)gridDim.x - 1) ? 1 : 0;
    __syncthreads();
    if (!*s_last) return;
    __threadfence();
    const int per_img = tiles_per_img * 16;
    constexpr int kRed = 512;
    for (int n = 0; n < p.N; ++n) {
        double s = 0.0, qq = 0.0;
        const float2* src = reinterpret_cast<const float2*>(p.ws) + (size_t)n * per_img;
        if (threadIdx.x < kRed) {
            for (int i = threadIdx.x; i < per_img; i += kRed) {
                const float2 v = __ldcg(src + i);
                s += (double)v.x;
                qq += (double)v.y;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                s += __shfl_xor_sync(0xffffffffu, s, o);
                qq += __shfl_xor_sync(0xffffffffu, qq, o);
            }
            if (lane == 0) { s_red[warp * 2] = s; s_red[warp * 2 + 1] = qq; }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            double a = 0.0, bsum = 0.0;
            for (int k = 0; k < kRed / 32; ++k) { a += s_red[k * 2]; bsum += s_red[k * 2 + 1]; }
            p.logdet[n] = (p.accumulate ? p.logdet[n] : 0.f) + (float)a;
            if (p.sumsq) p.sumsq[n] = (float)bsum;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) *p.ticket = 0;
}

// ------------------------------------------------------------------------------------------ Haar on the F8 detail half
// One thread = 4 consecutive pixels x one 8-channel group of the detail half (= 8 channel PAIRS of the full tensor):
// NCHW side: 16 (x) / 8 (lo) float4 accesses, each coalesced over the warp; F8 side: 4 pixels x 32 B = 128 contiguous bytes.
template <bool INV>
__global__ void __launch_bounds__(256) haar1d_f8_kernel(const float* __restrict__ a, const float* __restrict__ hi_in,
                                                        float* __restrict__ o1, float* __restrict__ hi_out, int B, int h, int64_t P) {
    // fwd: a = x (B,2h,P) -> o1 = lo (B,h,P), hi_out F8.   inv: a = lo, hi_in F8 -> o1 = x.
    const int G = (h + 7) >> 3;
    const int64_t P4 = P >> 2;
    const int64_t total = (int64_t)B * G * P4;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t p4 = idx % P4;
        const int64_t r = idx / P4;
        const int g = (int)(r % G);
        const int b = (int)(r / G);
        const int64_t pix = p4 * 4;
        float4 hv[4][2];                                   // [pixel][half of the group]
        const int64_t f8o = (((int64_t)b * G + g) * P + pix) * 8;
        if constexpr (INV) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                hv[k][0] = __ldg(reinterpret_cast<const float4*>(hi_in + f8o + k * 8));
                hv[k][1] = __ldg(reinterpret_cast<const float4*>(hi_in + f8o + k * 8 + 4));
            }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int i = g * 8 + j;                       // channel of lo / hi
            float hj[4];                                   // hi of channel i at the 4 pixels
            if (i < h) {
                if constexpr (!INV) {
                    const int64_t xo = ((int64_t)b * 2 * h + 2 * i) * P + pix;
                    const float4 e = __ldg(reinterpret_cast<const float4*>(a + xo));
                    const float4 o = __ldg(reinterpret_cast<const float4*>(a + xo + P));
                    float4 l;
                    l.x = (e.x + o.x) * INV_SQRT2; hj[0] = (e.x - o.x) * INV_SQRT2;
                    l.y = (e.y + o.y) * INV_SQRT2; hj[1] = (e.y - o.y) * INV_SQRT2;
                    l.z = (e.z + o.z) * INV_SQRT2; hj[2] = (e.z - o.z) * INV_SQRT2;
                    l.w = (e.w + o.w) * INV_SQRT2; hj[3] = (e.w - o.w) * INV_SQRT2;
                    *reinterpret_cast<float4*>(o1 + ((int64_t)b * h + i) * P + pix) = l;
                } else {
                    const float4 l = __ldg(reinterpret_cast<const float4*>(a + ((int64_t)b * h + i) * P + pix));
#pragma unroll
                    for (int k = 0; k < 4; ++k) hj[k] = reinterpret_cast<const float*>(&hv[k][j >> 2])[j & 3];
                    float4 e, o;
                    e.x = (l.x + hj[0]) * INV_SQRT2; o.x = (l.x - hj[0]) * INV_SQRT2;
                    e.y = (l.y + hj[1]) * INV_SQRT2; o.y = (l.y - hj[1]) * INV_SQRT2;
                    e.z = (l.z + hj[2]) * INV_SQRT2; o.z = (l.z - hj[2]) * INV_SQRT2;
                    e.w = (l.w + hj[3]) * INV_SQRT2; o.w = (l.w - hj[3]) * INV_SQRT2;
                    const int64_t xo = ((int64_t)b * 2 * h + 2 * i) * P + pix;
                    *reinterpret_cast<float4*>(o1 + xo) = e;
                    *reinterpret_cast<float4*>(o1 + xo + P) = o;
                }
            } else {
                hj[0] = hj[1] = hj[2] = hj[3] = 0.f;       // channel padding of the F8 group
            }
            if constexpr (!INV) {
#pragma unroll
                for (int k = 0; k < 4; ++k) reinterpret_cast<float*>(&hv[k][j >> 2])[j & 3] = hj[k];
            }
        }
        if constexpr (!INV) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                *reinterpret_cast<float4*>(hi_out + f8o + k * 8) = hv[k][0];
                *reinterpret_cast<float4*>(hi_out + f8o + k * 8 + 4) = hv[k][1];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------ posterior statistics
// Split^-1 + IDWT of K latent samples fused with their per-voxel mean and unbiased standard deviation: the K merged volumes
// exist only in registers.  Sample k: lo row k (or row 0 for every k: lo_shared) and hi row k, hi in F8 (HI_F8) or NCHW.
// One thread = VEC pixels x 4 channels of lo / hi (= 8 output channels); the two lanes of a pair hold the two halves of one
// F8 group, so a warp's 128-bit F8 loads cover whole 32-byte pixel groups and its NCHW accesses are 256-byte runs.
// Welford's update (mean, M2) per output: stable when the spread is many orders below the mean, and M2 stays exactly 0 when
// every sample gives the same value.  The merged values are the haar1d kernels' (l +- h) * INV_SQRT2, bit for bit.
template <bool HI_F8, int VEC>
__global__ void __launch_bounds__(256) haar1d_inv_stats_kernel(const float* __restrict__ lo, const float* __restrict__ hi,
                                                               float* __restrict__ mean, float* __restrict__ stdev, int K,
                                                               int lo_shared, int h, int64_t P) {
    const int G = (h + 7) >> 3;
    const int64_t Pv = P / VEC;
    const int64_t total = (int64_t)2 * G * Pv;
    const int64_t lo_row = lo_shared ? 0 : (int64_t)h * P;
    const int64_t hi_row = HI_F8 ? (int64_t)G * P * 8 : (int64_t)h * P;
    const float inv_km1 = 1.f / (float)(K - 1);
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int half = (int)(idx & 1);
        const int64_t r = idx >> 1;
        const int64_t pix = (r % Pv) * VEC;
        const int g = (int)(r / Pv);
        const int c0 = g * 8 + half * 4;                   // first lo / hi channel of this thread
        float mu[4][2][VEC], m2[4][2][VEC];                // [channel][even / odd output][pixel]
        float lv[4][VEC];
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int v = 0; v < VEC; ++v) { mu[j][0][v] = mu[j][1][v] = m2[j][0][v] = m2[j][1][v] = 0.f; lv[j][v] = 0.f; }
#pragma unroll 1
        for (int k = 0; k < K; ++k) {
            if (k == 0 || !lo_shared) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (c0 + j < h) {
                        const float* lp = lo + (int64_t)k * lo_row + (int64_t)(c0 + j) * P + pix;
                        if constexpr (VEC == 4) {
                            const float4 l4 = __ldg(reinterpret_cast<const float4*>(lp));
                            lv[j][0] = l4.x; lv[j][1] = l4.y; lv[j][2] = l4.z; lv[j][3] = l4.w;
                        } else {
                            lv[j][0] = __ldg(lp);
                        }
                    }
                }
            }
            float hv[4][VEC];
            if constexpr (HI_F8) {
#pragma unroll
                for (int v = 0; v < VEC; ++v) {
                    const float4 h4 = __ldg(reinterpret_cast<const float4*>(hi + (int64_t)k * hi_row + (((int64_t)g * P + pix + v) * 8) + half * 4));
                    hv[0][v] = h4.x; hv[1][v] = h4.y; hv[2][v] = h4.z; hv[3][v] = h4.w;
                }
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (c0 + j < h) {
                        const float* hp = hi + (int64_t)k * hi_row + (int64_t)(c0 + j) * P + pix;
                        if constexpr (VEC == 4) {
                            const float4 h4 = __ldg(reinterpret_cast<const float4*>(hp));
                            hv[j][0] = h4.x; hv[j][1] = h4.y; hv[j][2] = h4.z; hv[j][3] = h4.w;
                        } else {
                            hv[j][0] = __ldg(hp);
                        }
                    } else {
#pragma unroll
                        for (int v = 0; v < VEC; ++v) hv[j][v] = 0.f;
                    }
                }
            }
            const float rk = 1.f / (float)(k + 1);
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int v = 0; v < VEC; ++v) {
                    // __fmul_rn: the merged value is rounded once, as the merge kernels store it; a product contracted into
                    // the subtractions below would leave its rounding residual in M2 (std != 0 for identical samples)
                    const float x2[2] = {__fmul_rn(lv[j][v] + hv[j][v], INV_SQRT2), __fmul_rn(lv[j][v] - hv[j][v], INV_SQRT2)};
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const float d = x2[e] - mu[j][e][v];
                        mu[j][e][v] = fmaf(d, rk, mu[j][e][v]);
                        m2[j][e][v] = fmaf(d, x2[e] - mu[j][e][v], m2[j][e][v]);
                    }
                }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (c0 + j < h) {
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int64_t o = (int64_t)(2 * (c0 + j) + e) * P + pix;
                    float sd[VEC];
#pragma unroll
                    for (int v = 0; v < VEC; ++v) sd[v] = sqrtf(fmaxf(m2[j][e][v], 0.f) * inv_km1);
                    if constexpr (VEC == 4) {
                        *reinterpret_cast<float4*>(mean + o) = make_float4(mu[j][e][0], mu[j][e][1], mu[j][e][2], mu[j][e][3]);
                        *reinterpret_cast<float4*>(stdev + o) = make_float4(sd[0], sd[1], sd[2], sd[3]);
                    } else {
                        mean[o] = mu[j][e][0];
                        stdev[o] = sd[0];
                    }
                }
            }
        }
    }
}

// NCHW <-> F8 with an optional channel map: F8 slot j holds NCHW channel map[j] (to_f8) / NCHW channel c reads F8 slot map[c]
// (to_nchw).  map == NULL: identity.  4 pixels per thread (128-bit NCHW accesses).
template <bool TO_F8>
__global__ void __launch_bounds__(256) f8_convert_kernel(const float* __restrict__ src, float* __restrict__ dst, const int* __restrict__ map,
                                                         int B, int C, int64_t P) {
    const int G = (C + 7) >> 3;
    const int64_t P4 = P >> 2;
    const int64_t total = (int64_t)B * G * P4;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t p4 = idx % P4;
        const int64_t r = idx / P4;
        const int g = (int)(r % G);
        const int b = (int)(r / G);
        const int64_t pix = p4 * 4;
        if constexpr (TO_F8) {
            float v[4][8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int slot = g * 8 + j;
                float4 x4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (slot < C) {
                    const int c = map ? __ldg(map + slot) : slot;
                    x4 = __ldg(reinterpret_cast<const float4*>(src + ((int64_t)b * C + c) * P + pix));
                }
                v[0][j] = x4.x; v[1][j] = x4.y; v[2][j] = x4.z; v[3][j] = x4.w;
            }
            float* o = dst + (((int64_t)b * G + g) * P + pix) * 8;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                *reinterpret_cast<float4*>(o + k * 8) = make_float4(v[k][0], v[k][1], v[k][2], v[k][3]);
                *reinterpret_cast<float4*>(o + k * 8 + 4) = make_float4(v[k][4], v[k][5], v[k][6], v[k][7]);
            }
        } else {
            // output channels c = g*8 + j read F8 slot map[c] (any group): scalar 4-byte reads of 4 pixels, 128-bit NCHW store
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int c = g * 8 + j;
                if (c < C) {
                    const int slot = map ? __ldg(map + c) : c;
                    const float* s = src + (((int64_t)b * G + (slot >> 3)) * P + pix) * 8 + (slot & 7);
                    *reinterpret_cast<float4*>(dst + ((int64_t)b * C + c) * P + pix) = make_float4(__ldg(s), __ldg(s + 8), __ldg(s + 16), __ldg(s + 24));
                }
            }
        }
    }
}

int grid_for(int64_t total) {
    int64_t blocks = (total + 255) / 256;
    const int64_t maxb = (int64_t)kNumSMs * 16;
    if (blocks > maxb) blocks = maxb;
    return (int)(blocks < 1 ? 1 : blocks);
}
}  // namespace

// ---- C ABI ---------------------------------------------------------------------------------------------------------
extern "C" int cwfa_haar1d_fwd_f8(const float* x, float* lo, float* hi_f8, int B, int C, int64_t P, void* stream) {
    if (B <= 0 || C <= 0 || (C & 1) || P <= 0 || (P & 3) || !aligned16(x) || !aligned16(lo) || !aligned16(hi_f8)) {
        set_error("haar1d_fwd_f8: needs even C, P %% 4 == 0 and 16-byte aligned pointers");
        return CWFA_EINVAL;
    }
    const int h = C / 2;
    haar1d_f8_kernel<false><<<grid_for((int64_t)B * ((h + 7) / 8) * (P / 4)), 256, 0, (cudaStream_t)stream>>>(x, nullptr, lo, hi_f8, B, h, P);
    return check_launch("haar1d_fwd_f8");
}
extern "C" int cwfa_haar1d_inv_f8(const float* lo, const float* hi_f8, float* x, int B, int C, int64_t P, void* stream) {
    if (B <= 0 || C <= 0 || (C & 1) || P <= 0 || (P & 3) || !aligned16(x) || !aligned16(lo) || !aligned16(hi_f8)) {
        set_error("haar1d_inv_f8: needs even C, P %% 4 == 0 and 16-byte aligned pointers");
        return CWFA_EINVAL;
    }
    const int h = C / 2;
    haar1d_f8_kernel<true><<<grid_for((int64_t)B * ((h + 7) / 8) * (P / 4)), 256, 0, (cudaStream_t)stream>>>(lo, hi_f8, x, nullptr, B, h, P);
    return check_launch("haar1d_inv_f8");
}
// Posterior statistics of the last merge: see haar1d_inv_stats_kernel.  lo: K rows (lo_shared = 0) or one row for all samples;
// hi: K rows, F8 (hi_f8 = 1) or NCHW; mean / std: one (C, P) volume each.  F8 needs P % 4 == 0 and 16-byte aligned pointers;
// NCHW uses 128-bit accesses when P % 4 == 0 and they are aligned, scalar ones otherwise.
extern "C" int cwfa_haar1d_inv_stats(const float* lo, int lo_shared, const float* hi, int hi_f8, float* mean, float* stdev, int K, int C,
                                     int64_t P, void* stream) {
    const bool vec = (P & 3) == 0 && aligned16(lo) && aligned16(hi) && aligned16(mean) && aligned16(stdev);
    if (K < 2 || C <= 0 || (C & 1) || P <= 0 || !lo || !hi || !mean || !stdev || (hi_f8 && !vec)) {
        set_error("haar1d_inv_stats: needs K >= 2 samples, even C, and for an F8 detail half P %% 4 == 0 and 16-byte aligned pointers");
        return CWFA_EINVAL;
    }
    const int h = C / 2;
    const int64_t work = (int64_t)2 * ((h + 7) / 8) * (vec ? P / 4 : P);
    const int grid = grid_for(work);
    cudaStream_t st = (cudaStream_t)stream;
    if (hi_f8) haar1d_inv_stats_kernel<true, 4><<<grid, 256, 0, st>>>(lo, hi, mean, stdev, K, lo_shared, h, P);
    else if (vec) haar1d_inv_stats_kernel<false, 4><<<grid, 256, 0, st>>>(lo, hi, mean, stdev, K, lo_shared, h, P);
    else haar1d_inv_stats_kernel<false, 1><<<grid, 256, 0, st>>>(lo, hi, mean, stdev, K, lo_shared, h, P);
    return check_launch("haar1d_inv_stats");
}
extern "C" int cwfa_nchw_to_f8(const float* x, const int32_t* map, float* y_f8, int B, int C, int64_t P, void* stream) {
    if (B <= 0 || C <= 0 || P <= 0 || (P & 3) || !aligned16(x) || !aligned16(y_f8)) { set_error("nchw_to_f8: bad arguments (P %% 4 == 0, aligned pointers)"); return CWFA_EINVAL; }
    f8_convert_kernel<true><<<grid_for((int64_t)B * ((C + 7) / 8) * (P / 4)), 256, 0, (cudaStream_t)stream>>>(x, y_f8, map, B, C, P);
    return check_launch("nchw_to_f8");
}
extern "C" int cwfa_f8_to_nchw(const float* x_f8, const int32_t* map, float* y, int B, int C, int64_t P, void* stream) {
    if (B <= 0 || C <= 0 || P <= 0 || (P & 3) || !aligned16(x_f8) || !aligned16(y)) { set_error("f8_to_nchw: bad arguments (P %% 4 == 0, aligned pointers)"); return CWFA_EINVAL; }
    f8_convert_kernel<false><<<grid_for((int64_t)B * ((C + 7) / 8) * (P / 4)), 256, 0, (cudaStream_t)stream>>>(x_f8, y, map, B, C, P);
    return check_launch("f8_to_nchw");
}

// Shared launcher of cwfa_coupling_f8 (samples == 1), cwfa_coupling_f8_samples and cwfa_coupling_f8_map (nll_map != NULL).
static int coupling_f8_launch(const char* name, const void* b_c8, const void* w_packed, const float* bias, int N, int samples, int H,
                              int W, int BN, int chp8, const float* cx, float* cy, const float* ct, float t_scale, const int32_t* perm,
                              int perm_axis, float clamp, float k_atan, int inverse, float* workspace, float* logdet, float* sumsq,
                              int accumulate, int32_t* ticket, int in_total_chunks, int in_chunk_off, int is_bf16, void* stream,
                              float* nll_map = nullptr, const int32_t* row_src = nullptr, const int32_t* col_src = nullptr,
                              int map_mode = 0) {
    const bool ms = samples > 1;
    const bool map = nll_map != nullptr;
    if (samples < 1 || (ms && (!inverse || !cx || sumsq || (int64_t)samples * chp8 * H * W >= (1ll << 31)))) {
        set_error("%s: samples must be >= 1; with samples > 1 the coupling is inverse-only, needs x, has no sum of squares, and "
                  "samples * chp8 * H * W must stay below 2^31", name);
        return CWFA_EINVAL;
    }
    if (N <= 0 || H <= 0 || W <= 0 || (int64_t)chp8 * H * W >= (1ll << 31) || !cy || !workspace || chp8 <= 0 || chp8 > 48 || (chp8 & 7) ||
        BN > kMaxBN || (BN % 16) || (ct ? BN < chp8 : BN < 2 * chp8) || (perm && perm_axis != 2 && perm_axis != 3) || (!cx && !inverse) ||
        (ticket && !logdet) || in_chunk_off < 0 || in_chunk_off + kChunks > in_total_chunks) {
        set_error("%s: unsupported arguments (needs 64 -> BN <= 96 in one n-block, chp8 <= 48 multiple of 8, row / column perms only)", name);
        return CWFA_EINVAL;
    }
    if ((reinterpret_cast<uintptr_t>(b_c8) & 15) || (reinterpret_cast<uintptr_t>(w_packed) & 15) || !aligned16(cy) || (cx && !aligned16(cx)) ||
        (ct && !aligned16(ct)) || (map && !aligned16(nll_map))) {
        set_error("%s: pointers must be 16-byte aligned", name);
        return CWFA_EINVAL;
    }
    F8Params p{};
    p.N = N; p.H = H; p.W = W;
    p.tiles_x = ceil_div(W, kTW); p.tiles_y = ceil_div(H, kTH);
    const int64_t nt = (int64_t)p.tiles_x * p.tiles_y * N;
    if (nt > 0x7fffffff) { set_error("%s: too many tiles", name); return CWFA_EINVAL; }
    p.num_tiles = (int)nt;
    p.BN = BN; p.chp8 = chp8; p.axis = perm ? perm_axis : 0;
    p.w = (const uint8_t*)w_packed; p.bias = bias; p.x = cx; p.y = cy; p.t_ext = ct; p.perm = perm; p.ws = workspace;
    const float kk = clamp * k_atan;
    p.kk = inverse ? -kk : kk;
    p.c2 = (inverse ? -kk : kk) * 1.4426950408889634f;
    p.tscale = t_scale;
    p.logdet = logdet; p.sumsq = sumsq; p.ticket = ticket; p.accumulate = accumulate; p.samples = samples;
    p.map = nll_map; p.map_row = row_src; p.map_col = col_src; p.map_mode = map_mode;
    CUtensorMap tmap;
    p.in_chunk_off = in_chunk_off;
    int rc = make_c8_tensor_map(&tmap, b_c8, N, in_total_chunks, H, W, kBW, kBH, kChunks, is_bf16);
    if (rc) return rc;
    typedef void (*KernT)(const CUtensorMap, const F8Params);
    static const KernT table[2][4] = {
        {coupling_f8_kernel<false, false, false>, coupling_f8_kernel<false, true, false>, coupling_f8_kernel<false, false, true>, coupling_f8_kernel<false, true, true>},
        {coupling_f8_kernel<true, false, false>, coupling_f8_kernel<true, true, false>, coupling_f8_kernel<true, false, true>, coupling_f8_kernel<true, true, true>}};
    static const KernT table_ms[2][2] = {
        {coupling_f8_kernel<false, true, false, true>, coupling_f8_kernel<false, true, true, true>},
        {coupling_f8_kernel<true, true, false, true>, coupling_f8_kernel<true, true, true, true>}};
    static const KernT table_map[2][2] = {
        {coupling_f8_kernel<false, false, false, false, true>, coupling_f8_kernel<false, false, true, false, true>},
        {coupling_f8_kernel<true, false, false, false, true>, coupling_f8_kernel<true, false, true, false, true>}};
    const int mode = (ct ? 2 : 0) + (inverse ? 1 : 0);
    KernT kern = ms ? table_ms[is_bf16 ? 1 : 0][ct ? 1 : 0] : map ? table_map[is_bf16 ? 1 : 0][ct ? 1 : 0] : table[is_bf16 ? 1 : 0][mode];
    static bool attr_done[16] = {};
    const int ki = ms ? 8 + (is_bf16 ? 2 : 0) + (ct ? 1 : 0) : map ? 12 + (is_bf16 ? 2 : 0) + (ct ? 1 : 0) : (is_bf16 ? 4 : 0) + mode;
    if (!attr_done[ki]) {
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        attr_done[ki] = true;
    }
    const uint32_t wbytes = 9u * kChunks * BN * 16u;
    p.off_a = (kOffW + wbytes + 127u) & ~127u;
    int stages = (int)((227u * 1024u - 1024u - p.off_a) / kA1Bytes);
    p.a_stages = stages > 3 ? 3 : stages;
    const size_t smem_bytes = 1024 + p.off_a + (size_t)p.a_stages * kA1Bytes;
    const int grid = p.num_tiles < kNumSMs ? p.num_tiles : kNumSMs;
    kern<<<grid, kThreads, smem_bytes, (cudaStream_t)stream>>>(tmap, p);
    return check_launch(name);
}

// ---- C ABI: the coupling kernels --------------------------------------------------------------------------------------
// Last conv of a coupling sub-network + affine coupling on the F8 detail half.  w_packed: cwfa_tc_pack_weights output for a
// 3x3 conv 64 -> BN channels in ONE n-block whose columns are [s of slot 0..chp8-1 | t of slot 0..chp8-1] (or s alone when
// ct != NULL), slots = storage channels of the F8 tensors (chp8 = 8 * ceil(ch / 8); padding slots: zero weights and bias).
// cx: F8 input (NULL = zeros, inverse only); cy: F8 output; ct: F8 external shift or NULL; perm: int32 row (perm_axis 2) or
// column (perm_axis 3) gather indices applied to cx, or NULL.  workspace / logdet / sumsq / accumulate / ticket as in
// cwfa_coupling_tc (ticket may be NULL: reduce with cwfa_coupling_finalize over cwfa_coupling_tc_tiles(H, W) partials).
extern "C" int cwfa_coupling_f8(const void* b_c8, const void* w_packed, const float* bias, int N, int H, int W, int BN, int chp8,
                                const float* cx, float* cy, const float* ct, float t_scale, const int32_t* perm, int perm_axis,
                                float clamp, float k_atan, int inverse, float* workspace, float* logdet, float* sumsq, int accumulate,
                                int32_t* ticket, int in_total_chunks, int in_chunk_off, int is_bf16, void* stream) {
    return coupling_f8_launch("coupling_f8", b_c8, w_packed, bias, N, 1, H, W, BN, chp8, cx, cy, ct, t_scale, perm, perm_axis, clamp,
                              k_atan, inverse, workspace, logdet, sumsq, accumulate, ticket, in_total_chunks, in_chunk_off, is_bf16, stream);
}
// cwfa_coupling_f8 with ``samples`` latent samples per condition image (inverse only): cx / cy hold N * samples F8 rows, row
// n * samples + k being sample k of condition image n; b_c8, ct and the log-det stay per condition image (N rows).  s and t
// are computed once per tile and applied to every sample; sample k's output is bitwise that of cwfa_coupling_f8 on its row.
// sumsq must be NULL.  samples == 1 is cwfa_coupling_f8.
extern "C" int cwfa_coupling_f8_samples(const void* b_c8, const void* w_packed, const float* bias, int N, int samples, int H, int W,
                                        int BN, int chp8, const float* cx, float* cy, const float* ct, float t_scale,
                                        const int32_t* perm, int perm_axis, float clamp, float k_atan, int inverse, float* workspace,
                                        float* logdet, float* sumsq, int accumulate, int32_t* ticket, int in_total_chunks,
                                        int in_chunk_off, int is_bf16, void* stream) {
    return coupling_f8_launch("coupling_f8_samples", b_c8, w_packed, bias, N, samples, H, W, BN, chp8, cx, cy, ct, t_scale, perm,
                              perm_axis, clamp, k_atan, inverse, workspace, logdet, sumsq, accumulate, ticket, in_total_chunks,
                              in_chunk_off, is_bf16, stream);
}
// cwfa_coupling_f8 in the forward direction that also accumulates the per-element NLL terms of the level into nll_map (F8, the
// layout of cx / cy).  Every coupling of a level is elementwise (s and t come from the conditions only), so each detail element
// follows its own chain of affine maps and its NLL is 0.5 z^2 - sum over blocks of s.  nll_map is indexed by the element's
// coordinate at the level's INPUT: this block adds its term at map[n, c, row_src[h], col_src[w]] for the element it writes at
// (h, w) (row_src / col_src NULL = identity; the caller composes them from the level's row / column permutations; channels need
// no table, F8 slots keep the order in which the detail half entered the flow).  map_mode: CWFA_NLL_MAP_FIRST writes -s without
// reading nll_map (no memset needed), 0 (a middle block) adds -s, CWFA_NLL_MAP_LAST also adds 0.5 y^2 of the value it writes;
// FIRST | LAST for a level of one block.  Padding slots come out 0.  cy, the log-det and sumsq are bitwise cwfa_coupling_f8's.
// Rejected: inverse != 0, cx == NULL, nll_map == NULL, an unknown map_mode.
extern "C" int cwfa_coupling_f8_map(const void* b_c8, const void* w_packed, const float* bias, int N, int H, int W, int BN, int chp8,
                                    const float* cx, float* cy, const float* ct, float t_scale, const int32_t* perm, int perm_axis,
                                    float clamp, float k_atan, int inverse, float* workspace, float* logdet, float* sumsq, int accumulate,
                                    int32_t* ticket, int in_total_chunks, int in_chunk_off, int is_bf16, void* stream, float* nll_map,
                                    const int32_t* row_src, const int32_t* col_src, int map_mode) {
    if (inverse || !cx || !nll_map || map_mode < 0 || map_mode > (kMapFirst | kMapLast)) {
        set_error("coupling_f8_map: forward only (inverse = 0), needs x and nll_map, map_mode in 0..3 (FIRST = 1 | LAST = 2)");
        return CWFA_EINVAL;
    }
    return coupling_f8_launch("coupling_f8_map", b_c8, w_packed, bias, N, 1, H, W, BN, chp8, cx, cy, ct, t_scale, perm, perm_axis,
                              clamp, k_atan, inverse, workspace, logdet, sumsq, accumulate, ticket, in_total_chunks, in_chunk_off,
                              is_bf16, stream, nll_map, row_src, col_src, map_mode);
}
