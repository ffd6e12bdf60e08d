// Fused, persistent residual block of the coupling sub-network trunk (networks.py:624-634, :659-663):
//     y = ELU( W1x1 * ELU( W3x3 (*) x + b3 ) + b1 + x ),   64 -> 64 -> 64 channels, C8 in / C8 out.
// One persistent CTA per SM walks 16x16-pixel tiles.  Per tile:
//   TMA halo tile (18x18x64ch)  ->  GEMM1: 9 taps x (M=128,N=64,K=64) x 2 M-blocks into TMEM acc1
//   EPI1 warps: acc1 -> +b3 -> ELU -> half -> shared memory in the K-major UMMA layout (A operand of GEMM2)
//   GEMM2: (M=128,N=64,K=64) x 2 M-blocks into TMEM acc2 with the resident 1x1 weights
//   EPI2 warps: acc2 -> +b1 + x (residual, L2-hot re-read) -> ELU -> half -> global (16-byte stores)
// The 3x3->ELU->1x1 intermediate never leaves the SM; both weight sets stay resident in shared memory;
// acc1/acc2 are double buffered in TMEM (512 columns) so GEMM1 of tile i+1 overlaps the epilogues of tile i.
// Warp roles (448 threads): warp0 TMA producer, warp1 MMA issuer, warps2-5 EPI1, warps6-13 EPI2 (4 warps per M-block).
//
// Entry form (KS > 0): the FIRST block of a sub-network trunk, whose input b = Win * lf + bin is the trunk's 1x1 input conv of
// the LF condition lf (no activation in between, networks.py:60-87).  Since W3 (*) b = (W3 Win) (*) lf + W3 (*) bin, the block
// reads lf (Cin_p = 16 KS channels) directly: GEMM1 runs KS K-steps per tap with the composed weights W3' = W3_tap Win, and the
// residual b joins acc2 through KS more MMAs (Win on the centre tap of the same halo tile).  b never exists in memory.  The
// network zero-pads b, not lf: the composed bias b3 + sum_tap W3_tap bin holds inside the image, and EPI1 subtracts the
// contributions of the out-of-image taps on edge pixels (per-set fp32 table of the 16 edge classes).
#include "tc_common.cuh"
#include "cwfa_b200_debug.h"
using namespace cwfa;
using namespace cwfa::tcx;

namespace {

constexpr int kC = 64, kChunks = 8;
constexpr int kTH = 16, kTW = 16, kBH = 18, kBW = 18;
constexpr uint32_t kW1Bytes = kChunks * kC * 16;             // 8192
constexpr uint32_t kA2MbBytes = kChunks * 128 * 16;           // 16384 per M-block
constexpr uint32_t kHeader = 2048;
constexpr uint32_t kOnesBytes = 2 * 128 * 16;                // A tile of the bias MMA: [2 chunks][128 rows][8], e0 = e1 = 1
constexpr int kMaxSets = 5;                                  // weight sets (sub-networks) one launch can walk
constexpr uint32_t kBiasRow = kC * 16;                       // chunk 0 of one bias B tile: [64 n][8], e0 = hi, e1 = lo (1 KB)
// bias tiles: [set][conv 0 = 3x3 | 1 = 1x1] chunk-0 rows, then ONE shared all-zero chunk (chunk 1 of every tile: LBO points at it)
constexpr uint32_t kBiasBytes = (2 * kMaxSets + 1) * kBiasRow;

// Shared-memory plan of the block (KS = 0) and of the entry form with KS K-steps of 16 input channels.  The entry form keeps
// a halo tile alive until GEMM2 of its tile (the residual MMAs read it), so it runs three A slots where they fit.
template <int KS>
struct RbLayout {
    static constexpr bool kEntry = KS > 0;
    static constexpr int kKSteps = kEntry ? KS : 4;
    static constexpr int kInChunks = 2 * kKSteps;
    static constexpr int kSlots = kEntry && KS <= 3 ? 3 : 2;
    static constexpr uint32_t kA1Bytes = kInChunks * kBH * kBW * 16;    // 41472 at 8 chunks
    static constexpr uint32_t kTapBytes = kInChunks * kC * 16;          // 8192 at 8 chunks
    static constexpr uint32_t kW3Bytes = 9 * kTapBytes;                 // 73728 at 8 chunks
    static constexpr uint32_t kWinBytes = kEntry ? kTapBytes : 0;       // entry form: Win [chunk][64][8]
    static constexpr uint32_t kOffW3 = kHeader, kOffW1 = kOffW3 + kW3Bytes, kOffWin = kOffW1 + kW1Bytes,
                              kOffA1 = kOffWin + kWinBytes, kOffA2 = kOffA1 + kSlots * kA1Bytes,
                              kOffOnes = kOffA2 + 2 * kA2MbBytes, kOffBias = kOffOnes + kOnesBytes,
                              kOffZero = kOffBias + 2 * kMaxSets * kBiasRow, kSmemTotal = kOffBias + kBiasBytes;
    static_assert(kSmemTotal + 1024 <= 227 * 1024, "resblock_tc: shared memory");
};
// A-slot ring position of tile i (the two-slot form keeps the block's original bit arithmetic)
template <int NS> __device__ __forceinline__ int ring_slot(int i) { return NS == 2 ? (i & 1) : i % NS; }
template <int NS> __device__ __forceinline__ int ring_phase(int i) { return NS == 2 ? ((i >> 1) & 1) : ((i / NS) & 1); }
constexpr int kThreads = 448;        // warp0 TMA, warp1 MMA, warps2-5 EPI1, warps6-13 EPI2 (one M-block per warp set)

struct RbParams {
    int N, H, W, tiles_x, tiles_y, num_tiles;        // num_tiles = n_sets * tiles_per_set
    int n_sets, tiles_per_set;                       // weight sets (independent sub-network blocks) walked by ONE launch
    int in_total_chunks, out_total_chunks;
    int in_chunk_off[kMaxSets], out_chunk_off[kMaxSets];
    const uint8_t* x;        // input C8 tensor base (also the residual)
    uint8_t* y;              // output C8 tensor base
    const uint8_t* w3[kMaxSets];       // packed [9][8][64][8] (entry form: composed W3', [9][2 KS][64][8])
    const uint8_t* w1[kMaxSets];       // packed [8][64][8]
    const float* b3[kMaxSets];         // 64
    const float* b1[kMaxSets];         // 64
    unsigned long long* dbg;  // optional profiling stamps: [cta][tile<8][8]
    const uint8_t* win[kMaxSets];      // entry form: packed input conv [2 KS][64][8]
    const float* edge[kMaxSets];       // entry form: [16 edge classes][64] fp32, subtracted from acc1 on image-edge pixels
};
__device__ __forceinline__ void rb_stamp(const RbParams& p, int tile, int slot) {
    if (p.dbg && tile < 8) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        p.dbg[((size_t)blockIdx.x * 8 + tile) * 8 + slot] = t;
    }
}

template <bool BF16, int KS>
__global__ void __launch_bounds__(kThreads, 1) resblock_tc_kernel(const __grid_constant__ CUtensorMap tmap, const RbParams p) {
    using L = RbLayout<KS>;
    constexpr int NS = L::kSlots;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const uint32_t s0 = smem_u32(smem);
    // barriers (8 bytes each)
    const uint32_t w_full = s0;
    // three A slots: their barriers sit behind the TMEM slot (bytes 136..183)
    auto a1_full = [&](int b) { return NS == 2 ? s0 + 8u * (1 + b) : s0 + 8u * (17 + b); };
    auto a1_empty = [&](int b) { return NS == 2 ? s0 + 8u * (3 + b) : s0 + 8u * (20 + b); };
    auto acc1_full = [&](int b) { return s0 + 8u * (5 + b); };
    auto acc1_empty = [&](int b) { return s0 + 8u * (7 + b); };
    auto acc2_full = [&](int b) { return s0 + 8u * (9 + b); };
    auto acc2_empty = [&](int b) { return s0 + 8u * (11 + b); };
    const uint32_t a2_full = s0 + 8u * 13, a2_empty = s0 + 8u * 14, w_empty = s0 + 8u * 15;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 128);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        mbar_init(w_full, 1);
        for (int b = 0; b < 2; ++b) {
            mbar_init(a1_full(b), 1);
            mbar_init(a1_empty(b), 1);
            mbar_init(acc1_full(b), 1);
            mbar_init(acc1_empty(b), 128);
            mbar_init(acc2_full(b), 1);
            mbar_init(acc2_empty(b), 256);
        }
        if constexpr (NS == 3) {
            mbar_init(a1_full(2), 1);
            mbar_init(a1_empty(2), 1);
        }
        mbar_init(a2_full, 128);
        mbar_init(a2_empty, 1);
        mbar_init(w_empty, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // Biases enter the accumulators through one extra K=16 MMA per GEMM: A = "ones" tile (columns k=0,1 are 1),
    // B rows k=0 / k=1 = bf16 hi / lo parts of the fp32 bias (hi + lo reproduces it to ~2^-17 relative).
    for (int i = threadIdx.x; i < (int)(kOnesBytes + kBiasBytes) / 16; i += kThreads) {
        uint4 v = make_uint4(0, 0, 0, 0);
        const int ones_units = kOnesBytes / 16;
        if (i < 128) {
            v.x = pack2<BF16>(1.f, 1.f);                                  // chunk 0 of the ones tile: e0 = e1 = 1
        } else if (i >= ones_units) {
            const int j = i - ones_units;                                 // [set][conv][64 rows], then the zero chunk
            const int tile = j / kC, r = j % kC;
            if (tile < 2 * p.n_sets) {
                const float bv = __ldg(((tile & 1) ? p.b1[tile >> 1] : p.b3[tile >> 1]) + r);
                float hi;
                if constexpr (BF16) hi = __bfloat162float(__float2bfloat16_rn(bv));
                else hi = __half2float(__float2half_rn(bv));
                v.x = pack2<BF16>(hi, bv - hi);
            }
        }
        *reinterpret_cast<uint4*>(smem + L::kOffOnes + (size_t)i * 16) = v;
    }
    fence_proxy_async();
    if (warp == 1) tmem_alloc(smem_u32(tmem_slot), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    // several weight sets: each CTA walks a CONTIGUOUS range of the (set, sample, tile) space (at most one or two weight switches
    // per CTA and launch); one set: tiles strided over the CTAs (the CTAs sweep the image together: best DRAM / L2 locality)
    const bool strided = p.n_sets == 1;
    const int t_begin = strided ? (int)blockIdx.x : (int)((int64_t)blockIdx.x * p.num_tiles / gridDim.x);
    const int t_step = strided ? (int)gridDim.x : 1;
    const int my_tiles = strided ? (p.num_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x
                                 : (int)((int64_t)(blockIdx.x + 1) * p.num_tiles / gridDim.x) - t_begin;
    const int tiles_per_img = p.tiles_x * p.tiles_y;
    const size_t plane = (size_t)p.H * p.W;

    if (warp == 0) {
        // ============================ TMA producer ============================
        if (lane == 0) {
            int cur = -1;
            uint32_t wsw = 0;                                   // weight switches so far
            for (int i = 0; i < my_tiles; ++i) {
                const int t = t_begin + i * t_step;
                const int k = t / p.tiles_per_set, ts = t - k * p.tiles_per_set;
                if (k != cur) {                                 // (re)load the resident weights of set k
                    if (cur >= 0) { mbar_wait(w_empty, wsw & 1); ++wsw; }      // every MMA reading the old set has completed
                    mbar_expect_tx(w_full, L::kW3Bytes + kW1Bytes + L::kWinBytes);
                    bulk_load(s0 + L::kOffW3, p.w3[k], L::kW3Bytes, w_full);
                    bulk_load(s0 + L::kOffW1, p.w1[k], kW1Bytes, w_full);
                    if constexpr (L::kEntry) bulk_load(s0 + L::kOffWin, p.win[k], L::kWinBytes, w_full);
                    cur = k;
                }
                const int n = ts / tiles_per_img, r = ts % tiles_per_img;
                const int h0 = (r / p.tiles_x) * kTH, w0 = (r % p.tiles_x) * kTW;
                const int b = ring_slot<NS>(i);
                mbar_wait(a1_empty(b), ring_phase<NS>(i) ^ 1);
                mbar_expect_tx(a1_full(b), L::kA1Bytes);
                tma_load_4d(s0 + L::kOffA1 + b * L::kA1Bytes, &tmap, a1_full(b), (w0 - 1) * 8, h0 - 1, p.in_chunk_off[k], n);
            }
        }
    } else if (warp == 1) {
        // ============================ MMA issuer ============================
        const uint32_t idesc = idesc_f16(kC, BF16 ? 1 : 0);
        constexpr uint32_t a1_lbo = kBH * kBW * 16, a1_sbo = kBW * 16;
        constexpr uint32_t w_lbo = kC * 16, w_sbo = 128;
        constexpr uint32_t a2_lbo = 128 * 16, a2_sbo = 128;
        const uint32_t a1_hi = desc_hi(a1_sbo), w_hi = desc_hi(w_sbo), a2_hi = desc_hi(a2_sbo);
        const uint32_t w3_lo0 = desc_lo(s0 + L::kOffW3, w_lbo), w1_lo0 = desc_lo(s0 + L::kOffW1, w_lbo);
        const uint32_t ones_lo = desc_lo(s0 + L::kOffOnes, 128 * 16);         // same geometry as an A2 M-block (LBO 2048, SBO 128)
        // bias B tile of (set k, conv c): chunk 0 at kOffBias + (2k + c) KB, chunk 1 = the shared zero chunk (LBO = distance to it)
        auto bias_lo = [&](int k, int c) {
            const uint32_t base = L::kOffBias + (uint32_t)(2 * k + c) * kBiasRow;
            return desc_lo(s0 + base, L::kOffZero - base);
        };
        const uint32_t leader = elect_one();
        int cur_set = -1;
        uint32_t wph = 0;

        auto gemm2 = [&](int j, int kset) {
            const int bj = j & 1;
            const uint32_t b1_lo = bias_lo(kset, 1);
            mbar_wait(a2_full, j & 1);
            mbar_wait(acc2_empty(bj), ((j >> 1) & 1) ^ 1);
            tc_fence_after();
            if (leader) {
#pragma unroll
                for (int mb = 0; mb < 2; ++mb) {
                    const uint32_t d = tmem + 256 + (bj * 2 + mb) * kC;
                    const uint32_t a_lo0 = desc_lo(s0 + L::kOffA2 + mb * kA2MbBytes, a2_lbo);
                    tc_mma_f16_split(d, ones_lo, a2_hi, b1_lo, w_hi, idesc, 0u);          // acc = bias1
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
                        tc_mma_f16_split(d, a_lo0 + kk * ((2 * a2_lbo) >> 4), a2_hi, w1_lo0 + kk * ((2 * w_lbo) >> 4), w_hi,
                                         idesc, 1u);
                    if constexpr (L::kEntry) {
                        // residual b = Win * lf (its bias is in bias1): the centre tap of the tile's halo tile
                        const uint32_t r_lo0 = desc_lo(s0 + L::kOffA1 + ring_slot<NS>(j) * L::kA1Bytes + (kBW + 1) * 16, a1_lbo);
                        const uint32_t win_lo0 = desc_lo(s0 + L::kOffWin, w_lbo);
#pragma unroll
                        for (int kk = 0; kk < KS; ++kk)
                            tc_mma_f16_split(d, r_lo0 + mb * 8 + kk * ((2 * a1_lbo) >> 4), a1_hi, win_lo0 + kk * ((2 * w_lbo) >> 4),
                                             w_hi, idesc, 1u);
                    }
                }
                tc_commit(a2_empty);
                if constexpr (L::kEntry) tc_commit(a1_empty(ring_slot<NS>(j)));
                tc_commit(acc2_full(bj));
            }
            __syncwarp();
        };

        bool g2_done = true;                                    // GEMM2 of tile i-1 already issued?
        int prev_set = -1;
        for (int i = 0; i < my_tiles; ++i) {
            const int b = i & 1, ph = (i >> 1) & 1;
            const int kset = (t_begin + i * t_step) / p.tiles_per_set;
            if (kset != cur_set) {
                if (cur_set >= 0) {
                    // weight switch: GEMM2 of the last tile of the old set still needs W1 -- issue it now (drains the
                    // pipeline once), then tell the producer that the resident weights may be overwritten
                    if (!g2_done) { gemm2(i - 1, prev_set); g2_done = true; }
                    if (leader) tc_commit(w_empty);
                    __syncwarp();
                }
                mbar_wait(w_full, wph);
                wph ^= 1;
                cur_set = kset;
            }
            const uint32_t b3_lo = bias_lo(kset, 0);
            const int sa = ring_slot<NS>(i);                    // A slot (== b with two slots)
            mbar_wait(a1_full(sa), ring_phase<NS>(i));
            mbar_wait(acc1_empty(b), ph ^ 1);
            tc_fence_after();
            if (leader) rb_stamp(p, i, 0);
            if (leader) {
                const uint32_t a_base = s0 + L::kOffA1 + sa * L::kA1Bytes;
#pragma unroll
                for (int mb = 0; mb < 2; ++mb)                                             // acc = bias3
                    tc_mma_f16_split(tmem + (b * 2 + mb) * kC, ones_lo, a2_hi, b3_lo, w_hi, idesc, 0u);
#pragma unroll 1
                for (int tap = 0; tap < 9; ++tap) {
                    const int kh = tap / 3, kw = tap - kh * 3;
                    const uint32_t w_lo = w3_lo0 + tap * (L::kTapBytes >> 4);
                    const uint32_t a_lo0 = desc_lo(a_base + (uint32_t)((kh * kBW + kw) * 16), a1_lbo);
                    // interleave the two M-blocks: back-to-back MMAs never accumulate into the same TMEM tile
#pragma unroll
                    for (int kk = 0; kk < L::kKSteps; ++kk) {
#pragma unroll
                        for (int mb = 0; mb < 2; ++mb)
                            tc_mma_f16_split(tmem + (b * 2 + mb) * kC, a_lo0 + mb * 8 + kk * ((2 * a1_lbo) >> 4), a1_hi,
                                             w_lo + kk * ((2 * w_lbo) >> 4), w_hi, idesc, 1u);
                    }
                }
                if constexpr (!L::kEntry) tc_commit(a1_empty(b));    // entry form: released after GEMM2 (residual MMAs)
                tc_commit(acc1_full(b));
                rb_stamp(p, i, 1);
            }
            __syncwarp();
            if (i >= 1 && !g2_done) gemm2(i - 1, prev_set);
            g2_done = false;                                    // GEMM2 of THIS tile is outstanding
            prev_set = kset;
        }
        if (my_tiles > 0) gemm2(my_tiles - 1, prev_set);
    } else if (warp < 6) {
        // ============================ EPI1: acc1 -> ELU -> shared (A of GEMM2) ============================
        const int q = warp & 3;
        const int m = q * 32 + lane;
        for (int i = 0; i < my_tiles; ++i) {
            const int b = i & 1, ph = (i >> 1) & 1;
            mbar_wait(acc1_full(b), ph);
            if (threadIdx.x == 64) rb_stamp(p, i, 2);
            mbar_wait(a2_empty, (i & 1) ^ 1);
            tc_fence_after();
            if (threadIdx.x == 64) rb_stamp(p, i, 3);
#pragma unroll 1
            for (int mb = 0; mb < 2; ++mb) {
                const uint32_t a2 = s0 + L::kOffA2 + mb * kA2MbBytes + m * 16;
                uint32_t r[64];
                __syncwarp();
                const uint32_t ta = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)((b * 2 + mb) * kC);
                tmem_ld32_nowait(ta, r);
                tmem_ld32_nowait(ta + 32, r + 32);
                tmem_ld_wait();
                if constexpr (L::kEntry) {
                    // the zero padding of b: drop the out-of-image taps' W3_tap * bin from the composed bias
                    const int t = t_begin + i * t_step;
                    const int kset = t / p.tiles_per_set, rr = (t - kset * p.tiles_per_set) % tiles_per_img;
                    const int orow = (rr / p.tiles_x) * kTH + (m >> 3), ocol = (rr % p.tiles_x) * kTW + mb * 8 + (m & 7);
                    const int cls = ((orow == 0) | ((orow == p.H - 1) << 1)) * 4 + ((ocol == 0) | ((ocol == p.W - 1) << 1));
                    if (cls) {
                        const float4* e = reinterpret_cast<const float4*>(p.edge[kset] + cls * kC);
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const float4 v = __ldg(e + j);
                            r[4 * j + 0] = __float_as_uint(__uint_as_float(r[4 * j + 0]) - v.x);
                            r[4 * j + 1] = __float_as_uint(__uint_as_float(r[4 * j + 1]) - v.y);
                            r[4 * j + 2] = __float_as_uint(__uint_as_float(r[4 * j + 2]) - v.z);
                            r[4 * j + 3] = __float_as_uint(__uint_as_float(r[4 * j + 3]) - v.w);
                        }
                    }
                }
#pragma unroll
                for (int ch = 0; ch < 8; ++ch) {
                    uint4 ov;
                    ov.x = pack2<BF16>(elu5(__uint_as_float(r[ch * 8 + 0])), elu5(__uint_as_float(r[ch * 8 + 1])));
                    ov.y = pack2<BF16>(elu5(__uint_as_float(r[ch * 8 + 2])), elu5(__uint_as_float(r[ch * 8 + 3])));
                    ov.z = pack2<BF16>(elu5(__uint_as_float(r[ch * 8 + 4])), elu5(__uint_as_float(r[ch * 8 + 5])));
                    ov.w = pack2<BF16>(elu5(__uint_as_float(r[ch * 8 + 6])), elu5(__uint_as_float(r[ch * 8 + 7])));
                    sts128(a2 + ch * (128 * 16), ov);
                }
            }
            tc_fence_before();
            fence_proxy_async();                // make the generic-proxy smem writes visible to the tensor core
            mbar_arrive(acc1_empty(b));
            mbar_arrive(a2_full);
            if (threadIdx.x == 64) rb_stamp(p, i, 4);
        }
    } else {
        // ============================ EPI2: acc2 + b1 + x -> ELU -> global ============================
        const int q = warp & 3;
        const int m = q * 32 + lane;
        for (int i = 0; i < my_tiles; ++i) {
            const int b = i & 1, ph = (i >> 1) & 1;
            const int t = t_begin + i * t_step;
            const int kset = t / p.tiles_per_set, ts = t - kset * p.tiles_per_set;
            const int n = ts / tiles_per_img, rr = ts % tiles_per_img;
            const int h0 = (rr / p.tiles_x) * kTH, w0 = (rr % p.tiles_x) * kTW;
            const int orow = h0 + (m >> 3);
            const int mb = (warp - 6) >> 2;               // warps 6-9 -> M-block 0, warps 10-13 -> M-block 1
            const int ocol = w0 + mb * 8 + (m & 7);
            const bool ok = orow < p.H && ocol < p.W;
            const size_t pix = (size_t)orow * p.W + ocol;
            // prefetch the residual x BEFORE waiting on the accumulator (L2-hot: the halo tile of this very tile
            // was just fetched by TMA); 8 x 16-byte loads in flight per thread
            uint4 rx[8];
            if constexpr (!L::kEntry) {
                const uint8_t* xin = p.x + (((size_t)n * p.in_total_chunks + p.in_chunk_off[kset]) * plane + pix) * 16;
#pragma unroll
                for (int ch = 0; ch < 8; ++ch)
                    rx[ch] = ok ? __ldg(reinterpret_cast<const uint4*>(xin + (size_t)ch * plane * 16)) : make_uint4(0, 0, 0, 0);
            }
            mbar_wait(acc2_full(b), ph);
            tc_fence_after();
            if (threadIdx.x == 192) rb_stamp(p, i, 5);
            {
                uint8_t* yout = p.y + (((size_t)n * p.out_total_chunks + p.out_chunk_off[kset]) * plane + pix) * 16;
                uint32_t r[64];
                __syncwarp();
                const uint32_t ta = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(256 + (b * 2 + mb) * kC);
                tmem_ld32_nowait(ta, r);
                tmem_ld32_nowait(ta + 32, r + 32);
                tmem_ld_wait();
#pragma unroll
                for (int ch = 0; ch < 8; ++ch) {
                    if constexpr (L::kEntry) {                // the residual is already in acc2
                        uint4 ov;
                        ov.x = pack2<BF16>(elu5(__uint_as_float(r[ch * 8 + 0])), elu5(__uint_as_float(r[ch * 8 + 1])));
                        ov.y = pack2<BF16>(elu5(__uint_as_float(r[ch * 8 + 2])), elu5(__uint_as_float(r[ch * 8 + 3])));
                        ov.z = pack2<BF16>(elu5(__uint_as_float(r[ch * 8 + 4])), elu5(__uint_as_float(r[ch * 8 + 5])));
                        ov.w = pack2<BF16>(elu5(__uint_as_float(r[ch * 8 + 6])), elu5(__uint_as_float(r[ch * 8 + 7])));
                        if (ok) *reinterpret_cast<uint4*>(yout + (size_t)ch * plane * 16) = ov;
                        continue;
                    }
                    const float2 x0 = unpack2<BF16>(rx[ch].x), x1 = unpack2<BF16>(rx[ch].y),
                                 x2 = unpack2<BF16>(rx[ch].z), x3 = unpack2<BF16>(rx[ch].w);
                    uint4 ov;
                    ov.x = pack2<BF16>(elu5(__uint_as_float(r[ch * 8 + 0]) + x0.x), elu5(__uint_as_float(r[ch * 8 + 1]) + x0.y));
                    ov.y = pack2<BF16>(elu5(__uint_as_float(r[ch * 8 + 2]) + x1.x), elu5(__uint_as_float(r[ch * 8 + 3]) + x1.y));
                    ov.z = pack2<BF16>(elu5(__uint_as_float(r[ch * 8 + 4]) + x2.x), elu5(__uint_as_float(r[ch * 8 + 5]) + x2.y));
                    ov.w = pack2<BF16>(elu5(__uint_as_float(r[ch * 8 + 6]) + x3.x), elu5(__uint_as_float(r[ch * 8 + 7]) + x3.y));
                    if (ok) *reinterpret_cast<uint4*>(yout + (size_t)ch * plane * 16) = ov;
                }
            }
            tc_fence_before();
            mbar_arrive(acc2_empty(b));
            if (threadIdx.x == 192) rb_stamp(p, i, 6);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem, 512);
    }
}

}  // namespace

static unsigned long long* g_rb_dbg = nullptr;
extern "C" int cwfa_resblock_set_debug_buffer(void* buf) { g_rb_dbg = (unsigned long long*)buf; return CWFA_OK; }

static int resblock_launch(const void* x_c8, void* y_c8, int n_sets, const void* const* w3, const void* const* w1, const float* const* b3,
                           const float* const* b1, int N, int H, int W, int in_total_chunks, const int* in_chunk_off, int out_total_chunks,
                           const int* out_chunk_off, const void* const* win, const float* const* edge, int in_chunks, int is_bf16,
                           void* stream) {
    if (N <= 0 || H <= 0 || W <= 0 || n_sets < 1 || n_sets > kMaxSets) {
        set_error("resblock_tc: bad arguments (1..%d weight sets)", kMaxSets);
        return CWFA_EINVAL;
    }
    if ((reinterpret_cast<uintptr_t>(x_c8) & 15) || (reinterpret_cast<uintptr_t>(y_c8) & 15)) {
        set_error("resblock_tc: pointers must be 16-byte aligned");
        return CWFA_EINVAL;
    }
    const int ks = win ? in_chunks / 2 : 0;             // entry form: K-steps of 16 input channels
    if (win && (in_chunks < 2 || in_chunks > 8 || (in_chunks & 1) || !edge)) {
        set_error("resblock_tc: the entry form needs 2, 4, 6 or 8 input chunks and the edge-class tables");
        return CWFA_EINVAL;
    }
    const int chunks_in = win ? in_chunks : kChunks;
    RbParams p{};
    p.N = N; p.H = H; p.W = W;
    p.tiles_x = ceil_div(W, kTW); p.tiles_y = ceil_div(H, kTH);
    const int64_t per_set = (int64_t)p.tiles_x * p.tiles_y * N;
    if (per_set * n_sets > 0x7fffffff) { set_error("resblock_tc: too many tiles"); return CWFA_EINVAL; }
    p.n_sets = n_sets; p.tiles_per_set = (int)per_set; p.num_tiles = (int)(per_set * n_sets);
    p.in_total_chunks = in_total_chunks; p.out_total_chunks = out_total_chunks;
    for (int k = 0; k < n_sets; ++k) {
        if (in_chunk_off[k] < 0 || out_chunk_off[k] < 0 || in_chunk_off[k] + chunks_in > in_total_chunks ||
            out_chunk_off[k] + kChunks > out_total_chunks || !b3[k] || !b1[k] || (reinterpret_cast<uintptr_t>(w3[k]) & 15) ||
            (reinterpret_cast<uintptr_t>(w1[k]) & 15)) {
            set_error("resblock_tc: bad chunk offsets / missing bias / unaligned weights in set %d", k);
            return CWFA_EINVAL;
        }
        if (win && (!win[k] || !edge[k] || (reinterpret_cast<uintptr_t>(win[k]) & 15) || (reinterpret_cast<uintptr_t>(edge[k]) & 15))) {
            set_error("resblock_tc: missing / unaligned input-conv weights or edge table in set %d", k);
            return CWFA_EINVAL;
        }
        p.in_chunk_off[k] = in_chunk_off[k]; p.out_chunk_off[k] = out_chunk_off[k];
        p.w3[k] = (const uint8_t*)w3[k]; p.w1[k] = (const uint8_t*)w1[k]; p.b3[k] = b3[k]; p.b1[k] = b1[k];
        if (win) { p.win[k] = (const uint8_t*)win[k]; p.edge[k] = edge[k]; }
    }
    p.x = (const uint8_t*)x_c8; p.y = (uint8_t*)y_c8;
    p.dbg = g_rb_dbg;
    CUtensorMap tmap;
    int rc = make_c8_tensor_map(&tmap, x_c8, N, in_total_chunks, H, W, kBW, kBH, chunks_in, is_bf16);
    if (rc) return rc;
    typedef void (*KernT)(const CUtensorMap, const RbParams);
    static const KernT table[2][5] = {
        {resblock_tc_kernel<false, 0>, resblock_tc_kernel<false, 1>, resblock_tc_kernel<false, 2>, resblock_tc_kernel<false, 3>,
         resblock_tc_kernel<false, 4>},
        {resblock_tc_kernel<true, 0>, resblock_tc_kernel<true, 1>, resblock_tc_kernel<true, 2>, resblock_tc_kernel<true, 3>,
         resblock_tc_kernel<true, 4>}};
    static const uint32_t smem[5] = {RbLayout<0>::kSmemTotal, RbLayout<1>::kSmemTotal, RbLayout<2>::kSmemTotal,
                                     RbLayout<3>::kSmemTotal, RbLayout<4>::kSmemTotal};
    const KernT kern = table[is_bf16 ? 1 : 0][ks];
    static bool attr_done[2][5] = {};
    if (!attr_done[is_bf16 ? 1 : 0][ks]) {
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        attr_done[is_bf16 ? 1 : 0][ks] = true;
    }
    const int grid = p.num_tiles < kNumSMs ? p.num_tiles : kNumSMs;
    kern<<<grid, kThreads, smem[ks] + 1024, (cudaStream_t)stream>>>(tmap, p);
    return check_launch("resblock_tc");
}

extern "C" int cwfa_resblock_tc(const void* x_c8, void* y_c8, const void* w3_packed, const void* w1_packed, const float* b3,
                                const float* b1, int N, int H, int W, int in_total_chunks, int in_chunk_off,
                                int out_total_chunks, int out_chunk_off, int is_bf16, void* stream) {
    return resblock_launch(x_c8, y_c8, 1, &w3_packed, &w1_packed, &b3, &b1, N, H, W, in_total_chunks, &in_chunk_off, out_total_chunks,
                           &out_chunk_off, nullptr, nullptr, 0, is_bf16, stream);
}

// The same block for n_sets (<= 5) INDEPENDENT sub-networks in ONE launch: set k reads the 64-channel slice at in_chunk_off[k] of
// x and writes the slice at out_chunk_off[k] of y with its own weights / biases.  Every CTA walks a contiguous range of the
// (set, sample, tile) space and re-loads its resident weights at most once, so prologue, tail and wave quantisation are paid once
// per block row of a level (5 sub-networks, networks.py:305-366) instead of once per sub-network.
// win_packed != NULL selects the entry form (see the top of this file): set k reads in_chunks chunks of the LF condition at
// in_chunk_off[k]; w3 / b3 are the composed W3' and interior bias, b1 is b1 + bin, edge[k] the [16][64] edge-class table.
extern "C" int cwfa_resblock_tc_batched(const void* x_c8, void* y_c8, int n_sets, const void* const* w3_packed, const void* const* w1_packed,
                                        const float* const* b3, const float* const* b1, int N, int H, int W, int in_total_chunks,
                                        const int* in_chunk_off, int out_total_chunks, const int* out_chunk_off,
                                        const void* const* win_packed, const float* const* edge, int in_chunks, int is_bf16, void* stream) {
    return resblock_launch(x_c8, y_c8, n_sets, w3_packed, w1_packed, b3, b1, N, H, W, in_total_chunks, in_chunk_off, out_total_chunks,
                           out_chunk_off, win_packed, edge, in_chunks, is_bf16, stream);
}
