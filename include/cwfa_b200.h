/*
 * cwfa_b200 C ABI -- the drop-in boundary of the B200-native CWFA hot path.
 *
 * Every entry point is `extern "C"`, takes raw DEVICE pointers, sizes and a cudaStream_t
 * (passed as void*), allocates nothing, takes no ownership, is safe to call concurrently
 * on distinct streams, and returns 0 on success or a CWFA_E* code.  No torch types.
 * The reference (pvjosue/CWFA) is pure Python, so there is no FFI in it to replace; each
 * function instead names the reference Python function whose arithmetic it implements
 * (file:line into the reference tree).  The Python mirror of the reference module API
 * (cwfa_b200/modules.py, networks.py) is the only caller.  See INTEGRATION.md.
 *
 * Layouts:
 *   "NCHW"  fp32, contiguous, the reference's tensor layout (API side).
 *   "C8"    bf16 (or fp16), [N][Cp/8][H][W][8] with Cp = channels padded to a multiple
 *           of 16 with zeros -- the tensor-core side layout (DESIGN.md section 3).
 */
#ifndef CWFA_B200_H
#define CWFA_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CWFA_OK 0
#define CWFA_EINVAL 1   /* bad argument / unsupported shape */
#define CWFA_ECUDA 2    /* CUDA runtime / launch error (see cwfa_last_error) */
#define CWFA_ENOTSUP 3  /* device is not sm_100 */

/* activation codes used by conv epilogues */
#define CWFA_ACT_NONE 0
#define CWFA_ACT_ELU 1      /* alpha = 1   (networks.py:620) */
#define CWFA_ACT_PRELU 2    /* scalar slope read from device pointer (nn.PReLU(), networks.py:209, unet.py:22) */
#define CWFA_ACT_RELU 3
#define CWFA_ACT_GELU 4     /* exact erf GELU (networks.py:492) */
#define CWFA_ACT_SIGMOID 5

const char* cwfa_version(void);
const char* cwfa_last_error(void);
/* 0 if the current device is compute capability 10.x, else CWFA_ENOTSUP. */
int cwfa_device_check(void);

/* ---- K1: depth-wise Haar DWT / IDWT  (INN_utils.py:142-161 HaarTransform1D.forward,
 *      absorbs Split/cat of FrEIA/modules/graph_topology.py:73-80) ------------------------
 * fwd: lo[b,i,p] = (x[b,2i,p]+x[b,2i+1,p])/sqrt2, hi[b,i,p] = (x[b,2i,p]-x[b,2i+1,p])/sqrt2
 * inv: x[b,2i,p] = (lo+hi)/sqrt2, x[b,2i+1,p] = (lo-hi)/sqrt2
 * x is (B,C,P) contiguous; lo/hi are (B,C/2,P) with batch strides ld_lo/ld_hi (elements),
 * so one (B,C,P) buffer (lo=out, hi=out+C/2*P, ld=C*P) or two separate buffers both work. */
int cwfa_haar1d_fwd(const float* x, float* lo, float* hi, int B, int C, int64_t P,
                    int64_t ld_lo, int64_t ld_hi, void* stream);
int cwfa_haar1d_inv(const float* lo, const float* hi, float* x, int B, int C, int64_t P,
                    int64_t ld_lo, int64_t ld_hi, void* stream);

/* ---- K1b: FrEIA 2-D Haar down/up-sampling (FrEIA/modules/reshapes.py:273-300) ------------
 * down: x (B,C,H,W) -> y (B,4C,H/2,W/2); channel of (c, wavelet k): 4c+k, or k*C+c when
 * order_by_wavelet != 0.  y = fac * haar(x).  up is the exact inverse map with factor fac. */
int cwfa_haar2d_down(const float* x, float* y, int B, int C, int H, int W,
                     int order_by_wavelet, float fac, void* stream);
int cwfa_haar2d_up(const float* y, float* x, int B, int C, int H, int W,
                   int order_by_wavelet, float fac, void* stream);

/* ---- K4: permutations (fixed_transforms.py:37-41 PermuteRandom; INN_utils.py:73-81 PermuteDim)
 * axis 1: y[b,c,h,w] = x[b,perm[c],h,w]; axis 2: x[b,c,perm[h],w]; axis 3: x[b,c,h,perm[w]].
 * perm is int32 on the device, length = size of that axis. */
int cwfa_permute(const float* x, float* y, const int32_t* perm, int axis,
                 int B, int C, int H, int W, void* stream);

/* ---- K3: affine coupling + per-sample log-det (+ optional sum of squares of the output)
 *      (FrEIA/modules/coupling_layers.py:490-500, clamp const :52) ---------------------------
 * s = clamp * k_atan * atan(a_s[b,c,p]);  t = t_scale * a_t[b,c,p]
 * fwd: y = exp(s)*x + t, logdet[b] = +sum s;   inv: y = (x - t)*exp(-s), logdet[b] = -sum s.
 * a_s/a_t have batch strides ld_s/ld_t (elements) so they may alias the two halves of one
 * subnet output, or a_t may be the mean-volume condition with t_scale = -1/sqrt2
 * (networks.py:671).  x may be NULL in inv mode (z = 0, CWFA.py:906-907).
 * flags: bit0 = inverse; bit1 = a_s already holds the final s (no clamp applied; GIN blocks,
 * coupling_layers.py:360-361); bit2 = TANH clamp of AllInOneBlock: s = clamp * tanh(k_atan * a_s)
 * (all_in_one_block.py:206-211, k_atan = t_scale = 0.1).
 * logdet (B) and sumsq (B, may be NULL: sum over c,p of y^2, CWFA.py:183) are OVERWRITTEN;
 * workspace must hold 2*B*cwfa_affine_workspace_blocks() floats (deterministic 2-stage sum). */
int cwfa_affine_workspace_blocks(void);
int cwfa_affine(const float* x, const float* a_s, const float* a_t, float* y,
                float* logdet, float* sumsq, float* workspace,
                int B, int ch, int64_t P, int64_t ld_s, int64_t ld_t,
                float clamp, float k_atan, float t_scale, int flags, void* stream);

/* ---- generic fp32 direct convolution, NCHW, stride 1, "same" zero padding (KH,KW odd) -----
 * y = act2( act1(conv(x,w)+bias [+ res if res_mode==1]) [+ res if res_mode==2] ) ... precisely:
 *   v = conv + bias; if (res_mode==1) v += res; v = act(v); if (res_mode==2) v += res.
 * Covers every Conv2d/Conv1d of the path at reference precision
 * (networks.py:211-219,250-254,488-492,537,621-638; unet.py:67,99,104).
 * w is (Cout,Cin,KH,KW); bias may be NULL; slope = device pointer to the PReLU scalar. */
int cwfa_conv2d_f32(const float* x, const float* w, const float* bias, const float* res,
                    const float* slope, float* y, int N, int Cin, int H, int W, int Cout,
                    int KH, int KW, int act, int res_mode, void* stream);
/* ConvTranspose2d(k=2,s=2) (unet.py:166): x (N,Cin,H,W), w (Cin,Cout,2,2) -> y (N,Cout,2H,2W);
 * optional skip tensor added (unet.py:190). */
int cwfa_convT2x2_f32(const float* x, const float* w, const float* bias, const float* skip,
                      float* y, int N, int Cin, int H, int W, int Cout, void* stream);

/* ---- conditioning network's depth stencil: Conv3d(1,Cm,3,p1) -> PReLU -> Conv3d(Cm,1,3,p1)
 *      applied to (B,ch,H,W) viewed as a (H,W,ch) volume (networks.py:221-225,239) ---------
 * w1 (Cm,1,3,3,3) b1 (Cm) over (kh,kw,kd); w2 (1,Cm,3,3,3) b2 (1). Fused; the Cm-channel
 * hidden volume is never written to HBM. */
int cwfa_depth_stencil3d_f32(const float* x, const float* w1, const float* b1,
                             const float* slope, const float* w2, const float* b2, float* y,
                             int B, int ch, int H, int W, int Cm, void* stream);

/* ---- normalisation / pooling helpers of the LRNN (unet.py:72-113, networks.py:490) --------
 * channel_stats: per-channel sum and sum of squares over (N,H,W) -> stats[2*C] (overwritten;
 * workspace >= 2*C*cwfa_stats_workspace_blocks() floats).  bn_finalize turns them (or running
 * stats) into scale/shift.  scale_shift applies y = x*scale[c]+shift[c]. */
int cwfa_stats_workspace_blocks(void);
int cwfa_channel_stats_f32(const float* x, float* stats, float* workspace,
                           int N, int C, int64_t P, void* stream);
int cwfa_bn_finalize_f32(const float* stats, const float* gamma, const float* beta,
                         float* scale, float* shift, int C, double count, float eps, void* stream);
int cwfa_scale_shift_f32(const float* x, const float* scale, const float* shift, float* y,
                         int N, int C, int64_t P, void* stream);
int cwfa_maxpool2_f32(const float* x, float* y, int N, int C, int H, int W, void* stream);
/* LayerNorm over (C,H,W) per sample with element-wise affine (networks.py:490);
 * workspace >= 2*N*cwfa_layernorm_workspace_blocks() floats. */
int cwfa_layernorm_workspace_blocks(void);
int cwfa_layernorm_chw_f32(const float* x, const float* gamma, const float* beta, float* y,
                           float* workspace, int N, int64_t CHW, float eps, void* stream);
/* Fused GlobalAttention gate (networks.py:244-262,554): g = sigmoid(Conv1d_1(relu(Conv1d_3(v flattened over H*W))));
 * x += m * 2 * (g - 0.5).  v = mean volume (B,C,L), w1 (C,C,3), w2 (C,C,1), C <= 16. */
int cwfa_attention_gate_f32(float* x, const float* m, const float* v, const float* w1, const float* b1,
                            const float* w2, const float* b2, int B, int C, int64_t L, void* stream);
/* Lenslet crop + normalisation in one gather (XLFMDataset.extract_views XLFMDataset.py:212-242 followed by
 * (x - mean) / std, CWFA.py:797): image (B,1,Hi,Wi) -> out (B,L,SH,SW) fp32; image_dtype 0 = fp32, 1 = fp16, 2 = uint16 (a raw
 * sensor frame); coords int32 (L,2) = (row, col) lenslet centres on the device; patches are bottom/right aligned in the view
 * exactly as the reference does. */
int cwfa_extract_views(const void* image, int image_dtype, const int32_t* coords, float* out, int B, int Hi,
                       int Wi, int L, int SH, int SW, float mean, float stdv, int normalise, void* stream);
/* The same crop + normalisation written straight into the tensor-core input layout (csrc/sensor.cu): out is the C8 tensor
 * [B][Cp/8][SH][SW][8] bf16 (out_is_bf16) or fp16, 16-byte aligned, Cp >= L and a multiple of 8.  Bitwise equal to
 * cwfa_extract_views followed by cwfa_nchw_to_c8; lenslet slots L..Cp-1 are 0.  One pass, no fp32 intermediate. */
int cwfa_extract_views_c8(const void* image, int image_dtype, const int32_t* coords, void* out, int B, int Hi, int Wi, int L,
                          int Cp, int SH, int SW, float mean, float stdv, int normalise, int out_is_bf16, void* stream);
/* x += m * 2 * (g - 0.5)   (networks.py:554) */
int cwfa_gate_add_f32(float* x, const float* m, const float* g, int64_t n, void* stream);
/* fp32 -> fp16 narrowing of n elements (x, y 16-byte aligned): optional half-size host transfer of a finished volume (the
 * reference's own GPU output is fp16 under autocast, CWFA.py:845). */
int cwfa_cast_f32_f16(const float* x, void* y, int64_t n, void* stream);

/* ---- K2: tcgen05 / TMEM / TMA implicit-GEMM convolution (bf16 or fp16 operands, fp32 accumulate) --
 * The throughput path for every wide convolution of the path: coupling sub-network trunk
 * (networks.py:621-638), conditioning-net 2-D convs (:211-219), LRNN U-Net (unet.py:99-104,166) and
 * the ConvNeXt 7x7 (networks.py:489).  'same' zero padding, stride 1, KH/KW odd <= 7.
 * x_c8: C8 activations with Cin_p channels (multiple of 16).  w_packed: from cwfa_tc_pack_weights.
 * bias: Cout_p floats (zero padded) or NULL.  v = conv + bias; res_mode 1: v += res; v = act(v);
 * res_mode 2: v += res.  out_mode 0: C8 (Cout_p channels; res is C8), out_mode 1: NCHW fp32 with Cout
 * channels (res is NCHW fp32), out_mode 2: ConvTranspose2d(k=2,s=2) (unet.py:166) run as a 1x1 conv to
 * 4*Cout_p channels (weights packed with transposed=1) and scattered to a C8 (2H,2W) tensor, res = the
 * skip tensor added at the output location (unet.py:190; for out_mode 2 an n-block holds BN/2 channels of both horizontal
 * sub-pixels so that 32-byte sectors are written whole: BN % 32 == 0 and BN divides 2*Cout_p).  BN = output channels per CTA (multiple of 16, <= 256, divides Cout_p),
 * MB = number of 16x8-pixel M=128 blocks per CTA (1 or 2), MB*BN <= 512 TMEM columns.
 * cwfa_tc_packed_weight_elems = half elements to allocate for w_packed: the packed tiles followed by one uint32 per
 * (n-block, k-block) whose bit ks says "K-step ks has a nonzero weight" (written by cwfa_tc_pack_weights; cwfa_conv_tc
 * skips the zero K-steps -- the depth-banded stencil weights of the conditioning net, networks.py:221-225, are 2/3 zero). */
int cwfa_tc_kc(int cin_p);
int64_t cwfa_tc_packed_weight_elems(int Cin_p, int Cout_tot_p, int KH, int KW, int BN);
int cwfa_tc_pack_weights(const float* w, void* packed, int Cout, int Cin, int KH, int KW, int Cin_p,
                         int Cout_p, int BN, int transposed, int is_bf16, void* stream);
int cwfa_conv_tc(const void* x_c8, const void* w_packed, const float* bias, const float* slope,
                 const void* res, void* out, int N, int H, int W, int Cin_p, int Cout, int Cout_p,
                 int KH, int KW, int BN, int MB, int act, int res_mode, int out_mode, int is_bf16,
                 void* stream);
/* The launch plan cwfa_conv_tc (out_mode 0-2), cwfa_conv_tc_bn (stats != 0) or cwfa_conv_tc_coupling (out_mode 3, with the
 * coupling direction cpl_inverse and shift source cpl_ext) would use for these shapes; has_slope = a PReLU slope pointer is
 * passed.  Launches nothing.  plan[9] = {kernel index 0-25, A stages, B stages, resident weights, TMEM accumulator buffers,
 * wide (576-thread) kernel, grid, work items, dynamic shared memory bytes}.  Kernel index: 0-11 ring path
 * (fp16 | bf16) x (generic | wide) x epilogue (generic, lean none, lean PReLU); 12-19 fused coupling (fp16 | bf16) x
 * (fwd, inv, fwd + external shift, inv + external shift); 20-25 resident weights (fp16 | bf16) x epilogue. */
int cwfa_conv_tc_plan(int N, int H, int W, int Cin_p, int Cout_p, int KH, int KW, int BN, int MB, int act, int res_mode,
                      int out_mode, int has_slope, int stats, int cpl_inverse, int cpl_ext, int is_bf16, int* plan);
/* cwfa_conv_tc with the BatchNorm statistics of its (activated) output produced by the epilogue -- no separate pass over the
 * tensor (unet.py:100-107: conv -> PReLU -> BatchNorm in batch-statistics mode): one (sum, sum of squares) partial per 32-pixel
 * warp row and channel, plain stores, then a fixed-order two-stage sum (bit-reproducible).  stats_partial:
 * cwfa_conv_tc_stats_floats(N, H, W, Cout_p, MB) floats, no initialisation; cwfa_bn_partial_finalize turns it into the BatchNorm
 * scale / shift (and the raw (sum, sumsq) when stats_out != NULL).  C8 output, no residual, act none / PReLU, MB * BN > 256. */
int64_t cwfa_conv_tc_stats_floats(int N, int H, int W, int Cout_p, int MB);
int cwfa_conv_tc_bn(const void* x_c8, const void* w_packed, const float* bias, const float* slope, void* out, int N, int H,
                    int W, int Cin_p, int Cout, int Cout_p, int KH, int KW, int BN, int MB, int act, int is_bf16,
                    float* stats_partial, void* stream);
int cwfa_bn_partial_finalize(float* stats_partial, int N, int H, int W, int Cout_p, int MB, const float* gamma, const float* beta,
                             float eps, float* scale, float* shift, float* stats_out, void* stream);
/* ---- fused persistent residual block of the coupling sub-network trunk (networks.py:624-634,659-663):
 * y = ELU( W1x1 * ELU( W3x3 (*) x + b3 ) + b1 + x ), 64 -> 64 -> 64 channels.  x / y are 64-channel slices
 * (8 chunks starting at *_chunk_off) of C8 tensors with *_total_chunks chunks; y must not alias x.
 * w3_packed / w1_packed: cwfa_tc_pack_weights output with Cin_p = Cout_p = BN = 64. */
int cwfa_resblock_tc(const void* x_c8, void* y_c8, const void* w3_packed, const void* w1_packed,
                     const float* b3, const float* b1, int N, int H, int W, int in_total_chunks,
                     int in_chunk_off, int out_total_chunks, int out_chunk_off, int is_bf16, void* stream);
/* The same block for n_sets (<= 5) independent sub-networks in ONE launch (the block row of a level's five coupling
 * sub-networks, networks.py:305-366): set k reads the slice at in_chunk_off[k] of x, writes the slice at out_chunk_off[k] of y,
 * with its own packed weights / biases (host arrays of n_sets pointers / offsets).
 * win_packed == NULL: the block above (edge and in_chunks are ignored).  Otherwise the ENTRY form, the first block of a trunk
 * whose input b = Win * x + bin is the trunk's 1x1 input conv of the LF condition x: set k reads in_chunks (2, 4, 6 or 8) chunks
 * of x at in_chunk_off[k] and computes y = ELU( W1 * ELU( W3 (*) b + b3 ) + b1 + b ) with b zero-padded, without b in memory.
 * Per set: w3_packed = the composed 3x3 conv W3'_tap = W3_tap Win (cwfa_tc_pack_weights, Cin_p = 8 in_chunks, BN = 64),
 * b3 = b3 + sum_tap W3_tap bin, b1 = b1 + bin, win_packed = Win (1x1, Cin_p = 8 in_chunks, BN = 64), edge = fp32 [16][64]:
 * row (r * 4 + c) = sum of W3_tap bin over the taps outside the image for a pixel of row class r (bit 0: first image row,
 * bit 1: last) and column class c (bit 0: first column, bit 1: last); all 16-byte aligned. */
int cwfa_resblock_tc_batched(const void* x_c8, void* y_c8, int n_sets, const void* const* w3_packed,
                             const void* const* w1_packed, const float* const* b3, const float* const* b1, int N, int H, int W,
                             int in_total_chunks, const int* in_chunk_off, int out_total_chunks, const int* out_chunk_off,
                             const void* const* win_packed, const float* const* edge, int in_chunks, int is_bf16, void* stream);
/* ---- C8 helpers of the LRNN U-Net: per-channel (sum, sumsq) over (N,H,W) -> stats[2*Cp]
 * (workspace >= cwfa_c8_stats_workspace_floats(Cp) floats; feed to cwfa_bn_finalize_f32), and BatchNorm
 * apply y = x*scale+shift, optionally also writing the 2x2 max-pooled tensor (unet.py:79).
 * scale / shift must be 16-byte aligned; N * Cp/8 <= 65535. */
/* PReLU on a C8 tensor (y = x >= 0 ? x : slope[0] * x) and its adjoint g = dy * PReLU'(pre) with the per-channel sums
 * stats[c] = sum g (bias gradient of the producing convolution), stats[Cp + c] = sum dy * min(pre, 0) (its sum over c is the
 * slope gradient); workspace: cwfa_c8_stats_workspace_floats(Cp).  Training path of the conditioning net's depth stencil
 * (networks.py:221-225): the hidden tensor stays in the C8 half layout between the two tensor-core convolutions. */
int cwfa_c8_prelu(const void* x, const float* slope, void* y, int N, int Cp, int64_t P, int is_bf16, void* stream);
int cwfa_c8_prelu_bwd(const void* dy, const void* pre, const float* slope, void* g, float* stats, float* workspace, int N,
                      int Cp, int64_t P, int is_bf16, void* stream);
/* ELU adjoint on C8 tensors from the activation's OUTPUT y: g = dy * (y > 0 ? 1 : y + 1); stats[c] = sum g (the bias gradient of
 * the convolution whose epilogue applied the ELU), stats[Cp + c] = 0.  Training path of the coupling sub-networks
 * (networks.py:624-638) with activations and cotangents kept in the C8 layout. */
int cwfa_c8_elu_bwd(const void* dy, const void* y, void* g, float* stats, float* workspace, int N, int Cp, int64_t P, int is_bf16,
                    void* stream);
int cwfa_c8_stats_workspace_floats(int Cp);
int cwfa_c8_channel_stats(const void* x, float* stats, float* workspace, int N, int Cp, int64_t P,
                          int is_bf16, void* stream);
/* BatchNorm in batch-statistics mode on a C8 tensor: per-channel sums (cwfa_c8_channel_stats' first pass) and, in the same
 * finalize launch, scale = gamma / sqrt(var + eps), shift = beta - mean * scale (biased variance, unet.py:100-107).
 * workspace: cwfa_c8_stats_workspace_floats(Cp) floats. */
int cwfa_c8_bn_batch_scale_shift(const void* x, const float* gamma, const float* beta, float eps, float* scale, float* shift,
                                 float* workspace, int N, int Cp, int64_t P, int is_bf16, void* stream);
int cwfa_c8_bn_apply(const void* x, const float* scale, const float* shift, void* y, void* ypool,
                     int N, int Cp, int H, int W, int is_bf16, void* stream);
/* col2im of a 3x3 convolution evaluated as ONE 1x1 tensor-core convolution to 9 partial products per output channel
 * (second depth-stencil conv of the conditioning net, networks.py:221-225,239: Cin = 32*D, Cout = D):
 * out[n,d,y,x] = bias[d] + sum_{ky,kx} g[n, (d/8)*72 + (ky*3+kx)*8 + d%8, y+ky-1, x+kx-1].  g: C8 with Gp >= 9*Dp channels,
 * out: C8 with Dp channels (Dp % 8 == 0; 8-channel chunks beyond Gp/72 are channel padding and are written as zeros),
 * bias: Dp floats or NULL. */
int cwfa_c8_col2im3x3(const void* g, const float* bias, void* out, int N, int Dp, int Gp, int H, int W,
                      int is_bf16, void* stream);

/* The conditioning net's depth stencil Conv3d(1 -> 32, 3) -> PReLU -> Conv3d(32 -> 1, 3) over the (H, W, depth) volume
 * (networks.py:221-225 applied at :239) as ONE fused tcgen05 kernel in its true 3-D form (csrc/stencil_tc.cu): GEMM rows are
 * voxels, the 32-channel hidden volume stays in shared / tensor memory.
 * x: C8 tensor [N][cin_chunks][H][W][8] whose first D channels are the depths; y: C8 [N][cout_chunks][H][W][8] (channels >= D
 * are written as zeros; cout_chunks even).  wpack (half precision of the tensor's kind, 6144 bytes):
 *   W1[kd] [2 chunks][32 hidden][8], kd = 0..2: k = kh*3+kw < 9 the first conv's spatial taps at depth tap kd; for kd = 1,
 *   k = 9 / 10 hold the [hi | lo] split of its bias;
 *   W2[kd] [4 chunks][16][8], kd = 0..2: row n = kh*3+kw (< 9), k = hidden channel: the second conv's taps.
 * b2: the second conv's bias (1 float), slope: the PReLU slope (1 float); both read on the device.
 * rows_max: GEMM rows per pixel-row of a strip (multiple of 128, <= 768; 0 = default). 1 <= D <= 64. */
int cwfa_stencil3d_tc(const void* x, void* y, const void* wpack, const float* b2, const float* slope, int N, int H, int W,
                      int D, int cin_chunks, int cout_chunks, int rows_max, int is_bf16, void* stream);

/* LayerNorm([C,H,W]) of the LRNN's ConvNeXt blocks (networks.py:486-503) on C8 tensors: per-sample statistics over the
 * C*H*W true elements (channel padding must be zero), y = (x - mean) * rstd * gamma + beta with the element-wise affine
 * parameters given as C8 tensors of shape (1, Cp, H, W) (zero in the padding).  workspace: cwfa_c8_layernorm_workspace_floats(N). */
int cwfa_c8_layernorm_workspace_floats(int N);
int cwfa_c8_layernorm(const void* x, const void* gamma, const void* beta, void* y, float* workspace, int N, int C, int Cp,
                      int64_t P, float eps, int is_bf16, void* stream);
/* ---- K2+K3+K4 fused: the LAST conv of a coupling sub-network (networks.py:635-638) with the affine coupling
 * (coupling_layers.py:490-500), the per-sample log-det partial sums and the preceding permutation's gather
 * (fixed_transforms.py:37-41, INN_utils.py:73-81) in its epilogue.  Conv columns [0,ch) = s_raw, [ch,2ch) = t,
 * or t = t_scale * ct when ct != NULL (networks.py:671).  cx (may be NULL = zeros in inverse mode) is read as
 * cx[gather]; cy is written densely.  workspace: 2 * N * cwfa_conv_tc_coupling_tiles(H,W,MB) floats; reduce it
 * with cwfa_coupling_finalize (fixed order => bit-reproducible): logdet[n] (+)= sum s (sign per direction),
 * sumsq[n] = sum y^2. */
int cwfa_conv_tc_coupling_tiles(int H, int W, int MB);
int cwfa_conv_tc_coupling(const void* x_c8, const void* w_packed, const float* bias, int N, int H, int W,
                          int Cin_p, int Cout, int Cout_p, int KH, int KW, int MB, const float* cx, float* cy,
                          const float* ct, float t_scale, const int32_t* perm, int perm_axis, int ch,
                          float clamp, float k_atan, int inverse, float* workspace, int is_bf16, void* stream);
int cwfa_coupling_finalize(const float* workspace, float* logdet, float* sumsq, int N, int tiles,
                           int accumulate, void* stream);
/* Persistent variant of cwfa_conv_tc_coupling for the CWFA sub-network shape (3x3 conv from 64 hidden channels to
 * Cout_p <= 96 in one N block, ch <= 48): weights resident in shared memory, accumulators double buffered in TMEM,
 * 16 epilogue warps.  workspace: 2 * N * cwfa_coupling_tc_tiles(H, W) floats (one (sum s, sum y^2) partial per tile and
 * epilogue warp).  ticket != NULL (one int32 that is zero on entry; left zero on exit): the last CTA to finish reduces the
 * partials in a fixed order inside the kernel, logdet[n] = (accumulate ? logdet[n] : 0) + sum, sumsq[n] = sum y^2 (may be
 * NULL) -- no finalize launch.  ticket == NULL: reduce with cwfa_coupling_finalize(..., tiles = cwfa_coupling_tc_tiles(H, W), ...). */
int cwfa_coupling_tc_tiles(int H, int W);
int cwfa_coupling_tc(const void* b_c8, const void* w_packed, const float* bias, int N, int H, int W, int Cout,
                     int Cout_p, const float* cx, float* cy, const float* ct, float t_scale, const int32_t* perm,
                     int perm_axis, int ch, float clamp, float k_atan, int inverse, float* workspace, float* logdet,
                     float* sumsq, int accumulate, int32_t* ticket, int in_total_chunks, int in_chunk_off, int is_bf16,
                     void* stream);
/* ---- the coupling path on the "F8" layout of a level's detail half: [N][ceil(ch/8)][H][W][8] fp32, channel padding zero
 * (csrc/coupling_f8.cu).  cwfa_coupling_f8 = cwfa_coupling_tc with a lean epilogue: x / y / external shift as 128-bit
 * vectors, no channel gather (the caller permutes the OUTPUT CHANNELS of w_packed so that [s | t] arrive in storage order:
 * columns [0,chp8) = s of slot j, [chp8,2 chp8) = t of slot j; with ct != NULL columns [0,chp8) = s only), bias through an
 * extra MMA, row (perm_axis 2) / column (perm_axis 3) permutations as a gather on cx.  chp8 = 8 * ceil(ch / 8) <= 48; BN =
 * number of conv output columns (one n-block, multiple of 16, <= 96).  b_c8 is the 64-channel slice (8 chunks from in_chunk_off)
 * of a C8 tensor with in_total_chunks chunks (cwfa_coupling_tc likewise).  workspace / logdet / sumsq / accumulate / ticket as in
 * cwfa_coupling_tc (tiles = cwfa_coupling_tc_tiles(H, W)). */
int cwfa_coupling_f8(const void* b_c8, const void* w_packed, const float* bias, int N, int H, int W, int BN, int chp8,
                     const float* cx, float* cy, const float* ct, float t_scale, const int32_t* perm, int perm_axis,
                     float clamp, float k_atan, int inverse, float* workspace, float* logdet, float* sumsq, int accumulate,
                     int32_t* ticket, int in_total_chunks, int in_chunk_off, int is_bf16, void* stream);
/* cwfa_coupling_f8 for `samples` latent samples of each condition image (inverse only; posterior statistics): cx / cy hold
 * N * samples F8 rows, row n * samples + k = sample k of condition image n; b_c8, ct and logdet stay per condition image.  s and
 * t are computed once per tile and applied to every sample, each sample's y bitwise equal to cwfa_coupling_f8 on its row.
 * samples >= 1 (1 = cwfa_coupling_f8); with samples > 1: inverse = 1, cx != NULL, sumsq = NULL, samples * chp8 * H * W < 2^31. */
int cwfa_coupling_f8_samples(const void* b_c8, const void* w_packed, const float* bias, int N, int samples, int H, int W, int BN,
                             int chp8, const float* cx, float* cy, const float* ct, float t_scale, const int32_t* perm, int perm_axis,
                             float clamp, float k_atan, int inverse, float* workspace, float* logdet, float* sumsq, int accumulate,
                             int32_t* ticket, int in_total_chunks, int in_chunk_off, int is_bf16, void* stream);
/* cwfa_coupling_f8 in the forward direction (inverse = 0, cx != NULL) that also accumulates each detail element's NLL term into
 * nll_map (F8, fp32, the layout of cx / cy): the couplings of a level are elementwise, so an element's NLL is 0.5 z^2 - sum of s
 * over the level's blocks.  nll_map is indexed by the element's coordinate at the level's INPUT: the block adds -s (and, in the
 * last block, 0.5 y^2) at [n][c / 8][row_src[h]][col_src[w]][c % 8] for the element it writes at (h, w); row_src / col_src are
 * int32 tables composed from the level's row / column permutations (NULL = identity).  map_mode: CWFA_NLL_MAP_FIRST writes
 * without reading nll_map, 0 adds to it, CWFA_NLL_MAP_LAST adds 0.5 y^2 too (FIRST | LAST for a level of one block).  Padding
 * slots come out 0; cy, logdet and sumsq are bitwise those of cwfa_coupling_f8. */
#define CWFA_NLL_MAP_FIRST 1
#define CWFA_NLL_MAP_LAST 2
int cwfa_coupling_f8_map(const void* b_c8, const void* w_packed, const float* bias, int N, int H, int W, int BN, int chp8,
                         const float* cx, float* cy, const float* ct, float t_scale, const int32_t* perm, int perm_axis,
                         float clamp, float k_atan, int inverse, float* workspace, float* logdet, float* sumsq, int accumulate,
                         int32_t* ticket, int in_total_chunks, int in_chunk_off, int is_bf16, void* stream, float* nll_map,
                         const int32_t* row_src, const int32_t* col_src, int map_mode);
/* cwfa_coupling_f8 in the inverse direction (inverse = 1) that also carries each detail element's scale along the level's chain
 * of couplings: s and t come from the conditions only, so a level's detail half is affine in its latent, hi = beta + alpha * z
 * with alpha = exp(-sum of the blocks' s).  scale_in (F8, fp32, the layout of cx; NULL = 1, the first block in inverse order) is
 * gathered through perm like cx; scale_out = scale_in * exp(-s) is written where cy is.  cy, logdet and sumsq are bitwise those
 * of cwfa_coupling_f8.  Rejected: inverse == 0, scale_out == NULL, scale_out == scale_in (in-place use races with the gather). */
int cwfa_coupling_f8_scale(const void* b_c8, const void* w_packed, const float* bias, int N, int H, int W, int BN, int chp8,
                           const float* cx, float* cy, const float* ct, float t_scale, const int32_t* perm, int perm_axis,
                           float clamp, float k_atan, int inverse, float* workspace, float* logdet, float* sumsq, int accumulate,
                           int32_t* ticket, int in_total_chunks, int in_chunk_off, int is_bf16, void* stream,
                           const float* scale_in, float* scale_out);
/* cwfa_haar1d_inv_f8 fused with the exact per-voxel standard deviation of the merged volume when the detail half is
 * hi + sigma * scale * z with independent unit-variance latents z and lo carries the independent std std_lo (NULL = 0):
 * std_x[2i] = std_x[2i+1] = sqrt(0.5 (std_lo_i^2 + sigma^2 scale_i^2)), correctly rounded sqrt.  x is bitwise cwfa_haar1d_inv_f8's.
 * Rejected: sigma < 0 or not finite, a NULL lo / hi_f8 / scale_f8 / x / std_x, odd C, P % 4 != 0, unaligned pointers. */
int cwfa_haar1d_inv_std_f8(const float* lo, const float* std_lo, const float* hi_f8, const float* scale_f8, float sigma, float* x,
                           float* std_x, int B, int C, int64_t P, void* stream);
/* Posterior mean and exact standard deviation of R region readouts r = sum_v w_v V_v of each of B volumes, when every level's
 * detail half is hi_n + sigma * scale_n * z_n with independent unit-variance latents (cwfa_coupling_f8_scale):
 * mean[b, r] = sum_v w_v vol[b, v] and std[b, r] = sigma sqrt(sum_n sum_e (coef_n[e] scale_n[b, e])^2), fp64 sums, written (B, R).
 * vol: B items of vol_stride floats (the z = 0 volume).  scale_f8, scale_stride: HOST arrays of L device pointers to the F8 scale
 * tensors and their floats per batch item.  Tables (device, RoiSet in cwfa_b200/data.py): mean_ptr (R + 1) int64 and
 * (mean_idx, mean_w), a CSR over ROIs of (offset into one volume, weight); coef_ptr (L, R + 1) int64 and (coef_idx, coef_val),
 * level n's CSR over ROIs of (offset into one item of scale_f8[n], coefficient), offsets into the shared arrays.  One warp per
 * (b, ROI), no atomics: bitwise reproducible.  Rejected before any device access: L outside 1..8, sigma < 0 or not finite,
 * R < 1, B < 1, a stride < 1, a NULL pointer (also in scale_f8[0..L-1]). */
int cwfa_roi_readout_f8(const float* vol, int64_t vol_stride, const float* const* scale_f8, const int64_t* scale_stride, int L,
                        const int64_t* mean_ptr, const int32_t* mean_idx, const float* mean_w, const int64_t* coef_ptr,
                        const int32_t* coef_idx, const float* coef_val, int B, int R, float sigma, float* mean, float* std,
                        void* stream);
/* Split^-1 + IDWT of K >= 2 latent samples fused with their per-voxel mean and unbiased standard deviation (Welford): the K
 * merged volumes are never written.  lo: K rows (B, C/2, P) or, lo_shared = 1, one row for every sample; hi: K rows in F8
 * (hi_f8 = 1; P % 4 == 0, 16-byte aligned) or NCHW; mean, std: (C, P) each. */
int cwfa_haar1d_inv_stats(const float* lo, int lo_shared, const float* hi, int hi_f8, float* mean, float* std, int K, int C,
                          int64_t P, void* stream);
/* Depth-wise Haar DWT + Split (INN_utils.py:142-161, graph_topology.py:73-80) with the detail half written / read in F8:
 * fwd: x (B,C,P) -> lo (B,C/2,P) NCHW, hi F8;  inv: lo, hi F8 -> x.  P % 4 == 0, pointers 16-byte aligned; every access 128-bit. */
int cwfa_haar1d_fwd_f8(const float* x, float* lo, float* hi_f8, int B, int C, int64_t P, void* stream);
int cwfa_haar1d_inv_f8(const float* lo, const float* hi_f8, float* x, int B, int C, int64_t P, void* stream);
/* NCHW fp32 <-> F8 with an optional int32 channel map (NULL = identity): to_f8: slot j = channel map[j]; to_nchw: channel c =
 * slot map[c] (the flow's accumulated channel permutation, fixed_transforms.py:37-41, applied once at the boundary). */
int cwfa_nchw_to_f8(const float* x, const int32_t* map, float* y_f8, int B, int C, int64_t P, void* stream);
int cwfa_f8_to_nchw(const float* x_f8, const int32_t* map, float* y, int B, int C, int64_t P, void* stream);
/* Layout converters NCHW fp32 <-> C8 half (channels padded with zeros up to Cp). */
int cwfa_nchw_to_c8(const float* x, void* y, int N, int C, int Cp, int64_t P, int is_bf16, void* stream);
int cwfa_c8_to_nchw(const void* x, float* y, int N, int C, int Cp, int64_t P, int is_bf16, void* stream);

/* ==== training-time adjoints of the fp32 module path (csrc/backward.cu) =========================================
 * The reference trains one flow level at a time with torch autograd (CWFA.py:928-1015: inverse pass WITH gradients for
 * the MSE term, forward pass for the NLL term, backward, Lion step).  These are the hand-written adjoints of the forward
 * kernels above; cwfa_b200/autograd.py is the only caller. */
/* conv2d weight gradient dW[co,ci,kh,kw] = sum_{n,h,w} dy[n,co,h,w] * x[n,ci,h+kh-p,w+kw-p] of the stride-1 'same' convs
 * (square kernels 1x1 / 3x3 / 7x7: every conv of the coupling sub-networks networks.py:611-638, of the conditioning net's
 * 2-D part :211-219 and the ConvNeXt 7x7 of the LRNN :489).  Deterministic two-stage sum; workspace >= cwfa_conv2d_wgrad_workspace_floats(...) floats.
 * accumulate != 0: dw += result.  The DATA gradient is cwfa_conv2d_f32(dy, wt) with wt from cwfa_conv2d_dgrad_weights_f32
 * (wt[ci,co,kh,kw] = w[co,ci,KH-1-kh,KW-1-kw]); the bias gradient is cwfa_channel_stats_f32(dy). */
int64_t cwfa_conv2d_wgrad_workspace_floats(int N, int Cin, int H, int W, int Cout, int KH, int KW);
int cwfa_conv2d_wgrad_f32(const float* x, const float* dy, float* dw, float* workspace, int N, int Cin, int H, int W,
                          int Cout, int KH, int KW, int accumulate, void* stream);
int cwfa_conv2d_dgrad_weights_f32(const float* w, float* wt, int Cout, int Cin, int KH, int KW, void* stream);
/* Convolution weight gradient on the tcgen05 tensor cores (csrc/wgrad_tc.cu): x and dy are C8 half tensors (Cin_p / Cout_p
 * channels; output channels in M blocks of 128), dW is (Cout,Cin,KH,KW) fp32, square kernels 1x1 / 3x3, stride 1, 'same'.  The contraction over
 * pixels runs as M=128 x N<=64 x K=16 MMAs on MN-major operands (the C8 tile is the operand as TMA lands it; a tap is a
 * descriptor offset); one fp32 partial per CTA, fixed-order final sum.  workspace >= cwfa_wgrad_tc_workspace_floats(...). */
int64_t cwfa_wgrad_tc_workspace_floats(int N, int H, int W, int Cin, int Cin_p, int Cout, int Cout_p, int KH);
int cwfa_wgrad_tc(const void* x_c8, const void* dy_c8, float* dw, float* workspace, int N, int H, int W, int Cin, int Cin_p,
                  int Cout, int Cout_p, int KH, int KW, int is_bf16, void* stream);
/* ELU(alpha=1) adjoint from the layer OUTPUT y: dv = dy * (y > 0 ? 1 : y + 1)  (dv may alias dy). */
int cwfa_elu_bwd_f32(const float* dy, const float* y, float* dv, int64_t n, void* stream);
/* Cotangent preparation of a tensor-core convolution's backward pass in ONE pass over dy: g = dy * ELU'(y) when y != NULL (else
 * g = dy), written as the C8 half tensor g8 [N][Cp/8][P][8] the data / weight gradient MMAs read (channels >= C zero), optionally
 * also as fp32 NCHW (g32, may be NULL), and db[c] = sum over (n, pixels) of g = the bias gradient (db may be NULL; deterministic
 * two-stage sum).  workspace: cwfa_dy_prep_workspace_floats(N, Cp) floats (needed when db != NULL).
 * Replaces cwfa_elu_bwd_f32 + cwfa_nchw_to_c8 + cwfa_channel_stats in the autograd of nn.Conv2d (CWFA.py:996). */
int cwfa_dy_prep_workspace_floats(int N, int Cp);
int cwfa_dy_prep(const float* dy, const float* y, void* g8, float* g32, float* db, float* workspace, int N, int C, int Cp,
                 int64_t P, int is_bf16, void* stream);
/* out = alpha*a + beta*b (b may be NULL). */
int cwfa_axpby_f32(const float* a, const float* b, float* out, float alpha, float beta, int64_t n, void* stream);
/* nn.PReLU() with one shared slope (networks.py:209) as a stand-alone op and its adjoint: dv = v > 0 ? dy : a*dy,
 * dslope[0] = sum_{v<=0} v*dy (torch's convention at 0).  workspace >= cwfa_reduce_workspace_blocks() floats. */
int cwfa_prelu_f32(const float* v, const float* slope, float* y, int64_t n, void* stream);
int cwfa_reduce_workspace_blocks(void);
int cwfa_prelu_bwd_f32(const float* dy, const float* v, const float* slope, float* dv, float* dslope, float* workspace,
                       int64_t n, void* stream);
/* Adjoint of cwfa_affine (same argument meaning; coupling_layers.py:490-500).  dy = cotangent of y, g_logdet (B, may be NULL)
 * = cotangent of logdet.  Outputs (each may be NULL): dx (B,ch,P); da_s / da_t with batch strides ld_ds / ld_dt so that both
 * halves of one (B,2ch,P) sub-network output gradient are written in place. */
int cwfa_affine_bwd(const float* x, const float* a_s, const float* a_t, const float* dy, const float* g_logdet, float* dx,
                    float* da_s, float* da_t, int B, int ch, int64_t P, int64_t ld_s, int64_t ld_t, int64_t ld_ds,
                    int64_t ld_dt, float clamp, float k_atan, float t_scale, int flags, void* stream);
/* The conditioning net's depth stencil (networks.py:221-225,239) UNFUSED, for training: Conv3d(1,Cm,3,p1) and
 * Conv3d(Cm,1,3,p1) over the (H,W,depth) volume of a (B,D,H,W) tensor; hidden tensors are (B,Cm,D,H,W); weights (Cm,27)
 * with tap = (kh*3+kw)*3+kd.  flip != 0 applies the point-reflected kernel = the adjoint of the OTHER conv
 * (d hidden = 1toC(dy, w2, flip); dx = Cto1(d pre-activation, w1, flip)).  bias may be NULL.
 * wgrad: dw[c,t] = sum multi[b,c,pos] * single[b,pos+t] (1->Cm weights: single = x, multi = d pre-activation, flip 0;
 * Cm->1 weights: single = dy, multi = hidden, flip 1).  workspace >= cwfa_stencil3d_wgrad_workspace_floats(Cm) floats. */
int cwfa_stencil3d_1toC_f32(const float* x, const float* w, const float* bias, float* out, int B, int D, int H, int W,
                            int Cm, int flip, void* stream);
int cwfa_stencil3d_Cto1_f32(const float* hid, const float* w, const float* bias, float* out, int B, int D, int H, int W,
                            int Cm, int flip, void* stream);
int cwfa_stencil3d_wgrad_workspace_floats(int Cm);
int cwfa_stencil3d_wgrad_f32(const float* single, const float* multi, float* dw, float* workspace, int B, int D, int H,
                             int W, int Cm, int flip, void* stream);
/* LRNN U-Net adjoints (unet.py:72-113,161-195).  channel_dot_stats: out[c] = sum dy, out[C+c] = sum dy*x over (N,H,W)
 * (workspace >= 2*C*cwfa_channel_dot_workspace_blocks() floats); bn_bwd_apply: dx = a[c]*dy + b[c]*x + c0[c] (the BatchNorm
 * adjoint once the per-channel coefficients are known); maxpool2_bwd: gradient to the first maximum of each 2x2 window
 * (x is the pooling INPUT (N,C,H,W), dy (N,C,H/2,W/2)); pixel_shuffle2: y[n,c,2h+i,2w+j] = z[n,4c+2i+j,h,w] (+ skip), C = channels
 * of y, (H,W) = size of z -- with a 1x1 convolution in front this is ConvTranspose2d(k=2,s=2) + skip add (unet.py:166,190);
 * inverse != 0 is its adjoint (un-shuffle of src = y into dst = z). */
int cwfa_channel_dot_workspace_blocks(void);
int cwfa_channel_dot_stats_f32(const float* x, const float* dy, float* out, float* workspace, int N, int C, int64_t P, void* stream);
int cwfa_bn_bwd_apply_f32(const float* dy, const float* x, const float* a, const float* b, const float* c0, float* dx,
                          int N, int C, int64_t P, void* stream);
int cwfa_maxpool2_bwd_f32(const float* x, const float* dy, float* dx, int N, int C, int H, int W, void* stream);
int cwfa_pixel_shuffle2_f32(const float* src, const float* skip, float* dst, int N, int C, int H, int W, int inverse, void* stream);
/* LRNN mean-volume branch adjoints (networks.py:244-262, 486-503, 554).  act_bwd: adjoint of ELU / ReLU / sigmoid from the layer
 * OUTPUT (kind = CWFA_ACT_*).  gelu_add: dy == NULL: out = gelu(v) + r (r may be NULL); else out = dy * gelu'(v).
 * ln_bwd_stats: out[b] = sum dy*gamma, out[B+b] = sum dy*gamma*x over the n = C*H*W elements of sample b
 * (workspace >= 2*B*cwfa_channel_dot_workspace_blocks() floats); ln_bwd_apply: coef = B x (mean, rstd, mean g, mean g*xhat):
 * dx = rstd*(gamma*dy - mean g - xhat*mean(g xhat)), dgamma[p] = sum_b dy*xhat, dbeta[p] = sum_b dy (each output may be NULL).
 * gate: dy == NULL: out0 = x + m*2*(g-0.5); else out0 = dy*2*(g-0.5) (= dm), out1 = dy*2*m (= dg). */
int cwfa_act_bwd_f32(const float* dy, const float* y, float* dv, int64_t n, int kind, void* stream);
int cwfa_gelu_add_f32(const float* v, const float* r, const float* dy, float* out, int64_t n, void* stream);
int cwfa_ln_bwd_stats_f32(const float* x, const float* dy, const float* gamma, float* out, float* workspace, int B, int64_t n, void* stream);
int cwfa_ln_bwd_apply_f32(const float* x, const float* dy, const float* gamma, const float* coef, float* dx, float* dgamma,
                          float* dbeta, int B, int64_t n, void* stream);
int cwfa_gate_f32(const float* x, const float* m, const float* g, const float* dy, float* out0, float* out1, int64_t n, void* stream);
/* Lion update on a flat fp32 buffer (lion_pytorch 0.0.7, requirements.txt:1; call sites CWFA.py:381,608-610):
 * p *= 1 - lr*wd; p -= lr*sign(beta1*m + (1-beta1)*g); m = beta2*m + (1-beta2)*g, with g read as g*grad_scale. */
int cwfa_lion_step_f32(float* p, const float* g, float* m, int64_t n, float lr, float beta1, float beta2,
                       float weight_decay, float grad_scale, void* stream);
/* The same with a per-element byte mask (may be NULL): elements with mask 0 are left untouched -- lion_pytorch skips parameters whose
 * .grad is None (e.g. the unused block_grad_up / block1|block12 / block7|block72 weights of the sub-networks). */
int cwfa_lion_step_masked_f32(float* p, const float* g, float* m, const uint8_t* mask, int64_t n, float lr, float beta1,
                              float beta2, float weight_decay, float grad_scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CWFA_B200_H */
