/* e2fgvi_b200 — C ABI of the sm_100a hot-path kernels behind E2FGVI's InpaintGenerator.forward.
 *
 * The reference (MCG-NKU/E2FGVI) is pure Python and has no C ABI of its own; each entry point below replaces
 * one operator boundary of the reference and cites it.  A reference maintainer binds these with ctypes (see
 * INTEGRATION.md).  Conventions:
 *   - every pointer is a DEVICE pointer owned by the caller; the library never allocates or frees caller memory
 *     and keeps no persistent device state (TMA descriptors are built per call on the host);
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream); calls are asynchronous on it and
 *     re-entrant across streams;
 *   - return value: 0 = OK, negative = argument error (E2F_ERR_*), positive = cudaError_t of the launch;
 *     e2f_last_error() returns a thread-local human-readable message for the last non-zero return;
 *   - activation layout is NHWC ("channels last"), i.e. [N][H][W][C] contiguous; token tensors are
 *     [B][T][H][W][C] contiguous.
 */
#ifndef E2FGVI_B200_H_
#define E2FGVI_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define E2F_OK 0
#define E2F_ERR_BAD_ARG (-1)
#define E2F_ERR_UNSUPPORTED (-2)
#define E2F_ERR_ALIGNMENT (-3)
#define E2F_ERR_DRIVER (-4)

/* layouts of the deformable-conv input x */
#define E2F_X_NHWC 0     /* [N][H][W][Cin] */
#define E2F_X_GROUPED 1  /* [N][G][H][W][Cin/G] with G = deform_groups (group-major, see e2f_dcn_pack_input) */

/* element types */
#define E2F_F32 0
#define E2F_F16 1
#define E2F_SPLIT_BF16 2 /* e2f_focal_window_attention only: out = [2][B][T][H][W][C] bf16, the (hi, lo) two-term split
                          * of the fp32 result = the A operand pair of the following e2f_linear_bf16x3 (attn.proj) */

/* padding modes of e2f_flow_warp (reference: F.grid_sample padding_mode) */
#define E2F_PAD_ZEROS 0
#define E2F_PAD_BORDER 1

/* Library / build identification: "e2fgvi_b200 <version> sm_100a". */
const char* e2f_version(void);
/* Thread-local message describing the last failing call on this thread ("" if none). */
const char* e2f_last_error(void);

/* flow_warp — replaces model/modules/flow_comp.py:345-383 (bilinear grid_sample at pixel+flow,
 * align_corners=True, so the normalise/denormalise round trip cancels: sample at (x+flow[...,0], y+flow[...,1])).
 *   x    [N][H][W][C]  (dtype: E2F_F32 or E2F_F16)        flow [N][H][W][2] fp32 (u = x-displacement first)
 *   out  [N][H][W][C]  (same dtype as x)
 * C must be a multiple of 4 (fp32) / 8 (fp16), or C <= 4 for the small-channel path (flows, RGB). */
int e2f_flow_warp(const void* x, const float* flow, void* out, int n, int h, int w, int c, int dtype,
                  int pad_mode, void* stream);

/* flow_warp on NCHW fp32 tensors (the reference's native layout), used for few-channel inputs
 * (2-channel flows in feat_prop.py:120, 3-channel images in flow_comp.py:127). */
int e2f_flow_warp_nchw(const float* x, const float* flow, float* out, int n, int c, int h, int w, int pad_mode,
                       void* stream);

/* Pack a DCN weight [Cout][Cin][3][3] fp32 (mmcv / torch layout, feat_prop.py:13 via ModulatedDeformConv2d)
 * into the fp16 GEMM operand [Cout][K], K = 9*Cin, k = (g*9 + tap)*cpg + c_in_group with cpg = Cin/deform_groups.
 * This K order makes one 64-wide K block = 64/cpg consecutive sample points of the sampler. */
int e2f_dcn_pack_weight(const float* w, void* w_packed_f16, int cout, int cin, int deform_groups, void* stream);

/* modulated_deform_conv2d — replaces mmcv.ops.modulated_deform_conv2d as called at feat_prop.py:55-58
 * (3x3, stride 1, padding 1, dilation 1, groups 1).  Sampling + im2col are fused into the tcgen05 GEMM; no
 * column buffer is materialised.
 *   x        fp16, [N][H][W][Cin] (x_layout = E2F_X_NHWC) or group-major (E2F_X_GROUPED)     offset [N][H][W][2*9*dg] fp32, channel (g*9+tap)*2 + {0:dy, 1:dx}
 *   mask     [N][H][W][9*dg] fp32 (already sigmoid-ed), channel g*9+tap
 *   w_packed [Cout][9*Cin] fp16 from e2f_dcn_pack_weight      bias [Cout] fp32 or NULL
 *   out      [N][H][W][Cout] (out_dtype E2F_F32 or E2F_F16)
 * Supported: Cin = 256, Cout = 128, dg = 16 (the only instance on the path). */
int e2f_modulated_deform_conv2d(const void* x, const float* offset, const float* mask, const void* w_packed,
                                const float* bias, void* out, int n, int h, int w, int cin, int cout,
                                int deform_groups, int out_dtype, int x_layout, void* stream);

/* cat([a, b], channel).half() in the group-major layout E2F_X_GROUPED (feat_prop.py:126 builds the DCN input as
 * cat([feat_prop, feat_n2])): a [N][H][W][Ca], b [N][H][W][Cb] fp32 NHWC -> xg [N][(Ca+Cb)/16][H][W][16] fp16.
 * Ca, Cb multiples of 16. */
int e2f_dcn_pack_input(const float* a, const float* b, void* xg, int n, int h, int w, int ca, int cb, void* stream);

/* Fused SecondOrderDeformableAlignment tail — replaces feat_prop.py:41-58: takes the raw 27*dg-channel output of
 * conv_offset (`head`, [N][H][W][27*dg] fp32: o1 | o2 | mask), applies offset = max_residue * tanh(o) +
 * flow_k.flip(1) (first half of the groups uses flow_1, second half flow_2), mask = sigmoid(.), then the DCN.
 *   flow1, flow2 [N][H][W][2] fp32 (u, v). */
int e2f_deform_align_fused(const void* x, const float* head, const float* flow1, const float* flow2,
                           const void* w_packed, const float* bias, void* out, int n, int h, int w, int cin,
                           int cout, int deform_groups, float max_residue, int out_dtype, int x_layout,
                           void* stream);

/* e2f_deform_align_fused with fp32 output PLUS the bf16 (hi, lo) split of the same values ([N][H][W][Cout] each): the
 * operand pair of the backbone conv that consumes the aligned features (feat_prop.py:131-136), written by the DCN
 * epilogue so that no separate split pass sits on the serial propagation chain. */
int e2f_deform_align_fused_split(const void* x, const float* head, const float* flow1, const float* flow2,
                                 const void* w_packed, const float* bias, float* out, void* out_hi, void* out_lo, int n,
                                 int h, int w, int cin, int cout, int deform_groups, float max_residue, int x_layout,
                                 void* stream);

/* Temporal focal window attention core — replaces model/modules/tfocal_transformer.py:226-396 (everything in
 * WindowAttention.forward between the qkv Linear and the proj Linear): window partition of q, the own-window keys,
 * the 4 circularly rolled ring key sets (with their duplicated tokens), the pooled-window keys with the -100
 * logit on zero-padded neighbours, softmax and P*V, written back un-partitioned (fuses window_reverse :528).
 *   qkv        [B][T][H][W][3*C] fp16  (q | k | v, each C = heads*head_dim, head-major inside C)
 *   qkv_pooled [B][T][nWh][nWw][3*C] fp16 (the same Linear applied to the pooled window tokens; q part unused)
 *   out        [B][T][H][W][C] (out_dtype)
 *   window (wh, ww); expand (eh, ew) = window//2; focal window (fh, fw) (pooled neighbourhood, odd sizes);
 *   nWh = H/wh, nWw = W/ww.  scale multiplies q.k (head_dim^-0.5).  head_dim must be 128.
 *   use_pooled = 0 runs focal_level 1 (no pooled keys). */
int e2f_focal_window_attention(const void* qkv, const void* qkv_pooled, void* out, int b, int t, int h, int w,
                               int heads, int head_dim, int wh, int ww, int eh, int ew, int fh, int fw,
                               int use_pooled, float scale, int out_dtype, void* stream);

/* T2T token <-> image transforms, replacing F.unfold / F.fold as used by SoftSplit (tfocal_transformer.py:39-43),
 * SoftComp (:65-72) and FusionFeedForward (:89-96).  img [BT][C][H][W] fp32 (NCHW), tokens [BT][L][C*k*k] fp32 with
 * L = fh*fw, fh = (H+2p-k)/s+1, channel = c*k*k + ky*k + kx (torch.nn.Unfold order), i.e. the token-major layout
 * the Linears produce / consume (no transposes).
 *   e2f_t2t_unfold: tokens = unfold(img); gelu != 0 applies the exact (erf) GELU of FusionFeedForward.conv2[0].
 *                   Outputs (at least one): tokens fp32 and/or tokens_hi, tokens_lo bf16 (the split operand pair of
 *                   the following e2f_linear_bf16x3).
 *   e2f_t2t_fold  : img = fold(tokens); normalize != 0 divides by fold(ones) (the overlap count, :92-96);
 *                   bias (NULL or [C][H][W]) is added after (SoftComp.bias, :60-63,71). */
int e2f_t2t_unfold(const float* img, float* tokens, void* tokens_hi, void* tokens_lo, int bt, int c, int h, int w,
                   int k, int stride, int pad, int gelu, void* stream);
int e2f_t2t_fold(const float* tokens, const float* bias, float* img, int bt, int c, int h, int w, int k, int stride,
                 int pad, int normalize, void* stream);
/* e2f_t2t_fold writing a channels_last image [BT][H][W][C] = fold(tokens) (/ fold(ones)) (+ bias [C][H][W]) (+ residual
 * [BT][H][W][C]): SoftComp's output with "enc_feat + trans_feat" (e2fgvi.py:263) fused into the store, in the layout
 * the decoder's convs read.  Only k=7, stride=3, pad=3 with C % 8 == 0 (E2F_ERR_UNSUPPORTED otherwise). */
int e2f_t2t_fold_nhwc(const float* tokens, const float* bias, const float* residual_nhwc, float* img_nhwc, int bt, int c,
                      int h, int w, int k, int stride, int pad, int normalize, void* stream);
/* e2f_t2t_unfold reading a channels_last image [BT][H][W][C] (what the conv / linear epilogues write), so SoftSplit
 * needs no NHWC -> NCHW copy.  Only k=7, stride=3, pad=3 with C % 8 == 0 (E2F_ERR_UNSUPPORTED otherwise). */
int e2f_t2t_unfold_nhwc(const float* img_nhwc, float* tokens, void* tokens_hi, void* tokens_lo, int bt, int c, int h, int w,
                        int k, int stride, int pad, int gelu, void* stream);

/* FusionFeedForward's middle (tfocal_transformer.py:89-96) in ONE launch:
 *   out = gelu?( unfold( fold(tokens_in) / fold(ones) ) ), tokens [BT][L][C*k*k] -> tokens [BT][L][C*k*k];
 * the folded image stays in shared memory.  Fused for k=7, stride=3, pad=3 (the only geometry on the path); returns
 * E2F_ERR_UNSUPPORTED otherwise, and the caller composes e2f_t2t_fold(normalize=1) + e2f_t2t_unfold.  Outputs as
 * e2f_t2t_unfold (fp32 and/or bf16 hi/lo pair), with rows of out_pitch elements (0 = C*k*k; otherwise a multiple of 4
 * >= C*k*k, columns past C*k*k written as zeros): 1960 -> 1984 makes every row of the following GEMM's A operand
 * start on a 128-byte line, which its TMA loads want. */
int e2f_t2t_fold_unfold(const float* tokens_in, float* tokens, void* tokens_hi, void* tokens_lo, int bt, int c, int h,
                        int w, int k, int stride, int pad, int gelu, int out_pitch, void* stream);

/* Window pooling of the focal attention's coarse level: pool_layers[0] = nn.Linear(wh*ww, 1) across the tokens of
 * every window, per channel (tfocal_transformer.py:508-516, the permute/Linear/squeeze chain):
 *   out[bt][wi][wj][c] = bias[0] + sum_{r<wh, q<ww} x[bt][wi*wh + r][wj*ww + q][c] * weight[r*ww + q]
 * x_hi / x_lo [BT][H][W][C] bf16 = the split LayerNorm output (e2f_layernorm_split), weight [wh*ww] fp32, bias [1]
 * fp32 or NULL.  Outputs (at least one): out [BT][H/wh][W/ww][C] fp32 and/or its bf16 (hi, lo) split — the operand of
 * the pooled qkv Linear.  (The reference orders the pooled tokens (B, nWh, nWw, T, C); this is its
 * permute(0,3,1,2,4), which is what the qkv Linear + attention consume.) */
int e2f_window_pool(const void* x_hi, const void* x_lo, const float* weight, const float* bias, float* out, void* out_hi,
                    void* out_lo, int bt, int h, int w, int c, int wh, int ww, void* stream);

/* norm1 + focal window pooling in ONE pass (tfocal_transformer.py:470 and :508-516): LayerNorm of every token and, from
 * the normalised values still in registers, the pooled token of every (frame, window),
 *   pooled[bt][wi][wj][c] = pool_b[0] + sum_{r<wh, q<ww} pool_w[r*ww + q] * LN(x)[bt][wi*wh + r][wj*ww + q][c].
 * x [BT][H][W][C] fp32 (C = 512, H % wh == W % ww == 0).  out_hi / out_lo: bf16 [(BT*H*W + BT*(H/wh)*(W/ww))][C] — rows
 * [0, BT*H*W) hold the split normalised tokens, the following BT*nW rows the split pooled tokens ordered (bt, wi, wj):
 * one e2f_linear_bf16x3 over all rows yields qkv and qkv_pooled of e2f_focal_window_attention back to back. */
int e2f_layernorm_pool_split(const float* x, const float* gamma, const float* beta, const float* pool_w,
                             const float* pool_b, void* out_hi, void* out_lo, int bt, int h, int w, int c, int wh, int ww,
                             float eps, void* stream);

/* x2 bilinear upsample, align_corners=True (F.interpolate in deconv.forward, e2fgvi.py:125-129) of an NHWC fp32
 * tensor [N][H][W][C] (C % 8 == 0), written directly as the bf16 (hi, lo) split [N][2H][2W][C] consumed by
 * e2f_conv3x3_bf16x3 — the 4x larger fp32 intermediate is never materialised.  x must be 32-byte aligned (256-bit loads). */
int e2f_upsample2x_split(const float* x, void* out_hi, void* out_lo, int n, int h, int w, int c, void* stream);

/* nn.LayerNorm over the last dimension (tfocal_transformer.py:470 norm1, :533 norm2; C = 512):
 * y = (x - mean) / sqrt(var + eps) * gamma + beta, biased variance.  Outputs (at least one): out fp32 [rows][C]
 * and/or out_hi, out_lo bf16 (split operand pair of the following e2f_linear_bf16x3). */
int e2f_layernorm_split(const float* x, const float* gamma, const float* beta, float* out, void* out_hi, void* out_lo,
                        int64_t rows, int c, float eps, void* stream);

/* fp32 -> two-term bf16 split (x = hi + lo, hi = bf16(x), lo = bf16(x - hi)); n must be a multiple of 8. */
int e2f_split_bf16(const float* x, void* hi_bf16, void* lo_bf16, int64_t n, void* stream);

/* nn.Linear replacement (tfocal_transformer.py:44, :68, :89, :97, :221, :398) with fp32-level accuracy on the bf16
 * tensor pipe:  out[M][N] = A[M][K] . W[N][K]^T + bias[N] (+ residual[M][N]),  evaluated as Ah.Wh + Ah.Wl + Al.Wh
 * with fp32 accumulation (relative error ~2^-17; TF32 would be 2^-11).
 *   a_hi/a_lo [M][K] bf16, w_hi/w_lo [N][K] bf16 (from e2f_split_bf16), bias [N] fp32 or NULL,
 *   residual [M][N] fp32 or NULL, out [M][N] fp32 (E2F_F32) or fp16 (E2F_F16).
 *   K % 8 == 0; N % 4 == 0 (fp32 out) / N % 8 == 0 (fp16 out).  tile_hint: 0 = auto, 128 or 256 = N tile. */
int e2f_linear_bf16x3(const void* a_hi, const void* a_lo, const void* w_hi, const void* w_lo, const float* bias,
                      const float* residual, void* out, int m, int n, int k, int out_dtype, int tile_hint,
                      void* stream);

/* 3x3 / stride 1 / pad 1 convolution (nn.Conv2d at e2fgvi.py:75-94,143-150; feat_prop.py:20-28,73-77) as a tcgen05
 * implicit GEMM with fp32-level accuracy (bf16 3-term split, like e2f_linear_bf16x3):
 *   out = leaky_relu(conv(cat(src_0 .. src_{nsrc-1}, channel dim), W) + bias, slope) (+ residual)
 * without materialising the concatenation or an im2col buffer (TMA boxes with zero-filled out-of-bounds = padding).
 *   src_hi[i], src_lo[i]  [N][H][W][C_i] bf16 (e2f_split_bf16 of the NHWC fp32 activation), C_i % 8 == 0, nsrc <= 4
 *   groups G: group g convolves channels [g*C_i/G, (g+1)*C_i/G) of every source (in source order) into output
 *             channels [g*Cout/G, (g+1)*Cout/G)   (== nn.Conv2d(groups=G) on the group-wise concatenation of
 *             e2fgvi.py:103-108)
 *   w_hi, w_lo [Cout][9 * T * 64] bf16 with T = sum_i ceil((C_i/G)/64): k = ((tap*T + chunk_base_i + j)*64 + c),
 *             zero where c >= C_i/G - 64 j (see e2fgvi_b200.ops.pack_conv3x3_weight)
 *   bias [Cout] fp32 or NULL; residual [N][H][W][Cout] fp32 or NULL; leaky_slope = 1 disables the activation.
 *   Outputs (at least one): out [N][H][W][Cout] fp32 and/or out_hi, out_lo [N][H][W][Cout] bf16 = the two-term
 *   split of the result, i.e. directly the operand format of a following e2f_conv3x3_bf16x3 (Cout % 8 == 0). */
int e2f_conv3x3_bf16x3(int nsrc, const void* const* src_hi, const void* const* src_lo, const int* src_channels,
                       const void* w_hi, const void* w_lo, const float* bias, const float* residual, float* out,
                       void* out_hi, void* out_lo, int n, int h, int w, int cout, int groups, float leaky_slope,
                       void* stream);

/* Generalisation of e2f_conv3x3_bf16x3 to square k x k kernels (k = 3, 7), stride 1 or 2 and any zero padding:
 * the stride-2 encoder convs (e2fgvi.py:76,80) and SPyNet's 7x7 convs (flow_comp.py:181-215; leaky_slope = 0 is
 * ReLU).  h, w are the INPUT spatial size; outputs are [N][Ho][Wo][Cout] with Ho = (h + 2 pad - k)/stride + 1.
 * Weights: [Cout][k*k * T * 64] in the same tap-major order. */
int e2f_conv2d_bf16x3(int nsrc, const void* const* src_hi, const void* const* src_lo, const int* src_channels,
                      const void* w_hi, const void* w_lo, const float* bias, const float* residual, float* out,
                      void* out_hi, void* out_lo, int n, int h, int w, int cout, int groups, float leaky_slope,
                      int ksize, int stride, int pad, void* stream);

/* Small-channel convolutions (SPyNet's 7x7 convs with 8 / 32 / 16 input channels, flow_comp.py:181-215; the 3-channel
 * stride-2 stem, e2fgvi.py:76) with "window-packed" K, and the row-gapped layout that feeds them.
 *
 * Row-gapped NHWC: [N][H][P][C] bf16 (hi, lo) followed by e2f_conv_rows_tail(lead, C) pixels, with the row pitch
 * P = e2f_conv_rows_pitch(W, lead, C) = lead + W (rounded up to a 16-byte row for C = 4); pixel (y, x) lives at
 * y*P + lead + x; the `lead` pixels in front of every row, any rounding pixel behind it and the tail are zero.  With lead = the consuming conv's padding the gap is the left
 * padding of its row and the right padding of the previous one, and 64/C consecutive pixels x C channels form one
 * contiguous 64-element K chunk — a whole slice of a kernel row — that TMA fetches as a sliding window (tensor-map
 * pixel stride = one pixel).  A 7x7 conv over 8 channels takes 7 K chunks per tile instead of 49 zero-padded ones.
 *
 *   e2f_pack_rows_bf16     : NCHW fp32 [N][C][H][W] (C <= cin, cin in {4, 8, 16, 32}) -> row-gapped (hi, lo) with cin
 *                            channels (extra channels zero).
 *   e2f_conv2d_rows_bf16x3 : e2f_conv2d_bf16x3 plus
 *       in_rows  != 0: src_hi[0] / src_lo[0] is ONE row-gapped source with lead == pad and src_channels[0] = cin
 *                      (nsrc == 1, groups == 1, stride*cin*2 % 16 == 0).  Weights: [Cout][k * G * 64] with
 *                      G = ceil(k / PX), PX = 64 / cin:  K index ((ky*G + g)*64 + px*cin + c)  <->  W[co][c][ky][g*PX+px],
 *                      zero for g*PX + px >= k (see e2fgvi_b200.ops.pack_conv_rows_weight).
 *       out_lead  > 0: out_hi / out_lo are written row-gapped with this lead ([N][Ho][out_lead + Wo][Cout] + tail, Cout >= 8,
 *                      gaps and tail zeroed by the kernel) for a following window-packed conv; 0 = dense NHWC.
 *   e2f_conv_rows_pitch / e2f_conv_rows_tail : row pitch and number of tail pixels of a row-gapped buffer (host
 *                            arithmetic, no CUDA call). */
int e2f_conv_rows_pitch(int w, int lead, int channels);
int e2f_conv_rows_tail(int lead, int channels);
int e2f_pack_rows_bf16(const float* x, void* out_hi, void* out_lo, int n, int c, int h, int w, int cin, int lead,
                       void* stream);
int e2f_conv2d_rows_bf16x3(int nsrc, const void* const* src_hi, const void* const* src_lo, const int* src_channels,
                           int in_rows, const void* w_hi, const void* w_lo, const float* bias, const float* residual,
                           float* out, void* out_hi, void* out_lo, int out_lead, int n, int h, int w, int cout, int groups,
                           float leaky_slope, int ksize, int stride, int pad, void* stream);

/* The decoder's output conv with its tanh and the NCHW layout of the result fused into the epilogue — replaces
 * `torch.tanh(self.decoder(...))` (model/e2fgvi.py:149-150 last nn.Conv2d(64, 3, 3, 1, 1) and :262) and the
 * channels-last -> NCHW copy of the prediction: out [N][Cout][H][W] fp32 = tanh(conv3x3(x) + bias), x as one NHWC bf16
 * (hi, lo) source with cin channels (cin % 8 == 0), weights packed like e2f_conv3x3_bf16x3, Cout <= 32 and not a
 * multiple of 4 (the 3-channel image). */
int e2f_conv3x3_tanh_nchw(const void* src_hi, const void* src_lo, int cin, const void* w_hi, const void* w_lo,
                          const float* bias, float* out, int n, int h, int w, int cout, void* stream);

/* "kx-in-N" k x k / stride 1 / pad k/2 convolution for layers with FEW output channels — SPyNet's 64 -> 32, 32 -> 16 and
 * 16 -> 2 7x7 convs (model/modules/flow_comp.py:181-215) and the decoder's 64 -> 3 output conv (model/e2fgvi.py:149-150).
 * The kernel-COLUMN taps go into the GEMM's N dimension, D[(y, xin), (kx, co)] = sum_{ky, c} X[y+ky-pad, xin, c] * W[co,c,ky,kx],
 * and the epilogue adds the kx columns with a horizontal shift (warp shuffles: one warp per tile row), out[y, x, co] =
 * sum_kx D[(y, x+kx-pad), (kx, co)]: one read of an A tile feeds k times more output columns, so these layers are bound
 * by tensor math instead of by re-reading the A operand for every tap.
 * Also the encoder's groups-of-32 conv (model/e2fgvi.py:97, 640 -> 256, groups 8: 32 + 48 input and 32 output channels per
 * group), whose 64-wide N tiles / K chunks were half zero padding in the plain kernel: a tile is (pixels, group).
 *   src_hi / src_lo: nsrc <= 2 NHWC bf16 (hi, lo) sources [N][H][W][src_channels[i]] (multiples of 8 and of `groups`); the
 *                    group-local input channel axis is the concatenation of the sources' per-group slices (the
 *                    group-wise torch.cat of e2fgvi.py:103-108), never materialised
 *   w_hi / w_lo:     [groups * k*co_pad rows][k*chunks*64] bf16: row = g*k*co_pad + kx*co_pad + co, column =
 *                    (ky*chunks + chunk)*64 + c, chunks = sum_i ceil(src_channels[i]/groups/64) with source 0's chunks
 *                    first (zeros for co >= Cout/groups and padded channels); co_pad % 8 == 0, <= 32, k*co_pad % 16 == 0
 *   epilogue: + bias[Cout], LeakyReLU(leaky_slope) (1 = none, 0 = ReLU), + residual (NHWC fp32 [N][H][W][Cout] or NULL),
 *             flags bit 0: tanh, bit 1: fp32 output stored NCHW ([N][Cout][H][W]); outputs: out fp32 NHWC (or NCHW) and / or
 *             the bf16 (hi, lo) split NHWC [N][H][W][Cout] (Cout/groups % 8 == 0). */
int e2f_conv_kxn_bf16x3(int nsrc, const void* const* src_hi, const void* const* src_lo, const int* src_channels,
                        const void* w_hi, const void* w_lo, const float* bias, const float* residual, float* out, void* out_hi,
                        void* out_lo, int n, int h, int w, int cout, int groups, int co_pad, int ksize, float leaky_slope,
                        int flags, void* stream);

/* "Gather conv": the same implicit GEMM with an explicit TAP TABLE, OUTPUT PHASES and tile shape (groups == 1).
 * Replaces, without ever building the unfolded operand:
 *   - SoftSplit (model/modules/tfocal_transformer.py:39-46; HQ _hq.py:39-46): F.unfold(7x7, stride 3, pad 3) + nn.Linear
 *     IS a 7x7 / stride-3 conv 128 -> 512: one phase, 49 taps (dy = ky - 3, dx = kx - 3), stride = 3, GEMM grid = the
 *     token grid, tokens written as the NHWC output [BT][fh][fw][512].  The 49x larger unfolded token matrix
 *     (1.3 GB per call at 8 clips) does not exist.
 *   - SoftComp (tfocal_transformer.py:65-72; _hq.py:67-79): nn.Linear(512 -> 49*128) + F.fold IS the transposed conv.
 *     Output pixel (3a + ry, 3b + rx) sums token (a + 1 - dy, b + 1 - dx) times W[(c, 3dy + ry, 3dx + rx), :] over the
 *     taps with 3dy + ry <= 6, 3dx + rx <= 6: nine phases (ry, rx) with 9 / 6 / 4 taps, stride = 1, GEMM grid = token
 *     grid, ostep = 3.  The 6272-wide token matrix and the fold pass do not exist; the folded Linear bias (+ the base
 *     model's sc.bias[c, y, x], tfocal_transformer.py:60-63) arrives as `bias_map`, `enc_feat + trans_feat`
 *     (e2fgvi.py:263) as `residual`.
 * Tap i reads input pixel (y*stride + tap_dy[i], x*stride + tap_dx[i]) (zero outside); phase ph owns taps
 * [ph_tap0[ph], ph_tap0[ph+1]) and writes output pixel (y*ostep + ph_oy[ph], x*ostep + ph_ox[ph]) of the
 * out_h x out_w image for every GEMM-grid pixel (y, x) in grid_h x grid_w.  Weights: [Cout][ntaps * T * 64] bf16
 * (hi, lo), tap-major (in table order), then source, then 64-channel chunk (T = chunks over all sources).
 * tile_w * tile_h <= 128 grid pixels per tile (12 x 10 tiles the 20x36 / 60x108 / 90x162 token grids exactly).
 * bias: per-channel [Cout] or NULL; bias_map: fp32 [out_h][out_w][Cout] or NULL; residual: fp32 NHWC of the output.
 * Batch strides (pixels between consecutive images; NULL / 0 = dense) let a source or the output be ONE FRAME of a
 * (b, t, h, w, c) buffer — the per-frame tensors of BidirectionalPropagation (feat_prop.py:88-149) are then read and
 * written in place, with no gather / stack copies: src_nstride[i] for source i, out_nstride for out, out_hi / out_lo and
 * the residual alike. */
int e2f_conv_gather_bf16x3(int nsrc, const void* const* src_hi, const void* const* src_lo, const int* src_channels,
                           const void* w_hi, const void* w_lo, const float* bias, const float* bias_map,
                           const float* residual, float* out, void* out_hi, void* out_lo, int n, int h_in, int w_in,
                           int cout, float leaky_slope, int stride, int grid_h, int grid_w, int tile_w, int tile_h,
                           int ntaps, const int8_t* tap_dy, const int8_t* tap_dx, int nphase, const uint8_t* ph_tap0,
                           const uint8_t* ph_oy, const uint8_t* ph_ox, int ostep, int out_h, int out_w,
                           const int64_t* src_nstride, int64_t out_nstride, void* stream);

/* Fused prologue of one propagation step (SURVEY 8(f) rank 3) — replaces feat_prop.py:106-126 up to the offset-head conv:
 * the two feature warps, the second-order flow (flow_n1 + warp(flow_prev, flow_n1)), the operand splits of the offset
 * head's conv sources and the fp16 group-major DCN input, in one launch.
 *   prop, feat_n2     [N][H][W][C] fp32 NHWC (feat_n2 may be NULL: second frame of a sweep -> cond_n2, flow_n2, the second
 *                     half of x are zeros); C % 16 == 0
 *   flow_n1, flow_prev  fp32 planes [2][H][W] per image (u then v), image i at + i*bstride elements (a slice of the
 *                     [B][T-1][2][H][W] flow tensor); flow_prev NULL iff feat_n2 NULL
 *   cond1_hi/lo, cond2_hi/lo  [N][H][W][C] bf16: (hi, lo) split of flow_warp(prop, flow_n1) / flow_warp(feat_n2, flow_n2)
 *   flow1_out, flow2_out      [N][H][W][2] fp32: flow_n1 and flow_n2 in the layout e2f_deform_align_fused reads
 *   flows_hi/lo       [N][H][W][8] bf16 split of cat(flow_n1, flow_n2) (4 channels + 4 zero), conv operand
 *   x_grouped         [N][2C/16][H][W][16] fp16 = e2f_dcn_pack_input(prop, feat_n2)
 * Bit-identical to the unfused sequence of e2f_flow_warp / e2f_flow_warp_nchw / add / e2f_split_bf16 / e2f_dcn_pack_input. */
int e2f_prop_prologue(const float* prop, const float* feat_n2, const float* flow_n1, int64_t flow_n1_bstride,
                      const float* flow_prev, int64_t flow_prev_bstride, void* cond1_hi, void* cond1_lo, void* cond2_hi,
                      void* cond2_lo, float* flow1_out, float* flow2_out, void* flows_hi, void* flows_lo, void* x_grouped,
                      int n, int h, int w, int c, void* stream);

/* SPyNet glue (model/modules/flow_comp.py:84-169, model/e2fgvi.py:210-234) — one bidirectional flow estimate is
 * 1 + 6 x (1 + five 7x7 convs) + 1 launches.
 *   e2f_spynet_pyramid: frames (b, t, 3, H, W) fp32 in [-1, 1] -> for every LOCAL frame (j < l_t; index bi*l_t + j) the
 *     six normalised pyramid levels: (x + 1) / 2 (e2fgvi.py:247), 1/4 bilinear downsample to h x w (align_corners=True,
 *     e2fgvi.py:214-218), bilinear resize to h_up x w_up = multiples of 32 (align_corners=False, flow_comp.py:152-158),
 *     (v - mean) / std (mean3 / std3: device pointers to the 3 buffer values, flow_comp.py:95-96), five 2x2 average
 *     pools (:101-115).  `pyramid`: levels 0..5 back to back, level k = [b*l_t][3][h_up >> k][w_up >> k] fp32.
 *   e2f_spynet_level_input: one pyramid level -> the level's network input for all P = 2*b*(l_t-1) (ref, supp) pairs
 *     (direction-major: forward pairs (j, j+1) of every clip, then the backward pairs (j+1, j); e2fgvi.py:221-229):
 *     flow_up = 2 * bilinear_x2(prev_flow) (align_corners=True, flow_comp.py:121-126; prev_flow NULL = level 0, zero
 *     flow), border-mode warp of the support image (:128-132), cat([ref, warped, flow_up]) (:127-133) written as the
 *     row-gapped 8-channel bf16 (hi, lo) operand of e2f_conv2d_rows_bf16x3 (lead zero pixels per row + tail, see
 *     e2f_conv_rows_pitch / _tail) and flow_up [P][hk][wk][2] fp32 — the residual the level's last conv adds.
 *     prev_flow: [P][hk/2][wk/2][2] fp32.
 *   e2f_spynet_final: level-5 flow [P][h_up][w_up][2] fp32 -> bilinear resize to h x w (align_corners=False) and the
 *     u * w / w_up, v * h / h_up rescale (flow_comp.py:160-167), written as flows_forward / flows_backward
 *     (b, l_t - 1, 2, h, w) fp32 — pred_flows of InpaintGenerator.forward. */
int e2f_spynet_pyramid(const float* frames, float* pyramid, int b, int t, int l_t, int H, int W, int h, int w, int h_up,
                       int w_up, const float* mean3, const float* std3, void* stream);
int e2f_spynet_level_input(const float* level_img, const float* prev_flow, void* rows_hi, void* rows_lo, float* flow_up,
                           int b, int l_t, int hk, int wk, int lead, void* stream);
int e2f_spynet_final(const float* flow, float* flows_forward, float* flows_backward, int b, int l_t, int h, int w, int h_up,
                     int w_up, void* stream);

/* Output stitch over NVLink / NVSwitch peer memory (SURVEY 8(e): clips are the sharding unit, the only exchange is the
 * all-gather of the output frames — the multi-GPU form of test.py:168-179 collecting every window's frames into one list).
 * Each rank owns a landing buffer and PUSHES its block of frames into every peer's buffer with DMA copies (copy engines,
 * no SMs: an NCCL all-gather kernel takes SMs from the persistent kernels of the next forward, csrc/peer.cu).
 *   e2f_peer_alloc : cudaMalloc `bytes` (an IPC handle names a whole allocation, so no caching allocator) and export
 *                    the 64-byte CUDA IPC handle other processes open.
 *   e2f_peer_open  : map a peer's buffer into this process (lazily enables peer access); e2f_peer_close unmaps it.
 *   e2f_peer_copy  : asynchronous device-to-device copy of one block on `stream` (local or peer destination).
 *   e2f_peer_signal: 32-bit flag word (local or peer memory) := value, stream-ordered (cuStreamWriteValue32, no kernel).
 *   e2f_peer_wait  : `stream` stalls until (int32)(*flag - value) >= 0 (cuStreamWaitValue32); flag in LOCAL memory.
 * Protocol (e2fgvi_b200/clips.py, PeerStitcher): per step a rank tells every peer "my landing buffer k may be
 * overwritten", waits for the same word from the peer, pushes its block, then raises the peer's "block landed" word. */
int e2f_peer_alloc(size_t bytes, void** ptr, unsigned char* handle64);
int e2f_peer_open(const unsigned char* handle64, void** ptr);
int e2f_peer_close(void* ptr);
int e2f_peer_free(void* ptr);
int e2f_peer_copy(void* dst, const void* src, size_t bytes, void* stream);
int e2f_peer_signal(void* flag, unsigned int value, void* stream);
int e2f_peer_wait(void* flag, unsigned int value, void* stream);

/* Video-level driver (SURVEY 8(f) rank 4) — replaces the per-window host / eager-torch code of test.py:132-179.
 * All buffers are device memory; `frames` [N][H][W][3] uint8 RGB, `masks` [N][H][W] uint8 (non-zero = hole, already
 * dilated like test.py:55-68), `ids` int32 frame indices of the window (neighbours first, then reference frames).
 *   e2f_video_prepare_clip : out[k][c][y][x] fp32, k < t, y < hp, x < wp  =  (frames[ids[k]]/255*2-1) * (1-mask),
 *                            mirror-padded from (h, w) to (hp, wp) exactly like test.py:156-165
 *                            (cat(x, flip(x))[:h + h_pad]); needs h <= hp <= 2h, w <= wp <= 2w.
 *   e2f_video_compose      : img[k][y][x][c] uint8, k < n_local = hole ? uint8(((pred+1)/2)*255) : frame
 *                            (test.py:167-174); pred is [>= n_local][3][hp][wp] fp32.
 *   e2f_video_blend        : comp[ids[k]] = first[k] ? img[k] : comp*0.5 + img[k]*0.5, comp fp32 [N][frame_elems]
 *                            (test.py:175-179); windows must be blended in schedule order.
 *   e2f_video_finalize     : out uint8 = truncation of comp (test.py:195).
 * Results are bit-identical to the reference's numpy / torch-CPU arithmetic. */
int e2f_video_prepare_clip(const uint8_t* frames, const uint8_t* masks, const int* ids, float* out, int t, int h, int w,
                           int hp, int wp, void* stream);
int e2f_video_compose(const float* pred, const uint8_t* frames, const uint8_t* masks, const int* ids, uint8_t* img,
                      int n_local, int h, int w, int hp, int wp, void* stream);
int e2f_video_blend(const uint8_t* img, const int* ids, const int* first, float* comp, int n_local, int64_t frame_elems,
                    void* stream);
int e2f_video_finalize(const float* comp, uint8_t* out, int64_t count, void* stream);

/* Per-frame PSNR and SSIM of evaluate.py (core/metrics.py:20-53: calculate_psnr, and scikit-image 0.16
 * compare_ssim(ref, test, data_range, multichannel=True, win_size) with scipy's uniform window), in fp64.
 *   ref  [N][H][W][3] uint8 (the original frames), test [N][H][W][3] fp32 (the canvas), psnr / ssim [N] fp64.
 *   psnr[f] = 20 log10(data_range / sqrt(mean((ref - test)^2))), +inf when the frames are equal;
 *   ssim[f] = mean over the 3 channels and over the outputs whose win_size x win_size window lies inside the frame
 *             of skimage's S, with C1 = (0.01 data_range)^2, C2 = (0.03 data_range)^2 and sample covariances.
 * win_size must be odd, >= 3 and <= min(H, W) (skimage raises ValueError otherwise), and <= 255 (E2F_ERR_UNSUPPORTED).
 * `workspace` is device memory of at least e2f_psnr_ssim_workspace_bytes(n, h, w, win_size) bytes, 8-byte aligned;
 * a smaller one is not detected.  e2f_psnr_ssim_workspace_bytes returns 0 for arguments e2f_psnr_ssim rejects.
 * Deterministic: a frame's result does not depend on the other frames of the call, and no atomics are used. */
size_t e2f_psnr_ssim_workspace_bytes(int n, int h, int w, int win_size);
int e2f_psnr_ssim(const uint8_t* ref, const float* test, double* psnr, double* ssim, int n, int h, int w, int win_size,
                  double data_range, void* workspace, void* stream);

/* Number of kernel launches issued through this library since load (all threads); used by bench.py's
 * "gpu_launches" accounting. */
int64_t e2f_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* E2FGVI_B200_H_ */
