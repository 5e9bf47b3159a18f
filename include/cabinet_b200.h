/* libcabinet_b200.so — C-ABI of the B200-native CABiNet forward hot path.
 *
 * Plain pointers and sizes only (no torch types).  Every pointer is a DEVICE pointer unless the
 * parameter is documented as host; every entry point enqueues work on `stream` (a cudaStream_t
 * passed as void*) and returns without synchronising.  Return value: 0 = ok, CABINET_ERR_INVALID
 * = rejected arguments, CABINET_ERR_CUDA = CUDA runtime/driver failure; cabinet_last_error()
 * gives the message (thread-local).  The library allocates no persistent device memory: the
 * caller (PyTorch's caching allocator in the shipped host code) owns all buffers.
 *
 * Activations are NHWC; `ld*` arguments are the PIXEL stride in elements (>= channels), which is
 * how channel-concatenation (reference torch.cat) is expressed without a copy.  Element types are
 * CABINET_F32, CABINET_BF16 and, in the training entry points the fp16 training mode calls, CABINET_F16; an entry point
 * given a type it does not implement returns CABINET_ERR_INVALID before it launches anything.  The `*_dt` variants of
 * the tensor-core and staging entry points take the 2-byte operand type (CABINET_BF16 or CABINET_F16) as their last
 * argument before `stream`; the names without the suffix are the CABINET_BF16 case.  The reference is pure PyTorch (SURVEY F1): each entry point cites
 * the reference Python it replaces (paths relative to the reference repo root); there is no
 * pre-existing FFI in the reference, INTEGRATION.md shows the binding a maintainer would add.
 */
#ifndef CABINET_B200_H
#define CABINET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CABINET_ABI_VERSION 2

enum { CABINET_OK = 0, CABINET_ERR_INVALID = 1, CABINET_ERR_CUDA = 2 };
enum { CABINET_F32 = 0, CABINET_BF16 = 1, CABINET_F16 = 2 };
enum {
    CABINET_ACT_NONE = 0,
    CABINET_ACT_RELU = 1,     /* nn.ReLU */
    CABINET_ACT_HSWISH = 2,   /* src/models/mobilenetv3.py:53-65 */
    CABINET_ACT_HSIGMOID = 3, /* src/models/mobilenetv3.py:38-50 */
    CABINET_ACT_SIGMOID = 4   /* nn.Sigmoid */
};
/* OR into the `act` argument of the cabinet_conv_tc* entry points: walk the output tiles back to front, so a layer whose
 * input is larger than L2 starts on the part its producer wrote last (still L2 resident).  Results are identical. */
#define CABINET_CONV_REVERSE_TILES 0x100

/* One unit of the 64-bit fixed-point per-(image, channel) pooling sums that the depthwise kernels accumulate for the
 * squeeze-excite gate: value = raw * 2^-24.  Integer accumulation is associative, which makes the sums (and everything
 * downstream) bit-reproducible whatever the order in which the thread blocks finish. */
#define CABINET_GAP_FIXED_ONE 16777216.0f

typedef void* cabinet_stream_t; /* cudaStream_t */

const char* cabinet_last_error(void);
int cabinet_abi_version(void);
/* Fills SM count and compute capability of the current device. */
int cabinet_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* Kernel-development switches (bench/debug only; 0 = normal operation). Returns the previous value. */
int cabinet_debug_flags(int flags);
int cabinet_debug_read(long long* host_out, int n);

/* ---------------------------------------------------------------------------------------------
 * Dense convolution + folded-BN bias + activation + residual, CUDA-core implicit GEMM
 * (fp32 accumulate).  The fp32 parity mode of the whole path and the Cin=3 stems run here.
 * Replaces nn.Conv2d -> nn.BatchNorm2d(eval) -> {ReLU,HardSwish,-} [-> x + .] at
 *   src/models/cabinet.py:19-44 (ConvBNReLU), :59-63,68-72 (conva, convb, b1-b4),
 *   src/models/mobilenetv3.py:86-99 (stems), :126-151 (pw convs), src/models/cab.py:58-63,107-128.
 * Also used as a batched GEMM (grid over `batches`) for the fp32-mode attention products
 *   src/models/cab.py:149-153 (torch.bmm).
 *   out[b][m][co] = act( sum_k x_patch[b][m][k] * w[b][co*w_sco + k*w_sk] + bias[co] ) + res[b][m][co]
 * x is addressed with explicit element strides (sxn, sxh, sxw, sxc) so both NHWC activations and the
 * fp32 NCHW network input are read in place; k runs over (ky, kx, c) with c fastest.
 */
int cabinet_conv2d_simt(const void* x, int x_dtype, long long sxn, long long sxh, long long sxw, long long sxc,
                        long long x_batch_stride,
                        const void* w, int w_dtype, long long w_sco, long long w_sk, long long w_batch_stride,
                        const float* bias,
                        const void* res, long long ldres,
                        void* y, int y_dtype, long long ldy, long long y_batch_stride,
                        int batches, int N, int H, int W, int Cin, int Cout, int KH, int KW, int stride, int pad,
                        int OH, int OW, int act, float alpha, cabinet_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * The same convolution on the tensor cores: tcgen05.mma (bf16 x bf16 -> fp32 in TMEM), operands staged by TMA
 * (im2col-free implicit GEMM: one shifted 4-D box per filter tap, zero padding = TMA out-of-bounds fill).
 * bf16 NHWC input (16-byte aligned pixels), stride 1 or 2, any kernel size / padding.
 * w_packed: bf16 [ceil16(Cout)][KH*KW][ceil64(Cin)] (zero padded, BN folded).  y: bf16 or fp32 NHWC.
 * Replaces the same reference call sites as cabinet_conv2d_simt in the bf16 mode; the dense k x k layers
 * (src/models/cabinet.py:59-63,68,111-114,159) are the tensor-bound ones.
 *   out[m][co] = act( sum_k x_patch[m][k] * w[co][k] + bias[co] ) + res[m][co] */
int cabinet_conv_tc(const void* x, long long ldx, int N, int H, int W, int Cin, const void* w_packed, int Cout,
                    int KH, int KW, int stride, int pad, const float* bias, const void* res, long long ldres,
                    void* y, int y_dtype, long long ldy, int OH, int OW, int act, cabinet_stream_t stream);
/* The same with bf16 or fp16 operands (op_dtype; x, w_packed and a 2-byte y all of that type). */
int cabinet_conv_tc_dt(const void* x, long long ldx, int N, int H, int W, int Cin, const void* w_packed, int Cout,
                       int KH, int KW, int stride, int pad, const float* bias, const void* res, long long ldres,
                       void* y, int y_dtype, long long ldy, int OH, int OW, int act, int op_dtype, cabinet_stream_t stream);

/* cabinet_conv_tc (stride 1, no activation / residual, bf16) writing a strided VIEW of a larger NHWC tensor: output pixel
 * (n, oh, ow) lands at y + ((n * y_sn) + oh * y_sh + ow * y_sw) * ldy (pitches in pixels).  With the sub-filters of
 * cabinet_pack_conv_weight_parity, four calls (one per input parity) are the data gradient of a stride-2 convolution
 * on the tensor cores (backward of sb.conv2 / sb.conv3, src/models/cabinet.py:112-113). */
int cabinet_conv_tc_view(const void* x, long long ldx, int N, int H, int W, int Cin, const void* w_packed, int Cout, int KH,
                         int KW, int pad, const float* bias, void* y, long long ldy, int OH, int OW, long long y_sw,
                         long long y_sh, long long y_sn, cabinet_stream_t stream);
int cabinet_conv_tc_view_dt(const void* x, long long ldx, int N, int H, int W, int Cin, const void* w_packed, int Cout, int KH,
                            int KW, int pad, const float* bias, void* y, long long ldy, int OH, int OW, long long y_sw,
                            long long y_sh, long long y_sn, int op_dtype, cabinet_stream_t stream);

/* cabinet_conv_tc with the squeeze-excite apply fused in front (A-operand prologue): the GEMM consumes
 * act(x[n][p][c] * a_scale[n][c]) (a_scale fp32 [N][Cin]) without that tensor ever being written:
 * SELayer's x * y (src/models/mobilenetv3.py:83) and the activation that follows it (:143) run in shared memory
 * between the TMA load and the MMA.  Linear project convs only (act must be CABINET_ACT_NONE, bf16 output). */
int cabinet_conv_tc_se(const void* x, long long ldx, int N, int H, int W, int Cin, const float* a_scale, int a_act,
                       const void* w_packed, int Cout, int KH, int KW, int stride, int pad, const float* bias,
                       const void* res, long long ldres, void* y, int y_dtype, long long ldy, int OH, int OW, int act,
                       cabinet_stream_t stream);

/* Both network stems in one tensor-core kernel: sb.conv1 (7x7 s2 p3, 3->64, BN, ReLU; src/models/cabinet.py:111)
 * and the backbone stem (3x3 s2 p1, 3->16, BN, HardSwish; src/models/mobilenetv3.py:86-91,173) read the fp32 NCHW
 * image x [N][3][H][W] once (W % 4 == 0) and write their bf16 NHWC outputs.  w_packed: bf16 [80][192] with
 * k = (c*7 + ky)*8 + kx (rows 0-63 = 7x7 filters at kx 1..7, rows 64-79 = the 3x3 filters embedded at ky 2..4,
 * kx 3..5; zero elsewhere), BN-folded; the folded bias rides in K slots 168 / 169 as bf16 hi / lo parts (the kernel
 * feeds 1.0 there), so the `bias` argument is unused and may be NULL. */
int cabinet_stem_tc(const float* x, int N, int H, int W, const void* w_packed, const float* bias, void* y_sb,
                    long long ld_sb, void* y_stem, long long ld_stem, int OH, int OW, cabinet_stream_t stream);

/* The same two stems without an im2col tile: the converter warps write a pixel-interleaved bf16 copy (r, g, b, 1.0) of
 * the fp32 window and the tensor core reads the overlapping stride-2 rows of the implicit GEMM straight out of it (no-
 * swizzle K-major descriptor, rows 16 bytes = two pixels apart).  16 x 8 output patches.
 * w_packed2: bf16 [7 ky][2 K halves][2 k chunks][80 out][8] = UMMA core matrices of W[o][ky][kx][c] (kx = 0..7 with
 *            kx = 0 zero, c = 0..3 with c = 3 zero except the bias: hi part at (ky 3, kx 4), lo part at (ky 3, kx 5);
 *            element e = (kx % 2) * 4 + c of chunk (kx / 2) % 2 of half kx / 4); BN folded, rows 64..79 = backbone stem. */
int cabinet_stem_tc2(const float* x, int N, int H, int W, const void* w_packed2, void* y_sb, long long ld_sb, void* y_stem,
                     long long ld_stem, int OH, int OW, cabinet_stream_t stream);

/* sb.conv1 alone (a standalone SpatialBranch: 7x7 s2 p3, 3 -> 64, BN folded, ReLU): the kernel of cabinet_stem_tc2 at
 * N = 64, one TMA store per tile.  x fp32 NCHW [N][3][H][W] (W % 4 == 0); y bf16 NHWC [N][OH][OW] with pixel stride ld_y
 * (a multiple of 8, >= 64; channels 64.. of a pixel are not written).
 * w_packed7: rows 0..63 of the cabinet_stem_tc2 pack, bf16 [7 ky][2 K halves][2 k chunks][64 out][8]. */
int cabinet_stem7_tc(const float* x, int N, int H, int W, const void* w_packed7, void* y, long long ld_y, int OH, int OW,
                     cabinet_stream_t stream);

/* The backbone stem alone (a standalone MobileNetV3: 3x3 s2 p1, 3 -> 16, BN folded, HardSwish) in the formulation of
 * cabinet_stem_tc2, one K16 slice per tap row.  x fp32 NCHW [N][3][H][W] (W % 4 == 0); y bf16 NHWC [N][OH][OW] with pixel
 * stride ld_y (a multiple of 8, >= 16).
 * w_packed3: bf16 [3 ky][2 k chunks][16 out][8] = UMMA core matrices of W[o][ky][s][c], s = 0..3, c = 0..3: slot s = kx + 1
 * holds the filter tap kx (c < 3), slot 0 is zero except the bias on the constant-1 channel c = 3 (hi part at ky 1, lo
 * part at ky 0); element e = (s % 2) * 4 + c of chunk s / 2. */
int cabinet_stem3_tc(const float* x, int N, int H, int W, const void* w_packed3, void* y, long long ld_y, int OH, int OW,
                     cabinet_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Depthwise k x k (k in {3,5}, stride in {1,2}, pad (k-1)/2) + folded-BN bias + activation,
 * optional per-(image, channel) sum of the written values for the SE / GAP consumers.
 * Replaces the groups=C nn.Conv2d + BatchNorm2d (+act) at src/models/mobilenetv3.py:112-123,130-141
 * and src/models/cab.py:18-38 (DWConv).  w is [k*k][C] fp32 (BN scale folded), bias [C] fp32.
 * gap_sum ([N][C] fp32, may be NULL) must be zeroed by the caller; it is accumulated atomically.
 */
int cabinet_dwconv(const void* x, long long ldx, const float* w, const float* bias, void* y, long long ldy,
                   int dtype, int N, int H, int W, int C, int k, int stride, int OH, int OW, int act,
                   float* gap_sum, cabinet_stream_t stream);

/* The same depthwise convolution for bf16 with the input patch (+halo) staged in shared memory by one TMA box per
 * CTA (zero padding = TMA out-of-bounds fill).  Same arguments / semantics as cabinet_dwconv (bf16 only), except that
 * the pooling sums are DETERMINISTIC: gap_sum is [N][C] int64 fixed point (CABINET_GAP_FIXED_ONE), zeroed by the caller;
 * every CTA adds its fixed-order fp32 partial sum with one 64-bit integer atomic per channel. */
int cabinet_dwconv_tma(const void* x, long long ldx, const float* w, const float* bias, void* y, long long ldy, int N,
                       int H, int W, int C, int k, int stride, int OH, int OW, int act, long long* gap_sum,
                       cabinet_stream_t stream);
int cabinet_dwconv_tma_dt(const void* x, long long ldx, const float* w, const float* bias, void* y, long long ldy, int N,
                          int H, int W, int C, int k, int stride, int OH, int OW, int act, long long* gap_sum, int op_dtype,
                          cabinet_stream_t stream);

/* Whole no-expand inverted-residual block in one kernel (inp == hidden, no SE, stride 1, identity):
 *   y = x + W_pw * act(dw3x3(x) + b_dw) + b_pw     (src/models/mobilenetv3.py:110-125,154-159; Large f1)
 * bf16 NHWC in/out, C in {8,16,32}; w_dw fp32 [9][C], w_pw fp32 [C][C] (cout, cin), biases fp32, all BN-folded. */
int cabinet_mbconv_noexpand_fused(const void* x, long long ldx, const float* w_dw, const float* b_dw,
                                  const float* w_pw, const float* b_pw, void* y, long long ldy, int N, int H, int W,
                                  int C, int act, cabinet_stream_t stream);

/* conv_tc whose epilogue adds a bilinearly upsampled (align_corners=False) low-resolution fp32 map before the
 * activation:  y = act(conv(x) + bias + bilinear(up [N][up_h][up_w][Cout] -> OH x OW)).
 * A 1x1 convolution commutes with bilinear interpolation, so the part of `FeatureFusionModule.convblk` that reads the
 * upsampled attention features (src/models/cabinet.py:228-231,143-144) is computed at 1/32 resolution (with
 * `AttentionBranch.convb`, cabinet.py:86, folded into its weights) and added here: the x4-upsampled 256-channel
 * tensor is never written and the GEMM's K shrinks from 384 to 128.  bf16 output, Cout % 16 == 0, act ReLU or none. */
int cabinet_conv_tc_up(const void* x, long long ldx, int N, int H, int W, int Cin, const void* w_packed, int Cout,
                       int KH, int KW, int stride, int pad, const float* bias, const float* up, int up_h, int up_w,
                       void* y, long long ldy, int OH, int OW, int act, cabinet_stream_t stream);

/* cabinet_conv_tc whose activation applies to the first act_cols output channels only (act_cols % 16 == 0): several
 * convolutions of the SAME input merged into one GEMM, e.g. GlobalContextAttention's to_query | to_key (Conv+BN+ReLU) |
 * to_value (plain conv), src/models/cab.py:107-128, as one 256 -> 384 projection with act_cols = 256. */
int cabinet_conv_tc_split_act(const void* x, long long ldx, int N, int H, int W, int Cin, const void* w_packed, int Cout,
                              int KH, int KW, int stride, int pad, const float* bias, void* y, int y_dtype, long long ldy,
                              int OH, int OW, int act, int act_cols, cabinet_stream_t stream);

/* cabinet_conv_tc with one weight matrix PER IMAGE (w_packed_per_image + n * w_image_stride elements, each in the
 * cabinet_conv_tc packing); 1x1 convolutions need H * W % 128 == 0.  Used to fold a per-(image, input-channel) scale of
 * the INPUT into the weights instead of rewriting the input tensor: FeatureFusionModule's feat * atten + feat
 * (src/models/cabinet.py:152-153) feeding CABiNetOutput.conv (cabinet.py:166): W'_n = W * (1 + atten_n); and the
 * squeeze-excite scale of ReLU blocks, relu(s * d) = s * relu(d) for s >= 0 (src/models/mobilenetv3.py:83,143):
 * W'_n = W_project * s_n. */
int cabinet_conv_tc_imgw(const void* x, long long ldx, int N, int H, int W, int Cin, const void* w_packed_per_image,
                         long long w_image_stride, int Cout, int KH, int KW, int stride, int pad, const float* bias,
                         const void* res, long long ldres, void* y, int y_dtype, long long ldy, int OH, int OW, int act,
                         cabinet_stream_t stream);
int cabinet_conv_tc_imgw_dt(const void* x, long long ldx, int N, int H, int W, int Cin, const void* w_packed_per_image,
                            long long w_image_stride, int Cout, int KH, int KW, int stride, int pad, const float* bias,
                            const void* res, long long ldres, void* y, int y_dtype, long long ldy, int OH, int OW, int act,
                            int op_dtype, cabinet_stream_t stream);

/* out[n][r][t][c] = bf16(w[r][t][c] * (scale[n][c] + plus_one)): per-image copies of a cabinet_conv_tc weight pack
 * ([rows][taps][cin_pad] bf16, cin_pad % 8 == 0; channels >= Cin stay 0); scale is fp32 [N][Cin]. */
int cabinet_scale_weights(const void* w_packed, const float* scale, void* out, int N, int rows, int taps, int cin_pad,
                          int Cin, int plus_one, cabinet_stream_t stream);

/* cabinet_gate_fc x 2 + cabinet_scale_weights in ONE launch: every block recomputes the gate of its image
 *   gate[n][c] = act(b2 + W2 relu(b1 + W1 (sum[n] * inv_hw)))     (SELayer.fc, mobilenetv3.py:68-83; FFM conv1/conv2,
 *                                                                    cabinet.py:146-150)
 * in shared memory and writes out[n][r][t][c] = bf16(w[r][t][c] * (gate[n][c] + plus_one)).  gap_sum: fp32 [N][C], or the
 * int64 fixed-point sums of the depthwise kernels (in_fixed != 0).  C <= cin_pad, C, Cmid <= 1024. */
int cabinet_gate_scale_weights(const void* gap_sum, int in_fixed, float inv_hw, const float* w1, const float* b1,
                               const float* w2, const float* b2, int gate, int C, int Cmid, const void* w_packed, void* out,
                               int N, int rows, int taps, int cin_pad, int plus_one, cabinet_stream_t stream);

/* Fused inverted-residual block with expansion (src/models/mobilenetv3.py:126-159), bf16 NHWC, Cin <= 248:
 *   h = act_expand(W_e * x + b_e)            1x1 expand + BN + act          (mobilenetv3.py:128-131)
 *   d = act_dw(dw_kxk(h) + b_dw)             depthwise + BN                 (mobilenetv3.py:132-141)
 *   w_project != NULL:  y = W_p * d + b_p (+ x when residual)                (mobilenetv3.py:145-159), y has Cout channels
 *   w_project == NULL:  y = d (Cexp channels) and gap_sum[n][c] += sum over pixels of (dw_kxk(h) + b_dw), i.e. of the
 *                       values BEFORE act_dw (blocks with squeeze-excite: the gate needs the global mean of the BN
 *                       output before the project conv); gap_sum is [N][Cexp] int64 fixed point (CABINET_GAP_FIXED_ONE),
 *                       zeroed by the caller: fixed-order fp32 sum per tile, then 64-bit integer atomics (deterministic).  act_dw = NONE leaves the activation to the SE apply;
 *                       act_dw = RELU is for the identity relu(s * d) = s * relu(d), s >= 0, with the scale folded
 *                       into per-image project weights (cabinet_scale_weights + cabinet_conv_tc_imgw).
 * The expanded activation h never reaches HBM (TMEM -> shared memory -> depthwise).
 * w_expand: bf16 [ceil16(Cexp)][64 * KB], KB = Cin / 64 + 1 K blocks, row = expanded channel: columns 0..Cin-1 = W_e (BN
 *           folded), columns Cin, Cin+1 = b_e split into bf16 (hi, lo) -- the kernel feeds 1.0 into those two K slots,
 *           the bias is part of the GEMM -- remaining columns 0.  Needs Cin % 8 == 0, Cin % 64 <= 56 and Cin <= 248.
 * w_project: the cabinet_conv_tc packing (bf16 [ceil16(Cout)][1][ceil64(Cexp)]); b_project fp32 [Cout].
 * aux_packed: fp32 [ceil(Cexp/64)][k*k + 2][64], zero padded, BN folded: rows 0..k*k-1 = depthwise taps of the chunk's
 *           64 channels, row k*k = reserved (0), row k*k+1 = depthwise bias (one bulk copy per chunk).
 * k in {3,5}, stride in {1,2}, pad (k-1)/2; Cexp % 8 == 0; Cout <= 160; gap_sum may be NULL.  Shapes whose tiles do not
 * fit 113 KB of shared memory / 256 TMEM columns (two CTAs per SM) return CABINET_ERR_INVALID ("budget"). */
int cabinet_mbconv_fused(const void* x, long long ldx, int N, int H, int W, int Cin, const void* w_expand,
                         const float* aux_packed, int Cexp, int act_expand, int k, int stride, int act_dw,
                         const void* w_project, const float* b_project, int Cout, int residual, void* y, long long ldy,
                         int OH, int OW, long long* gap_sum, cabinet_stream_t stream);

/* The same block (same semantics, arguments and modes as cabinet_mbconv_fused) in the channel-major formulation: the
 * expand GEMM is computed transposed (TMEM lane = expanded channel, TMEM column = pixel of the input patch), so the
 * depthwise conv reads its rows straight from TMEM into fp32 registers -- the expanded activation is neither staged in
 * shared memory nor rounded to bf16.  One persistent CTA per SM (16 compute warps + TMA warp + MMA warp).
 * w_expand_t: bf16 [nc * 128][64 * KB], KB = Cin / 64 + 1: chunk c, row l = expanded channel c * CH + (l % CH) with
 *           CH = 64 (Cexp <= 64: one chunk, rows 64..127 repeat rows 0..63) or 128; columns as in cabinet_mbconv_fused
 *           (W_e, then the bias as bf16 hi / lo in columns Cin, Cin + 1); rows of channels >= Cexp are 0.
 * aux_t:    fp32 [nc][k*k + 1][128]: rows 0..k*k-1 = depthwise taps, row k*k = depthwise bias, same row -> channel map.
 * se_scale (project mode only, may be NULL): fp32 [N][Cexp] squeeze-excite gate; the block then computes
 *           d = act_dw(se_scale[n][c] * (dw_kxk(h) + b_dw)) -- a whole SE block in one launch once the gate is known
 *           (cabinet_expand_sums + cabinet_gate_fc obtain it without running the depthwise conv).
 * Supported: k = 3 with stride 1 | 2, k = 5 with stride 1; Cout <= 128, Cout % 8 == 0.
 * Everything else returns CABINET_ERR_INVALID (the caller falls back to cabinet_mbconv_fused / the unfused kernels). */
int cabinet_mbconv_t(const void* x, long long ldx, int N, int H, int W, int Cin, const void* w_expand_t, const float* aux_t,
                     int Cexp, int act_expand, int k, int stride, int act_dw, const void* w_project,
                     const float* b_project, int Cout, int residual, void* y, long long ldy, int OH, int OW,
                     long long* gap_sum, const float* se_scale, cabinet_stream_t stream);

/* Squeeze-excite pooling sums without the depthwise conv (stride-1 blocks; src/models/mobilenetv3.py:68-83,126-143): the
 * sum of d = dw_kxk(h) + b_dw over the pixels is linear in the expanded activation h = act_expand(W_e x + b_e):
 *   sum d = HW b_dw + sum_taps w_dw[ky][kx] * R(ky - p, kx - p),  R(dy, dx) = T - (border rows the tap never reads)
 *   - (border columns it never reads) + (their corner overlap),  p = (k - 1) / 2,
 * i.e. it only takes the total T of h, the sums of its first / last p rows and columns and 2p x 2p corner values.
 * The expand GEMM runs on tcgen05, channel-major (TMEM lane = channel): a thread adds up the columns of its lane.
 * gap_sum: [N][Cexp] int64 fixed point (CABINET_GAP_FIXED_ONE), zeroed by the caller: receives sum d exactly like the
 *          pooling output of cabinet_dwconv_tma / cabinet_mbconv_fused (nsplit + 1 integer atomics per entry:
 *          deterministic) -> cabinet_gate_fc(in_fixed = 1) -> cabinet_mbconv_t(se_scale) runs the block in one launch.
 * w_expand_t, aux_t as in cabinet_mbconv_t; needs 64 < Cexp, 2p <= H, W <= 256; nsplit in [1, ceil(H / max(1, 256 / W))]
 * = parts of an image that are added up as separate work units (<= 0: chosen by the library). */
int cabinet_expand_sums(const void* x, long long ldx, int N, int H, int W, int Cin, const void* w_expand_t,
                        const float* aux_t, int Cexp, int act_expand, int k, int nsplit, long long* gap_sum,
                        cabinet_stream_t stream);

/* Squeeze-excite / FFM channel gate: scale[n][c] = gate(b2 + W2 * relu(b1 + W1 * (sum[n]/HW))).
 * Replaces src/models/mobilenetv3.py:68-83 (gate = CABINET_ACT_HSIGMOID, biases present) and
 * src/models/cabinet.py:146-150 (gate = CABINET_ACT_SIGMOID, b1 = b2 = NULL).  All fp32. */
int cabinet_gate_mlp(const float* gap_sum, float inv_hw, const float* w1, const float* b1, const float* w2,
                     const float* b2, float* scale, int N, int C, int Cmid, int gate, cabinet_stream_t stream);

/* One layer of that gate for the whole batch at once (each weight is read once for all images):
 *   out[n][j] = act(b[j] + sum_c W[j][c] * in[n][c] * in_scale),  in [N][C], W [J][C], out [N][J], all fp32.
 * in_fixed != 0: in is [N][C] int64 fixed point (CABINET_GAP_FIXED_ONE): the pooling sums of cabinet_dwconv_tma /
 * cabinet_mbconv_fused.
 * The engine runs the SE / FFM gate as gate_fc(ReLU, in_scale = 1/HW) -> gate_fc(hard-sigmoid | sigmoid). */
int cabinet_gate_fc(const float* in, float in_scale, const float* W, const float* b, float* out, int N, int C, int J,
                    int act, int in_fixed, cabinet_stream_t stream);

/* In place: x[n][p][c] = act(x * scale[n][c])            (plus_one = 0; SE apply, mobilenetv3.py:83 + act)
 *           x[n][p][c] = x * scale[n][c] + x             (plus_one = 1; FFM, src/models/cabinet.py:152-153) */
int cabinet_scale_act(void* x, long long ldx, int dtype, const float* scale, int N, long long HW, int C, int act,
                      int plus_one, cabinet_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * PSP (src/models/cab.py:46-76).  psp_pool: adaptive average pools of sizes (1,3,6,8) -> pooled
 * [N][110][C] fp32 (bins floor(i*H/s) .. ceil((i+1)*H/s)).  psp_concat: writes the 5C-channel
 * tensor [x, up(pool1), up(pool3), up(pool6), up(pool8)] (bilinear, align_corners=False) that the
 * 1x1 `project` conv consumes.  psp_pool is deterministic: bins larger than 128 pixels are split over several blocks
 * whose partial sums are parked in `scratch` and added in a fixed order by the last block to arrive.  scratch: device
 * memory, >= 256 + 440 * N (rounded up to 256) + N * 256 * C * 4 bytes; its first 440 * N bytes (per-bin tickets)
 * must be zero before the first call, the kernel leaves them zero. */
int cabinet_psp_pool(const void* x, long long ldx, int dtype, float* pooled, int N, int H, int W, int C,
                     float* scratch, long long scratch_bytes, cabinet_stream_t stream);
int cabinet_psp_concat(const void* x, long long ldx, const float* pooled, void* out, long long ldo, int dtype,
                       int N, int H, int W, int C, cabinet_stream_t stream);

/* Row softmax, in place semantics split: s [rows][cols] fp32 (already scaled) -> p [rows][cols] (dtype).
 * Replaces F.softmax(attn, dim=-1) at src/models/cab.py:151 in the fp32 parity mode. */
int cabinet_softmax_rows(const float* s, void* p, int p_dtype, long long rows, int cols, cabinet_stream_t stream);

/* Fused attention on the tensor cores: ctx[n] = softmax(q[n] k[n]^T * scale) v[n]  (src/models/cab.py:149-153) for
 * bf16 q, k, v [N][L][128] (row strides ld*), never materialising the L x L scores.  vt_workspace: bf16
 * [N][128][ceil8(L)] scratch for the transposed values.  ctx: bf16 [N][L][128] (row stride ldc). */
int cabinet_attention_tc(const void* q, long long ldq, const void* k, long long ldk, const void* v, long long ldv,
                         void* vt_workspace, void* ctx, long long ldc, int N, int L, int d, float scale,
                         cabinet_stream_t stream);

/* The same with separate query / key width dk and value / output width dv (a ContextAggregationBlock(C, V) has dk = C / 2,
 * dv = V): q, k bf16 [N][L][dk], v bf16 [N][L][dv], ctx bf16 [N][L][dv], vt_workspace bf16 [N][dv][ceil8(L)].
 * dk in {64, 128, 256}, dv in {64, 128}; scale is the caller's (the reference's dk^-0.5).  At dk = dv = 128 it computes
 * exactly what cabinet_attention_tc computes. */
int cabinet_attention_tc_dkdv(const void* q, long long ldq, const void* k, long long ldk, const void* v, long long ldv,
                              void* vt_workspace, void* ctx, long long ldc, int N, int L, int dk, int dv, float scale,
                              cabinet_stream_t stream);

/* out[p][0:C] = gamma * g + x + x * sigmoid(r)   (src/models/cab.py:182-184,213-216).  g, x, r are dense
 * [n_pixels][C]; out has pixel stride ldo (it is written straight into the b1 concat buffer,
 * src/models/cabinet.py:87).  gamma is a DEVICE scalar (the nn.Parameter itself). */
int cabinet_cab_combine(const void* g, const void* x, const void* r, void* out, long long ldo, const float* gamma,
                        int dtype, long long n_pixels, int C, cabinet_stream_t stream);

/* out[n][c] = sum over pixels of x[n][p][c]  (out fp32, overwritten): the global average pool of
 * src/models/cabinet.py:146.  Deterministic (no floating-point atomics): blocks write partial sums, the last block of
 * an image adds them in block order.  scratch: device memory, >= 256 + 4 * N (rounded up to 256) + N * 64 * C * 4 bytes,
 * whose first 4 * N bytes (the per-image tickets) must be zero before the first call; the kernel leaves them zero. */
int cabinet_channel_sum(const void* x, long long ldx, int dtype, int N, long long HW, int C, float* out, float* scratch,
                        long long scratch_bytes, cabinet_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Bilinear resize, align_corners=False, NHWC -> NHWC (src/models/cabinet.py:228-233). */
int cabinet_bilinear_nhwc(const void* x, long long ldx, int x_dtype, void* y, long long ldy, int y_dtype, int N,
                          int IH, int IW, int C, int OH, int OW, cabinet_stream_t stream);

/* Final x8 bilinear of fp32 NHWC class logits [N][IH][IW][C] (src/models/cabinet.py:240-245):
 *   _nchw   -> NCHW logits (fp32 or bf16), the tensors CABiNet.forward returns;
 *   _argmax -> uint8 mask [N][OH][OW] = argmax_c (first maximum wins, like torch.argmax), logits never stored
 *              (src/scripts/evaluate.py:222); if hist != NULL also accumulates the confusion matrix
 *              hist[pred*C + label] (int64, src/scripts/evaluate.py:162-191) for labels != ignore_label;
 *              labels are int64 (label_dtype 0) or uint8 (label_dtype 1), values clipped to [0, C-1]. */
int cabinet_upsample_logits_nchw(const float* x, int N, int IH, int IW, int C, void* y, int y_dtype, int OH, int OW,
                                 cabinet_stream_t stream);
int cabinet_upsample_argmax(const float* x, int N, int IH, int IW, int C, uint8_t* mask, int OH, int OW,
                            const void* labels, int label_dtype, int ignore_label, long long* hist,
                            cabinet_stream_t stream);

/* uint8 HWC image batch [N][H][W][3] -> normalised fp32 NCHW [N][3][H][W]: (x/255 - mean[c]) / std[c], i.e.
 * torchvision ToTensor + Normalize of the reference datasets (src/datasets/uavid.py:175-183,
 * src/datasets/cityscapes.py:102-109) on the device, so only 3 bytes per pixel cross PCIe.  H*W % 4 == 0. */
int cabinet_normalize_u8(const uint8_t* x, float* y, int N, int H, int W, float mean0, float mean1, float mean2,
                         float std0, float std1, float std2, cabinet_stream_t stream);

/* Confusion matrix of an existing prediction map (pred int64 or uint8 like labels):
 * hist[clip(pred)*C + clip(label)] += 1 where label != ignore_label (src/scripts/evaluate.py:162-191). */
int cabinet_confusion_hist(const void* pred, int pred_dtype, const void* labels, int label_dtype, long long n_pixels,
                           int C, int ignore_label, long long* hist, cabinet_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Evaluator tail (MscEvalV0, src/scripts/evaluate.py:74-159,216-228) on fp32 NCHW probability accumulators.
 *
 * _upsample_softmax_accum: eval_chip + the window accumulation of crop_eval (evaluate.py:74-87,139-146) for one chip:
 *   prob[n][c][dst_y0+oh][dst_x0+ow] += weight * weight_y[oh] * weight_x[ow] * P[n][c][oh][ow],
 *   P = softmax_c(bilinear(x -> OH x OW)), or with x_flip != NULL the mean of that and the mirrored softmax of the
 *   upsampled class map of the horizontally flipped chip (flip TTA).  x, x_flip: fp32 NHWC class maps [N][IH][IW][C]
 *   (the 1/8-resolution output of the head, src/models/cabinet.py:236-243); prob: plane strides in floats; chip
 *   pixels whose destination falls outside [0,dst_h) x [0,dst_w) are dropped (the un-pad crop, evaluate.py:152-156);
 *   weight_y [OH] / weight_x [OW] (NULL = 1) carry 1 / overlap count of the window's rows / columns (the count map of
 *   a window grid is the outer product of per-axis counts, evaluate.py:149-150).
 * _prob_resize_accum: dst[n][c] += bilinear(src[n][c][crop] -> H x W), align_corners=False (evaluate.py:157-158,218).
 * _argmax_hist_nchw: uint8 mask = argmax_c probs (first maximum wins) and / or hist[pred*C + label] += 1 for labels !=
 *   ignore_label, labels int64 (label_dtype 0) or uint8 (1), clipped to [0, C-1] (evaluate.py:222-228,162-191). */
int cabinet_upsample_softmax_accum(const float* x, const float* x_flip, int N, int IH, int IW, int C, int OH, int OW,
                                   float* prob, long long stride_n, long long stride_c, long long stride_row,
                                   int dst_y0, int dst_x0, int dst_h, int dst_w, const float* weight_y,
                                   const float* weight_x, float weight, cabinet_stream_t stream);
int cabinet_prob_resize_accum(const float* src, int N, int C, int src_h, int src_w, int crop_y0, int crop_x0,
                              int crop_h, int crop_w, float* dst, int H, int W, cabinet_stream_t stream);
int cabinet_argmax_hist_nchw(const float* probs, int N, int C, long long HW, uint8_t* mask, const void* labels,
                             int label_dtype, int ignore_label, long long* hist, cabinet_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Training-step loss (BASELINE config 5): OhemCELoss (src/utils/loss.py:38-80; src/scripts/train.py:344-349,435)
 * forward + backward without the reference's full sort of the per-pixel losses.
 *   loss_i = weight[label_i] * (logsumexp_c(logits_i) - logits_i[label_i]) for label_i != ignore_label;
 *   k = min(n_min, #valid); if #(loss > thresh) >= k: mean of the losses above thresh, else mean of the k largest
 *   (exact k-th value by a 3-level radix select over the float bit patterns); no valid pixel: 0.
 * logits: NCHW [N][C][HW] fp32 or bf16 (`dtype`); labels int64 (label_dtype 0) or uint8 (1); weight: [C] fp32 or NULL;
 * loss_px: fp32 [N*HW] scratch kept for the backward pass (-1 marks ignored pixels); workspace:
 * cabinet_ohem_workspace_bytes() bytes of device memory, 8-byte aligned, zeroed by the call itself and read again by
 * _backward; loss_out: one fp32 on the device.  Labels outside [0, C) other than ignore_label are treated as ignored.
 * _backward: grad_logits (same dtype / shape as logits, fully overwritten) = *grad_out * d loss / d logits. */
long long cabinet_ohem_workspace_bytes(void);
int cabinet_ohem_ce_forward(const void* logits, int dtype, const void* labels, int label_dtype, int N, int C, long long HW,
                            const float* weight, int ignore_label, float thresh, long long n_min, float* loss_px,
                            void* workspace, float* loss_out, cabinet_stream_t stream);
int cabinet_ohem_ce_backward(const void* logits, int dtype, const void* labels, int label_dtype, int N, int C,
                             long long HW, const float* weight, const float* loss_px, const void* workspace,
                             const float* grad_out, void* grad_logits, cabinet_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Training step (BASELINE config 5; src/scripts/train.py:429-441: net(im) in .train() mode -> 2 x OhemCELoss ->
 * backward).  NHWC activations (fp32, bf16 or fp16), fp32 statistics and parameter gradients.  Every reduction has a fixed
 * summation order (two-level sums, no floating-point atomics).  Scratch buffers are uninitialised device memory of
 * cabinet_train_scratch_floats(rows, C, quantities) floats unless stated otherwise.
 */
long long cabinet_train_scratch_floats(long long M, int C, int nq);

/* PyTorch OIHW fp32 weight -> [rows_pad][KH*KW][k_pad] (k fastest, zero padded), fp32 or bf16.
 *   transpose_flip = 0: rows = output channels, k = input channels: the layout of cabinet_conv2d_simt (w_sco =
 *     KH*KW*k_pad, w_sk = 1), cabinet_conv_tc (rows_pad = ceil16(Cout), k_pad = ceil64(Cin), bf16), cabinet_conv_dgrad;
 *   transpose_flip = 1: rows = input channels, taps mirrored, k = output channels: the weights with which the data
 *     gradient of a stride-1 convolution is itself a cabinet_conv_tc call (pad' = K - 1 - pad).
 * Depthwise [C][1][k][k] -> [k*k][C] fp32 (cabinet_dwconv / cabinet_dwconv_tma / cabinet_dwconv_dgrad); flip = 1 mirrors
 * the taps (stride-1 data gradient = the depthwise convolution of dy with the mirrored filter). */
int cabinet_pack_conv_weight(const float* w_oihw, int Cout, int Cin, int KH, int KW, void* out, int out_dtype,
                             int rows_pad, int k_pad, int transpose_flip, cabinet_stream_t stream);
int cabinet_pack_dw_weight(const float* w, int C, int k, int flip, float* out, cabinet_stream_t stream);
/* Sub-filter of the input-parity class (py, px) of a stride-2 convolution's data gradient, transposed for cabinet_conv_tc:
 * out bf16 [rows_pad >= Cin][KH2*KW2][k_pad >= Cout]; tap (jy, jx) holds w[co][ci][py + pad - 2 (jy - pad2)][px + pad - 2 (jx - pad2)]
 * (zero outside the filter): dx[2a+py][2b+px] = conv(dy, out, pad2)[a][b]. */
int cabinet_pack_conv_weight_parity(const float* w_oihw, int Cout, int Cin, int K, int pad, int py, int px, int KH2, int KW2,
                                    int pad2, void* out, int rows_pad, int k_pad, cabinet_stream_t stream);
int cabinet_pack_conv_weight_parity_dt(const float* w_oihw, int Cout, int Cin, int K, int pad, int py, int px, int KH2,
                                       int KW2, int pad2, void* out, int rows_pad, int k_pad, int out_dtype,
                                       cabinet_stream_t stream);

/* im2col of the fp32 NCHW network input for the stem convolutions (sb.conv1 7x7 s2 p3, src/models/cabinet.py:111; backbone
 * stem 3x3 s2 p1 = the centre of the same footprint, src/models/mobilenetv3.py:86-91): out bf16 [N*OH*OW][ld], column
 * ci*k*k + ky*k + kx (the OIHW flattening of the filter; columns >= Cin*k*k are zeroed).  Both stems and their weight
 * gradients then run as 1x1 GEMMs on the tensor cores (cabinet_conv_tc / cabinet_conv_wgrad_tc) on this matrix.
 * cabinet_embed_filter: w_big[co][ci*K*K + (ky+o)*K + kx+o] = w_small[co][ci][ky][kx], o = (K-k)/2 (extract_add = 0), or
 * w_small += that slice of w_big (extract_add = 1: the gradient of the embedded filter). */
int cabinet_im2col_nchw(const float* x, int N, int Cin, int H, int W, int k, int stride, int pad, void* out, long long ld,
                        cabinet_stream_t stream);
int cabinet_im2col_nchw_dt(const float* x, int N, int Cin, int H, int W, int k, int stride, int pad, void* out, long long ld,
                           int out_dtype, cabinet_stream_t stream);
int cabinet_embed_filter(float* w_small, int Cout, int Cin, int k, int K, float* w_big, long long ld_big, int extract_add,
                         cabinet_stream_t stream);

/* Train-mode BatchNorm2d statistics (nn.BatchNorm2d in .train(): src/models/cabinet.py:30-31, mobilenetv3.py:88-98,
 * cab.py:26-27) of x [M][C] (M = N*H*W): stats[4][C] = batch mean, 1/sqrt(biased var + eps), scale = gamma * invstd,
 * shift = beta - mean * scale; running_mean / running_var (may be NULL) are updated in place with `momentum` and the
 * unbiased variance.  scratch: (M, C, 2). */
int cabinet_bn_train_stats(const void* x, long long ldx, int dtype, long long M, int C, const float* gamma,
                           const float* beta, float eps, float momentum, float* running_mean, float* running_var,
                           float* stats, float* scratch, cabinet_stream_t stream);

/* y[m][c] = act((z * scale[c] + shift[c]) * (gate[n][c] + gate_plus)) + res[m][c]; scale/shift, gate ([N][C], n = m / HW)
 * and res are optional.  BN apply (+activation), SE / FFM scale (+activation), residual add. */
int cabinet_affine_act(const void* z, long long ldz, int z_dtype, const float* scale, const float* shift, const float* gate,
                       float gate_plus, const void* res, long long ldres, void* y, long long ldy, int y_dtype, long long M,
                       long long HW, int C, int act, cabinet_stream_t stream);

/* Backward of y = act(BN_train(z)): g = dy * act'(u), dgamma += sum g * xhat, dbeta += sum g,
 * dz (+)= scale * (g - mean(g) - xhat * mean(g * xhat)).  stats as written by cabinet_bn_train_stats.  scratch: (M, C, 4). */
int cabinet_bn_train_backward(const void* dy, long long lddy, const void* z, long long ldz, int dtype, const float* stats,
                              int act, float* dgamma, float* dbeta, void* dz, long long lddz, long long M, int C,
                              int accumulate, float* scratch, cabinet_stream_t stream);

/* Eval-mode BatchNorm2d inside a training step (bn.eval() in a .train() model, e.g. frozen BN for fine-tuning): stats[4][C]
 * in the layout of cabinet_bn_train_stats, from the running statistics: mean = running_mean, invstd =
 * 1/sqrt(running_var + eps), scale = gamma * invstd, shift = beta - mean * scale (gamma / beta may be NULL: 1 / 0).  Runs
 * on the device, so a replayed graph reads the running statistics of replay time; they are never written.  The forward
 * apply is cabinet_affine_act with stats[2] / stats[3]. */
int cabinet_bn_frozen_stats(const float* gamma, const float* beta, const float* running_mean, const float* running_var,
                            float eps, int C, float* stats, cabinet_stream_t stream);

/* Backward of y = act(BN_eval(z)) with stats from cabinet_bn_frozen_stats: g = dy * act'(u), dz (+)= scale * g,
 * dgamma += sum g * xhat, dbeta += sum g.  One pass over dy and z writes dz and the per-block column partials; a
 * fixed-order second-level sum gives the parameter gradients (bit-reproducible).  dgamma and dbeta NULL: no reduction;
 * dz NULL: no store (at least one output).  With the batch statistics of cabinet_bn_train_stats and dz NULL it gives the
 * parameter gradients of a train-mode BN whose input needs no gradient.  scratch: (M, C, 2) (the block partials), unused
 * without a reduction. */
int cabinet_bn_frozen_backward(const void* dy, long long lddy, const void* z, long long ldz, int dtype, const float* stats,
                               int act, float* dgamma, float* dbeta, void* dz, long long lddz, long long M, int C,
                               int accumulate, float* scratch, cabinet_stream_t stream);

/* Data gradient of both stride-2 stems (sb.conv1 7x7 / pad 3, 64 outputs, src/models/cabinet.py:111; mobile.features.0.0
 * 3x3 / pad 1, 16 outputs, src/models/mobilenetv3.py:86-91) into the fp32 NCHW network input: dx [N][3][H][W] = the sum
 * of both transposed convolutions (overwritten, not accumulated).  dy7 / dy3: NHWC [N][OH][OW] with pixel strides ld7 /
 * ld3, element type dtype (fp32, bf16 or fp16); either may be NULL (that stem received no gradient), not both.  w7 / w3:
 * the raw fp32 filters [64][3][7][7] / [16][3][3][3], read (and for 2-byte dy rounded to dtype) on every call.  OH =
 * (H - 1) / 2 + 1, OW = (W - 1) / 2 + 1.  2-byte dy runs on the tensor cores; fixed summation order, no atomics. */
int cabinet_stem_dgrad(const void* dy7, long long ld7, const void* dy3, long long ld3, int dtype, const float* w7,
                       const float* w3, float* dx, int N, int H, int W, int OH, int OW, cabinet_stream_t stream);

/* Backward of y = act(v * (s[n][c] + plus)) (SE apply, mobilenetv3.py:83,143; FFM feat * atten + feat, cabinet.py:152):
 *   _scale_backward: ds[n][c] = sum_p dy * act'(v s') * v          (scratch: (HW, C, 1) * N floats)
 *   _apply_backward: dv (+)= dy * act'(v s') * s' + dm[n][c] * inv_hw  (dm = gradient of the pooled mean, may be NULL;
 *                    s may be NULL: plain activation backward) */
int cabinet_gate_scale_backward(const void* dy, long long lddy, const void* v, long long ldv, int dtype, const float* s,
                                float plus, int act, float* ds, int N, long long HW, int C, float* scratch,
                                cabinet_stream_t stream);
int cabinet_gate_apply_backward(const void* dy, long long lddy, const void* v, long long ldv, int dtype, const float* s,
                                float plus, const float* dm, float inv_hw, int act, void* dv, long long lddv, int N,
                                long long HW, int C, int accumulate, cabinet_stream_t stream);
/* Backward of the gate MLP s = gate(W2 relu(W1 m + b1) + b2), m = mean * mean_scale (SELayer.fc, FFM conv1/conv2; pass
 * the pooling SUMS and mean_scale = 1/HW): parameter gradients are accumulated (+=), dmean [N][C] (gradient with respect
 * to m) is overwritten.  scratch: N * (C + J) floats. */
int cabinet_gate_mlp_backward(const float* mean, float mean_scale, const float* w1, const float* w2, const float* hidden, const float* s,
                              const float* ds, int gate, int N, int C, int J, float* dw1, float* db1, float* dw2,
                              float* db2, float* dmean, float* scratch, cabinet_stream_t stream);

/* out[c] (+)= sum over the M rows of x[m][c] (bias gradients).  scratch: (M, C, 1). */
int cabinet_col_sum(const void* x, long long ldx, int dtype, long long M, int C, float* out, int accumulate, float* scratch,
                    cabinet_stream_t stream);

/* Dense convolution gradients (nn.Conv2d backward).  w_packed: cabinet_pack_conv_weight layout, element strides w_sco
 * (per output channel) and w_stap (per tap).  _dgrad: dx [N][H][W][Cin] (+)= conv_transpose(dy, w).  _wgrad: dw (OIHW
 * fp32) += dy^T * im2col(x), split over the pixels with a fixed-order second-level sum; x is addressed with element
 * strides (NHWC maps and the fp32 NCHW network input); scratch: cabinet_conv_wgrad_scratch_floats(...) floats. */
int cabinet_conv_dgrad(const void* dy, long long lddy, int dtype, const void* w_packed, int w_dtype, long long w_sco,
                       long long w_stap, void* dx, long long lddx, int N, int H, int W, int Cin, int Cout, int KH, int KW,
                       int stride, int pad, int OH, int OW, int accumulate, cabinet_stream_t stream);
long long cabinet_conv_wgrad_scratch_floats(int N, int OH, int OW, int Cin, int Cout, int KH, int KW);
int cabinet_conv_wgrad(const void* dy, long long lddy, int dtype, const void* x, int x_dtype, long long sxn, long long sxh,
                       long long sxw, long long sxc, float* dw_oihw, int N, int H, int W, int Cin, int Cout, int KH, int KW,
                       int stride, int pad, int OH, int OW, float* scratch, cabinet_stream_t stream);
/* The weight gradient of a stride-1 "same" convolution (2 * pad == k - 1; every 1x1 and the 3x3 stride-1 layers) or a
 * stride-2 convolution (one tensor map per input parity) on the tensor cores: per tap a GEMM over the pixel index with both bf16 NHWC operands consumed as MN-major UMMA tiles
 * straight from TMA boxes (tcgen05.mma, fp32 accumulation in TMEM), split over the pixels, fixed-order second-level
 * sum.  dy [N][OH][OW][Cout], x [N][H][W][Cin] bf16 (pixel strides multiples of 8); dw (OIHW fp32) +=;
 * scratch: cabinet_conv_wgrad_tc_scratch_floats(...) floats. */
long long cabinet_conv_wgrad_tc_scratch_floats(int N, int H, int W, int Cin, int Cout, int KH, int KW, int stride, int pad);
int cabinet_conv_wgrad_tc(const void* dy, long long lddy, const void* x, long long ldx, float* dw_oihw, int N, int H, int W,
                          int Cin, int Cout, int KH, int KW, int stride, int pad, float* scratch, cabinet_stream_t stream);
int cabinet_conv_wgrad_tc_dt(const void* dy, long long lddy, const void* x, long long ldx, float* dw_oihw, int N, int H,
                             int W, int Cin, int Cout, int KH, int KW, int stride, int pad, float* scratch, int op_dtype,
                             cabinet_stream_t stream);

/* Batched form for per-image products (training-mode attention: dV = P^T dO, dK = dS^T Q, src/models/cab.py:149-153):
 * out[n][co][ci] = sum over the H * W pixels of image n of a[n][pix][co] * x[n][pix][ci]   (fp32, overwritten; one launch,
 * no second-level sum).  H * W must be a multiple of 64. */
int cabinet_conv_wgrad_tc_batched(const void* a, long long lda, const void* x, long long ldx, float* out, int N, int H, int W,
                                  int Cin, int Cout, cabinet_stream_t stream);
int cabinet_conv_wgrad_tc_batched_dt(const void* a, long long lda, const void* x, long long ldx, float* out, int N, int H,
                                     int W, int Cin, int Cout, int op_dtype, cabinet_stream_t stream);

/* Depthwise convolution gradients; w_packed [k*k][C] fp32; dw ([C][1][k][k] fp32) +=; scratch: (N*OH*OW, C, k*k). */
int cabinet_dwconv_dgrad(const void* dy, long long lddy, int dtype, const float* w_packed, void* dx, long long lddx, int N,
                         int H, int W, int C, int k, int stride, int OH, int OW, int accumulate, cabinet_stream_t stream);
int cabinet_dwconv_wgrad(const void* dy, long long lddy, const void* x, long long ldx, int dtype, float* dw, int N, int H,
                         int W, int C, int k, int stride, int OH, int OW, float* scratch, cabinet_stream_t stream);

/* Separable sparse resampling  out[n][oy][ox][c] (+)= sum_{iy, ix} Ry[oy][iy] Rx[ox][ix] in[n][iy][ix][c]  with the row
 * operators as CSR tables (start[O+1], index[], weight[]).  Given the TRANSPOSED matrices of a bilinear resize
 * (align_corners=False) or an adaptive average pool it is the exact adjoint: the backward of F.interpolate
 * (src/models/cabinet.py:228-245, cab.py:70-72) and nn.AdaptiveAvgPool2d (cab.py:55-57).  Element strides on both
 * sides (NHWC maps, NCHW logit gradients).  accumulate: bit 0 = add to out; bit 1 = the input is planar (isx = 1,
 * isy = the dense line length) with many taps per output (the x8 adjoint): one block per output row adds the band of
 * input rows into a shared-memory line, then applies the x operator; bit 2 = an output has few taps (an upsample, the
 * adjoint of a pool): channel-contiguous maps then take the 8-channel vector kernel. */
int cabinet_resample_sep(const void* in, int in_dtype, long long isn, long long isy, long long isx, long long isc,
                         void* out, int out_dtype, long long osn, long long osy, long long osx, long long osc, int N, int OH,
                         int OW, int C, const int* y_start, const int* y_index, const float* y_weight, const int* x_start,
                         const int* x_index, const float* x_weight, int accumulate, cabinet_stream_t stream);

/* ds = p * (dp - rowsum(dp * p)) * alpha over rows of `cols` fp32 (softmax backward, cab.py:150-151). */
int cabinet_softmax_backward(const float* p, const float* dp, float* ds, long long rows, int cols, float alpha,
                             cabinet_stream_t stream);

/* Training-mode attention with its GEMMs on the tensor cores (bf16 mode; src/models/cab.py:149-153 and its autograd
 * backward): S = Q K^T, P V, dO V^T and dS K run as cabinet_conv_tc_imgw calls (the per-image K / V / K^T / V^T maps ARE
 * cabinet_conv_tc weight matrices when their row stride equals their width), P^T dO and dS^T Q as per-image
 * cabinet_conv_wgrad_tc calls.  Between them:
 *   _attn_softmax: p = softmax(scale * s) per row, as fp32 (kept for the backward) and as bf16 (GEMM operand);
 *   _attn_softmax_backward: ds = p * (dp - rowsum(dp * p)) * alpha as bf16;
 *   _transpose_tokens: out[n][c][l] = x[n][l][c], bf16 (x rows ldx apart, out dense). */
int cabinet_attn_softmax(const float* s, float scale, float* p, void* p_bf16, long long rows, int cols,
                         cabinet_stream_t stream);
int cabinet_attn_softmax_backward(const float* p, const float* dp, void* ds_bf16, long long rows, int cols, float alpha,
                                  cabinet_stream_t stream);
int cabinet_transpose_tokens(const void* x, long long ldx, void* out, int N, int L, int C, cabinet_stream_t stream);
/* The same with the 2-byte outputs / operands of type op_dtype (CABINET_BF16 or CABINET_F16). */
int cabinet_attn_softmax_dt(const float* s, float scale, float* p, void* p_half, long long rows, int cols, int op_dtype,
                            cabinet_stream_t stream);
int cabinet_attn_softmax_backward_dt(const float* p, const float* dp, void* ds_half, long long rows, int cols, float alpha,
                                     int op_dtype, cabinet_stream_t stream);
int cabinet_transpose_tokens_dt(const void* x, long long ldx, void* out, int N, int L, int C, int op_dtype,
                                cabinet_stream_t stream);

/* Backward of out = gamma * g + x + x * sigmoid(r) (cab.py:175-184,213-216), dense [n_pixels][C] operands:
 * dg = gamma * dout, dx (+)= dout * (1 + sigmoid(r)), dr = dout * x * sigmoid'(r), *dgamma += sum dout * g.
 * scratch: (n_pixels, C, 1). */
int cabinet_cab_combine_backward(const void* dout, long long ldo, const void* g, const void* x, const void* r,
                                 const float* gamma, int dtype, void* dg, void* dx, void* dr, float* dgamma,
                                 long long n_pixels, int C, int accumulate_dx, float* scratch, cabinet_stream_t stream);
/* out[m][c] = a[m][c] + b[m][c] (gradient fan-in). */
int cabinet_add(const void* a, long long lda, const void* b, long long ldb, void* out, long long ldo, int dtype, long long M,
                int C, cabinet_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CABINET_B200_H */
