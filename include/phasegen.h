/* phasegen -- C ABI of the B200-native magnitude -> phase -> waveform path.
 *
 * The reference (LemonATsu/UNet-PhaseGen) is pure Python and has no FFI of its own; its
 * "interface" for this path is the Python call surface (SURVEY.md section 8b).  Each entry
 * point below names the reference call it stands behind.  The Python shims in
 * unet-phasegen_b200/{model,utils}.py bind these with ctypes (see INTEGRATION.md).
 *
 * Conventions: every function returns 0 (PG_OK) or a negative error code and records a
 * message retrievable with pg_last_error() (thread-local); no C++ exception crosses the
 * boundary.  All data pointers are caller-owned DEVICE memory; the library allocates
 * nothing.  Calls are asynchronous on the given stream (a cudaStream_t passed as void*).
 * Activations are "channels-last": [clip][row][channel], row = STFT frame / conv position.
 */
#ifndef PHASEGEN_H_
#define PHASEGEN_H_
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PG_OK 0
#define PG_ERR_INVALID (-1)
#define PG_ERR_CUDA (-2)
#define PG_ERR_UNSUPPORTED (-3)

typedef void* pg_stream;

const char* pg_last_error(void);
int pg_abi_version(void);
/* Fails (PG_ERR_UNSUPPORTED) unless the current device is compute capability 10.x. */
int pg_check_device(int* sm_count, int* cc_major, int* cc_minor);

/* ---------------------------------------------------------------- STFT front end
 * Replaces librosa.stft(c, n_fft, hop) + np.delete(.., 0, axis=0) at preproc_mdb.py:93 and
 * utils.py:120-121, the re/im split of preproc_mdb.py:94-95 (PG_STFT_REIM) and the
 * abs/log1p/angle of data.py:39-47 (PG_STFT_LOGMAG).  center=True, reflect padding, periodic
 * Hann of length n_fft.  wave [B][N] fp32 -> out_a/out_b fp32 [B][T][n_fft/2] (frame-major,
 * DC bin dropped), T = 1 + N/hop.  out_a or out_b may be NULL.  op_hi/op_lo (may be NULL): out_a as
 * 16-bit hi/lo planes (op_fmt: PG_FMT_BF16 or PG_FMT_F16) [B][..][n_fft/2] with op_batch_stride
 * elements between clips -- the operand of the first convolution.  twiddle: float2[n_fft] = exp(-2*pi*i*m/n_fft).
 * n_fft in {256,512,1024,2048}, hop = n_fft/4. */
enum { PG_STFT_LOGMAG = 0, PG_STFT_REIM = 1, PG_STFT_PROJECT = 2 /* pg_stft_project only */, PG_STFT_PAIRS = 3 /* pg_stft_pairs only */ };
int pg_stft_num_frames(int n_samples, int hop);
int pg_stft(const float* wave, int B, int N, int n_fft, int hop, const float* twiddle, int mode,
            float* out_a, float* out_b, uint16_t* op_hi, uint16_t* op_lo, int64_t op_batch_stride,
            int op_fmt, pg_stream stream);

/* One Griffin-Lim projection (utils.py:119-124: recon_spec = stft(recon_aud) without the DC row; new_spec =
 * spec * exp(1j * angle(recon_spec))): out = mag * X / |X| as (re, im) planes, frame-major [B][T][n_fft/2],
 * ready for pg_istft(PG_SPEC_CARTESIAN).  mag: the target magnitude [B][T][n_fft/2]. */
int pg_stft_project(const float* wave, int B, int N, int n_fft, int hop, const float* twiddle,
                    const float* mag, float* out_re, float* out_im, pg_stream stream);

/* Online training-pair producer: the STFT of preproc_mdb.py:93-96, the dataset-wide standardisation of the (re, im)
 * values (preproc_mdb.py:182: (x - mean) / std) and data.py:39-47 (log1p|.|, angle) in one kernel:
 * wave [B][N] -> log-magnitude and phase planes [B][T][n_fft/2], the channels-last pair TrainStep consumes. */
int pg_stft_pairs(const float* wave, int B, int N, int n_fft, int hop, const float* twiddle, float mean, float std,
                  float* out_logmag, float* out_phase, pg_stream stream);

/* ---------------------------------------------------------------- ISTFT back end
 * Replaces utils.generate_audio (utils.py:11-44): zero DC row (:38-39), librosa.istft (:40:
 * inverse real FFT, periodic Hann, overlap-add, / window sum-of-squares, trim n_fft/2),
 * finiteness check (:41 -> nonfinite[b] != 0), peak normalisation (:42 -> pg_peak_normalize),
 * with the polar->complex step of demo.py:39 / train.py:83 fused in (PG_SPEC_POLAR_LOG:
 * a = log1p-magnitude, b = phase; PG_SPEC_CARTESIAN: a = re, b = im; PG_SPEC_POLAR_MAG:
 * a = magnitude; in both polar modes b may be NULL for zero phase: the "no phase" reconstruction of train.py:86).  Inputs frame-major [B][T][n_fft/2]
 * (bins 1..n_fft/2); wave [B][(T-1)*hop].  peak [B] (max |wave|) and nonfinite [B] may be NULL. */
enum { PG_SPEC_POLAR_LOG = 0, PG_SPEC_CARTESIAN = 1, PG_SPEC_POLAR_MAG = 2 };
/* b_scale_shift (may be NULL): float2 (scale, shift) per bin, [B][n_fft/2] when b_ss_per_clip else [n_fft/2]; the kernel
 * reads in_b as in_b*scale + shift.  This is the train-mode norm that ends the U-Net (model.py:83,91) applied while the
 * last convolution's raw output is read, so that tensor is never re-written normalised. */
int pg_istft(const float* in_a, const float* in_b, int mode, int B, int T, int n_fft, int hop,
             const float* twiddle, float* wave, float* peak, int* nonfinite,
             const float* b_scale_shift, int b_ss_per_clip, pg_stream stream);
int pg_peak_normalize(float* wave, const float* peak, int B, int N, pg_stream stream);

/* ---------------------------------------------------------------- ragged batches
 * Clips of different lengths in one [B][N] buffer: clip b holds its first n_b <= N samples.  Its frame count is T_b, the
 * smallest multiple of 8 with (T_b - 1)*hop >= n_b, and it is computed as if it were alone, zero-padded to (T_b - 1)*hop
 * samples.  Each entry below is the NULL-lengths entry above with per-clip int32 arrays in device memory [B]; every
 * layer of the U-Net then holds clip b's valid rows L_b (the convolution length chain from T_b) and ZEROS in rows
 * [L_b, L), which is the zero padding the next convolution of the standalone clip would read.  Table entries larger
 * than the call's extent (N, T, L_out, L) are clamped to it, so a bad table never reaches another clip's rows.
 *
 * pg_stft_ragged: PG_STFT_LOGMAG only (else PG_ERR_UNSUPPORTED).  Samples >= clip_samples[b] are never read; reflect
 *   padding at (T_b - 1)*hop; frames >= T_b = clip_frames[b] are written as 0 in every plane.
 * pg_conv_tc_ragged: out_rows[b] = valid output rows L_b.  PG_EPI_RAW: statistics records count those rows only (a part
 *   with none gets n = 0, which pg_bn_finalize skips); y beyond them is unspecified.  PG_EPI_ACT / NORM_ACT: the norm
 *   uses those rows only and rows [L_b, L_out) of both destinations are written as 0.
 * pg_bn_act_ragged: clip_rows[b] = valid rows; y is not read beyond them and rows [L_b, L) of every destination are 0.
 * pg_istft_ragged: frames >= clip_frames[b] are not read; the window sum of squares at the clip's end is the one of
 *   T_b frames; peak and non-finite flags cover samples [0, (T_b - 1)*hop); samples [clip_samples[b], (T-1)*hop) are
 *   written as 0 (pg_peak_normalize keeps them 0).
 *
 * Packed clips: the same clips laid end to end in one flat buffer of n samples, clip b at [o_b, o_b + n_b) with
 * o_b = clip_offsets[b] (device int64 [B+1], o_0 = 0, o_B = n).  The executor's frame count T is given; the U-Net and ISTFT
 * entries above run unchanged on [B][T] and [B][(T-1)*hop] buffers.  Offsets are clamped to [0, n] and n_b to >= 0.
 * pg_stft_packed: pg_stft_ragged of the padded [B][(T-1)*hop] buffer that holds clip b in row b (bit-identical), with the
 *   clip read from wave[o_b ..] instead; n_b is further clamped to (T-1)*hop.  PG_STFT_LOGMAG only (else PG_ERR_UNSUPPORTED).
 * pg_peak_normalize_packed: dst[o_b + i] = src[b][i] / peak[b] for i < n_b (src: [B][src_pitch], the pg_istft_ragged output;
 *   the pg_peak_normalize rule, so bit-identical to it); a copy when peak is NULL.  n_b is clamped to src_pitch, and
 *   dst [n_dst] is written at [o_b, o_b + n_b) only. */
int pg_stft_packed(const float* wave, int64_t n_wave, const int64_t* clip_offsets, int B, int T, int n_fft, int hop,
                   const float* twiddle, int mode, float* out_a, float* out_b, uint16_t* op_hi, uint16_t* op_lo,
                   int64_t op_batch_stride, int op_fmt, const int* clip_frames, pg_stream stream);
int pg_peak_normalize_packed(const float* src, int B, int64_t src_pitch, const float* peak, const int64_t* clip_offsets,
                             float* dst, int64_t n_dst, pg_stream stream);
int pg_stft_ragged(const float* wave, int B, int N, int n_fft, int hop, const float* twiddle, int mode,
                   float* out_a, float* out_b, uint16_t* op_hi, uint16_t* op_lo, int64_t op_batch_stride,
                   int op_fmt, const int* clip_samples, const int* clip_frames, pg_stream stream);
int pg_istft_ragged(const float* in_a, const float* in_b, int mode, int B, int T, int n_fft, int hop,
                    const float* twiddle, float* wave, float* peak, int* nonfinite,
                    const float* b_scale_shift, int b_ss_per_clip, const int* clip_frames, const int* clip_samples,
                    pg_stream stream);

/* Long-form stitching (BASELINE.json config 4; the reference cuts long audio into independent slices,
 * preproc_mdb.py:66-82, and never stitches them): n_windows windows of `win` samples, one every `step` samples
 * (win/2 <= step <= win), cross-faded over the shared samples with complementary periodic-Hann ramps -> out [n_out].
 * Window i is read from slot (i % world) * per_rank + i / world of `windows` [world * per_rank][win]: the layout an
 * all-gather of round-robin-dealt windows produces (world = 1, per_rank = n_windows: plain order).  peak (may be NULL):
 * one float, max |out|, for a single pg_peak_normalize(out, peak, 1, n_out) of the whole recording. */
int pg_stitch(const float* windows, int n_windows, int win, int step, int world, int per_rank, float* out,
              int64_t n_out, float* peak, pg_stream stream);

/* ---------------------------------------------------------------- U-Net layers
 * Replace the nn.Conv1d / nn.ConvTranspose1d / norm / activation / torch.cat calls of
 * model.py:77-113.  A layer is: convolution -> per-channel statistics records -> finalize
 * (scale, shift) -> apply + activation written as the operand(s) of the consumer(s). */
enum { PG_CONV = 0, PG_CONV_TRANSPOSE = 1 };
/* Tensor-core precisions.  Operands are 16-bit planes (hi, lo) with x = hi + lo; fp32 accumulate.
 *   BF16X3: Whi*Xhi + Whi*Xlo + Wlo*Xhi, bf16 planes   (rel. error per product ~2^-16)
 *   BF16  : Whi*Xhi, bf16                              (~2^-8; the separately stated loose mode)
 *   F16X3 : same three products on fp16 planes          (~2^-22; operands must stay inside the fp16 range)
 *   F16X2 : Whi*Xhi + Whi*Xlo, fp16: activations exact to 2^-22, weights rounded to fp16 (2^-11, the
 *           rounding of a TF32 operand) -- the cost of ONE TF32 pass with half of its rounding error
 *   F16   : Whi*Xhi, fp16: both operands rounded to 11 significant bits -- exactly the operand rounding of a
 *           TF32 pass (10-bit mantissa), at twice its tensor rate */
enum { PG_PREC_FP32_SIMT = 0, PG_PREC_BF16X3 = 1, PG_PREC_BF16 = 2, PG_PREC_F16X3 = 3, PG_PREC_F16X2 = 4, PG_PREC_F16 = 5 };
enum { PG_DT_NONE = 0, PG_DT_F32 = 1, PG_DT_BF16_SPLIT = 2, PG_DT_BF16 = 3, PG_DT_F16_SPLIT = 4, PG_DT_F16 = 5 };
enum { PG_FMT_BF16 = 0, PG_FMT_F16 = 1 };   /* 16-bit format of operand planes written by a kernel */

typedef struct pg_conv_desc {
    int kind;                 /* PG_CONV (model.py:77) or PG_CONV_TRANSPOSE (model.py:88,94,101) */
    int B, C_in, C_out, L_in, L_out, k, stride, pad;
    int in_rows, in_ld;       /* input buffer: allocated rows per clip (zero beyond L_in), row pitch */
    int out_rows, out_ld;     /* fp32 output buffer geometry */
    int precision;            /* PG_PREC_* */
    int taps_per_group;       /* tensor-core path: taps sharing one activation strip (0 = default 16, 1 = off) */
    int tc_base_offset_mode;  /* tensor-core path: descriptor base-offset handling of shifted strips */
    int tc_max_ctas;          /* tensor-core path: cap on the persistent grid (0 = one per SM) */
    int max_clips_per_tile;   /* tensor-core path: clips packed into one tile for short time axes (0 = auto, 1 = off) */
    int weights_mn_major;     /* tensor-core path: weight planes are [k][C_in][C_out] (the packed layout of the MIRRORED
                                 layer) and are fed to the MMA as an MN-major operand: the data gradient of a layer
                                 reuses that layer's forward weight planes, no second packing */
    int tc_cta_pair;          /* tensor-core path: 256-channel tiles on CTA pairs (cta_group::2 MMAs, each SM reads half
                                 of the activation strip): 0 = auto (C_out % 256 == 0), 1 = off, 2 = required */
    int tc_whole_clip;        /* tensor-core path, planning only (pg_conv_tc_plan): tile = every output position of a clip
                                 (all phases x position tiles side by side in the accumulator); pg_conv_tc sets it itself
                                 from the epilogue mode */
} pg_conv_desc;

/* weights: torch layout (Conv1d [C_out][C_in][k], ConvTranspose1d [C_in][C_out][k], SURVEY 8a9)
 * -> 16-bit hi/lo planes [k][C_out][C_in] (tensor-core path; fmt = PG_FMT_*) and/or fp32
 * [k][C_in][C_out] (SIMT). */
int pg_pack_weight(const float* w, int kind, int C_in, int C_out, int k, uint16_t* w_hi,
                   uint16_t* w_lo, float* w_simt, int fmt, pg_stream stream);

/* tcgen05 implicit GEMM.  x: bf16 planes [B][in_rows][in_ld]; y fp32 [B][out_rows][out_ld];
 * stats (may be NULL): float4 {n, mean, M2, 0} [B][P][C_out], P = pg_conv_stat_parts(). */
/* fp32 -> 16-bit hi/lo planes (fmt = PG_FMT_*), elementwise (weights kept in the packed layout need no re-ordering) */
int pg_cast_split(const float* src, int64_t n, uint16_t* hi, uint16_t* lo, int fmt, int* range_flag, pg_stream stream);

/* Destination of an activated tensor (the operand buffer of a consumer layer, or an fp32 tensor). */
typedef struct pg_act_dst {
    void* hi; void* lo;       /* PG_DT_F32: hi = float*; PG_DT_{BF16,F16}_SPLIT: two 16-bit planes; PG_DT_{BF16,F16}: hi only */
    int64_t batch_stride;     /* elements between clips */
    int ld, ch_off;           /* row pitch and first channel written (skip-concat offset, model.py:113) */
    int dtype;                /* PG_DT_* */
    float slope;              /* 0 = ReLU (model.py:82), 0.2 = LeakyReLU (model.py:80), 1 = identity */
    int* range_flag;          /* may be NULL; device int, bit 0 is OR-ed in when a value written to an FP16 plane lies outside
                                 the fp16 range (|v| > 65504) or is not finite: the fp16 operand modes are then invalid for
                                 this input and the caller must fall back to the bf16 planes (same bytes, fp32 range) */
} pg_act_dst;

/* Fused epilogue of pg_conv_tc (model.py:80-83,113 inside the convolution kernel).
 *   PG_EPI_RAW      y fp32 + statistics records (batch statistics need a second pass: pg_bn_finalize + pg_bn_act)
 *   PG_EPI_ACT      layer without norm (model.py:90,96): act(conv) written straight into the consumers' operand planes
 *   PG_EPI_NORM_ACT train-mode norm with the clip's OWN statistics (what the demo.py:33-42 batch-1 loop computes), then
 *                   the activation(s): statistics are complete inside the tile because the tile holds every output
 *                   position of the clip (pg_conv_epilogue_supported says whether it fits); y and stats are not written */
enum { PG_EPI_RAW = 0, PG_EPI_ACT = 1, PG_EPI_NORM_ACT = 2 };
typedef struct pg_conv_epilogue {
    int mode;
    const float* gamma; const float* beta;   /* [C_out], may be NULL (1, 0) */
    float eps;
    pg_act_dst dst0, dst1;                   /* dst1.dtype = PG_DT_NONE when unused */
    float* scale_shift;                      /* NORM_ACT, may be NULL: float2 [B][C_out], the (scale, shift) applied */
} pg_conv_epilogue;
int pg_conv_epilogue_supported(const pg_conv_desc* d, int mode);

int pg_conv_tc(const pg_conv_desc* d, const uint16_t* x_hi, const uint16_t* x_lo,
               const uint16_t* w_hi, const uint16_t* w_lo, float* y, float* stats,
               const pg_conv_epilogue* epilogue /* NULL = PG_EPI_RAW */, pg_stream stream);
/* ragged batch (see pg_stft_ragged): out_rows [B] device int32, valid output rows of each clip */
int pg_conv_tc_ragged(const pg_conv_desc* d, const uint16_t* x_hi, const uint16_t* x_lo,
                      const uint16_t* w_hi, const uint16_t* w_lo, float* y, float* stats,
                      const pg_conv_epilogue* epilogue, const int* out_rows, pg_stream stream);
int pg_conv_stat_parts(const pg_conv_desc* d);
/* Tiling plan of pg_conv_tc for a layer, host-only: out[16] = {n_tile, n_ntiles, clips per tile, strip rows, CTA pair,
 * merged clips, MMA groups per weight tile, TMEM accumulator stages, C_in/64, C_out/128, output phases, input
 * parities, taps of phase 0, of phase 1, tap groups of phase 0, of phase 1 [, whole-clip tile]} (the 17th when n_out >= 17). */
int pg_conv_tc_plan(const pg_conv_desc* d, int* out, int n_out);
/* exact fp32 on CUDA cores; x fp32 [B][in_rows][in_ld], w_simt from pg_pack_weight. */
int pg_conv_simt(const pg_conv_desc* d, const float* x, const float* w_simt, float* y, pg_stream stream);
int pg_channel_stats(const float* y, int B, int L, int C, int rows, int ld, float* stats, pg_stream stream);

/* train-mode batch norm (model.py:81,83; the reference never calls .eval()): combine the
 * partial records over (B, L) (per_clip = 0, train.py:42) or over L of each clip
 * (per_clip = 1, the demo.py:33-42 batch-1 loop).  scale_shift: float2 [G][C], G = per_clip ?
 * B : 1; mean_var (may be NULL): float2 [G][C] (mean, biased variance). */
int pg_bn_finalize(const float* stats, int B, int P, int C, int per_clip, const float* gamma,
                   const float* beta, float eps, float* scale_shift, float* mean_var, pg_stream stream);

/* Train-mode side effect of nn.BatchNorm (model.py:81,83 in train mode): running = (1 - momentum) * running + momentum * batch value,
 * the variance unbiased by `unbias` = n / (n - 1).  mean_var: float2 [C] (mean, biased variance) as written by pg_bn_finalize. */
int pg_bn_running_update(const float* mean_var, float* running_mean, float* running_var, int C, float momentum, float unbias,
                         pg_stream stream);

/* eval-mode norm (nn.BatchNorm after .eval(); the reference never calls it, kept for API parity): scale/shift from the
 * running statistics, replicated into G groups so that per-clip consumers can index it by clip. */
int pg_bn_from_running(const float* running_mean, const float* running_var, const float* gamma, const float* beta,
                       float eps, int C, int G, float* scale_shift, float* mean_var, pg_stream stream);

/* v = y*scale+shift (scale_shift NULL = identity), then per destination act(v).  C = number
 * of leading channels of y processed. */
int pg_bn_act(const float* y, int B, int L, int C, int rows, int ld, const float* scale_shift,
              int per_clip, const pg_act_dst* dst0, const pg_act_dst* dst1, pg_stream stream);
/* ragged batch (see pg_stft_ragged): clip_rows [B] device int32, valid rows of each clip */
int pg_bn_act_ragged(const float* y, int B, int L, int C, int rows, int ld, const float* scale_shift,
                     int per_clip, const pg_act_dst* dst0, const pg_act_dst* dst1, const int* clip_rows, pg_stream stream);

/* [B][R][S] fp32 -> [B][S][R] fp32 and/or 16-bit hi/lo planes (fmt = PG_FMT_*) (reference [B,C,T] <-> channels-last). */
int pg_transpose(const float* src, int B, int R, int S, int64_t src_batch_stride, float* dst,
                 uint16_t* dst_hi, uint16_t* dst_lo, int64_t dst_batch_stride, int dst_ld, int fmt, int* range_flag /* may be NULL */,
                 pg_stream stream);

/* ---------------------------------------------------------------- training step (train.py:37-62)
 * Replace loss.backward() (autograd through cuDNN, train.py:61), the loss of train.py:45-60 and
 * torch.optim.Adam (train.py:26-27,62).  Gradients w.r.t. activations flow as fp32 channels-last
 * buffers; the data gradient of a layer is the forward kernel run on the mirrored geometry
 * (pg_conv_tc / pg_conv_simt with kind swapped and the weight packed with the other `kind`). */

/* loss3[0..3] = total, MSE(cos), MSE(sin), MSE(mag); total = cos + sin + mag_weight*mag (0.2 at
 * train.py:60).  out [rows][2C] channels-last; d_out (may be NULL) same shape; partial: double[3*n_blocks]. */
int pg_phase_loss(const float* out, const float* logmag, const float* phase, int64_t rows, int C,
                  float mag_weight, float* d_out, double* partial, int n_blocks, float* loss3, pg_stream stream);

typedef struct pg_grad_src {
    const float* g;           /* upstream gradient w.r.t. an activated copy of h, fp32 [B*L][ld] */
    int ld, ch_off;
    float slope;              /* slope of that activation for h <= 0 (0 ReLU, 0.2 LeakyReLU, 1 identity) */
} pg_grad_src;
/* Backward of [conv output z -> train-mode norm -> activation fan-out] (model.py:80-83).
 * scale_shift / mean_var: what pg_bn_finalize produced in the forward pass (batch statistics), or
 * NULL for a layer without norm.  Outputs: dgamma, dbeta [C] (may be NULL), and dZ as operand
 * planes [B][dz_rows][C] (dz_dtype: PG_DT_F32 / PG_DT_BF16 / PG_DT_BF16_SPLIT).  Workspace:
 * partial float2[n_chunks*C], coef float2[C]. */
int pg_bn_bwd(const float* z, int B, int L, int C, const float* scale_shift, const float* mean_var, float eps,
              const pg_grad_src* g0, const pg_grad_src* g1, float* partial, int n_chunks, float* coef,
              float* dgamma, float* dbeta, void* dz_hi, void* dz_lo, int dz_rows, int dz_dtype, pg_stream stream);

/* weight gradient, packed fp32 [k][C_out][C_in]; d describes the FORWARD convolution; x = its input
 * operand, g = dZ operand planes [B][g_rows][C_out]. */
int pg_wgrad_tc(const pg_conv_desc* d, const uint16_t* x_hi, const uint16_t* x_lo, const uint16_t* g_hi,
                const uint16_t* g_lo, int g_rows, void* dw_packed, int dw_dtype /* PG_DT_F32 | PG_DT_BF16 */, pg_stream stream);
int pg_wgrad_simt(const pg_conv_desc* d, const float* x, const float* g, int g_rows, float* dw_packed, pg_stream stream);
/* packed [k][C_out][C_in] -> torch layout (Conv1d [C_out][C_in][k] / ConvTranspose1d [C_in][C_out][k]) */
int pg_unpack_grad(const float* packed, int kind, int C_in, int C_out, int k, float* out, pg_stream stream);
/* torch.optim.Adam semantics (bias-corrected, eps outside the sqrt), fp32 state; step >= 1.
 * w_hi / w_lo (may be NULL): also write the updated parameter as bf16 operand planes (same element
 * order), which fuses the re-pack of packed-layout weights into the optimiser step. */
int pg_adam_step(float* p, const void* g, int g_dtype /* PG_DT_F32 | PG_DT_BF16 */, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                 float eps, int step, float grad_scale, uint16_t* w_hi, uint16_t* w_lo, pg_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* PHASEGEN_H_ */
