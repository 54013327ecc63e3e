/* hifigan_b200.h — C-ABI of libhifigan_b200.so (sm_100a kernels for the HiFi-GAN vocoder hot path).
 *
 * The reference (AlonKellner/hifi-gan) has no FFI layer: its hot path is the Python module API
 * of src/models.py and src/meldataset.py, whose arithmetic is delegated to torch / torchaudio
 * library ops (SURVEY.md §2.2, §8b).  Each entry point below replaces one of those library call
 * sites; the Python host in hifi-gan_b200/ mirrors the reference classes and calls these through
 * ctypes.  No torch types cross this boundary: plain device pointers, sizes and a cudaStream_t
 * passed as void*.
 *
 * Conventions
 *   - every function returns 0 on success, a negative code on failure; hg_last_error() returns
 *     the message of the last failure on the calling thread.
 *   - all pointers are DEVICE pointers unless the parameter name starts with `host_`.
 *   - the library never allocates device memory; workspaces are supplied by the caller.
 *   - activations between kernels are channels-last in time: bf16 [B][T][C] ("NLC"), so that the
 *     GEMM K dimension (channels) is contiguous for TMA / UMMA.  The public Python API keeps the
 *     reference's fp32 [B][C][T] tensors at its edges.
 *   - arithmetic: bf16 operands, fp32 accumulate (tcgen05.mma kind::f16), fp32 epilogue math.
 */
#ifndef HIFIGAN_B200_H
#define HIFIGAN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HG_ABI_VERSION 3

/* Library identity / diagnostics. */
const char* hg_version(void);
const char* hg_last_error(void);
int hg_abi_version(void);
/* Number of kernel launches issued by this library since load (bench.py's gpu_launches). */
int64_t hg_launch_count(void);
/* Diagnostics: a one-thread kernel on `stream` stores the GPU's %globaltimer (ns) to *dst (device memory).  Unlike a
 * CUDA event it can be read after a graph replay: the training step marks where each discriminator lane finishes its
 * backward, its gradient all-reduce and its generator-step pass (HG_LANE_STAMPS=1, tests/lane_stamps.py). */
int hg_timestamp(uint64_t* dst, void* stream);

/* ------------------------------------------------------------------------------------------
 * Weight preparation (replaces torch.nn.utils.weight_norm's per-forward recompute,
 * reference call sites src/models.py:16-31,56-59,81,86-88,96; fold = remove_weight_norm
 * src/models.py:44-48,70-72,118-125).
 *
 * hg_pack_conv1d_weight: v fp32 [Cout][Cin][k] (+ optional g fp32 [Cout]; w = g * v / ||v||_2
 * over (Cin,k) per output channel) -> bf16 [k][Cout][cin_pad], zero-filled for ci >= Cin.
 * With g == NULL, v is taken as the already-folded `weight`.
 */
int hg_pack_conv1d_weight(const float* v, const float* g, int cout, int cin, int k, int cin_pad,
                          void* w_packed, void* stream);

/* Polyphase geometry of ConvTranspose1d(k, stride, padding) (src/models.py:84-88): every output
 * phase p in [0,stride) of out[t*stride + p] reads inputs x[t + s] for a few shifts s; the union
 * over phases is the contiguous range [shift_min, shift_min + nshift).  Host-only helper. */
int hg_convtr1d_geometry(int k, int stride, int padding, int* host_nshift, int* host_shift_min);

/* hg_pack_convtr1d_weight: v fp32 [Cin][Cout][k] (+ optional g fp32 [Cin]; weight_norm dim 0 of a
 * ConvTranspose1d is the INPUT channel, SURVEY.md Appendix B.3) -> bf16
 * [nshift][stride*Cout][Cin]: slot (s, p*Cout+co, ci) holds w[ci][co][j] with
 * j = p + padding - (shift_min + s)*stride when 0 <= j < k, else 0.  Running hg_conv1d_fwd with
 * ktaps = nshift, pad_left = -shift_min on it yields [B][T_in][stride*Cout] == [B][T_in*stride][Cout]. */
int hg_pack_convtr1d_weight(const float* v, const float* g, int cin, int cout, int k, int stride,
                            int padding, void* w_packed, void* stream);

/* ------------------------------------------------------------------------------------------
 * hg_conv1d_fwd — stride-1 dilated Conv1d as a tcgen05/TMEM implicit GEMM fed by TMA.
 * Replaces torch Conv1d at src/models.py:35-42,63-68 (ResBlock1/2), :101 (conv_pre) and, through
 * the polyphase packing above, ConvTranspose1d at :104.
 *
 *   acc[b,t,co] = sum_{j<ktaps} sum_{ci<cin} x[b, t + j*dilation - pad_left, ci] * w[j][co][ci]
 *   v           = (acc + bias[co] + res0 + res1 + res2) * scale        (absent terms = 0)
 *   out_raw     = bf16(v)                     if out_raw != NULL
 *   out_act     = bf16(leaky_relu(v, slope))  if out_act != NULL
 *
 * x is read with zero padding outside [0,T).  x, res*, out_* are bf16 [B][T][C]; w_packed is
 * bf16 [ktaps][cout][cin]; bias fp32 [cout].  cin % 32 == 0, cout % 32 == 0.
 * The fused epilogue covers F.leaky_relu (models.py:36,38,64,103,112), the residual add (:41,67),
 * and the MRF branch average xs / num_kernels (:105-111).
 *
 * Ragged batches (the reference's drivers run one utterance per call, src/inference.py:55; stacking utterances of
 * different lengths must not change anyone's samples): item_len (optional, device int32 [B]) gives every batch item
 * its own length item_len[b] * item_mul <= t; rows between that and t are stored as ZEROS, so the next layer reads
 * exactly the zero padding the item would see when run alone and results stay bit-identical to the per-item call.
 */
int hg_conv1d_fwd(const void* x, const void* w_packed, const float* bias, int batch, int t, int cin,
                  int cout, int ktaps, int dilation, int pad_left, const void* res0,
                  const void* res1, const void* res2, float scale, void* out_raw, void* out_act,
                  float act_slope, const int* item_len, int item_mul, void* stream);
/* hg_conv1d_fwd_actres — hg_conv1d_fwd whose first residual is stored activated: res0 holds
 * bf16(leaky_relu(r, res0_slope)), 0 < res0_slope <= 1, and the epilogue adds r = min(res0, res0 / res0_slope)
 * (same 2^-9 relative rounding as a raw copy of r).  A tensor that feeds both a conv and a residual add is
 * then stored once, as the conv's input. */
int hg_conv1d_fwd_actres(const void* x, const void* w_packed, const float* bias, int batch, int t, int cin,
                         int cout, int ktaps, int dilation, int pad_left, const void* res0, float res0_slope,
                         const void* res1, const void* res2, float scale, void* out_raw, void* out_act,
                         float act_slope, const int* item_len, int item_mul, void* stream);

/* hg_conv1d_general_fwd — strided and/or grouped Conv1d on the same tcgen05 kernel (the discriminator stacks:
 * DiscriminatorS src/models.py:195-204 — k=41, stride 1/2/4, groups 4/16; DiscriminatorP :133-140 — (5,1)
 * kernels with stride (3,1), one independent 1-D problem per period column).
 *
 *   out[b,t,co] = leaky_relu(bias[co] + sum_{j,ci in group(co)} x[b, stride*t + j - pad_left, ci] * w[j][co][ci])
 *
 * x bf16 [B][t_in_rows][c_total] with t_in_rows a multiple of `stride` and rows past the true length zero
 * (they are the conv's zero padding); the kernel reads it through the view [B][t_in_rows/stride][stride*c_total]
 * so that taps of equal residue mod stride are row-shifted views of one TMA box.  w_packed bf16
 * [ktaps][cout][c_total/groups] with the taps in the order given by hg_conv1d_tap_order (identity for stride 1).
 * Per-group widths must be multiples of 32 (cin) and one of 32/64/128/256 (cout): callers merge narrower
 * groups into block-diagonal ones.  out_act / out_raw bf16 [B][t_out_rows][cout] (rows >= t_out are left
 * untouched so a zero-initialised buffer keeps its zero padding), either may be NULL.
 * Flat sequences (seq_pitch > 0, batch == 1): many short sequences laid end to end on the time axis, seq_pitch
 * output rows each (seq_pitch * stride input rows), the first seq_valid of them real; the zero rows between two
 * sequences stand in for the conv padding, and rows >= seq_valid of every sequence are never written.  The late
 * discriminator layers (10..51 rows per sequence, hundreds of sequences) fill 128-row tiles this way. */
int hg_conv1d_tap_order(int ktaps, int stride, int pad_left, int* host_order);
int hg_conv1d_general_fwd(const void* x, const void* w_packed, const float* bias, int batch, int t_in_rows,
                          int c_total, int t_out, int t_out_rows, int groups, int cout, int ktaps, int stride,
                          int pad_left,
                          void* out_act, float act_slope, void* out_raw, int seq_pitch, int seq_valid, void* stream);

/* ------------------------------------------------------------------------------------------
 * hg_resblock_pair_fwd — one fused ResBlock1 step (src/models.py:36-41) for the narrow stages:
 *
 *   t1 = leaky_relu(conv1d(leaky_relu(x, in_slope), w1, dilation=dil1) + b1, in_slope)
 *   v  = (conv1d(t1, w2, dilation=1) + b2 + x + res1 + res2) * scale
 *   out_raw = bf16(v), out_act = bf16(leaky_relu(v, out_slope))        (either may be NULL)
 *
 * x, res*, out_* bf16 [B][T][c]; w*_packed bf16 [ktaps][c][c] (hg_pack_conv1d_weight); b* fp32 [c].
 * Both convolutions use "same" zero padding ((k-1)*d/2).  The intermediate t1 stays in shared memory;
 * HBM traffic is one read of x and one write per requested output.  out_* must not alias x.
 * hg_resblock_pair_supported(c, ktaps, dil1) tells whether the shape fits (c in {32,64}, both filter
 * banks resident in shared memory); otherwise the caller composes two hg_conv1d_fwd calls.
 * With w2_packed == NULL (b2 ignored) the same kernel runs ONE ResBlock2 step (src/models.py:64-67):
 *   v = (conv1d(leaky_relu(x, in_slope), w1, dilation=dil1) + b1 + x + res1 + res2) * scale
 * (hg_resblock_single_supported). */
int hg_resblock_pair_supported(int c, int ktaps, int dil1);
int hg_resblock_single_supported(int c, int ktaps, int dil1);
int hg_resblock_pair_fwd(const void* x, const void* w1_packed, const float* b1, const void* w2_packed,
                         const float* b2, int batch, int t, int c, int ktaps, int dil1, float in_slope,
                         const void* res1, const void* res2, float scale, void* out_raw, void* out_act,
                         float out_slope, const int* item_len, int item_mul, void* stream);   /* item_*: hg_conv1d_fwd */
/* hg_resblock_pair_fwd_actin — hg_resblock_pair_fwd on x_act = bf16(leaky_relu(x, in_slope)), 0 < in_slope <= 1,
 * instead of x: the first leaky_relu is already applied, and the residual x is rebuilt as
 * min(x_act, x_act / in_slope) (see hg_conv1d_fwd_actres). */
int hg_resblock_pair_fwd_actin(const void* x_act, const void* w1_packed, const float* b1, const void* w2_packed,
                               const float* b2, int batch, int t, int c, int ktaps, int dil1, float in_slope,
                               const void* res1, const void* res2, float scale, void* out_raw, void* out_act,
                               float out_slope, const int* item_len, int item_mul, void* stream);

/* ------------------------------------------------------------------------------------------
 * Discriminator ends (bandwidth-bound CUDA-core kernels).
 * hg_disc_first_conv_fwd: the Cin = 1 layers — DiscriminatorS convs[0] (src/models.py:196; period = 1) and
 *   DiscriminatorP convs[0] (:134) with the right-side reflect pad and the [B,1,T] -> [B,1,H,p] view
 *   (:146-151) folded into the addressing.  y fp32 [B][T]; w fp32 [cout][k]; out bf16
 *   [B*period][h_rows_out][cout] = leaky_relu(conv + bias); rows >= H_out are not written.
 * hg_disc_last_conv_fwd: the Cout = 1 layers (conv_post :141,204): x bf16 [S][h_rows][c], w fp32 [c][k],
 *   out fp32 [S][h] (no activation).
 * hg_avgpool_4_2_2_fwd: AvgPool1d(4,2,padding=2), zero padding counted (:227-230); out length t/2 + 1.
 * hg_disc_export_fmap: bf16 [B*period][h_rows][c] -> the reference's fp32 [B][c][H][period]. */
int hg_disc_first_conv_fwd(const float* y, const float* w, const float* bias, int batch, int t, int period,
                           int k, int stride, int pad, int cout, int h_rows_out, void* out, float slope,
                           void* stream);
int hg_disc_last_conv_fwd(const void* x, const float* w, const float* bias, int nseq, int h, int h_rows, int c,
                          int k, float* out, void* stream);
int hg_avgpool_4_2_2_fwd(const float* x, int batch, int t, float* out, void* stream);
int hg_disc_export_fmap(const void* x, int batch, int period, int h, int h_rows, int c, float* out,
                        void* stream);
/* hg_disc_import_fmap — the inverse layout change: fp32 [B][c][H][period] -> bf16 [B*period][h_rows][c] (rows >= H
 * untouched).  Carries a gradient that arrives at an exported feature map (torch autograd through feature_loss,
 * src/models.py:251-257) into the data-gradient chain (hg_conv1d_dgrad's pre_add). */
int hg_disc_import_fmap(const float* in, int batch, int period, int h, int h_rows, int c, void* x, void* stream);

/* ------------------------------------------------------------------------------------------
 * Layout edges.
 * hg_ncl_to_nlc: fp32 [B][C][T] -> bf16 [B][T][c_pad] (zero-filled channels >= C); the mel input of
 *   Generator.forward (src/models.py:100-101).  `out` receives the values, `out_act` (optional)
 *   leaky_relu(., act_slope) of them; either may be NULL.
 * hg_nlc_to_ncl: bf16 [B][T][C] -> fp32 [B][C][T]; used by tests / feature-map export.
 */
int hg_ncl_to_nlc(const float* x, int batch, int c, int t, int c_pad, void* out, void* out_act,
                  float act_slope, void* stream);
int hg_nlc_to_ncl(const void* x, int batch, int t, int c, float* out, void* stream);

/* hg_float_to_int16 — out[i] = (int16) trunc(x[i] * scale): the `audio * MAX_WAV_VALUE` -> `astype('int16')` of the
 * reference's inference drivers (src/inference.py:57-58, src/inference_e2e.py:51-52) on the device. */
int hg_float_to_int16(const float* x, long long n, float scale, int16_t* out, void* stream);

/* hg_loss_sum — the reductions behind feature_loss / discriminator_loss / generator_loss (src/models.py:251-282)
 * and the mel L1: mode 0 accumulates sum |a[i] - b[i]|, mode 1 accumulates sum (c - a[i])^2 into *out_acc (fp32,
 * atomicAdd: zero it first; the caller divides by n for the mean).  a, b fp32 device arrays of n elements. */
int hg_loss_sum(const float* a, const float* b, long long n, int mode, float c, float* out_acc, void* stream);

/* hg_segment_gather — batched form of MelDataset.__getitem__'s crop / right zero-pad (src/meldataset.py:141-150):
 * out[b][i] = i < valid[b] ? pool[start[b] + i] : 0.  pool fp32 (all utterances concatenated, resident in HBM),
 * start int64 [B] (utterance offset + the drawn audio_start), valid int32 [B] (min(len, seg)), out fp32 [B][seg]. */
int hg_segment_gather(const float* pool, const long long* start, const int* valid, int batch, int seg,
                      float* out, void* stream);

/* Staging of a packed int16 corpus's crops (hifigan_b200.corpus, CorpusSampler): the host copies a batch's crops into
 * one buffer that moves to the device in one copy; these kernels turn them into what hg_segment_gather produces from
 * the in-memory fp32 pool, bit for bit.
 * hg_segment_stage_i16: staged int16 [B][seg] -> out fp32 [B][seg], zero for i >= valid[b].  Sample q of an utterance
 *   whose peak is peak[b] = max|q| over the whole utterance becomes what the host pipeline q / 32768 (read_wav)
 *   / 32768 (MAX_WAV_VALUE) followed by the normalisation gives:
 *     HG_STAGE_PEAK  (q / m) * 0.95f, IEEE division (normalize_peak; m = 0 gives 0)
 *     HG_STAGE_FORK  sign(q) * 0.95f                (normalize_fork)
 *     HG_STAGE_NONE  q * 2^-30                      (fine-tuning: no normalisation)
 *   peak, valid int32 [B].
 * hg_segment_stage_mel: staged fp32 [B][fps][num_mels] (frame-major fine-tuning mel crops) -> out fp32
 *   [B][num_mels][fps], zero for frames >= valid_frames[b] (int32 [B]). */
enum { HG_STAGE_PEAK = 0, HG_STAGE_FORK = 1, HG_STAGE_NONE = 2 };
int hg_segment_stage_i16(const int16_t* staged, const int* peak, const int* valid, int batch, int seg, int mode,
                         float* out, void* stream);
int hg_segment_stage_mel(const float* staged, const int* valid_frames, int batch, int fps, int num_mels, float* out,
                         void* stream);

/* hg_conv_post_tanh_fwd — conv_post + tanh (src/models.py:113-114).  x bf16 [B][T][C] already
 * holds leaky_relu(., 0.01) (models.py:112, fused into the producer's epilogue).  w fp32 [C][k]
 * (folded weight of the single output channel), y fp32 [B][T] == the reference's [B,1,T].
 * Bandwidth-bound CUDA-core kernel. */
int hg_conv_post_tanh_fwd(const void* x, const float* w, const float* bias, int batch, int t, int c,
                          int k, float* y, void* stream);

/* ------------------------------------------------------------------------------------------
 * mel_spectrogram (src/meldataset.py:56-85): reflect-pad (n_fft-hop)/2, frames of win_size with a
 * periodic Hann window, rFFT(n_fft), |X|^2, HTK mel filterbank (un-normalised triangles), and
 * log(clamp(., 1e-5)) in ONE kernel.  The plan owns the immutable tables (window, twiddles, sparse
 * filterbank), keyed like the reference's cache key (meldataset.py:57).
 * n_fft 256 / 512 / 1024 / 2048 (the 16 kHz, 22.05 kHz and 44.1 / 48 kHz HiFi-GAN recipes) run the fused kernel with
 * the FFT held in registers; any other even n_fft in [16, 4096] (the reference's other callers:
 * src/speech_distillation/lightning_model.py:513-522 pass 16 kHz / fmax None / n_fft = a layer's kernel size) runs a
 * general direct-DFT kernel, one block per frame.
 * win_size <= n_fft, hop_size <= n_fft, num_mels <= 128.
 */
typedef struct hg_mel_plan hg_mel_plan;
int hg_mel_plan_create(hg_mel_plan** out_plan, int n_fft, int num_mels, int sampling_rate,
                       int hop_size, int win_size, double fmin, double fmax /* <0: sr/2 */,
                       void* stream);
int hg_mel_plan_destroy(hg_mel_plan* plan);
/* frames produced for t input samples (center=False after the manual reflect pad) */
int hg_mel_num_frames(const hg_mel_plan* plan, int t);
/* y fp32 [B][T] -> out fp32 [B][num_mels][frames]; minmax (optional, fp32[2], must be preset to
 * {+inf,-inf}) receives min/max of y so the caller can reproduce the reference's range warning
 * (meldataset.py:74-77) without a blocking sync per call. */
int hg_mel_fwd(const hg_mel_plan* plan, const float* y, int batch, int t, float* out,
               float* minmax, void* stream);

/* hg_mel_bwd — backward of hg_mel_fwd: dmel fp32 [B][num_mels][frames] (gradient at the log-mel output) ->
 * dy fp32 [B][T] ADDED to (zero it first).  y is the forward input; the spectrum is recomputed with the forward
 * kernel's FFT and the adjoint is one more n_fft / 2-point transform per frame.  n_fft 256, 512, 1024 or 2048. */
int hg_mel_bwd(const hg_mel_plan* plan, const float* y, const float* dmel, int batch, int t, float* dy,
               void* stream);

/* Test hook: the backward kernel's phase functions on the HOST (threads serialised).  host_y fp32 [B][T], host_dmel
 * fp32 [B][num_mels][frames]; host_dy fp32 [B][T] is ADDED to.  n_fft 256, 512, 1024 or 2048. */
int hg_mel_bwd_emulate_host(const hg_mel_plan* plan, const float* host_y, const float* host_dmel, int batch, int t,
                            float* host_dy);

/* Test hook: runs the mel kernel's per-thread phase functions on the HOST (threads serialised) so
 * the FFT / un-pack / CSR-mel arithmetic can be pinned without a GPU.  host_y, host_out are HOST
 * pointers; works on a plan created without a device. */
int hg_mel_emulate_host(const hg_mel_plan* plan, const float* host_y, int batch, int t,
                        float* host_out);

/* ==========================================================================================
 * Training step (UPSTREAM train.py restated in SURVEY.md §3.3; the reference runs these through torch autograd
 * and torch.optim.AdamW).  Gradients between kernels are bf16 [B][T][C] like the activations; parameter
 * gradients are fp32.
 * ========================================================================================== */

/* hg_pack_dgrad_weight: bf16 [ktaps][n][c] -> bf16 [ktaps][c][n] with the taps reversed — the filter bank with
 * which hg_conv1d_dgrad computes the data gradient of a stride-1 (dilated) conv, pad_left' = (k-1)*dil - pad_left. */
int hg_pack_dgrad_weight(const void* w_packed, int ktaps, int n, int c, void* out, void* stream);

/* hg_conv1d_dgrad — data gradient on the tcgen05 implicit-GEMM kernel (replaces convolution_backward's input
 * half for src/models.py:35-42,63-68,104,153-158,208-214):
 *   out[b,t,n] = ((sum_{j,c} dy[b, t + j*dil - pad_left, blk(n) + c] * w[j][n][c] + fm_coef * sgn(fm_g - fm_r))
 *                 * (mask_src[b,t,n] > 0 ? 1 : mask_slope) + res0 + res1 + res2) * scale
 * dy bf16 [B][t_dy_rows][c_dy_total], rows >= t_dy_valid read as zero; w_packed bf16 [ktaps][cout][c_dy_total/groups];
 * mask_src / fm_r / fm_g / res* / out bf16 [B][t_out_rows][cout] (optional except out).  mask_src is the layer
 * input as the forward stored it (leaky_relu'd: its sign is the sign of the pre-activation); fm_* add the
 * feature-matching L1 gradient (src/models.py:251-257).  groups > 1: N tile nt (width n_tile) reads dy channel
 * block nt % groups — the polyphase (phase-major) output of a strided grouped conv's gradient.
 * Flat sequences (seq_pitch > 0, batch == 1, see hg_conv1d_general_fwd): output element (row t, channel n) is stored
 * only when (t % seq_pitch) * seq_mul + n / seq_div < seq_valid — for a polyphase gradient seq_mul = stride and
 * seq_div = the layer's input channel count, i.e. the input position the element stands for must be real.
 *
 * pre_add (optional, bf16, same layout as out) is added to the accumulator before the mask: a gradient arriving
 * at the layer's activated input from outside the chain (an exported feature map's gradient under autograd).
 * bias_grad0..2 (optional, fp32 [bias_mod]): the bias gradient of the layer whose output `out` is the gradient of
 * — bias_grad*[n % bias_mod] += sum_{b,t} out[b,t,n], summed in fp32 from the accumulators BEFORE `out` is rounded
 * to bf16 (replaces a separate column-sum pass over the bf16 tensor).  bias_mod = 0: cout; a polyphase gradient
 * passes the layer's input channel count so the `stride` phases of a channel fold together.  Up to three
 * destinations receive the same sums (the last convs of the MRF branches share one output gradient). */
int hg_conv1d_dgrad(const void* dy, const void* w_packed, int batch, int t_dy_valid, int t_dy_rows, int c_dy_total,
                    int t_out, int t_out_rows, int groups, int n_tile, int cout, int ktaps, int dilation, int pad_left,
                    const void* mask_src, float mask_slope, const void* fm_r, const void* fm_g, float fm_coef,
                    const void* res0, const void* res1, const void* res2, float scale, void* out, int seq_pitch,
                    int seq_valid, int seq_mul, int seq_div, const void* pre_add, float* bias_grad0,
                    float* bias_grad1, float* bias_grad2, int bias_mod, void* stream);

/* hg_conv1d_wgrad — weight gradient as a tcgen05 implicit GEMM contracting over time (MN-major operands):
 *   dw[q][co][ci] (+)= sum_{b, t < t_out} dy[b,t,co] * xv[b, t + row(q), col(q) + blk(co) + ci]
 * in the packed layout of the forward weight (tap order of hg_conv1d_tap_order, [ktaps][cout][c_total/groups]).
 * x bf16 [B][t_in_rows][c_total] is the forward input (same zero-padding-rows contract as hg_conv1d_general_fwd),
 * dy bf16 [B][t_out_rows][cout].  c_total/groups must be 32, 64 or a multiple of 128; cout/groups one of
 * 32/64/128/256 when groups > 1.  accumulate == 0 zeroes dw first.  Partial sums are added with fp32 atomics. */
int hg_conv1d_wgrad(const void* x, const void* dy, int batch, int t_in_rows, int c_total, int t_out, int t_out_rows,
                    int groups, int cout, int ktaps, int stride, int dilation, int pad_left, float* dw_packed,
                    int accumulate, void* stream);

/* Packed weight gradient -> parameter layout: dw fp32 [cout][cin_g][k] from [k][rows_p][cin_tile]
 * (host_tap_order = hg_conv1d_tap_order or NULL for identity; merge = groups merged per block-diagonal tile,
 * cout_g = output channels per original group). */
int hg_unpack_wgrad_conv(const float* dw_packed, int cout, int cin_g, int k, int rows_p, int cin_tile, int cout_g,
                         int merge, const int* host_tap_order, float* dw, void* stream);

/* hg_wgrad_finish_conv / _convtr — the unpack to parameter layout and hg_weight_norm_bwd in ONE launch per layer:
 * packed weight gradient -> (weight_v.grad, weight_g.grad), or -> weight.grad when g == NULL.  conv: the layout of
 * hg_unpack_wgrad_conv; convtr: dw [cin][cout][k] from the polyphase [nshift][stride*cout_p][cin_p].  Added to the
 * existing values when accumulate != 0. */
int hg_wgrad_finish_conv(const float* dw_packed, int cout, int cin_g, int k, int rows_p, int cin_tile, int cout_g,
                         int merge, const int* host_tap_order, const float* v, const float* g, int accumulate,
                         float* dv, float* dg, void* stream);
int hg_wgrad_finish_convtr(const float* dw_packed, int cin, int cout, int k, int stride, int padding, int cin_p,
                           int cout_p, const float* v, const float* g, int accumulate, float* dv, float* dg,
                           void* stream);

/* hg_weight_norm_bwd — backward of w = g * v / ||v|| (norm over all dims but 0): dw, v fp32 [dim0][rest],
 * g fp32 [dim0] -> dv, dg (added to the existing values when accumulate != 0). */
int hg_weight_norm_bwd(const float* dw, const float* v, const float* g, int dim0, int rest, int accumulate,
                       float* dv, float* dg, void* stream);

/* Discriminator weight preparation (replaces torch.nn.utils.weight_norm's per-forward recompute for
 * src/models.py:132-141,194-204).  hg_fold_weight_norm: w_eff fp32 [dim0][rest] = g * v / ||v|| (g == NULL copies).
 * hg_pack_disc_weight: w_eff fp32 [cout][cin/groups][k] -> w_fwd bf16 [k][cout][cin_tile] (taps in
 * hg_conv1d_tap_order order, `merge` adjacent groups merged into one block-diagonal tile) for
 * hg_conv1d_general_fwd, and / or w_dgrad bf16 [nshift][stride*cin][cout_tile] (polyphase data-gradient filter
 * bank, geometry of hg_convtr1d_geometry(k, stride, pad)) for hg_conv1d_dgrad. */
int hg_fold_weight_norm(const float* v, const float* g, int dim0, int rest, float* w_eff, void* stream);
int hg_pack_disc_weight(const float* w_eff, int cout, int cin, int groups, int merge, int k, int stride, int pad,
                        void* w_fwd, void* w_dgrad, void* stream);

/* Spectral norm (torch.nn.utils.spectral_norm as used by MultiScaleDiscriminator's first scale, src/models.py:194,
 * 222; dim 0, eps 1e-12).  hg_spectral_norm_fwd: w fp32 [rows][cols]; with iterate != 0 (train mode) one power
 * iteration v <- normalize(W^T u), u <- normalize(W v) updates the u / v buffers IN PLACE like torch; then
 * sigma = u . (W v), w_eff = W / sigma.  u_copy / v_copy (optional) receive the vectors this call used (the next
 * call moves them on; the backward of THIS call needs them), sigma_out fp32 [1] the scalar.  ws: >= rows + cols
 * floats.  hg_spectral_norm_bwd: dw_orig (+)= (dw_eff - <dw_eff, w_eff> u v^T) / sigma (u, v constants of sigma, as
 * torch computes them under no_grad).  ws: >= 1 float. */
int hg_spectral_norm_fwd(const float* w, float* u, float* v, int rows, int cols, int iterate, float* w_eff,
                         float* sigma_out, float* u_copy, float* v_copy, float* ws, void* stream);
int hg_spectral_norm_bwd(const float* dw_eff, const float* w_eff, const float* u, const float* v, const float* sigma,
                         int rows, int cols, int accumulate, float* dw_orig, float* ws, void* stream);
/* ------------------------------------------------------------------------------------------
 * Batched weight preparation / weight-gradient finishing: ONE launch for many layers.
 *
 * The per-layer entry points above (hg_pack_conv1d_weight, hg_pack_convtr1d_weight, hg_pack_dgrad_weight,
 * hg_fold_weight_norm, hg_pack_disc_weight, hg_wgrad_finish_conv / _convtr) cost one launch per layer and call; a
 * training step re-derives ~135 filter banks after every optimizer update (the reference's weight_norm hook recomputes
 * w = g * v / ||v|| on every forward, src/models.py:16-31,56-59,81,86-88,96,132-140,196-204).  hg_prep_batched runs any
 * mix of those per-layer jobs in one grid: `jobs` is a device array of hg_prep_job, `block_job` a device array of
 * (job index, block index within the job) int pairs, one per block; blocks [first_block, first_block + nblocks) are
 * launched with `smem_bytes` of dynamic shared memory (the largest any job in the range needs).  Jobs whose input is
 * another job's output (a data-gradient bank is packed from the forward bank / the effective weight) go into a later
 * range = a later launch.  Integer fields by kind (i[..], tab[..]):
 *   HG_JOB_GEN_CONV        one block per padded output channel.  src0 v fp32 [cout][cin][k], src1 g (NULL: folded weight),
 *                          src2 bias (optional) -> dst0 bf16 [k][cout_p][cin_p], dst1 bias_out fp32 [cout_p] (optional).
 *                          i = {cout, cin, k, cout_p, cin_p}
 *   HG_JOB_GEN_CONVTR      one block per padded input channel.  src0 v fp32 [cin][cout][k], src1 g, src2 bias ->
 *                          dst0 bf16 [nshift][stride*cout_p][cin_p] (polyphase), dst1 bias_out fp32 [stride*cout_p].
 *                          i = {cin, cout, k, cin_p, cout_p, stride, padding, nshift, shift_min}
 *   HG_JOB_GEN_POST        one block.  conv_post folded to fp32: src0 v [1][cin][k], src1 g, src2 bias -> dst0 fp32
 *                          [cin_p][k], dst1 fp32 [1].  i = {cin, k, cin_p}
 *   HG_JOB_DISC_ROW        one block per output channel; smem cin_g * k floats.  src0 v fp32 [cout][cin_g][k], src1 g
 *                          (NULL: src0 is the effective weight) -> dst0 effective weight fp32 (optional), dst1 forward
 *                          bank bf16 [q][cout][cin_tile] (optional).  i = {cout, cin_g, k, merge, cout_g, cin_tile},
 *                          tab = tap order (hg_conv1d_tap_order)
 *   HG_JOB_TRANSPOSE_TILE  one block per 32 x 32 tile; smem 2 176 B.  src0 bf16 [k][n][c] -> dst0 bf16 [k][c][n], taps
 *                          reversed (hg_pack_dgrad_weight).  i = {k, n, c, tiles_c, tiles_n}; blocks = k*tiles_c*tiles_n
 *   HG_JOB_DISC_DGRAD_TILE one block per [tci input channels] x [32 dy channels]; smem 32 * (tci*k + 1) floats.  src0
 *                          effective weight fp32 -> dst0 bf16 [nshift][stride*cin][cout_tile] (hg_pack_disc_weight's
 *                          w_dgrad).  i = {cout, cin_g, k, merge, cout_g, cin, stride, pad, nshift, shift_min, cout_tile,
 *                          tci, cin / tci}; blocks = (cin / tci) * (cout_tile / 32)
 *   HG_JOB_FINISH_ROW      one block per dim-0 index of the parameter; smem d1 * k floats.  src0 packed dW fp32, src1 g
 *                          (NULL: plain weight), src2 v -> dst0 dv, dst1 dg (hg_wgrad_finish_conv / _convtr).
 *                          i = {mode (0 conv, 1 convtr), d0, d1, k, rows_p, cin_tile, cout_g, merge, stride, padding,
 *                          shift_min, cout_p, accumulate}, tab = packed position of tap j (conv)
 *   HG_JOB_LOSS_SUM        one block per `chunk` elements: *dst0 += partial sum (the reductions of hg_loss_sum and
 *                          of the bf16 feature maps, for many tensors at once).  src0 a, src1 b.  i = {mode (0: fp32
 *                          |a - b|, 1: fp32 (c - a)^2, 2: bf16 |a - b| counted in 16-byte groups), n low 32 bits,
 *                          n high 32 bits, chunk, c as float bits}
 */
enum {
  HG_JOB_GEN_CONV = 0, HG_JOB_GEN_CONVTR = 1, HG_JOB_GEN_POST = 2, HG_JOB_DISC_ROW = 3, HG_JOB_TRANSPOSE_TILE = 4,
  HG_JOB_DISC_DGRAD_TILE = 5, HG_JOB_FINISH_ROW = 6, HG_JOB_LOSS_SUM = 7
};
typedef struct hg_prep_job {
  const void* src0;
  const void* src1;
  const void* src2;
  void* dst0;
  void* dst1;
  int32_t kind;
  int32_t i[16];
  int32_t tab[64];
  int32_t pad_;
} hg_prep_job;
int hg_prep_job_size(void);
int hg_prep_batched(const hg_prep_job* jobs, const int* block_job, int first_block, int nblocks, int smem_bytes,
                    void* stream);

/* hg_colsum_bf16 — bias gradient: out[c] (+)= sum_{b, t < t_valid} x[b][t][c]; x bf16 [B][t_rows][C]. */
int hg_colsum_bf16(const void* x, int batch, int t_valid, int t_rows, int c, int accumulate, float* out, void* stream);

/* hg_conv_post_tanh_bwd — backward of hg_conv_post_tanh_fwd.  x bf16 [B][T][C] (the activated input), y fp32 [B][T]
 * (the forward output), dy fp32 [B][T] -> dx bf16 [B][T][C] = dx_scale * gradient at the PRE-activation of x (the
 * leaky_relu(., in_slope) mask taken from x's sign; dx_scale = 1 / num_kernels hands every MRF branch its share,
 * src/models.py:111), dw fp32 [C][k] and db fp32 [1] (both ADDED to; may be NULL).  dpre_ws fp32 [B][T] receives
 * dy * (1 - y^2).  bias_grad0..2 (optional, fp32 [C]) += column sums of dx in fp32 (see hg_conv1d_dgrad). */
int hg_conv_post_tanh_bwd(const void* x, const float* w, const float* y, const float* dy, int batch, int t, int c,
                          int k, float in_slope, float dx_scale, void* dx, float* dpre_ws, float* dw, float* db,
                          float* bias_grad0, float* bias_grad1, float* bias_grad2, void* stream);

/* Discriminator ends, backward.  hg_disc_last_conv_bwd: dx bf16 [S][h_rows][C] = (conv^T(dlogit) + fm_coef *
 * sgn(x - fm_r) + pre_add) * lrelu'(x) (x = the last wide layer's activated output; fm_r, pre_add optional, layout
 * of x), dw fp32 [C][k] / db ADDED to (NULL to skip; dx may be NULL too); bias_grad_in (optional, fp32 [C]) +=
 * column sums of dx in fp32 = the bias gradient of the layer that produced x.  hg_disc_first_conv_bwd: dpre bf16 [B*period][h_rows][cout] is the
 * gradient at the first conv's output (mask applied) -> dw fp32 [cout][k], db fp32 [cout] (ADDED to; NULL to skip)
 * and / or dy fp32 [B][T] (ADDED to: the gradient reaching the audio, reflect-padded tail folded back).
 * hg_avgpool_4_2_2_bwd: din fp32 [B][T] += backward of AvgPool1d(4,2,2) from dout fp32 [B][T/2+1]. */
int hg_disc_last_conv_bwd(const void* x, const float* w, const float* dlogit, int nseq, int h, int h_rows, int c,
                          int k, float slope, const void* fm_r, float fm_coef, const void* pre_add, void* dx, float* dw,
                          float* db, float* bias_grad_in, void* stream);
int hg_disc_first_conv_bwd(const float* y, const float* w, const void* dpre, int batch, int t, int period, int k,
                           int stride, int pad, int cout, int h_rows, float* dw, float* db, float* dy, void* stream);
int hg_avgpool_4_2_2_bwd(const float* dout, int batch, int t, float* din, void* stream);

/* Loss gradients (src/models.py:251-282 and the mel L1): mode 0 out = coef * sgn(a - b); mode 1 out = coef * (a - c);
 * mode 2 out = coef * (a - c) + coef2 * sgn(a - b).  scale_dev (optional): device scalar multiplied into coef and
 * coef2 (the gradient arriving at the mean, under torch autograd). */
int hg_loss_grad(const float* a, const float* b, long long n, int mode, float c, float coef, float coef2,
                 const float* scale_dev, float* out, void* stream);

/* hg_adamw_step — torch.optim.AdamW on one flat fp32 tensor (decoupled weight decay, bias correction by `step`,
 * or by the device-resident counter *dev_step when non-NULL so that a captured CUDA graph advances it; *dev_lr,
 * when non-NULL, overrides lr the same way (learning-rate schedules without re-capture); gradients multiplied by
 * grad_scale first: 1/world_size after a sum all-reduce). */
int hg_adamw_step(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2,
                  float eps, float weight_decay, int step, const int* dev_step, const float* dev_lr, float grad_scale,
                  void* stream);

/* Gradient-norm clipping with the skip of a non-finite step (torch.nn.utils.clip_grad_norm_ followed by
 * `if torch.isfinite(total): optim.step()`), without a host sync:
 *   hg_grad_sumsq          sum of squares of x fp32 [n] (x 4-byte aligned; 16-byte loads when 16-byte aligned) as
 *                          per-block fp64 partials into ONE slot of hg_grad_norm_slot_size() doubles at `partials`
 *                          (the whole slot is written).  Deterministic: the block partition depends on n only, no
 *                          floating-point atomics; several calls on different streams may fill different slots.
 *   hg_grad_norm_finalize  one block after every slot is written: norm = sqrt(sum of slots [0, nslots)) * grad_scale
 *                          (grad_scale = 1/world after a sum all-reduce: the norm of the averaged gradient), summed in
 *                          fp64 in a fixed order.  Writes *norm, *clip_coef = min(1, max_norm / (norm + 1e-6)) (fp32,
 *                          as torch; max_norm may be +inf), *skip = !isfinite(norm); then *dev_step += 1 when the norm
 *                          is finite, else *skipped += 1 (either pointer may be NULL).
 *   hg_adamw_step_guarded  hg_adamw_step with the step counter on the device (dev_step required, NOT advanced here),
 *                          that writes nothing when *skip != 0 and otherwise scales the gradient by
 *                          grad_scale * *clip_coef (the product rounded to fp32). */
int hg_grad_norm_slot_size(void);
int hg_grad_sumsq(const float* x, long long n, double* partials, void* stream);
int hg_grad_norm_finalize(const double* partials, int nslots, float max_norm, float grad_scale, float* norm,
                          float* clip_coef, int* skip, int* dev_step, int* skipped, void* stream);
int hg_adamw_step_guarded(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1,
                          float beta2, float eps, float weight_decay, const int* dev_step, const float* dev_lr,
                          float grad_scale, const float* clip_coef, const int* skip, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HIFIGAN_B200_H */
