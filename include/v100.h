/*
 * v100.h -- C ABI of libv100.so: the B200 (sm_100a) kernels behind Voice100's batched
 * inference hot path.
 *
 * The reference (kaiidams/voice100) is pure Python and has no FFI: its operator interface for
 * this path is a handful of torch.nn.Module.forward methods.  Each entry point below replaces
 * the library kernels one such forward dispatches to; the citation says which
 * (paths relative to the reference repository).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller; the library allocates nothing;
 *  - activations are "NCW with pitch": x[b][c][t] at  base + (b*C + c)*pitch + t,  t < T,
 *    16-bit unless stated, pitch % 8 == 0 (16-byte rows) and base 16-byte aligned.  This is the
 *    reference's own layout inside ConvVoiceEncoder/VoiceDecoder (asr.py:111, tts.py:174);
 *  - `dtype` selects the 16-bit storage type of activations and weights: V100_DTYPE_BF16 (default of
 *    the Python modules) or V100_DTYPE_F16 (same tensor-core throughput, 3 more mantissa bits);
 *    accumulation, folded BatchNorm, ReLU6 and residual adds are fp32 either way;
 *  - `stream` is a cudaStream_t passed as void*; all calls are asynchronous on it and are
 *    CUDA-graph capturable;
 *  - return value 0 = ok; <0 = V100_E_* below; >0 = a cudaError_t.  v100_last_error() returns a
 *    thread-local description of the last failure.  There is no CPU fallback: an unsupported
 *    shape is an error, never a silent slow path.
 */
#ifndef V100_H_
#define V100_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define V100_ABI_VERSION 9

#define V100_E_INVALID   (-1)   /* bad argument (null pointer, misaligned pitch, size <= 0)   */
#define V100_E_UNSUPPORTED (-2) /* shape outside what the kernels implement                   */
#define V100_E_DRIVER    (-3)   /* could not resolve cuTensorMapEncodeTiled / wrong device    */

#define V100_DTYPE_BF16 0
#define V100_DTYPE_F16  1

/* waveform sample types of v100_logmel */
#define V100_WAV_F32 0   /* fp32 samples in [-1, 1] (what torchaudio.load returns)              */
#define V100_WAV_I16 1   /* int16 PCM; scaled by 1/32768 in the kernel = torchaudio.load of 16-bit WAV */

/* sticky bits OR-ed into the optional device status word of the index-consuming kernels */
#define V100_STATUS_BAD_INDEX 1  /* an embedding id outside [0, V) (nn.Embedding raises IndexError) */

#define V100_ACT_NONE  0
#define V100_ACT_RELU6 1

/* log-mel output selectors */
#define V100_MEL_LOG_BF16_NCW  0  /* log(mel+offset), bf16 [B][64][pitch], frames >= n_i = log(offset)  */
#define V100_MEL_LOG_F32_NTC   1  /* log(mel+offset), fp32 [B][T][64]  (the reference's feature layout) */
#define V100_MEL_POWER_F32_NCW 2  /* mel power, fp32 [B][64][pitch]    (MelSpectrogram.forward layout)  */
#define V100_MEL_LOG_F16_NCW   3  /* as 0 with fp16 storage                                             */

int v100_abi_version(void);
const char* v100_last_error(void);

/*
 * Log-mel front end.  Replaces MelSpectrogramAudioTransform.melspec + log
 * (voice100/data_modules.py:276-281,290-291; torchaudio MelSpectrogram: reflect pad 256,
 * 512-sample frames every 160, periodic Hann(400) centred, |rFFT|^2, 64 HTK mel filters) and
 * the BLANK_AUDIO feature padding of generate_audio_text_batch (data_modules.py:446-455).
 *   wav      [B][wav_pitch] samples of `wav_dtype` (V100_WAV_F32 | V100_WAV_I16); clip i is valid for len[i]
 *            samples; len[i] is clamped to [0, L_max] on the device (L_max <= wav_pitch = row capacity).
 *            torchaudio refuses clips of <= 256 samples (reflect padding); here they are evaluated with the
 *            reflected index clamped into the clip, and a clip of 0 samples yields BLANK_AUDIO only.
 *   fb_*     the sparse mel filterbank: filter m covers bins [fb_start[m], fb_start[m]+fb_count[m])
 *            with weights fb_w[fb_off[m] ...], fb_nnz weights in all (built by the host from the torchaudio formula)
 *   out      see V100_MEL_*;  T = frames written per clip (>= max_i 1 + len[i]/160)
 *   frames_out  optional int32 [B]: 1 + len[i]/160, the `audio_len` of the batch (data_modules.py:448)
 */
int v100_logmel(const void* wav, int wav_dtype, const int32_t* len, int B, int64_t wav_pitch, int L_max,
                const int32_t* fb_start, const int32_t* fb_count, const int32_t* fb_off,
                const float* fb_w, int fb_nnz, float log_offset,
                void* out, int T, int64_t out_pitch, int out_mode, int32_t* frames_out, void* stream);

/*
 * The same front end for any other MelSpectrogramAudioTransform configuration (the reference's constructor takes
 * sample_rate, n_fft, win_length, hop_length, n_mels -- data_modules.py:263-281 -- although its code only ever builds
 * 512 / 400 / 160 / 64, which v100_logmel serves): n_fft a power of two in [8, 2048], 0 < win_length <= n_fft,
 * hop_length > 0, any sparse filter bank with n_mels filters.  Outputs as v100_logmel with 64 replaced by n_mels and
 * 160 by hop_length; NCW pitches are not constrained.  A plain kernel (one CTA per frame), not a tuned one.
 */
int v100_logmel_generic(const void* wav, int wav_dtype, const int32_t* len, int B, int64_t wav_pitch, int L_max,
                        int n_fft, int win_length, int hop_length, int n_mels,
                        const int32_t* fb_start, const int32_t* fb_count, const int32_t* fb_off, const float* fb_w,
                        float log_offset, void* out, int T, int64_t out_pitch, int out_mode, int32_t* frames_out,
                        void* stream);

/*
 * fp32 [B][T][C] features -> 16-bit NCW [B][C][pitch].  Replaces the transpose at the top of
 * AudioToTextCTC.forward (voice100/models/asr.py:111) plus the storage cast.
 */
int v100_ntc_f32_to_ncw16(const float* x, void* y, int B, int T, int C, int64_t y_pitch, int dtype, void* stream);

/*
 * Dense fp32 NCW [B][C][T] <-> pitched 16-bit NCW.  Entry/exit casts of ConvVoiceEncoder.forward
 * (voice100/models/asr.py:78-79) and VoiceDecoder.forward (tts.py:28-29) when those sub-modules are
 * called on their own with the reference's fp32 NCW tensors.
 */
int v100_ncw_f32_to_16(const float* x, void* y, int64_t y_pitch, int B, int C, int T, int dtype, void* stream);
int v100_ncw_16_to_f32(const void* x, int64_t x_pitch, float* y, int B, int C, int T, int dtype, void* stream);

/*
 * Pointwise (1x1) Conv1d as a tcgen05 GEMM (bf16 or fp16 operands, fp32 accumulate) with TMA-staged
 * tiles and TMEM accumulators:
 *   y[b][co][t] = act(scale[co] * sum_ci W[co][ci] * x[b][ci][t] + shift[co]) (+ res[b][co][t])
 * Replaces Conv1d(k=1,bias=False) + BatchNorm1d(eval) + ReLU6 and the residual add of
 * InvertedResidual (voice100/models/asr.py:27-37,45-59); scale/shift are the folded BN.
 *   W [C_out][C_in] row-major, C_in % 8 == 0;  x, y, res NCW (all of `dtype`);  scale/shift fp32 [C_out]
 *   (scale may be NULL = 1);  res may be NULL; res shares y's pitch.
 */
int v100_conv1x1(const void* x, int64_t x_pitch, const void* W, const float* scale,
                 const float* shift, const void* res, void* y, int64_t y_pitch,
                 int B, int C_in, int C_out, int T, int act, int dtype, void* stream);

/*
 * Same GEMM, fp32 NCW output and bias only:  y[b][co][t] = sum_ci W[co][ci] x[b][ci][t] + bias[co].
 * Replaces the biased 1x1 heads: LinearCharDecoder (asr.py:89-94), TextToAlignTextModel's
 * Conv1d(512->2) (tts.py:77) and VoiceDecoder's Conv1d(256->260) (tts.py:26).
 */
int v100_conv1x1_f32out(const void* x, int64_t x_pitch, const void* W, const float* bias,
                        float* y, int64_t y_pitch, int B, int C_in, int C_out, int T, int dtype, void* stream);

/*
 * Depthwise Conv1d + folded BN + ReLU6:
 *   y[b][c][o] = act(scale[c] * sum_j w[c][j] * x[b][c][o*stride + j - (k-1)/2] + shift[c])
 * with zero padding, k odd, T_out = (T_in-1)/stride + 1.  Replaces ConvBNActivate with
 * groups=C (voice100/models/asr.py:27-37,49).  w [C][k] of `dtype`.
 */
int v100_dwconv1d(const void* x, int64_t x_pitch, const void* w, const float* scale,
                  const float* shift, void* y, int64_t y_pitch,
                  int B, int C, int T_in, int k, int stride, int act, int dtype, void* stream);

/* Same contract, always the plain CUDA-core kernel (any stride).  Used for stride != 1 internally;
 * exported so the tests can cross-check the tensor-core kernel against it on the device. */
int v100_dwconv1d_simt(const void* x, int64_t x_pitch, const void* w, const float* scale,
                       const float* shift, void* y, int64_t y_pitch,
                       int B, int C, int T_in, int k, int stride, int act, int dtype, void* stream);

/*
 * ConvTranspose1d(C_in -> C_out, kernel 5, stride 2, padding 2) + bias as a two-phase tcgen05
 * GEMM (even outputs: taps 0,2,4; odd outputs: taps 1,3; two TMEM accumulators interleaved in the
 * epilogue).  Replaces VoiceDecoder.layers[4] (voice100/models/tts.py:22).
 *   Wp [C_out][5*C_in], Wp[co][tap*C_in + ci] = weight[ci][co][tap];  y NCW, T_out = 2T-1;
 *   workspace: caller-provided 16-bit [B][3*C_in][x_pitch] scratch (the x(t+1) | x(t) | x(t-1) stack:
 *   TMA box coordinates must be 16-byte aligned, so one-step time shifts are materialised once).
 */
int v100_convtranspose1d_k5s2(const void* x, int64_t x_pitch, const void* Wp, const float* bias,
                              void* workspace, void* y, int64_t y_pitch,
                              int B, int C_in, int C_out, int T, int dtype, void* stream);

/*
 * Embedding lookup into NCW: y[b][c][t] = table[ids[b][t]][c].  Replaces nn.Embedding +
 * transpose (voice100/models/tts.py:81-83,174-175).  ids int64 [B][T]; table [V][C] of 16-bit elements
 * (either storage type: the rows are copied, not converted).  An id outside [0, V) -- an IndexError in the
 * reference -- yields a zero column and sets V100_STATUS_BAD_INDEX in *status (optional device int32, sticky:
 * the caller zeroes it and reads it back when it wants the check).
 */
int v100_embedding_ncw16(const int64_t* ids, const void* table, void* y, int64_t y_pitch,
                         int B, int T, int V, int C, int32_t* status, void* stream);

/*
 * CTC head tail: fp32 NCW logits [B][V][pitch] -> logits [B][T][V] fp32 (optional) and greedy
 * tokens int64 [B][T] (first maximal index).  Replaces transpose(1,2) (asr.py:114) and
 * logits.argmax(-1) (tests/test_onnx.py:40).  With audio_len/out_len (both or neither; int32 [B]) it also
 * writes out_len[b] = (audio_len[b] + 1) / 2 = AudioToTextCTC.output_length (asr.py:81-82,118-122).
 */
int v100_ctc_finalize(const float* y_ncw, int64_t y_pitch, float* logits_or_null, int64_t* tokens,
                      int B, int V, int T, const int32_t* audio_len, int32_t* out_len, void* stream);

/*
 * CTC collapse on the device: per row, within the first valid_len[b] tokens (all T when valid_len is
 * NULL), drop tokens equal to their predecessor, then drop `blank`; survivors are written in order to
 * out[b][0..out_len[b]) and the rest of the row is filled with `blank`.  Replaces the id-level effect of
 * CharTokenizer/BasicTokenizer.merge_repeated (voice100/text.py:99-104,140-145) so that only collapsed
 * ids need to cross PCIe (SURVEY.md section 8f #2).  tokens/out int64 [B][T] (distinct buffers).
 */
int v100_ctc_collapse(const int64_t* tokens, const int64_t* valid_len, int64_t* out, int32_t* out_len,
                      int B, int T, int blank, void* stream);

/*
 * Batched CTC forced alignment (Viterbi best path over the blank-expanded label sequence).  Replaces the
 * per-utterance numpy DP `ctc_best_path` (voice100/models/align.py:18-66, max_move = 3) that the v2 aligner
 * calls through .cpu().numpy() for every utterance (voice100/models/_asr_v2.py:100-119) -- SURVEY.md 8f #3.
 *   logprob  fp32 [B][T][V] log-probabilities, or raw logits with normalize != 0: the kernel then applies
 *            log_softmax over V itself (_asr_v2.py:95);  logit_len int32 [B] valid frames;
 *   text     int64 [B][L] labels (0 = blank never appears inside);  text_len int32 [B];
 *   workspace uint8 [B][T][2L+1] back-pointers (caller-provided scratch);
 *   score fp32 [B]; path int32 [B][T] = state index per frame (the reference's best_path);
 *   path_labels int64 [B][T] = expanded label per frame (best_labels); entries past logit_len are 0.
 * Where the reference raises IndexError the utterance gets score = NaN and path = -1: frames that cannot reach
 * state 2*text_len - 1 (exactly the reference's rule, align.py:57-58: with one state missing the result is valid
 * only if the last live score is not the larger one), an empty text, or a label outside [0, V).
 */
int v100_ctc_best_path(const float* logprob, const int32_t* logit_len, const int64_t* text,
                       const int32_t* text_len, uint8_t* workspace, float* score, int32_t* path,
                       int64_t* path_labels, int B, int T, int V, int L, int normalize, void* stream);

/*
 * WORLD head tail: fp32 NCW decoder output -> hasf0[B][T], f0[B][T], logspc[B][T][S], (hascodeap[B][T][A],)
 * codeap[B][T][A]; with `unnormalize` != 0: std*x+mean, f0 := 0 where hasf0 < 0 and (layout 2) codeap := 0 where
 * hascodeap < 0.  S = logspc_size (257, or 25 with use_mcep), A = codeap_size.
 *   layout 1: channels [hasf0 | f0 | logspc(S) | codeap(A)] -- AlignTextToAudioModel: split + WORLDNorm.unnormalize
 *             + where (tts.py:181-190,196-200; _layers_v1.py:131-138); hascodeap is ignored
 *   layout 2: channels [hasf0 | f0 | logspc(S) | hascodeap(A) | codeap(A)] -- AlignTextToAudio (_tts_v2.py:65-71,80-91)
 * mean/std fp32 [1 + S + A] ordered f0, logspc, codeap (ignored when unnormalize == 0).  hasf0/hascodeap may be NULL.
 */
int v100_world_finalize(const float* y_ncw, int64_t y_pitch, const float* mean, const float* std,
                        float* hasf0, float* f0, float* logspc, float* hascodeap, float* codeap,
                        int B, int T, int logspc_size, int codeap_size, int layout, int unnormalize, void* stream);

/* fp32 NCW [B][C][pitch] -> fp32 [B][T][C] (align head output [B][L][2]). */
int v100_ncw_f32_to_ntc(const float* y_ncw, int64_t y_pitch, float* out, int B, int C, int T, void* stream);

/*
 * Feature masking of a padded batch: out[b][t][c] = log(max(exp(audio[b][t][c]) * (t < audio_len[b]), log_offset)),
 * i.e. frames at or past an utterance's own length become log(log_offset) = BLANK_AUDIO and valid frames are floored
 * there.  audio / out fp32 [B][T][C] contiguous (out may alias audio), audio_len int32 [B].
 * Replaces BatchSpectrogramAugumentation.maskaudio (voice100/audio.py:106-108).
 */
int v100_maskaudio(const float* audio, const int32_t* audio_len, float* out, int B, int T, int C, float log_offset,
                   void* stream);

/* ------------------------------------------------------------------------------------------------
 * v2 models: ConvLayerBlock / ConvTransposeLayerBlock (voice100/models/_layers_v2.py:29-88) and the
 * bidirectional LSTM stacks of AudioToAlignText (_asr_v2.py:31-49), TextToAlignText (_align_v2.py:22-43)
 * and AlignTextToAudio (_tts_v2.py:35-60).
 *
 * Time-major layout ("TM") used around the recurrent layers: x[c][t * Bp + b], 16-bit, Bp = batch rounded up
 * to a multiple of 8.  A TM tensor is also a valid NCW tensor with B = 1, T = pitch = T * Bp, so the LSTM input
 * projection (weight_ih, bias_ih + bias_hh) and the dense heads are plain v100_conv1x1 / v100_conv1x1_f32out
 * calls on it.
 * ------------------------------------------------------------------------------------------------ */

/*
 * nn.Conv1d(C_in, C_out, k, stride, padding) of ConvLayerBlock (_layers_v2.py:41-48,52), dense (groups = 1):
 * y[b][co][to] = bias[co] + sum_{ci,j} Wp[co][j*C_in + ci] * x[b][ci][to*stride + j - pad], zero padded,
 * T_out = (T_in + 2*pad - k)/stride + 1.  Wp is the weight re-packed tap-major ([C_out][k*C_in]); bias fp32 [C_out]
 * (zeros when the layer has none).  k in {3,5}, stride in {1,2}, (k*C_in) % 8 == 0.
 * workspace: 16-bit [B][k*C_in][y_pitch] (the k shifted/strided views stacked along channels; TMA needs
 * 16-byte aligned box offsets, so tap shifts are materialised once and the conv becomes one GEMM).
 */
int v100_conv1d(const void* x, int64_t x_pitch, const void* Wp, const float* bias, void* workspace,
                void* y, int64_t y_pitch, int B, int C_in, int C_out, int T_in, int k, int stride, int pad,
                int dtype, void* stream);

/*
 * The same nn.Conv1d for stride 1 and padding (k-1)/2 on TIME-MAJOR tensors (x [C_in][T*Bp] -> y [C_out][T*Bp]):
 * a tap is a shift by (j - pad)*Bp columns, which is a 16-byte aligned TMA box offset, so the k taps accumulate in
 * one GEMM tile with no workspace and no data movement.  k odd, <= 5; C_in a multiple of 64; Wp and bias as above.
 * Columns b in [B, Bp) carry conv(0) = bias.
 */
int v100_conv1d_tm(const void* x, const void* Wp, const float* bias, void* y, int C_in, int C_out, int T, int Bp,
                   int k, int dtype, void* stream);

/*
 * transpose -> nn.LayerNorm(C) -> transpose -> gelu of ConvLayerBlock.forward (_layers_v2.py:53-57,84-88):
 * per (b, t) column, y = gelu((x - mean_c) * rsqrt(var_c + eps) * gamma[c] + beta[c]), biased variance,
 * exact (erf) GELU.  NCW in, NCW out (x and y may alias), statistics in fp32.
 */
int v100_layernorm_gelu(const void* x, int64_t x_pitch, const float* gamma, const float* beta, float eps,
                        void* y, int64_t y_pitch, int B, int C, int T, int dtype, void* stream);

/* NCW 16-bit [B][C][pitch] -> TM [C][T*Bp] (columns b in [B,Bp) zero) and back.
 * Replace the transposes + pack_padded_sequence / pad_packed_sequence around nn.LSTM (_asr_v2.py:44-47). */
int v100_ncw_to_tm(const void* x, int64_t x_pitch, void* y, int B, int C, int T, int Bp, void* stream);
int v100_tm_to_ncw(const void* x, void* y, int64_t y_pitch, int B, int C, int T, int Bp, void* stream);

/*
 * One bidirectional nn.LSTM layer in eval mode over a packed batch (_asr_v2.py:33-35,46; gate order i,f,g,o).
 * gx:  TM 16-bit [8H][T*Bp] = W_ih x + b_ih + b_hh for every step; rows [0,4H) forward, [4H,8H) reverse
 * w_hh: 16-bit [2][4H][H] (weight_hh_l{n}, weight_hh_l{n}_reverse)
 * lengths: int32 [B]; utterance b runs over steps [0, lengths[b]) (reverse direction starts at its last step
 *          with zero state), outputs past the length are zero (pad_packed_sequence)
 * y:   TM 16-bit [2H][T*Bp], rows [0,H) forward, [H,2H) reverse (= the concatenated nn.LSTM output)
 * workspace: v100_lstm_workspace_bytes(B, H) bytes, 1024-byte aligned (h exchange buffers + step counters)
 * H a multiple of 64, <= 512.  Cell state fp32, h rounded to the storage type each step.
 */
int64_t v100_lstm_workspace_bytes(int B, int H);
int v100_lstm_layer(const void* gx, const void* w_hh, const int32_t* lengths, void* y, void* workspace,
                    int B, int Bp, int T, int H, int dtype, void* stream);

/* ------------------------------------------------------------------------------------------------
 * TTS text alignment
 * ------------------------------------------------------------------------------------------------ */

/* per-utterance status codes of v100_tts_align; the reference raises where noted */
#define V100_ALIGN_OK       0
#define V100_ALIGN_INDEX    1   /* rule 1: a frame index outside [-total, total)          (IndexError)    */
#define V100_ALIGN_NEGATIVE 2   /* the total length is negative                            (RuntimeError)  */
#define V100_ALIGN_NAN      3   /* the duration sum is NaN                                 (ValueError)    */
#define V100_ALIGN_INF      4   /* the duration sum is +-inf                               (OverflowError) */
#define V100_ALIGN_TOO_LONG 5   /* total >= 2^31 frames: frame indices are int32                           */
#define V100_ALIGN_CAPACITY 6   /* total > T_cap: the first T_cap frames are written, the rest dropped      */

/*
 * Per-token (gap, duration) pairs -> aligned text, the int64 [B][T_cap] frame ids v100_embedding_ncw16 consumes.
 * Replaces TextToAlignTextModel.align (voice100/models/tts.py:89-110, rule = 1) and TextToAlignText.align
 * (voice100/models/_align_v2.py:54-82, rule = 2), each applied to one utterance at a time on the host, with the same
 * results bit for bit:
 *   rule 1: t = head + running sum of the entries in token order (float64); token i covers frames
 *           [rint(t + gap_i), rint(t + gap_i + dur_i)), or [s, max(0, s + 1)) when the two are equal; later tokens
 *           overwrite earlier ones; a frame j < 0 wraps to total + j; j outside [-total, total) is V100_ALIGN_INDEX.
 *           total = head + int(sum) + tail.
 *   rule 2: the first gap is skipped; s_i = max(trunc(t), e_{i-1}), e_i = max(trunc(t + dur_i), s_i + 1) (e_{-1} = 0);
 *           frames at or past total are dropped.  total = head + int(sum - gap_0) + tail, the subtraction in fp32.
 * The running position is summed by one thread per utterance, strictly in token order, as the reference's Python float
 * is.  `sum` is the float32 rounding of the sequential float64 sum (the reference's CPU torch.sum may round differently
 * when the sum lies within a few float32 ulps of an integer).
 *   durations  fp32, element (b, i, c) at durations[b*stride_b + i*stride_l + c*stride_c], c = 0 gap, 1 duration;
 *              this reads the align heads in place: the v1 NCW head [B][2][pitch] is (2*pitch, 1, pitch), the v2 dense
 *              head over a time-major tensor ([1][2][pitch >= T*Bp], column t*Bp + b) is (1, Bp, pitch)
 *   log1p_input  != 0: every value x is first replaced by expf(x) - 1, the exp(pred) - 1 the reference applies to the
 *              head output (TextToAlignText.predict, _align_v2.py:45-48)
 *   durations_out  optional fp32 [B][L][2]: the durations after that step, for all L tokens
 *   text       int64 [B][L], row stride text_stride;  text_len  optional int32 [B] (NULL = L; clamped to [0, L])
 *   aligntext  int64 [B][T_cap] or NULL (a plan-only call: lengths and status only, no capacity check); every element
 *              of [0, T_cap) is written: frames of failed utterances and frames past the length are 0
 *   aligntext_len  int32 [B]: the total length (also for V100_ALIGN_INDEX and V100_ALIGN_CAPACITY), 0 where undefined
 *   status     int32 [B]: V100_ALIGN_*
 *   filled_len optional int32 [B]: frames written = min(total, T_cap), 0 for a failed utterance (the LSTM lengths of
 *              the v2 audio model);  frame_len  optional int32 [B]: 2*filled_len - 1 (0 if filled_len is 0), the WORLD
 *              frames the audio models' stride-2 decoders produce from it
 * L <= 4096 (V100_E_UNSUPPORTED above).  One CTA per utterance; no host synchronisation, CUDA-graph capturable.
 */
int v100_tts_align(const float* durations, int64_t stride_b, int64_t stride_l, int64_t stride_c, int log1p_input,
                   float* durations_out, const int64_t* text, int64_t text_stride, const int32_t* text_len, int B,
                   int L, int rule, int head, int tail, int64_t* aligntext, int T_cap, int32_t* aligntext_len,
                   int32_t* status, int32_t* filled_len, int32_t* frame_len, void* stream);

/* ------------------------------------------------------------------------------------------------
 * WORLD waveform synthesis (fs = 16000, fft_size = 512, frame period 10 ms)
 *
 * Replaces WORLDVocoder.decode (voice100/vocoder.py:89-102): pyworld.decode_aperiodicity followed by
 * pyworld.synthesize, i.e. WORLD's DecodeAperiodicity (codec.cpp) and Synthesis (synthesis.cpp), run on the host one
 * utterance at a time.  The contract is the float64 restatement oracle/world.py; parity with pyworld itself has not
 * been checked (DESIGN.md section 3.8 lists the details a restatement could have wrong).
 * Inputs are fp32 device tensors read in place through strides (element strides):
 *   f0      (b, t)    at f0[b*f0_sb + t*f0_st]                       Hz; < 32.25 (and negative) = unvoiced
 *   logspc  (b, t, k) at logspc[b*sp_sb + t*sp_st + k*sp_sk], k < 257  natural log of the power spectrum (sp = exp)
 *   codeap  (b, t)    at codeap[b*ap_sb + t*ap_st]                    coded aperiodicity, one band at 16 kHz
 *   frame_len  optional int32 [B]: utterance b has min(max(frame_len[b], 0), T) frames (NULL = T)
 * ------------------------------------------------------------------------------------------------ */

/* per-utterance status codes of v100_world_timebase / v100_world_synthesize */
#define V100_WORLD_OK        0
#define V100_WORLD_SHORT     1   /* fewer than 2 frames (WORLD reads f0[-1] there)                           */
#define V100_WORLD_NONFINITE 2   /* a NaN or inf in f0, logspc or codeap of the utterance's frames            */

/*
 * WORLD's randn() stream after its reseed (matlabfunctions.cpp randn / initializeSeed): xorshift128 with state
 * (123456789, 362436069, 521288629, 88675123); value j sums (w >> 4) over 12 steps and is sum / 2^28 - 6, exact in
 * float64.  out: float64 [n] on the device.  One thread runs the recurrence (about 12 n dependent steps); the table
 * depends on n only, so build it once and keep it.
 */
int v100_world_noise(double* out, int64_t n, void* stream);

/*
 * Bytes of the workspace of v100_world_timebase / v100_world_synthesize for B utterances of at most y_len_max = 160 T
 * samples; it does not depend on the WORLD parameters.  Layout, Yp = y_len_max rounded up to a multiple of 32:
 *   int32 head[B][4]  (status, y_len, sample of the first pulse, number of pulses), padded to 256 bytes;
 *   int32 info[B][Yp] -1 where no pulse sits at the sample, else (noise size << 1) | vuv, padded to 256 bytes;
 *   double tau[B][Yp] the pulse's fractional time shift in s (defined at pulse samples only).
 */
int64_t v100_world_workspace_bytes(int B, int64_t y_len_max);

/*
 * The time base of Synthesis (GetTimeBase: GetTemporalParametersForTimeBase + interp1 + GetPulseLocationsForTimeBase)
 * into the workspace, one CTA per utterance: f0 < 32.25 Hz is unvoiced, a knot at T is extrapolated
 * (2 f[T-1] - f[T-2]), f0 and voicing are interpolated per sample with interp1's formula, vuv > 0.5 keeps f0 and
 * anything else takes 500 Hz; the phase sum((2 pi) f0 / fs) is accumulated by one thread in sample order in float64
 * and a pulse sits at sample i < y_len - 1 where |fmod(phi[i+1], 2 pi) - fmod(phi[i], 2 pi)| > pi.  No FMA
 * contraction: the pulse samples and shifts equal oracle/world.py's bit for bit.
 *   wav_len  int32 [B]: 160 frames (0 for a rejected utterance);  status  int32 [B]: V100_WORLD_*
 */
int v100_world_timebase(const float* f0, int64_t f0_sb, int64_t f0_st, const float* logspc, int64_t sp_sb,
                        int64_t sp_st, int64_t sp_sk, const float* codeap, int64_t ap_sb, int64_t ap_st,
                        const int32_t* frame_len, int B, int T, void* workspace, int32_t* wav_len, int32_t* status,
                        void* stream);

/*
 * DecodeAperiodicity + Synthesis: v100_world_timebase, then one CTA per (1024-sample tile, utterance) computes every
 * pulse response that reaches its tile (GetOneFrameSegment: spectral envelope and aperiodic ratio interpolated at the
 * pulse, periodic part min-phase(log(S (1 - A) + eps) / 2) with the fractional delay and DC removal, aperiodic part
 * min-phase(log(S A + eps) / 2) times the pulse's noise) in fp32 and adds them in pulse order.  Deterministic: the
 * same inputs give the same bits in any batch.
 *   noise      v100_world_noise output with noise_len >= 160 T values
 *   workspace  v100_world_workspace_bytes(B, 160 T) bytes, 256-byte aligned
 *   wav        fp32 [B][wav_pitch], wav_pitch >= 160 T: every sample of every row is written; samples at or past
 *              wav_len[b], and whole rows of rejected utterances, are 0
 *   wav_len, status as v100_world_timebase
 */
int v100_world_synthesize(const float* f0, int64_t f0_sb, int64_t f0_st, const float* logspc, int64_t sp_sb,
                          int64_t sp_st, int64_t sp_sk, const float* codeap, int64_t ap_sb, int64_t ap_st,
                          const int32_t* frame_len, int B, int T, const double* noise, int64_t noise_len,
                          void* workspace, float* wav, int64_t wav_pitch, int32_t* wav_len, int32_t* status,
                          void* stream);

/* ------------------------------------------------------------------------------------------------
 * WORLD analysis (fs = 16000, frame period 10 ms, fft_size 512)
 *
 * Replaces WORLDVocoder.encode (voice100/vocoder.py:66-88): pyworld.dio (f0_floor 71, f0_ceil 800, 2 channels an
 * octave, speed 1, allowed range 0.1), stonemask, cheaptrick (fft_size 512), d4c (threshold 0.85),
 * code_aperiodicity, then logspc = log(sp + 1e-15), run on the host one utterance at a time.  The contract is the
 * float64 restatement oracle/world_analysis.py; parity with pyworld itself has not been checked (DESIGN.md section
 * 3.10 lists the conventions a restatement could have wrong).  Status codes are V100_WORLD_*: V100_WORLD_SHORT for
 * fewer than 4 frames (L < 480 samples, where FixF0Contour returns early), V100_WORLD_NONFINITE for a NaN or inf
 * sample.
 * ------------------------------------------------------------------------------------------------ */

/*
 * Bytes of the workspace of v100_world_analyze for B utterances of at most L_max samples (vocoder.py:66-88).  It
 * depends on the shapes only; it is dominated by the refined zero crossings, 28 series of at most L_max / 2 + 1
 * float64 values per utterance (about 112 bytes a sample).
 */
int64_t v100_world_analysis_workspace_bytes(int B, int64_t L_max);

/*
 * WORLD analysis of a padded batch (vocoder.py:66-88): Dio + StoneMask + CheapTrick + D4C + CodeAperiodicity.
 *   wav        [B][wav_pitch] fp32 (wav_dtype 0) or int16 PCM (wav_dtype 1, scaled by 1 / 32768), unit stride along
 *              time; utterance b is wav[b][0, min(max(len[b], 0), L_max))
 *   taps       float64 [1633] on the device: DIO's low-cut filter (641 taps: w[i] = 0.5 - 0.5 cos(2 pi (i + 1) / 642),
 *              h = -w / sum(w), h[320] += 1), then the Nuttall windows of the 7 bands (320, 224, 160, 112, 80, 56, 40
 *              taps: 0.355768 - 0.487396 cos(2 pi u) + 0.144232 cos(4 pi u) - 0.012604 cos(6 pi u), u = i / (n - 1)),
 *              as the restatement's dio_taps() computes them
 *   noise      v100_world_noise output with noise_len >= 5290 (L_max / 160 + 1) values (CheapTrick's and D4C's dither)
 *   workspace  v100_world_analysis_workspace_bytes(B, L_max) bytes, 256-byte aligned
 *   T          frames of the outputs, T >= L_max / 160 + 1
 *   f0         fp32 [B][T] (Hz, 0 = unvoiced), logspc fp32 [B][T][257] (log(sp + 1e-15)), codeap fp32 [B][T]
 *              (20 log10 of the aperiodicity at 3000 Hz); every element is written, rows at or past frame_len[b] are 0
 *   frame_len  int32 [B]: len / 160 + 1 (0 for a rejected utterance);  status  int32 [B]: V100_WORLD_*
 * All float64.  The DIO stage (filters, crossings, contour, FixF0Contour) repeats the restatement's operations in its
 * order without FMA contraction, so its f0 contour is bit-identical to it.  Deterministic: an utterance's outputs do
 * not depend on the rest of the batch.  No host synchronisation; CUDA-graph capturable.  L_max above 2^30, or B or T
 * above 65535, is V100_E_UNSUPPORTED.
 */
int v100_world_analyze(const void* wav, int wav_dtype, int64_t wav_pitch, const int32_t* len, int B, int64_t L_max,
                       const double* taps, const double* noise, int64_t noise_len, void* workspace, int T, float* f0,
                       float* logspc, float* codeap, int32_t* frame_len, int32_t* status, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Resampling
 * ------------------------------------------------------------------------------------------------ */

/*
 * Polyphase sinc resampling of a padded batch.  Replaces torchaudio.functional.resample, which
 * MelSpectrogramAudioTransform.forward applies after load when a file is not at the transform's rate
 * (voice100/data_modules.py:288-289): torchaudio's _get_sinc_resample_kernel builds a dense [n][1][2w + o] kernel
 * and _apply_sinc_resample_kernel runs it as a conv1d at stride o.  Rates are reduced by their gcd (o -> n); the
 * non-zero taps of each phase p form one contiguous run, and only that run is stored:
 *   out[b][j n + p] = sum_{i < count[p]} taps[off[p] + i] * wav[b][j o + start[p] + i - w]
 * with wav taken as 0 outside [0, len[b]): padding past a row's length is never read into a result.  Each output is
 * one fp32 fmaf chain in i order, so the bits do not depend on the batch or the run.
 *   wav        [B][wav_pitch] samples of `wav_dtype` (V100_WAV_F32 | V100_WAV_I16, int16 scaled by 1/32768);
 *              len int32 [B] on the device, clamped to [0, L_in], L_in <= wav_pitch
 *   start, count, off  int32 [n] device arrays: phase p's run is taps[off[p] .. off[p] + count[p]) and covers dense
 *              kernel columns [start[p], start[p] + count[p]), which must lie in [0, 2w + o) (a run outside it is
 *              clipped, never read past);  taps fp32 [n_taps]
 *   out        fp32 [B][out_pitch], L_out <= out_pitch: every sample of [0, L_out) is written; out_len[b] is
 *              torchaudio's output length for len[b] samples, min(ceil(float32(n len / o)), n (len / o + 1), L_out):
 *              the float64 quotient rounded to float32 as torch.ceil(torch.as_tensor(...)) does, which is
 *              ceil(n len / o) until float32 can no longer resolve 1/o (n len / o >= 2^15 at o = 441); samples
 *              [out_len[b], L_out) are 0
 *   out_len    optional int32 [B]
 * Limits (V100_E_UNSUPPORTED beyond them): B <= 65535, n <= 16384 phases, L_in and L_out < 2^31, and the input span
 * of four frames, 3 o + 2w + o, at most 16384 samples.  One CTA per (tile of output frames, utterance); no host
 * synchronisation, CUDA-graph capturable.
 */
int v100_resample(const void* wav, int wav_dtype, const int32_t* len, int B, int64_t wav_pitch, int64_t L_in,
                  const int32_t* start, const int32_t* count, const int32_t* off, const float* taps, int n_taps,
                  int o, int n, int w, float* out, int64_t out_pitch, int64_t L_out, int32_t* out_len, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* V100_H_ */
