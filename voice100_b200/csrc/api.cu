// extern "C" surface of libv100.so (see include/v100.h) + host plumbing.
#include <cstdarg>
#include <cstdio>
#include <mutex>

#include "host.h"

namespace v100 {

static thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int num_sms() {
  static thread_local int dev_cached = -1, sms = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev != dev_cached) {
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    dev_cached = dev;
  }
  return sms > 0 ? sms : 148;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// libv100 does not link libcuda: the one driver call it needs is resolved through the runtime.
static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

static int encode(CUtensorMap* m, CUtensorMapDataType type, const void* base, int rank, const cuuint64_t* dims,
                  const cuuint64_t* strides, const cuuint32_t* box, CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B) {
  EncodeTiledFn fn = encode_fn();
  if (fn == nullptr) return fail(V100_E_DRIVER, "cuTensorMapEncodeTiled is not available from this driver");
  const cuuint32_t ones[3] = {1, 1, 1};
  CUresult r = fn(m, type, rank, const_cast<void*>(base), dims, strides, box, ones,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(V100_E_DRIVER, "cuTensorMapEncodeTiled failed (CUresult %d; rank %d dims %llu,%llu strides %llu)",
                int(r), rank, (unsigned long long)dims[0], (unsigned long long)dims[1],
                (unsigned long long)strides[0]);
  return 0;
}

int make_tmap_2d(CUtensorMap* m, CUtensorMapDataType type, const void* base, int64_t d0, int64_t d1, int64_t stride1_bytes, int box0, int box1) {
  const cuuint64_t dims[2] = {cuuint64_t(d0), cuuint64_t(d1)};
  const cuuint64_t strides[1] = {cuuint64_t(stride1_bytes)};
  const cuuint32_t box[2] = {cuuint32_t(box0), cuuint32_t(box1)};
  return encode(m, type, base, 2, dims, strides, box);
}

int make_tmap_3d(CUtensorMap* m, CUtensorMapDataType type, const void* base, int64_t d0, int64_t d1, int64_t d2, int64_t stride1_bytes,
                 int64_t stride2_bytes, int box0, int box1) {
  const cuuint64_t dims[3] = {cuuint64_t(d0), cuuint64_t(d1), cuuint64_t(d2)};
  const cuuint64_t strides[2] = {cuuint64_t(stride1_bytes), cuuint64_t(stride2_bytes)};
  const cuuint32_t box[3] = {cuuint32_t(box0), cuuint32_t(box1), 1};
  return encode(m, type, base, 3, dims, strides, box);
}

// NCW activations as a (T, C, B) tensor with a box of [box_t steps x 1 channel x box_b utterances]: the rows of one
// channel for several utterances in one TMA instruction, zero-filled outside [0, T) and [0, B).
int make_tmap_rows(CUtensorMap* m, CUtensorMapDataType type, const void* base, int64_t T, int64_t C, int64_t B,
                   int64_t pitch_bytes, int box_t, int box_b, CUtensorMapSwizzle swizzle) {
  const cuuint64_t dims[3] = {cuuint64_t(T), cuuint64_t(C), cuuint64_t(B)};
  const cuuint64_t strides[2] = {cuuint64_t(pitch_bytes), cuuint64_t(C) * cuuint64_t(pitch_bytes)};
  const cuuint32_t box[3] = {cuuint32_t(box_t), 1, cuuint32_t(box_b)};
  return encode(m, type, base, 3, dims, strides, box, swizzle);
}

}  // namespace v100

using namespace v100;
#define STREAM(s) reinterpret_cast<cudaStream_t>(s)

extern "C" {

int v100_abi_version(void) { return V100_ABI_VERSION; }
const char* v100_last_error(void) { return g_err; }

int v100_logmel(const void* wav, int wav_dtype, const int32_t* len, int B, int64_t wav_pitch, int L_max,
                const int32_t* fb_start, const int32_t* fb_count, const int32_t* fb_off, const float* fb_w, int fb_nnz,
                float log_offset, void* out, int T, int64_t out_pitch, int out_mode, int32_t* frames_out,
                void* stream) {
  return logmel(wav, wav_dtype, len, B, wav_pitch, L_max, fb_start, fb_count, fb_off, fb_w, fb_nnz, log_offset, out, T,
                out_pitch, out_mode, frames_out, STREAM(stream));
}

int v100_logmel_generic(const void* wav, int wav_dtype, const int32_t* len, int B, int64_t wav_pitch, int L_max,
                        int n_fft, int win_length, int hop_length, int n_mels, const int32_t* fb_start,
                        const int32_t* fb_count, const int32_t* fb_off, const float* fb_w, float log_offset, void* out,
                        int T, int64_t out_pitch, int out_mode, int32_t* frames_out, void* stream) {
  return logmel_generic(wav, wav_dtype, len, B, wav_pitch, L_max, n_fft, win_length, hop_length, n_mels, fb_start, fb_count,
                        fb_off, fb_w, log_offset, out, T, out_pitch, out_mode, frames_out, STREAM(stream));
}

int v100_ntc_f32_to_ncw16(const float* x, void* y, int B, int T, int C, int64_t y_pitch, int dtype, void* stream) {
  return ntc_f32_to_ncw16(x, y, B, T, C, y_pitch, dtype, STREAM(stream));
}

int v100_ncw_f32_to_16(const float* x, void* y, int64_t y_pitch, int B, int C, int T, int dtype, void* stream) {
  return ncw_f32_to_16(x, y, y_pitch, B, C, T, dtype, STREAM(stream));
}

int v100_ncw_16_to_f32(const void* x, int64_t x_pitch, float* y, int B, int C, int T, int dtype, void* stream) {
  return ncw_16_to_f32(x, x_pitch, y, B, C, T, dtype, STREAM(stream));
}

int v100_conv1x1(const void* x, int64_t x_pitch, const void* W, const float* scale, const float* shift,
                 const void* res, void* y, int64_t y_pitch, int B, int C_in, int C_out, int T, int act, int dtype,
                 void* stream) {
  return conv1x1(x, x_pitch, W, scale, shift, res, y, y_pitch, B, C_in, C_out, T, act, dtype, STREAM(stream));
}

int v100_conv1x1_f32out(const void* x, int64_t x_pitch, const void* W, const float* bias, float* y, int64_t y_pitch,
                        int B, int C_in, int C_out, int T, int dtype, void* stream) {
  return conv1x1_f32out(x, x_pitch, W, bias, y, y_pitch, B, C_in, C_out, T, dtype, STREAM(stream));
}

int v100_dwconv1d(const void* x, int64_t x_pitch, const void* w, const float* scale, const float* shift, void* y,
                  int64_t y_pitch, int B, int C, int T_in, int k, int stride, int act, int dtype, void* stream) {
  return dwconv1d(x, x_pitch, w, scale, shift, y, y_pitch, B, C, T_in, k, stride, act, dtype, 0, STREAM(stream));
}

// Same contract as v100_dwconv1d but always the plain CUDA-core kernel (any stride); exported so the tests can
// cross-check the tensor-core kernel against it on the GPU.
int v100_dwconv1d_simt(const void* x, int64_t x_pitch, const void* w, const float* scale, const float* shift,
                       void* y, int64_t y_pitch, int B, int C, int T_in, int k, int stride, int act, int dtype,
                       void* stream) {
  return dwconv1d(x, x_pitch, w, scale, shift, y, y_pitch, B, C, T_in, k, stride, act, dtype, 1, STREAM(stream));
}

int v100_convtranspose1d_k5s2(const void* x, int64_t x_pitch, const void* Wp, const float* bias, void* workspace,
                              void* y, int64_t y_pitch, int B, int C_in, int C_out, int T, int dtype, void* stream) {
  return convtranspose1d_k5s2(x, x_pitch, Wp, bias, workspace, y, y_pitch, B, C_in, C_out, T, dtype, STREAM(stream));
}

int v100_embedding_ncw16(const int64_t* ids, const void* table, void* y, int64_t y_pitch, int B, int T, int V, int C,
                         int32_t* status, void* stream) {
  return embedding_ncw16(ids, table, y, y_pitch, B, T, V, C, status, STREAM(stream));
}

int v100_ctc_finalize(const float* y_ncw, int64_t y_pitch, float* logits_or_null, int64_t* tokens, int B, int V,
                      int T, const int32_t* audio_len, int32_t* out_len, void* stream) {
  return ctc_finalize(y_ncw, y_pitch, logits_or_null, tokens, B, V, T, audio_len, out_len, STREAM(stream));
}

int v100_ctc_collapse(const int64_t* tokens, const int64_t* valid_len, int64_t* out, int32_t* out_len, int B, int T,
                      int blank, void* stream) {
  return ctc_collapse(tokens, valid_len, out, out_len, B, T, blank, STREAM(stream));
}

int v100_ctc_best_path(const float* logprob, const int32_t* logit_len, const int64_t* text, const int32_t* text_len,
                       uint8_t* workspace, float* score, int32_t* path, int64_t* path_labels, int B, int T, int V,
                       int L, int normalize, void* stream) {
  return ctc_best_path(logprob, logit_len, text, text_len, workspace, score, path, path_labels, B, T, V, L, normalize,
                       STREAM(stream));
}

int v100_world_finalize(const float* y_ncw, int64_t y_pitch, const float* mean, const float* std, float* hasf0,
                        float* f0, float* logspc, float* hascodeap, float* codeap, int B, int T, int logspc_size,
                        int codeap_size, int layout, int unnormalize, void* stream) {
  return world_finalize(y_ncw, y_pitch, mean, std, hasf0, f0, logspc, hascodeap, codeap, B, T, logspc_size,
                        codeap_size, layout, unnormalize, STREAM(stream));
}

int v100_ncw_f32_to_ntc(const float* y_ncw, int64_t y_pitch, float* out, int B, int C, int T, void* stream) {
  return ncw_f32_to_ntc(y_ncw, y_pitch, out, B, C, T, STREAM(stream));
}

int v100_maskaudio(const float* audio, const int32_t* audio_len, float* out, int B, int T, int C, float log_offset,
                   void* stream) {
  return maskaudio(audio, audio_len, out, B, T, C, log_offset, STREAM(stream));
}

int v100_conv1d(const void* x, int64_t x_pitch, const void* Wp, const float* bias, void* workspace, void* y,
                int64_t y_pitch, int B, int C_in, int C_out, int T_in, int k, int stride, int pad, int dtype,
                void* stream) {
  return conv1d(x, x_pitch, Wp, bias, workspace, y, y_pitch, B, C_in, C_out, T_in, k, stride, pad, dtype,
                STREAM(stream));
}

int v100_conv1d_tm(const void* x, const void* Wp, const float* bias, void* y, int C_in, int C_out, int T, int Bp,
                   int k, int dtype, void* stream) {
  return conv1d_tm(x, Wp, bias, y, C_in, C_out, T, Bp, k, dtype, STREAM(stream));
}

int v100_layernorm_gelu(const void* x, int64_t x_pitch, const float* gamma, const float* beta, float eps, void* y,
                        int64_t y_pitch, int B, int C, int T, int dtype, void* stream) {
  return layernorm_gelu(x, x_pitch, gamma, beta, eps, y, y_pitch, B, C, T, dtype, STREAM(stream));
}

int v100_ncw_to_tm(const void* x, int64_t x_pitch, void* y, int B, int C, int T, int Bp, void* stream) {
  return ncw_to_tm(x, x_pitch, y, B, C, T, Bp, STREAM(stream));
}

int v100_tm_to_ncw(const void* x, void* y, int64_t y_pitch, int B, int C, int T, int Bp, void* stream) {
  return tm_to_ncw(x, y, y_pitch, B, C, T, Bp, STREAM(stream));
}

int64_t v100_lstm_workspace_bytes(int B, int H) { return static_cast<int64_t>(lstm_workspace_bytes(B, H)); }

int v100_lstm_layer(const void* gx, const void* w_hh, const int32_t* lengths, void* y, void* workspace, int B,
                    int Bp, int T, int H, int dtype, void* stream) {
  return lstm_layer(gx, w_hh, lengths, y, workspace, B, Bp, T, H, dtype, STREAM(stream));
}

int v100_tts_align(const float* durations, int64_t stride_b, int64_t stride_l, int64_t stride_c, int log1p_input,
                   float* durations_out, const int64_t* text, int64_t text_stride, const int32_t* text_len, int B,
                   int L, int rule, int head, int tail, int64_t* aligntext, int T_cap, int32_t* aligntext_len,
                   int32_t* status, int32_t* filled_len, int32_t* frame_len, void* stream) {
  return tts_align(durations, stride_b, stride_l, stride_c, log1p_input, durations_out, text, text_stride, text_len, B,
                   L, rule, head, tail, aligntext, T_cap, aligntext_len, status, filled_len, frame_len,
                   STREAM(stream));
}

int v100_world_noise(double* out, int64_t n, void* stream) { return world_noise(out, n, STREAM(stream)); }

int64_t v100_world_workspace_bytes(int B, int64_t y_len_max) { return world_workspace_bytes(B, y_len_max); }

int v100_world_timebase(const float* f0, int64_t f0_sb, int64_t f0_st, const float* logspc, int64_t sp_sb,
                        int64_t sp_st, int64_t sp_sk, const float* codeap, int64_t ap_sb, int64_t ap_st,
                        const int32_t* frame_len, int B, int T, void* workspace, int32_t* wav_len, int32_t* status,
                        void* stream) {
  return world_timebase(f0, f0_sb, f0_st, logspc, sp_sb, sp_st, sp_sk, codeap, ap_sb, ap_st, frame_len, B, T,
                        workspace, wav_len, status, STREAM(stream));
}

int v100_world_synthesize(const float* f0, int64_t f0_sb, int64_t f0_st, const float* logspc, int64_t sp_sb,
                          int64_t sp_st, int64_t sp_sk, const float* codeap, int64_t ap_sb, int64_t ap_st,
                          const int32_t* frame_len, int B, int T, const double* noise, int64_t noise_len,
                          void* workspace, float* wav, int64_t wav_pitch, int32_t* wav_len, int32_t* status,
                          void* stream) {
  return world_synthesize(f0, f0_sb, f0_st, logspc, sp_sb, sp_st, sp_sk, codeap, ap_sb, ap_st, frame_len, B, T, noise,
                          noise_len, workspace, wav, wav_pitch, wav_len, status, STREAM(stream));
}

int64_t v100_world_analysis_workspace_bytes(int B, int64_t L_max) { return world_analysis_workspace_bytes(B, L_max); }

int v100_world_analyze(const void* wav, int wav_dtype, int64_t wav_pitch, const int32_t* len, int B, int64_t L_max,
                       const double* taps, const double* noise, int64_t noise_len, void* workspace, int T, float* f0,
                       float* logspc, float* codeap, int32_t* frame_len, int32_t* status, void* stream) {
  return world_analyze(wav, wav_dtype, wav_pitch, len, B, L_max, taps, noise, noise_len, workspace, T, f0, logspc,
                       codeap, frame_len, status, STREAM(stream));
}

int v100_resample(const void* wav, int wav_dtype, const int32_t* len, int B, int64_t wav_pitch, int64_t L_in,
                  const int32_t* start, const int32_t* count, const int32_t* off, const float* taps, int n_taps,
                  int o, int n, int w, float* out, int64_t out_pitch, int64_t L_out, int32_t* out_len, void* stream) {
  return resample(wav, wav_dtype, len, B, wav_pitch, L_in, start, count, off, taps, n_taps, o, n, w, out, out_pitch,
                  L_out, out_len, STREAM(stream));
}

}  // extern "C"
