// Host-side plumbing shared by the libv100 translation units: error reporting, device queries,
// TMA tensor-map construction, and the internal (C++) signatures behind the C ABI in include/v100.h.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/v100.h"

namespace v100 {

// Records a formatted message for v100_last_error() and returns `code`.
int fail(int code, const char* fmt, ...);
int num_sms();

#define V100_CUDA(expr)                                                                   \
  do {                                                                                    \
    cudaError_t e__ = (expr);                                                             \
    if (e__ != cudaSuccess)                                                               \
      return ::v100::fail(static_cast<int>(e__), "%s -> %s", #expr, cudaGetErrorString(e__)); \
  } while (0)

// 16-bit tensor maps, 128-byte swizzle, zero fill out of bounds.  Dimensions innermost first.
int make_tmap_2d(CUtensorMap* m, CUtensorMapDataType type, const void* base, int64_t d0, int64_t d1, int64_t stride1_bytes, int box0, int box1);
int make_tmap_3d(CUtensorMap* m, CUtensorMapDataType type, const void* base, int64_t d0, int64_t d1, int64_t d2, int64_t stride1_bytes,
                 int64_t stride2_bytes, int box0, int box1);

int make_tmap_rows(CUtensorMap* m, CUtensorMapDataType type, const void* base, int64_t T, int64_t C, int64_t B,
                   int64_t pitch_bytes, int box_t, int box_b, CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_NONE);

int conv1x1(const void* x, int64_t x_pitch, const void* W, const float* scale, const float* shift, const void* res,
            void* y, int64_t y_pitch, int B, int C_in, int C_out, int T, int act, int dtype, cudaStream_t stream);
int conv1x1_f32out(const void* x, int64_t x_pitch, const void* W, const float* bias, float* y, int64_t y_pitch,
                   int B, int C_in, int C_out, int T, int dtype, cudaStream_t stream);
int convtranspose1d_k5s2(const void* x, int64_t x_pitch, const void* Wp, const float* bias, void* workspace, void* y,
                         int64_t y_pitch, int B, int C_in, int C_out, int T, int dtype, cudaStream_t stream);
int dwconv1d(const void* x, int64_t x_pitch, const void* w, const float* scale, const float* shift, void* y,
             int64_t y_pitch, int B, int C, int T_in, int k, int stride, int act, int dtype, int force_simt,
             cudaStream_t stream);
int logmel(const void* wav, int wav_dtype, const int32_t* len, int B, int64_t wav_pitch, int L_max,
           const int32_t* fb_start, const int32_t* fb_count, const int32_t* fb_off, const float* fb_w, int fb_nnz,
           float log_offset, void* out, int T, int64_t out_pitch, int out_mode, int32_t* frames_out,
           cudaStream_t stream);
int logmel_generic(const void* wav, int wav_dtype, const int32_t* len, int B, int64_t wav_pitch, int L_max, int n_fft,
                   int win_length, int hop_length, int n_mels, const int32_t* fb_start, const int32_t* fb_count,
                   const int32_t* fb_off, const float* fb_w, float log_offset, void* out, int T, int64_t out_pitch,
                   int out_mode, int32_t* frames_out, cudaStream_t stream);
int ntc_f32_to_ncw16(const float* x, void* y, int B, int T, int C, int64_t y_pitch, int dtype, cudaStream_t stream);
int ncw_f32_to_16(const float* x, void* y, int64_t y_pitch, int B, int C, int T, int dtype, cudaStream_t stream);
int ncw_16_to_f32(const void* x, int64_t x_pitch, float* y, int B, int C, int T, int dtype, cudaStream_t stream);
int embedding_ncw16(const int64_t* ids, const void* table, void* y, int64_t y_pitch, int B, int T, int V, int C,
                    int32_t* status, cudaStream_t stream);
int ctc_finalize(const float* y_ncw, int64_t y_pitch, float* logits, int64_t* tokens, int B, int V, int T,
                 const int32_t* audio_len, int32_t* out_len, cudaStream_t stream);
int ctc_collapse(const int64_t* tokens, const int64_t* valid_len, int64_t* out, int32_t* out_len, int B, int T,
                 int blank, cudaStream_t stream);
int ctc_best_path(const float* logprob, const int32_t* logit_len, const int64_t* text, const int32_t* text_len,
                  uint8_t* workspace, float* score, int32_t* path, int64_t* path_labels, int B, int T, int V, int L,
                  int normalize, cudaStream_t stream);
int world_finalize(const float* y_ncw, int64_t y_pitch, const float* mean, const float* std, float* hasf0, float* f0,
                   float* logspc, float* hascodeap, float* codeap, int B, int T, int logspc_size, int codeap_size,
                   int layout, int unnormalize, cudaStream_t stream);
int ncw_f32_to_ntc(const float* y_ncw, int64_t y_pitch, float* out, int B, int C, int T, cudaStream_t stream);
int maskaudio(const float* audio, const int32_t* audio_len, float* out, int B, int T, int C, float log_offset,
              cudaStream_t stream);

// v2 models (seq.cu)
int conv1d(const void* x, int64_t x_pitch, const void* Wp, const float* bias, void* workspace, void* y,
           int64_t y_pitch, int B, int C_in, int C_out, int T_in, int k, int stride, int pad, int dtype,
           cudaStream_t stream);
int conv1d_tm(const void* x, const void* Wp, const float* bias, void* y, int C_in, int C_out, int T, int Bp, int k,
              int dtype, cudaStream_t stream);
int layernorm_gelu(const void* x, int64_t x_pitch, const float* gamma, const float* beta, float eps, void* y,
                   int64_t y_pitch, int B, int C, int T, int dtype, cudaStream_t stream);
int ncw_to_tm(const void* x, int64_t x_pitch, void* y, int B, int C, int T, int Bp, cudaStream_t stream);
int tm_to_ncw(const void* x, void* y, int64_t y_pitch, int B, int C, int T, int Bp, cudaStream_t stream);
size_t lstm_workspace_bytes(int B, int H);
int lstm_layer(const void* gx, const void* w_hh, const int32_t* lengths, void* y, void* workspace, int B, int Bp,
               int T, int H, int dtype, cudaStream_t stream);

// TTS text alignment (tts_align.cu)
int tts_align(const float* durations, int64_t stride_b, int64_t stride_l, int64_t stride_c, int log1p_input,
              float* durations_out, const int64_t* text, int64_t text_stride, const int32_t* text_len, int B, int L,
              int rule, int head, int tail, int64_t* aligntext, int T_cap, int32_t* aligntext_len, int32_t* status,
              int32_t* filled_len, int32_t* frame_len, cudaStream_t stream);

// WORLD synthesis (world.cu)
int64_t world_workspace_bytes(int B, int64_t y_len_max);
int world_noise(double* out, int64_t n, cudaStream_t stream);
int world_timebase(const float* f0, int64_t f0_sb, int64_t f0_st, const float* logspc, int64_t sp_sb, int64_t sp_st,
                   int64_t sp_sk, const float* codeap, int64_t ap_sb, int64_t ap_st, const int32_t* frame_len, int B,
                   int T, void* workspace, int32_t* wav_len, int32_t* status, cudaStream_t stream);
int world_synthesize(const float* f0, int64_t f0_sb, int64_t f0_st, const float* logspc, int64_t sp_sb,
                     int64_t sp_st, int64_t sp_sk, const float* codeap, int64_t ap_sb, int64_t ap_st,
                     const int32_t* frame_len, int B, int T, const double* noise, int64_t noise_len, void* workspace,
                     float* wav, int64_t wav_pitch, int32_t* wav_len, int32_t* status, cudaStream_t stream);

// WORLD analysis (world_analysis.cu)
int64_t world_analysis_workspace_bytes(int B, int64_t L_max);
int64_t world_analysis_noise_values(int64_t L_max);
int world_analyze(const void* wav, int wav_dtype, int64_t wav_pitch, const int32_t* len, int B, int64_t L_max,
                  const double* taps, const double* noise, int64_t noise_len, void* workspace, int T, float* f0,
                  float* logspc, float* codeap, int32_t* frame_len, int32_t* status, cudaStream_t stream);

// Resampling (resample.cu)
int resample(const void* wav, int wav_dtype, const int32_t* len, int B, int64_t wav_pitch, int64_t L_in,
             const int32_t* start, const int32_t* count, const int32_t* off, const float* taps, int n_taps, int o,
             int n, int w, float* out, int64_t out_pitch, int64_t L_out, int32_t* out_len, cudaStream_t stream);

}  // namespace v100
