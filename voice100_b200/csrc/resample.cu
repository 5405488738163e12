// Polyphase sinc resampling of a padded batch of waveforms (v100_resample in include/v100.h).
//
// Replaces torchaudio.functional.resample, which MelSpectrogramAudioTransform.forward calls between load and the mel
// spectrogram when a file is not at 16 kHz (voice100/data_modules.py:288-289).  torchaudio evaluates a dense
// conv1d with a [n, 1, 2w + o] kernel at stride o (_get_sinc_resample_kernel / _apply_sinc_resample_kernel, rates
// reduced by their gcd to o -> n); most of that kernel is zero.  Here every phase p keeps only its contiguous run of
// taps (the host packs them: start[p], count[p], off[p] into taps[]), and
//   y[b, j n + p] = sum_i taps[off[p] + i] * x[b, j o + start[p] + i - w],   x = 0 outside [0, len[b]).
//  - output-stationary: one CTA per (tile of JT frames = JT n outputs, utterance); the packed table is staged in shared
//    memory, and a CTA walks several tiles of its row so that the table is loaded once for all of them.
//  - the input span of a tile, (JT - 1) o + 2w + o samples, is staged in shared memory as fp32 with zeros outside
//    [0, len[b]), so padding content is never read into a result.
//  - a thread owns one phase and R frames of the tile (strided by JT / R, so that for n = 1 consecutive threads
//    write consecutive samples); each output is its own fixed-order fmaf chain over the phase's taps, so results are
//    bit-identical from run to run and do not depend on the rest of the batch.  One tap load serves R outputs.
//  - all sample indices are int64 (j o overflows int32 at 15 s x 441).
#include "common.cuh"
#include "host.h"

namespace v100 {

namespace {

constexpr int kResThreads = 256;
constexpr int kResR = 4;                  // frames per thread item: the taps of a phase are loaded once for R outputs
constexpr int kResMaxSpan = 16384;        // staged input samples per tile (64 KB)
constexpr int kResMaxSmemTaps = 16384;    // packed tables up to this size are staged in shared memory (64 KB)
constexpr int kResMaxPhases = 16384;      // n after the gcd reduction
constexpr int kResTargetOutputs = 1024;   // outputs per tile, before rounding to whole thread rounds

// torchaudio's output length: _apply_sinc_resample_kernel slices the conv1d output, n (floor(len / o) + 1) samples,
// at torch.ceil(torch.as_tensor(n * len / o)): a float64 quotient (exact operands, n len < 2^53) rounded to a float32
// tensor, then ceil.  That is ceil(n len / o) while the float32 rounding is finer than 1/o (about n len / o < 2^15 at
// o = 441) and can be a sample shorter or longer beyond; both ops round to nearest here as on the host.
__device__ __forceinline__ long long out_length(int len, int o, int n, int L_out) {
  const long long nl = static_cast<long long>(n) * len;
  long long ol = static_cast<long long>(ceilf(__double2float_rn(__ddiv_rn(static_cast<double>(nl), static_cast<double>(o)))));
  const long long conv = static_cast<long long>(n) * (len / o + 1);
  ol = ol < conv ? ol : conv;
  return ol < L_out ? ol : L_out;
}

template <bool I16, bool TAPS_SMEM>
__global__ void __launch_bounds__(kResThreads)
resample_kernel(const void* __restrict__ x, long long x_pitch, const int32_t* __restrict__ len, int L_in,
                const int32_t* __restrict__ start, const int32_t* __restrict__ count, const int32_t* __restrict__ off,
                const float* __restrict__ taps, int n_taps, int o, int n, int w, int JT, long long tiles,
                int tiles_per_cta, float* __restrict__ y, long long y_pitch, int L_out, int32_t* __restrict__ out_len) {
  extern __shared__ float smem[];
  const int K = 2 * w + o;                               // the dense kernel's width: every packed run lies in [0, K)
  const int span = (JT - 1) * o + K;
  float* xs = smem;
  const float* tp = taps;
  const int b = blockIdx.y;
  int lb = __ldg(len + b);
  lb = lb < 0 ? 0 : (lb > L_in ? L_in : lb);
  const long long ol = out_length(lb, o, n, L_out);
  if (out_len != nullptr && blockIdx.x == 0 && threadIdx.x == 0) out_len[b] = static_cast<int32_t>(ol);
  if (TAPS_SMEM) {
    float* ts = smem + span;
    for (int i = threadIdx.x; i < n_taps; i += kResThreads) ts[i] = __ldg(taps + i);
    tp = ts;                                               // made visible by the first tile's __syncthreads
  }
  const int G = JT / kResR;
  const int items = n * G;
  float* yb = y + b * y_pitch;
  const float* xf = static_cast<const float*>(x) + b * x_pitch;
  const int16_t* xi = static_cast<const int16_t*>(x) + b * x_pitch;

  for (int k = 0; k < tiles_per_cta; ++k) {
    const long long tile = static_cast<long long>(blockIdx.x) * tiles_per_cta + k;
    if (tile >= tiles) break;
    const long long j0 = tile * JT;
    const long long q0 = j0 * n;
    if (q0 >= ol) {                                        // the whole tile lies past out_len: zeros, no staging
      const long long q1 = min(q0 + static_cast<long long>(JT) * n, static_cast<long long>(L_out));
      for (long long q = q0 + threadIdx.x; q < q1; q += kResThreads) yb[q] = 0.0f;
      continue;
    }
    const long long base = j0 * o - w;                     // sample index of xs[0]
    __syncthreads();                                       // the previous tile is done reading xs
    for (int i = threadIdx.x; i < span; i += kResThreads) {
      const long long s = base + i;
      float v = 0.0f;
      if (s >= 0 && s < lb) v = I16 ? static_cast<float>(__ldg(xi + s)) * (1.0f / 32768.0f) : __ldg(xf + s);
      xs[i] = v;
    }
    __syncthreads();
    for (int it = threadIdx.x; it < items; it += kResThreads) {
      const int p = it % n, g = it / n;
      int s0 = __ldg(start + p), c = __ldg(count + p);
      const int o0 = __ldg(off + p);
      // a malformed table (a run outside [0, K) or past n_taps) stays inside the staged arrays
      s0 = s0 < 0 ? 0 : (s0 > K ? K : s0);
      c = c < 0 ? 0 : (c > K - s0 ? K - s0 : c);
      c = (o0 < 0 || o0 > n_taps) ? 0 : (c > n_taps - o0 ? n_taps - o0 : c);
      const float* t = tp + o0;
      const float* xr = xs + g * o + s0;
      float acc[kResR];
#pragma unroll
      for (int r = 0; r < kResR; ++r) acc[r] = 0.0f;
      for (int i = 0; i < c; ++i) {
        const float tv = TAPS_SMEM ? t[i] : __ldg(t + i);
#pragma unroll
        for (int r = 0; r < kResR; ++r) acc[r] = fmaf(tv, xr[r * G * o + i], acc[r]);
      }
#pragma unroll
      for (int r = 0; r < kResR; ++r) {
        const long long q = (j0 + g + r * G) * n + p;
        if (q < L_out) yb[q] = q < ol ? acc[r] : 0.0f;
      }
    }
  }
}

template <bool I16, bool TAPS_SMEM>
int launch(const void* x, long long x_pitch, const int32_t* len, int L_in, const int32_t* start, const int32_t* count,
           const int32_t* off, const float* taps, int n_taps, int o, int n, int w, int JT, long long tiles, int tpc,
           int B, float* y, long long y_pitch, int L_out, int32_t* out_len, size_t smem, cudaStream_t stream) {
  auto kern = resample_kernel<I16, TAPS_SMEM>;
  if (smem > 48 * 1024) V100_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  // at least one CTA per row, which writes out_len even when the rows are empty (L_out = 0)
  const dim3 grid(static_cast<unsigned>(tiles > 0 ? (tiles + tpc - 1) / tpc : 1), static_cast<unsigned>(B));
  kern<<<grid, dim3(kResThreads), smem, stream>>>(x, x_pitch, len, L_in, start, count, off, taps, n_taps, o, n, w, JT,
                                                  tiles, tpc, y, y_pitch, L_out, out_len);
  V100_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace

int resample(const void* wav, int wav_dtype, const int32_t* len, int B, int64_t wav_pitch, int64_t L_in,
             const int32_t* start, const int32_t* count, const int32_t* off, const float* taps, int n_taps, int o,
             int n, int w, float* out, int64_t out_pitch, int64_t L_out, int32_t* out_len, cudaStream_t stream) {
  if (wav == nullptr || len == nullptr || start == nullptr || count == nullptr || off == nullptr || out == nullptr ||
      (taps == nullptr && n_taps > 0))
    return fail(V100_E_INVALID, "resample: null pointer");
  if (wav_dtype != V100_WAV_F32 && wav_dtype != V100_WAV_I16)
    return fail(V100_E_INVALID, "resample: wav_dtype must be V100_WAV_F32 or V100_WAV_I16 (got %d)", wav_dtype);
  if (B <= 0 || o <= 0 || n <= 0 || w < 0 || n_taps < 0 || L_in < 0 || L_out < 0)
    return fail(V100_E_INVALID, "resample: need B, o, n > 0 and w, n_taps, L_in, L_out >= 0");
  if (wav_pitch < L_in || out_pitch < L_out)
    return fail(V100_E_INVALID, "resample: row pitches (%lld, %lld) below the row lengths (%lld, %lld)",
                (long long)wav_pitch, (long long)out_pitch, (long long)L_in, (long long)L_out);
  if (L_in > INT32_MAX || L_out > INT32_MAX)
    return fail(V100_E_UNSUPPORTED, "resample: rows of 2^31 samples or more (L_in %lld, L_out %lld)",
                (long long)L_in, (long long)L_out);
  if (B > 65535) return fail(V100_E_UNSUPPORTED, "resample: B = %d > 65535 utterances", B);
  if (n > kResMaxPhases) return fail(V100_E_UNSUPPORTED, "resample: %d phases > %d", n, kResMaxPhases);
  const long long K = 2LL * w + o;
  if ((kResR - 1) * static_cast<long long>(o) + K > kResMaxSpan)
    return fail(V100_E_UNSUPPORTED, "resample: o = %d, w = %d: the input span of %d frames exceeds %d samples", o, w,
                kResR, kResMaxSpan);

  // frames per tile: JT = G R, G the smallest count with at least kResTargetOutputs outputs whose items fill at
  // least 7/8 of their last thread round, within the span limit
  int G = 1;
  for (int g = 1; (kResR * g - 1) * static_cast<long long>(o) + K <= kResMaxSpan; ++g) {
    G = g;
    const long long items = static_cast<long long>(n) * g;
    const long long rounds = (items + kResThreads - 1) / kResThreads;
    if (items * kResR >= kResTargetOutputs && items * 8 >= rounds * kResThreads * 7) break;
    if (items >= 4 * kResThreads) break;
  }
  const int JT = G * kResR;
  const long long frames = (L_out + n - 1) / n;
  const long long tiles = (frames + JT - 1) / JT;
  const bool tsm = n_taps <= kResMaxSmemTaps;
  // with the table in shared memory a CTA walks several tiles of its row (the table is staged once per CTA), as many
  // as keeps about 8 CTAs per SM in the grid
  int tpc = 1;
  if (tsm) {
    const long long want = static_cast<long long>(num_sms()) * 8;
    const long long per_row = (want + B - 1) / B;
    tpc = static_cast<int>(tiles / (per_row > 0 ? per_row : 1));
    tpc = tpc < 1 ? 1 : (tpc > 16 ? 16 : tpc);
  }
  if ((tiles + tpc - 1) / tpc > INT32_MAX) return fail(V100_E_UNSUPPORTED, "resample: too many tiles");
  const size_t smem = sizeof(float) * (static_cast<size_t>((JT - 1) * static_cast<long long>(o) + K) + (tsm ? n_taps : 0));
  const bool i16 = wav_dtype == V100_WAV_I16;
#define V100_RES_LAUNCH(A, T)                                                                                        \
  return launch<A, T>(wav, wav_pitch, len, int(L_in), start, count, off, taps, n_taps, o, n, w, JT, tiles, tpc, B, \
                      out, out_pitch, int(L_out), out_len, smem, stream)
  if (i16) {
    if (tsm) V100_RES_LAUNCH(true, true);
    V100_RES_LAUNCH(true, false);
  }
  if (tsm) V100_RES_LAUNCH(false, true);
  V100_RES_LAUNCH(false, false);
#undef V100_RES_LAUNCH
}

}  // namespace v100
