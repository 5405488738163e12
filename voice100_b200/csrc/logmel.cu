// Fused log-mel front end: framing (reflect padding at the clip's own ends) + periodic Hann(400) in a
// 512 frame + 512-point real FFT + |.|^2 + sparse 64-filter HTK mel bank + log(. + offset), one kernel.
//
// Replaces reflect-pad + unfold + window + cuFFT R2C + abs/pow + sgemm + add/log + transpose
// (>= 6 library launches, and a 257-bin complex spectrum written to and read back from HBM).
//
// Round-2 structure (the round-1 kernel spent 6,144 CTA prologues on sincospif tables, 17 M bank-conflict
// wavefronts in the mel stage and ran at 24 % warp occupancy):
//   * persistent CTAs walk [clip, 32-frame] tiles; the window, the W256^(q k1) twiddle table and the filter
//     descriptors are built once per CTA;
//   * FFT phase: sixteen threads per frame (logmel_core.h), two 16-point FFTs in registers around one 16 x 16
//     transpose through a stride-17 shared buffer; the conjugate partner Z[256-k] of the real-FFT unpacking is
//     always an upper-half register of lane (16-q)&15, so it comes by warp shuffle, not through shared memory,
//     and one complex multiply serves both bins of a conjugate pair;
//   * the 257 power bins of the tile's 32 frames go to P[bin][frame] (stride 33, conflict-free for the two
//     half-warps of a warp, whose frames are 16 apart);
//   * mel phase: LANE = FRAME.  A warp applies one filter at a time to 32 frames: P[(s0+tap)*33 + lane] is one
//     conflict-free wavefront per tap and the weight is a warp-uniform broadcast;
//   * input is fp32 or int16 PCM (scaled by 1/32768 in the kernel = what torchaudio.load produces for 16-bit WAV,
//     so the two entry forms are bit-identical on such data) -- the int16 form halves the H2D stream.
// The kernel is bound by instruction issue and shared-memory wavefronts, not by HBM (64 KB in + 12.8 KB out per
// audio-second); see DESIGN.md.
#include "common.cuh"
#include "host.h"
#include "logmel_core.h"

namespace v100 {

constexpr int kNMels = 64;
constexpr int kNFft = 512, kWin = 400, kHop = 160, kWinLeft = (kNFft - kWin) / 2;  // data_modules.py:266-269
constexpr int kMelTile = 32;         // frames per tile
constexpr int kPStride = 33;
constexpr int kMelMaxNnz = 1024;     // accepted filter-bank size (the HTK bank at 512/16 kHz/64 has 500 weights)
constexpr int kMelWarps = 16;        // warps per CTA
constexpr int kMelCtasPerSm = 2;     // resident CTAs per SM: the launch bounds and the persistent grid

struct MelCfg {
  static constexpr int kHalfWarps = 2 * kMelWarps;
  static constexpr int kIters = kMelTile / kHalfWarps;          // FFT passes per tile
  static constexpr int kWinBytes = 256 * 8;                     // float2 window of samples (2n, 2n+1)
  static constexpr int kTwBytes = 16 * 16 * 8;                  // W256^(q k1) as [k1][q]
  static constexpr int kFbBytes = 3 * kNMels * 4 + (kMelMaxNnz + 4 * kNMels) * 4;   // start, count, offset; weights, each
                                                                // filter's run padded to a multiple of four
  static constexpr int kEBytes = kHalfWarps * 16 * 17 * 8;      // exchange buffers (reused as the NTC output tile)
  static constexpr int kPBytes = (257 * kPStride * 4 + 15) & ~15;
  static constexpr int kSmemBytes = kWinBytes + kTwBytes + kFbBytes + kEBytes + kPBytes;
  static_assert(kIters >= 1 && kIters * kHalfWarps == kMelTile, "a tile is a whole number of passes");
  static_assert(kEBytes >= kMelTile * (kNMels + 1) * 4, "the NTC output tile aliases the exchange buffers");
};

struct MelParams {
  const void* wav;
  const int32_t* len;
  long long wav_pitch;
  int L_max;
  const int32_t *fb_start, *fb_count, *fb_off;
  const float* fb_w;
  float log_offset;
  void* out;
  int T;
  long long out_pitch;
  int out_mode;
  int32_t* frames_out;
  int tiles_per_clip, total_tiles;
};

template <bool I16>
__global__ void __launch_bounds__(kMelWarps * 32, kMelCtasPerSm)
logmel_kernel(const MelParams p) {
  extern __shared__ __align__(16) uint8_t mel_smem[];
  float2* win2 = reinterpret_cast<float2*>(mel_smem);                                      // [256]
  cpx* twt = reinterpret_cast<cpx*>(mel_smem + MelCfg::kWinBytes);                          // [16 k1][16 q]
  int* fbs = reinterpret_cast<int*>(mel_smem + MelCfg::kWinBytes + MelCfg::kTwBytes);       // [3][64]
  cpx* exch = reinterpret_cast<cpx*>(mel_smem + MelCfg::kWinBytes + MelCfg::kTwBytes + MelCfg::kFbBytes);
  float* P = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(exch) + MelCfg::kEBytes);  // [257][33]
  float* otile = reinterpret_cast<float*>(exch);                                           // [32][65] (NTC mode)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float in_scale = I16 ? (1.0f / 32768.0f) : 1.0f;

  // ---- once per CTA: window, twiddles, filter descriptors ----
  for (int n = threadIdx.x; n < 256; n += kMelWarps * 32) {   // periodic Hann(400) centred in the 512 frame
    float w2[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int m = 2 * n + h - kWinLeft;
      w2[h] = (m >= 0 && m < kWin) ? (0.5f - 0.5f * cospif(float(2 * m) / float(kWin))) * in_scale : 0.0f;
    }
    win2[n] = make_float2(w2[0], w2[1]);
  }
  for (int i = threadIdx.x; i < 256; i += kMelWarps * 32) {   // twt[k1][q] = exp(-2 pi i q k1 / 256)
    const int k1 = i >> 4, qq = i & 15;
    float sn, cs;
    sincospif(-float((2 * qq * k1) & 511) / 256.0f, &sn, &cs);
    twt[i] = cpx{cs, sn};
  }
  float* fbw = reinterpret_cast<float*>(fbs + 3 * kNMels);     // filter m's weights at fbw[fbs[2*64 + m] ...], 16-byte aligned,
  if (threadIdx.x < 32) {                                      // zero-padded to a multiple of four taps
    int run = 0;                                               // (one warp: exclusive scan of the padded counts)
    for (int m0 = 0; m0 < kNMels; m0 += 32) {
      const int m = m0 + lane;
      const int cnt = __ldg(p.fb_count + m), pad = (cnt + 3) & ~3;
      int incl = pad;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += up;
      }
      const int off = run + incl - pad;
      fbs[m] = __ldg(p.fb_start + m);
      fbs[kNMels + m] = pad;
      fbs[2 * kNMels + m] = off;
      const float* src = p.fb_w + __ldg(p.fb_off + m);
      for (int i = 0; i < pad; ++i) fbw[off + i] = i < cnt ? __ldg(src + i) : 0.0f;
      run += __shfl_sync(0xffffffffu, incl, 31);
    }
  }
  const int q = lane & 15, half = lane >> 4;
  cpx wq;                                              // exp(-2 pi i q / 512)
  {
    float sn, cs;
    sincospif(-float(q) / 256.0f, &sn, &cs);
    wq = cpx{cs, sn};
  }
  cpx* E = exch + (warp * 2 + half) * (16 * 17);
  const int partner_lane = (lane & 16) | ((16 - q) & 15);
  const float blank = p.out_mode == V100_MEL_POWER_F32_NCW ? 0.0f : logf(p.log_offset);
  __syncthreads();

  for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
    const int b = tile / p.tiles_per_clip;
    const int f0 = (tile - b * p.tiles_per_clip) * kMelTile;
    const int L = min(max(__ldg(p.len + b), 0), p.L_max);
    const int n_frames = L > 0 ? 1 + L / kHop : 0;     // frames with data; the rest of the row is BLANK_AUDIO
    if (p.frames_out != nullptr && f0 == 0 && threadIdx.x == 0) p.frames_out[b] = 1 + L / kHop;
    const float* xf = static_cast<const float*>(p.wav) + static_cast<long long>(b) * p.wav_pitch;
    const short* xi = static_cast<const short*>(p.wav) + static_cast<long long>(b) * p.wav_pitch;
    const bool vec_ok = I16 ? ((reinterpret_cast<uintptr_t>(xi) & 3) == 0) : ((reinterpret_cast<uintptr_t>(xf) & 7) == 0);

    // ---------------- FFT phase: one frame per half-warp and pass ----------------
#pragma unroll 1
    for (int it = 0; it < MelCfg::kIters; ++it) {
      const int fl = warp + kMelWarps * it + 16 * half;   // the two frames of a warp are 16 apart (P bank layout)
      const int t = f0 + fl;
      const bool valid = t < n_frames;
      if (!__any_sync(0xffffffffu, valid)) continue;   // nothing to transform; the mel phase writes `blank`
      // frame t covers reflect-padded samples [160 t, 160 t + 512) = clip samples 160 t - 256 + m; this thread
      // takes the complex points n = q + 16 r (samples 2n, 2n+1); the window is zero for n < 28 and n >= 228
      cpx v[16];
      const int base = kHop * t - kNFft / 2;
      v[0] = cpx{0.0f, 0.0f};
      v[15] = cpx{0.0f, 0.0f};
      if (valid && vec_ok && base + kWinLeft >= 0 && base + kWinLeft + kWin <= L) {
#pragma unroll
        for (int r = 1; r < 15; ++r) {
          const int n = q + 16 * r;
          float2 sv = make_float2(0.0f, 0.0f);
          if (n >= kWinLeft / 2 && n < (kWinLeft + kWin) / 2) {
            if constexpr (I16) {
              const short2 s2 = __ldg(reinterpret_cast<const short2*>(xi + base + 2 * n));
              sv = make_float2(float(s2.x), float(s2.y));
            } else {
              sv = __ldg(reinterpret_cast<const float2*>(xf + base + 2 * n));
            }
          }
          const float2 w2 = win2[n];
          v[r] = cpx{sv.x * w2.x, sv.y * w2.y};
        }
      } else {
#pragma unroll
        for (int r = 1; r < 15; ++r) {
          const int n = q + 16 * r;
          const float2 w2 = win2[n];
          float sv[2] = {0.0f, 0.0f};
          if (valid && n >= kWinLeft / 2 && n < (kWinLeft + kWin) / 2) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              int i = base + 2 * n + h;
              i = i < 0 ? -i : i;
              i = i >= L ? 2 * (L - 1) - i : i;
              i = min(max(i, 0), L - 1);               // clips of <= 256 samples (torchaudio refuses them): stay in bounds
              sv[h] = I16 ? float(__ldg(xi + i)) : __ldg(xf + i);
            }
          }
          v[r] = cpx{sv[0] * w2.x, sv[1] * w2.y};
        }
      }
      fft16(v);                                              // over r:  Y[q][k1]
      E[q] = v[0];
#pragma unroll
      for (int k1 = 1; k1 < 16; ++k1) E[k1 * 17 + q] = cmul(v[k1], twt[k1 * 16 + q]);
      __syncwarp();
#pragma unroll
      for (int qq = 0; qq < 16; ++qq) v[qq] = E[q * 17 + qq]; // this thread is now k1 = q
      __syncwarp();                                          // E is free for the next pass
      fft16(v);                                              // over q:  v[k2] = Z[q + 16 k2]
      // conjugate pairs (k, 256 - k), k = q + 16 k2 < 128: Z[256 - k] is register 15 - k2 of lane (16 - q) & 15
      // (for q = 0: this thread's own register (16 - k2) & 15)
      float* Pf = P + fl;
#pragma unroll
      for (int k2 = 0; k2 < 8; ++k2) {
        cpx zn;
        zn.x = __shfl_sync(0xffffffffu, v[15 - k2].x, partner_lane);
        zn.y = __shfl_sync(0xffffffffu, v[15 - k2].y, partner_lane);
        if (q == 0) zn = v[(16 - k2) & 15];
        float ck, sk;
        sincospif(-float(k2) / 16.0f, &sk, &ck);             // exp(-2 pi i 16 k2 / 512): compile-time constants
        float pk, pn;
        rfft512_power_both(v[k2], zn, cmul(wq, cpx{ck, sk}), &pk, &pn);
        const int k = q + 16 * k2;
        Pf[k * kPStride] = pk;
        Pf[(256 - k) * kPStride] = pn;
      }
      if (q == 0) Pf[128 * kPStride] = rfft512_power_pair(v[8], v[8], cpx{0.0f, -1.0f});
    }
    __syncthreads();

    // ---------------- mel phase: lane = frame, one filter at a time per warp ----------------
    {
      const int t = f0 + lane;
      const bool valid = t < n_frames;
      const float* Pl = P + lane;
#pragma unroll 1
      for (int m = warp; m < kNMels; m += kMelWarps) {
        const int s0 = fbs[m], cnt4 = fbs[kNMels + m];            // taps, rounded up to four (zero weights)
        const float4* w4 = reinterpret_cast<const float4*>(fbw + fbs[2 * kNMels + m]);
        // (a padded tap may point one to three rows past the filter: clamp the row, its weight is zero)
        const float* Pm = Pl + s0 * kPStride;
        const int last = (256 - s0) * kPStride;
        float acc = 0.0f;
        for (int tap = 0; tap < cnt4; tap += 4) {                 // same summation order as a plain tap loop
          const float4 w = w4[tap >> 2];                          // warp-uniform address: one broadcast
          const int o = tap * kPStride;
          acc = fmaf(w.x, Pm[min(o, last)], acc);
          acc = fmaf(w.y, Pm[min(o + kPStride, last)], acc);
          acc = fmaf(w.z, Pm[min(o + 2 * kPStride, last)], acc);
          acc = fmaf(w.w, Pm[min(o + 3 * kPStride, last)], acc);
        }
        // __logf = lg2.approx * ln 2: <= 3 ulp of the result, i.e. < 4e-6 on log-mel values in [-13.8, 12] -- below the
        // FFT's own fp32 round-off in the quiet bins and 4 decades below the bf16 rounding that follows; logf was 9 % of
        // the kernel's instructions
        const float val = !valid ? blank : (p.out_mode == V100_MEL_POWER_F32_NCW ? acc : __logf(acc + p.log_offset));
        if (p.out_mode == V100_MEL_LOG_F32_NTC) {
          otile[lane * (kNMels + 1) + m] = val;
        } else if (t < p.out_pitch) {
          const long long o = (static_cast<long long>(b) * kNMels + m) * p.out_pitch + t;
          if (p.out_mode == V100_MEL_POWER_F32_NCW) static_cast<float*>(p.out)[o] = val;
          else if (p.out_mode == V100_MEL_LOG_F16_NCW) static_cast<unsigned short*>(p.out)[o] = f2h<DT_F16>(val);
          else static_cast<unsigned short*>(p.out)[o] = f2h<DT_BF16>(val);
        }
      }
    }
    __syncthreads();
    if (p.out_mode == V100_MEL_LOG_F32_NTC) {   // out[b][t][64]: transpose through the tile
      for (int i = threadIdx.x; i < kMelTile * (kNMels / 4); i += kMelWarps * 32) {
        const int fl = i >> 4, m4 = (i & 15) * 4;
        const int t = f0 + fl;
        if (t < p.T) {
          const float* s = otile + fl * (kNMels + 1) + m4;
          *reinterpret_cast<float4*>(static_cast<float*>(p.out) + (static_cast<long long>(b) * p.T + t) * kNMels + m4) =
              make_float4(s[0], s[1], s[2], s[3]);
        }
      }
      __syncthreads();
    }
  }
}

template <bool I16>
static int launch_logmel(const MelParams& p, cudaStream_t stream) {
  auto kern = logmel_kernel<I16>;
  static thread_local int configured_dev = -1;
  int dev = 0;
  V100_CUDA(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    V100_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, MelCfg::kSmemBytes));
    configured_dev = dev;
  }
  const int grid = p.total_tiles < kMelCtasPerSm * num_sms() ? p.total_tiles : kMelCtasPerSm * num_sms();
  kern<<<dim3(grid), dim3(kMelWarps * 32), MelCfg::kSmemBytes, stream>>>(p);
  V100_CUDA(cudaGetLastError());
  return 0;
}

int logmel(const void* wav, int wav_dtype, const int32_t* len, int B, int64_t wav_pitch, int L_max,
           const int32_t* fb_start, const int32_t* fb_count, const int32_t* fb_off, const float* fb_w, int fb_nnz,
           float log_offset, void* out, int T, int64_t out_pitch, int out_mode, int32_t* frames_out,
           cudaStream_t stream) {
  if (wav == nullptr || len == nullptr || out == nullptr || fb_start == nullptr || fb_count == nullptr ||
      fb_off == nullptr || fb_w == nullptr)
    return fail(V100_E_INVALID, "logmel: null pointer");
  if (wav_dtype != V100_WAV_F32 && wav_dtype != V100_WAV_I16) return fail(V100_E_INVALID, "logmel: wav_dtype must be V100_WAV_F32 or V100_WAV_I16");
  if (B <= 0 || T <= 0) return fail(V100_E_INVALID, "logmel: bad B=%d or T=%d", B, T);
  if (L_max < 0 || wav_pitch < L_max) return fail(V100_E_INVALID, "logmel: wav_pitch %lld < L_max %d", (long long)wav_pitch, L_max);
  if (fb_nnz < 0 || fb_nnz > kMelMaxNnz) return fail(V100_E_UNSUPPORTED, "logmel: filter bank with %d weights (max %d)", fb_nnz, kMelMaxNnz);
  if (out_mode == V100_MEL_LOG_BF16_NCW || out_mode == V100_MEL_LOG_F16_NCW) {
    if (out_pitch < T || (out_pitch & 7) || (reinterpret_cast<uintptr_t>(out) & 15))
      return fail(V100_E_INVALID, "logmel: 16-bit NCW pitch must be >= T and a multiple of 8, base 16B aligned");
  } else if (out_mode == V100_MEL_POWER_F32_NCW) {
    if (out_pitch < T || (out_pitch & 3) || (reinterpret_cast<uintptr_t>(out) & 15))
      return fail(V100_E_INVALID, "logmel: fp32 NCW pitch must be >= T and a multiple of 4, base 16B aligned");
  } else if (out_mode == V100_MEL_LOG_F32_NTC) {
    if (reinterpret_cast<uintptr_t>(out) & 15) return fail(V100_E_INVALID, "logmel: output base must be 16B aligned");
  } else {
    return fail(V100_E_INVALID, "logmel: unknown out_mode %d", out_mode);
  }
  MelParams p{};
  p.wav = wav; p.len = len; p.wav_pitch = wav_pitch; p.L_max = L_max;
  p.fb_start = fb_start; p.fb_count = fb_count; p.fb_off = fb_off; p.fb_w = fb_w;
  p.log_offset = log_offset; p.out = out; p.T = T; p.out_pitch = out_pitch; p.out_mode = out_mode;
  p.frames_out = frames_out;
  const long long cols = out_mode == V100_MEL_LOG_F32_NTC ? T : out_pitch;   // NCW rows are written to the pitch
  p.tiles_per_clip = int((cols + kMelTile - 1) / kMelTile);
  const long long total = static_cast<long long>(p.tiles_per_clip) * B;
  if (total > 2147483647LL) return fail(V100_E_UNSUPPORTED, "logmel: too many tiles");
  p.total_tiles = int(total);
  return wav_dtype == V100_WAV_I16 ? launch_logmel<true>(p, stream) : launch_logmel<false>(p, stream);
}

// ------------------------------------------------------------------------------------------------------------------
// Any other MelSpectrogramAudioTransform configuration (the reference's constructor is general, data_modules.py:263-281,
// although its code only ever builds 512 / 400 / 160 / 64): n_fft a power of two up to 2048, any win_length <= n_fft,
// any hop, any filter bank.  Not a tuned kernel -- one CTA per frame, an in-place radix-2 FFT in shared memory --
// but the same arithmetic contract as logmel_kernel: reflect padding at the clip's own ends, periodic Hann window
// centred in the frame, |rFFT|^2, sparse mel filters, log(. + offset), BLANK_AUDIO past the clip's own frames.
// ------------------------------------------------------------------------------------------------------------------
struct MelGenParams {
  const void* wav;
  const int32_t* len;
  long long wav_pitch;
  int L_max, n_fft, log2_fft, win, hop, n_mels;
  const int32_t *fb_start, *fb_count, *fb_off;
  const float* fb_w;
  float log_offset;
  void* out;
  int T;
  long long out_pitch;
  int out_mode;
  int32_t* frames_out;
};

template <bool I16>
__global__ void __launch_bounds__(128)
logmel_generic_kernel(const MelGenParams p) {
  __shared__ float2 z[2048];
  __shared__ float P[1025];
  const int b = blockIdx.y, t = blockIdx.x, tid = threadIdx.x;
  const int L = min(max(__ldg(p.len + b), 0), p.L_max);
  const int n_frames = L > 0 ? 1 + L / p.hop : 0;
  if (p.frames_out != nullptr && t == 0 && tid == 0) p.frames_out[b] = 1 + L / p.hop;
  const bool valid = t < n_frames;
  const int N = p.n_fft;
  if (valid) {
    const float* xf = static_cast<const float*>(p.wav) + static_cast<long long>(b) * p.wav_pitch;
    const short* xi = static_cast<const short*>(p.wav) + static_cast<long long>(b) * p.wav_pitch;
    const int base = p.hop * t - N / 2, left = (N - p.win) / 2;
    for (int n = tid; n < N; n += 128) {
      const int m = n - left;
      float v = 0.0f;
      if (m >= 0 && m < p.win) {
        const float w = 0.5f - 0.5f * cospif(float(2 * m) / float(p.win));     // periodic Hann(win)
        int i = base + n;
        i = i < 0 ? -i : i;
        i = i >= L ? 2 * (L - 1) - i : i;
        i = min(max(i, 0), L - 1);
        v = (I16 ? float(__ldg(xi + i)) * (1.0f / 32768.0f) : __ldg(xf + i)) * w;
      }
      z[__brev(unsigned(n)) >> (32 - p.log2_fft)] = make_float2(v, 0.0f);
    }
    __syncthreads();
    for (int len2 = 2; len2 <= N; len2 <<= 1) {
      const int half = len2 >> 1;
      for (int k = tid; k < N / 2; k += 128) {
        const int j = k & (half - 1), i0 = ((k - j) << 1) + j, i1 = i0 + half;
        float sn, cs;
        sincospif(-float(2 * j) / float(len2), &sn, &cs);
        const float2 a = z[i0], c = z[i1];
        const float2 wc = make_float2(c.x * cs - c.y * sn, c.x * sn + c.y * cs);
        z[i0] = make_float2(a.x + wc.x, a.y + wc.y);
        z[i1] = make_float2(a.x - wc.x, a.y - wc.y);
      }
      __syncthreads();
    }
    for (int k = tid; k <= N / 2; k += 128) P[k] = z[k].x * z[k].x + z[k].y * z[k].y;
    __syncthreads();
  }
  const float blank = p.out_mode == V100_MEL_POWER_F32_NCW ? 0.0f : logf(p.log_offset);
  for (int m = tid; m < p.n_mels; m += 128) {
    float val = blank;
    if (valid) {
      const int s0 = __ldg(p.fb_start + m), cnt = __ldg(p.fb_count + m);
      const float* w = p.fb_w + __ldg(p.fb_off + m);
      float acc = 0.0f;
      for (int i = 0; i < cnt; ++i) acc = fmaf(__ldg(w + i), P[s0 + i], acc);
      val = p.out_mode == V100_MEL_POWER_F32_NCW ? acc : logf(acc + p.log_offset);
    }
    if (p.out_mode == V100_MEL_LOG_F32_NTC) {
      static_cast<float*>(p.out)[(static_cast<long long>(b) * p.T + t) * p.n_mels + m] = val;
    } else {
      const long long o = (static_cast<long long>(b) * p.n_mels + m) * p.out_pitch + t;
      if (p.out_mode == V100_MEL_POWER_F32_NCW) static_cast<float*>(p.out)[o] = val;
      else if (p.out_mode == V100_MEL_LOG_F16_NCW) static_cast<unsigned short*>(p.out)[o] = f2h<DT_F16>(val);
      else static_cast<unsigned short*>(p.out)[o] = f2h<DT_BF16>(val);
    }
  }
}

int logmel_generic(const void* wav, int wav_dtype, const int32_t* len, int B, int64_t wav_pitch, int L_max, int n_fft,
                   int win_length, int hop_length, int n_mels, const int32_t* fb_start, const int32_t* fb_count,
                   const int32_t* fb_off, const float* fb_w, float log_offset, void* out, int T, int64_t out_pitch,
                   int out_mode, int32_t* frames_out, cudaStream_t stream) {
  if (wav == nullptr || len == nullptr || out == nullptr || fb_start == nullptr || fb_count == nullptr ||
      fb_off == nullptr || fb_w == nullptr)
    return fail(V100_E_INVALID, "logmel_generic: null pointer");
  if (wav_dtype != V100_WAV_F32 && wav_dtype != V100_WAV_I16) return fail(V100_E_INVALID, "logmel_generic: bad wav_dtype");
  if (B <= 0 || B > 65535 || T <= 0) return fail(V100_E_INVALID, "logmel_generic: bad B=%d or T=%d", B, T);
  if (L_max < 0 || wav_pitch < L_max) return fail(V100_E_INVALID, "logmel_generic: wav_pitch %lld < L_max %d", (long long)wav_pitch, L_max);
  int log2_fft = 0;
  while ((1 << log2_fft) < n_fft) ++log2_fft;
  if (n_fft < 8 || n_fft > 2048 || (1 << log2_fft) != n_fft)
    return fail(V100_E_UNSUPPORTED, "logmel_generic: n_fft=%d must be a power of two in [8, 2048]", n_fft);
  if (win_length <= 0 || win_length > n_fft || hop_length <= 0 || n_mels <= 0)
    return fail(V100_E_INVALID, "logmel_generic: need 0 < win_length <= n_fft, hop_length > 0, n_mels > 0");
  if (!(log_offset > 0.0f) && out_mode != V100_MEL_POWER_F32_NCW) return fail(V100_E_INVALID, "logmel_generic: log_offset must be positive");
  if (out_mode == V100_MEL_LOG_BF16_NCW || out_mode == V100_MEL_LOG_F16_NCW || out_mode == V100_MEL_POWER_F32_NCW) {
    if (out_pitch < T) return fail(V100_E_INVALID, "logmel_generic: NCW pitch must be >= T");
  } else if (out_mode != V100_MEL_LOG_F32_NTC) {
    return fail(V100_E_INVALID, "logmel_generic: unknown out_mode %d", out_mode);
  }
  MelGenParams p{};
  p.wav = wav; p.len = len; p.wav_pitch = wav_pitch; p.L_max = L_max;
  p.n_fft = n_fft; p.log2_fft = log2_fft; p.win = win_length; p.hop = hop_length; p.n_mels = n_mels;
  p.fb_start = fb_start; p.fb_count = fb_count; p.fb_off = fb_off; p.fb_w = fb_w;
  p.log_offset = log_offset; p.out = out; p.T = T; p.out_pitch = out_pitch; p.out_mode = out_mode; p.frames_out = frames_out;
  const long long cols = out_mode == V100_MEL_LOG_F32_NTC ? T : out_pitch;   // NCW rows are written to the pitch
  dim3 grid((unsigned)cols, B);
  if (wav_dtype == V100_WAV_I16) logmel_generic_kernel<true><<<grid, 128, 0, stream>>>(p);
  else logmel_generic_kernel<false><<<grid, 128, 0, stream>>>(p);
  V100_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace v100
