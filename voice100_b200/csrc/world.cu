// WORLD waveform synthesis on the device: f0 / log-spectrum / coded aperiodicity -> 16 kHz PCM (v100_world_* in
// include/v100.h).  Restates WORLD's DecodeAperiodicity (codec.cpp) and Synthesis (synthesis.cpp), the code behind
// pyworld.decode_aperiodicity / pyworld.synthesize that the reference's WORLDVocoder.decode (voice100/vocoder.py:89-102)
// runs one utterance at a time on a CPU core.  The contract is oracle/world.py (float64 numpy); parity with pyworld
// itself is unverified (DESIGN.md section 3.8).
//
// Three kernels:
//  - world_noise_kernel: WORLD's randn() stream (xorshift128, 12 draws a value) into a float64 table.  One thread
//    runs the recurrence; the table is a pure function of its length, so the Python layer builds it once per device.
//  - world_timebase_kernel: one CTA per utterance.  Per sample: the interpolated f0 / voicing (interp1 with WORLD's
//    histc intervals), the phase increment 2 pi f0 / fs, the running phase, fmod(., 2 pi) and the pulse test.  Every
//    float64 operation is an explicit _rn intrinsic (no FMA contraction), and the running phase is ONE dependent chain
//    of adds taken by one thread in sample order: pulse positions are integers compared exactly with the oracle, so
//    the phase must round as the sequential float64 sum does.  Then each pulse's noise run (distance to the next
//    pulse) is filled in.  The workspace it writes has a size that depends only on (B, 160 T).
//  - world_synth_kernel: output-stationary, one CTA per (1024-sample tile, utterance).  The CTA lists the pulses
//    whose 512-sample response overlaps its tile; each warp computes one pulse's whole response (four 512-point
//    complex FFTs, fp32) and the CTA adds the responses in pulse order.  A pulse near a tile edge is computed by both
//    CTAs; in exchange there are no float atomics and no buffer of data-dependent size, and the output is the same
//    bit for bit from run to run and whatever else is in the batch.
//
// Per pulse (one warp; FFT = fft512_warp, built from logmel_core.h's fft16):
//   1. both log-amplitudes, L1 = log(S (1 - A) + eps) / 2 (periodic) and L2 = log(S A + eps) / 2 or log(S) / 2
//      (aperiodic), mirrored to 512 points and packed as L1 + i L2: both are real and even, so ONE FFT gives both real
//      cepstra.  Fold (c0, 2c, c256, 0) and pack again: ONE FFT gives DFT(c1^) and DFT(c2^) (separated through
//      X[k] and conj X[N-k]); H = exp(.) for bins 0..256.
//   2. the noise run (mean removed in float64, exact) through one FFT.
//   3. P = H1 * fractional delay (cos - i sqrt(1 - cos^2) = cos - i |sin|), Q = H2 * noise: the two real inverse
//      transforms are one complex inverse of P + iQ (Hermitian-extended; the Nyquist bin of P keeps its real part only,
//      as a real inverse FFT reads it).  fftshift, DC removal, (h sqrt(n) + a) / N.
// The envelope is handled in the log domain (log S = logsumexp of the two frames' logspc) so that logspc anywhere in
// [-80, 20] neither underflows nor overflows in fp32; 1 - A is formed as d (2 - d) with d = 1 - ap = -expm1(.),
// which keeps it accurate where ap is close to 1.
#include <math.h>

#include "common.cuh"
#include "host.h"
#include "logmel_core.h"

namespace v100 {

namespace {

constexpr int kFs = 16000;
constexpr int kN = 512;
constexpr int kHalf = kN / 2;
constexpr int kHop = 160;                                   // samples per 10 ms frame at 16 kHz
constexpr double kPi = 3.1415926535897932384;
constexpr double kTwoPi = 2.0 * kPi;
constexpr double kPeriod = 10.0 / 1000.0;                   // frame period in s, as WORLD computes it
constexpr double kLowestF0 = static_cast<double>(kFs) / kN + 1.0;
constexpr double kDefaultF0 = 500.0;
constexpr double kApMax = 0.999999999999, kApMin = 0.001;
constexpr float kLogEps = -27.631021115928547f;             // log(1e-12)

constexpr int kTbThreads = 256;
constexpr int kTbChunk = 2048;

constexpr int kSynThreads = 256;
constexpr int kSynWarps = kSynThreads / 32;
constexpr int kTile = 1024;                                 // output samples per CTA
constexpr int kListMax = kTile + kN - 1;                    // pulse positions whose response can reach the tile
constexpr int kSBuf = 2 * (kHalf + 1) + 6;                  // per-warp spectra: P[257] | H2[257] (cpx)
constexpr int kEBuf = 32 * 17;                              // per-warp FFT exchange buffer (cpx)

__host__ __device__ inline long long ws_pitch(int T) { return static_cast<long long>(T) * kHop; }

struct WorldWs {
  int32_t* head;   // [B][4] status, y_len, first pulse sample, pulse count
  int32_t* info;   // [B][Yp] -1 = no pulse, else (noise size << 1) | vuv
  double* tau;     // [B][Yp] fractional pulse shift in s (at pulse samples only)
};

__host__ __device__ inline size_t align256(size_t x) { return (x + 255) & ~static_cast<size_t>(255); }

__host__ __device__ inline WorldWs ws_carve(void* base, int B, long long Yp) {
  uint8_t* p = static_cast<uint8_t*>(base);
  WorldWs w;
  w.head = reinterpret_cast<int32_t*>(p);
  p += align256(static_cast<size_t>(B) * 16);
  w.info = reinterpret_cast<int32_t*>(p);
  p += align256(static_cast<size_t>(B) * Yp * 4);
  w.tau = reinterpret_cast<double*>(p);
  return w;
}

struct WorldIn {
  const float* f0;
  long long f0_sb, f0_st;
  const float* sp;
  long long sp_sb, sp_st, sp_sk;
  const float* ap;
  long long ap_sb, ap_st;
  const int32_t* frame_len;
  int T;
};

// ------------------------------------------------------------------------------------------------ noise table

__global__ void world_noise_kernel(double* __restrict__ out, long long n) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  uint32_t x = 123456789u, y = 362436069u, z = 521288629u, w = 88675123u;
  for (long long j = 0; j < n; ++j) {
    uint32_t s = 0;
#pragma unroll
    for (int k = 0; k < 12; ++k) {
      const uint32_t t = x ^ (x << 11);
      x = y;
      y = z;
      z = w;
      w = (w ^ (w >> 19)) ^ (t ^ (t >> 8));
      s += w >> 4;
    }
    out[j] = __dadd_rn(__dmul_rn(static_cast<double>(s), 1.0 / 268435456.0), -6.0);   // both steps exact
  }
}

// ------------------------------------------------------------------------------------------------ time base

// coarse f0 / vuv knot t (t <= Tb): WORLD's GetTemporalParametersForTimeBase, the knot at Tb extrapolated
__device__ __forceinline__ double knot_f0(const float* f0, long long st, int t) {
  const double f = static_cast<double>(__ldg(f0 + t * st));
  return f < kLowestF0 ? 0.0 : f;
}

__device__ void knot_pair(const float* f0, long long st, int Tb, int j, double* f, double* v) {
  // knots j and j + 1 (j + 1 may be the extrapolated Tb)
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int t = j + u;
    if (t < Tb) {
      f[u] = knot_f0(f0, st, t);
      v[u] = f[u] == 0.0 ? 0.0 : 1.0;
    } else {
      const double a = knot_f0(f0, st, Tb - 1), b = knot_f0(f0, st, Tb - 2);
      const double va = a == 0.0 ? 0.0 : 1.0, vb = b == 0.0 ? 0.0 : 1.0;
      f[u] = __dsub_rn(__dmul_rn(a, 2.0), b);
      v[u] = __dsub_rn(__dmul_rn(va, 2.0), vb);
    }
  }
}

__global__ void __launch_bounds__(kTbThreads)
world_timebase_kernel(const WorldIn in, int B, WorldWs ws, long long Yp, int32_t* __restrict__ wav_len,
                      int32_t* __restrict__ status) {
  __shared__ double ph[kTbChunk];
  __shared__ unsigned char vv[kTbChunk];
  __shared__ double s_wprev;
  __shared__ int s_vprev;
  __shared__ int s_first[kTbThreads], s_next[kTbThreads];
  __shared__ int s_count;
  const int b = blockIdx.x, tid = threadIdx.x;
  int Tb = in.frame_len == nullptr ? in.T : __ldg(in.frame_len + b);
  Tb = Tb < 0 ? 0 : (Tb > in.T ? in.T : Tb);
  const float* f0 = in.f0 + b * in.f0_sb;
  const float* sp = in.sp + b * in.sp_sb;
  const float* ap = in.ap + b * in.ap_sb;
  int32_t* head = ws.head + 4 * b;

  int st = V100_WORLD_OK;
  if (Tb < 2) {
    st = V100_WORLD_SHORT;                 // WORLD reads f0[-1] for the extrapolated knot
  } else {
    bool bad = false;
    for (int t = tid; t < Tb; t += kTbThreads)
      bad |= !isfinite(__ldg(f0 + t * in.f0_st)) || !isfinite(__ldg(ap + t * in.ap_st));
    const long long n_sp = static_cast<long long>(Tb) * (kHalf + 1);
    for (long long i = tid; i < n_sp; i += kTbThreads) {
      const long long t = i / (kHalf + 1), k = i - t * (kHalf + 1);
      bad |= !isfinite(__ldg(sp + t * in.sp_st + k * in.sp_sk));
    }
    if (__syncthreads_or(bad)) st = V100_WORLD_NONFINITE;
  }
  if (st != V100_WORLD_OK) {
    if (tid == 0) {
      head[0] = st;
      head[1] = head[2] = head[3] = 0;
      wav_len[b] = 0;
      status[b] = st;
    }
    return;
  }

  const int y_len = Tb * kHop;
  int32_t* info = ws.info + b * Yp;
  double* tau = ws.tau + b * Yp;
  if (tid == 0) {
    s_wprev = 0.0;
    s_vprev = 0;
  }
  double run = 0.0;                                          // thread 0: the running phase
  for (int c0 = 0; c0 < y_len; c0 += kTbChunk) {
    const int n = min(kTbChunk, y_len - c0);
    for (int i = tid; i < n; i += kTbThreads) {
      const int gi = c0 + i;
      const double xi = __ddiv_rn(static_cast<double>(gi), static_cast<double>(kFs));
      // histc: the interval j with x_j <= xi < x_{j+1}, clamped to [0, Tb - 1]
      int j = static_cast<int>(xi * 100.0);
      j = j < 0 ? 0 : (j > Tb - 1 ? Tb - 1 : j);
      while (j > 0 && __dmul_rn(static_cast<double>(j), kPeriod) > xi) --j;
      while (j < Tb - 1 && __dmul_rn(static_cast<double>(j + 1), kPeriod) <= xi) ++j;
      const double xj = __dmul_rn(static_cast<double>(j), kPeriod), xj1 = __dmul_rn(static_cast<double>(j + 1), kPeriod);
      const double s = __ddiv_rn(__dsub_rn(xi, xj), __dsub_rn(xj1, xj));
      double f[2], v[2];
      knot_pair(f0, in.f0_st, Tb, j, f, v);
      const double fi = __dadd_rn(f[0], __dmul_rn(s, __dsub_rn(f[1], f[0])));
      const double vi = __dadd_rn(v[0], __dmul_rn(s, __dsub_rn(v[1], v[0])));
      const bool voiced = vi > 0.5;
      const double fr = voiced ? fi : kDefaultF0;
      ph[i] = __ddiv_rn(__dmul_rn(kTwoPi, fr), static_cast<double>(kFs));
      vv[i] = voiced ? 1 : 0;
    }
    __syncthreads();
    if (tid == 0) {                                          // the one sequential chain of float64 adds
      int i = 0;
      for (; i + 4 <= n; i += 4) {
        const double a0 = ph[i], a1 = ph[i + 1], a2 = ph[i + 2], a3 = ph[i + 3];
        run = __dadd_rn(run, a0);
        ph[i] = run;
        run = __dadd_rn(run, a1);
        ph[i + 1] = run;
        run = __dadd_rn(run, a2);
        ph[i + 2] = run;
        run = __dadd_rn(run, a3);
        ph[i + 3] = run;
      }
      for (; i < n; ++i) {
        run = __dadd_rn(run, ph[i]);
        ph[i] = run;
      }
    }
    __syncthreads();
    for (int i = tid; i < n; i += kTbThreads) ph[i] = fmod(ph[i], kTwoPi);
    __syncthreads();
    // the pulse test of sample gi = c0 + i - 1 compares w[gi] and w[gi + 1]
    for (int i = tid; i < n; i += kTbThreads) {
      const int gi = c0 + i - 1;
      if (gi < 0) continue;
      const double wi = i == 0 ? s_wprev : ph[i - 1], wn = ph[i];
      const int vi = i == 0 ? s_vprev : vv[i - 1];
      if (fabs(__dsub_rn(wn, wi)) > kPi) {
        const double y1 = __dsub_rn(wi, kTwoPi);
        const double x = __ddiv_rn(-y1, __dsub_rn(wn, y1));
        tau[gi] = __ddiv_rn(x, static_cast<double>(kFs));
        info[gi] = vi;
      } else {
        info[gi] = -1;
      }
    }
    __syncthreads();
    if (tid == 0) {
      s_wprev = ph[n - 1];
      s_vprev = vv[n - 1];
    }
    __syncthreads();
  }
  if (tid == 0) {
    info[y_len - 1] = -1;                                   // the last sample has no successor to test against
    s_count = 0;
  }
  __syncthreads();

  // noise size of each pulse = distance to the next pulse (0 for the last): contiguous segments per thread
  const int seg = (y_len + kTbThreads - 1) / kTbThreads;
  const int lo = min(y_len, tid * seg), hi = min(y_len, lo + seg);
  int first = INT_MAX, cnt = 0;
  for (int i = lo; i < hi; ++i)
    if (info[i] >= 0) {
      if (first == INT_MAX) first = i;
      ++cnt;
    }
  s_first[tid] = first;
  atomicAdd(&s_count, cnt);
  __syncthreads();
  if (tid == 0) {
    int nx = INT_MAX;
    for (int t = kTbThreads - 1; t >= 0; --t) {
      s_next[t] = nx;
      nx = min(nx, s_first[t]);
    }
    head[0] = V100_WORLD_OK;
    head[1] = y_len;
    head[2] = nx == INT_MAX ? 0 : nx;
    head[3] = s_count;
    wav_len[b] = y_len;
    status[b] = V100_WORLD_OK;
  }
  __syncthreads();
  int pend = -1;
  for (int i = lo; i < hi; ++i) {
    const int v = info[i];
    if (v < 0) continue;
    if (pend >= 0) info[pend] = ((i - pend) << 1) | (info[pend] & 1);
    pend = i;
  }
  if (pend >= 0) {
    const int nx = s_next[tid];
    info[pend] = ((nx == INT_MAX ? 0 : nx - pend) << 1) | (info[pend] & 1);
  }
}

// ------------------------------------------------------------------------------------------------ synthesis

// 512-point complex forward DFT across one warp.  In: lane q holds x[q + 32 r] in v[r], r = 0..15.  Out: lane
// (k1 = lane & 15, h = lane >> 4) holds X[k1 + 16 k2a + 256 h] in v[k2a].  n = q + 32 r, k = k1 + 16 k2:
// a 16-point DFT over r (fft16), twiddle W512^(q k1), exchange through E, a 16-point DFT over q' (q = 2 q' + h),
// twiddle W32^(h k2a), and one radix-2 butterfly between lanes h = 0 and h = 1 by shuffle.
__device__ __forceinline__ void fft512_warp(cpx* v, cpx* E, const cpx* tw, int lane) {
  fft16(v);
  E[lane * 17] = v[0];
#pragma unroll
  for (int k1 = 1; k1 < 16; ++k1) E[lane * 17 + k1] = cmul(v[k1], tw[lane * k1]);
  __syncwarp();
  const int k1 = lane & 15, h = lane >> 4;
#pragma unroll
  for (int qq = 0; qq < 16; ++qq) v[qq] = E[(2 * qq + h) * 17 + k1];
  __syncwarp();
  fft16(v);
  if (h) {
#pragma unroll
    for (int k = 1; k < 16; ++k) v[k] = cmul(v[k], tw[16 * k]);
  }
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const float ox = __shfl_xor_sync(0xffffffffu, v[k].x, 16), oy = __shfl_xor_sync(0xffffffffu, v[k].y, 16);
    v[k] = h ? cpx{ox - v[k].x, oy - v[k].y} : cpx{v[k].x + ox, v[k].y + oy};
  }
}

__device__ __forceinline__ int out_bin(int lane, int k2a) { return (lane & 15) + 16 * k2a + 256 * (lane >> 4); }

// decoded aperiodicity of bin m for coded value ca: a = clamp(ap, 0.001, 1 - 1e-12) and d = 1 - a, accurate near 1
__device__ __forceinline__ void ap_bin(float ca, int m, float* a, float* d) {
  if (ca > -0.5f) {
    *a = 1.0f;
    *d = 1e-12f;
    return;
  }
  const float fr = static_cast<float>(m) * 31.25f;          // k fs / N
  const float v = m < 96 ? -60.0f + (fr / 3000.0f) * (ca + 60.0f) : ca + ((fr - 3000.0f) / 5000.0f) * (-1e-12f - ca);
  const float e = v * 0.11512925464970229f;                 // ln(10) / 20
  *a = fmaxf(expf(e), 0.001f);
  *d = fminf(fmaxf(-expm1f(e), 1e-12f), 0.999f);
}

__device__ __forceinline__ float log_add_eps(float u) {    // log(exp(u) + 1e-12)
  const float m = fmaxf(u, kLogEps);
  return m + log1pf(expf(-fabsf(u - kLogEps)));
}

struct PulseFrame {
  const float* spf;
  const float* spc;
  long long sk;
  float w, caf, cac;
  bool same, vuv;
};

// (L1, L2) of bin m: periodic and aperiodic half log-amplitudes
__device__ __forceinline__ cpx bin_logs(const PulseFrame& p, int m) {
  const float sf = __ldg(p.spf + m * p.sk);
  float lS, a, d;
  float af, df;
  ap_bin(p.caf, m, &af, &df);
  if (p.same) {
    lS = sf;
    a = af;
    d = df;
  } else {
    const float sc = __ldg(p.spc + m * p.sk);
    const float mx = fmaxf(sf, sc);
    lS = mx + logf((1.0f - p.w) * expf(sf - mx) + p.w * expf(sc - mx));
    float ac, dc;
    ap_bin(p.cac, m, &ac, &dc);
    a = (1.0f - p.w) * af + p.w * ac;
    d = (1.0f - p.w) * df + p.w * dc;
  }
  const float L1 = 0.5f * log_add_eps(lS + logf(d) + logf(2.0f - d));
  const float L2 = p.vuv ? 0.5f * log_add_eps(lS + 2.0f * logf(a)) : 0.5f * lS;
  return cpx{L1, L2};
}

struct SynthParams {
  WorldIn in;
  WorldWs ws;
  long long Yp;
  const double* noise;
  float* wav;
  long long wav_pitch;
};

// one pulse's 512-sample response (fftshifted: sample n lands at y[pos - 255 + n]) into resp, by one warp
__device__ void pulse_response(const SynthParams& P, int b, int Tb, int first, int pos, cpx* S, cpx* E,
                               const cpx* tw, const float* dcr, int lane) {
  const int inf = P.ws.info[b * P.Yp + pos];
  const int nsz = inf >> 1;
  const bool vuv = (inf & 1) != 0;
  const double tau = P.ws.tau[b * P.Yp + pos];
  // frames around the pulse time (GetSpectralEnvelope / GetAperiodicRatio)
  const double q = __ddiv_rn(__ddiv_rn(static_cast<double>(pos), static_cast<double>(kFs)), kPeriod);
  const double qf = floor(q);
  const int fl = min(Tb - 1, static_cast<int>(qf)), ce = min(Tb - 1, static_cast<int>(ceil(q)));
  const double wd = q - qf;
  PulseFrame pf;
  pf.spf = P.in.sp + b * P.in.sp_sb + fl * P.in.sp_st;
  pf.spc = P.in.sp + b * P.in.sp_sb + ce * P.in.sp_st;
  pf.sk = P.in.sp_sk;
  pf.w = static_cast<float>(wd);
  pf.caf = __ldg(P.in.ap + b * P.in.ap_sb + fl * P.in.ap_st);
  pf.cac = __ldg(P.in.ap + b * P.in.ap_sb + ce * P.in.ap_st);
  pf.same = fl == ce;
  pf.vuv = vuv;
  bool periodic = vuv;
  {  // A[0] > 0.999 switches the periodic part off; bin 0 decodes to 0.001 or (clamped) 1 - 1e-12
    const double a0f = pf.caf > -0.5f ? kApMax : kApMin, a0c = pf.cac > -0.5f ? kApMax : kApMin;
    const double a0 = pf.same ? a0f : (1.0 - wd) * a0f + wd * a0c;
    periodic = periodic && a0 * a0 <= 0.999;
  }

  cpx v[16];
  // (1) cepstra of both log-amplitudes in one FFT
#pragma unroll
  for (int r = 0; r < 16; ++r) {
    const int n = lane + 32 * r;
    v[r] = bin_logs(pf, n <= kHalf ? n : kN - n);
  }
  fft512_warp(v, E, tw, lane);
#pragma unroll
  for (int k2a = 0; k2a < 16; ++k2a) {
    const int k = out_bin(lane, k2a);
    const float f = (k == 0 || k == kHalf) ? 1.0f / kN : (k < kHalf ? 2.0f / kN : 0.0f);
    S[k] = cpx{v[k2a].x * f, v[k2a].y * f};
  }
  __syncwarp();
#pragma unroll
  for (int r = 0; r < 16; ++r) v[r] = S[lane + 32 * r];
  __syncwarp();
  fft512_warp(v, E, tw, lane);
#pragma unroll
  for (int k2a = 0; k2a < 16; ++k2a) S[out_bin(lane, k2a)] = v[k2a];
  __syncwarp();
  // separate the two transforms, exponentiate, apply the fractional delay: P[k] (periodic), H2[k] (aperiodic)
  cpx pk[9], h2[9];
  const float xs = static_cast<float>(tau * kFs);
#pragma unroll
  for (int j = 0; j < 9; ++j) {
    const int k = lane + 32 * j;
    if (k > kHalf) continue;
    const cpx zk = S[k], zn = S[(kN - k) & (kN - 1)];
    const cpx x1{0.5f * (zk.x + zn.x), 0.5f * (zk.y - zn.y)};
    const cpx x2{0.5f * (zk.y + zn.y), -0.5f * (zk.x - zn.x)};
    float s1, c1, s2, c2;
    sincosf(x1.y, &s1, &c1);
    sincosf(x2.y, &s2, &c2);
    const float m1 = expf(x1.x), m2 = expf(x2.x);
    h2[j] = cpx{m2 * c2, m2 * s2};
    if (periodic) {
      float ss, cs;
      sincospif(xs * static_cast<float>(k) / static_cast<float>(kHalf), &ss, &cs);   // theta k = 2 pi tau fs k / N
      const cpx h1{m1 * c1, m1 * s1};
      cpx pp = cmul(h1, cpx{cs, -fabsf(ss)});
      if (k == kHalf) pp.y = 0.0f;                          // a real inverse FFT reads the Nyquist bin's real part
      pk[j] = pp;
    } else {
      pk[j] = cpx{0.0f, 0.0f};
    }
  }
  __syncwarp();
#pragma unroll
  for (int j = 0; j < 9; ++j) {
    const int k = lane + 32 * j;
    if (k > kHalf) continue;
    S[k] = pk[j];
    S[kHalf + 1 + k] = h2[j];
  }
  __syncwarp();

  // (2) the pulse's noise: WORLD's randn values [pos - first, + nsz), mean removed (exact in float64), first N kept
  const int off = pos - first;
  double sum = 0.0;
  for (int i = lane; i < nsz; i += 32) sum += P.noise[off + i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const double mean = nsz > 0 ? __ddiv_rn(sum, static_cast<double>(nsz)) : 0.0;
  const int nk = min(nsz, kN);
#pragma unroll
  for (int r = 0; r < 16; ++r) {
    const int n = lane + 32 * r;
    v[r] = cpx{n < nk ? static_cast<float>(__dsub_rn(P.noise[off + n], mean)) : 0.0f, 0.0f};
  }
  fft512_warp(v, E, tw, lane);

  // (3) Y = P + i Q, Hermitian-extended; the inverse is conj(FFT(conj Y))
#pragma unroll
  for (int k2a = 0; k2a < 16; ++k2a) {
    const int k = out_bin(lane, k2a);
    cpx pp, hh;
    if (k <= kHalf) {
      pp = S[k];
      hh = S[kHalf + 1 + k];
    } else {
      pp = S[kN - k];
      pp.y = -pp.y;
      hh = S[kHalf + 1 + kN - k];
      hh.y = -hh.y;
    }
    const cpx qq = cmul(v[k2a], hh);
    v[k2a] = cpx{pp.x - qq.y, -(pp.y + qq.x)};             // conj(P + i Q)
  }
  __syncwarp();
#pragma unroll
  for (int k2a = 0; k2a < 16; ++k2a) S[out_bin(lane, k2a)] = v[k2a];
  __syncwarp();
#pragma unroll
  for (int r = 0; r < 16; ++r) v[r] = S[lane + 32 * r];
  __syncwarp();
  fft512_warp(v, E, tw, lane);
  // v[k2a] = conj(p + i q)[j], j = out_bin: p = N irfft(P) (periodic), q = N irfft(Q) (aperiodic), before fftshift.
  // After fftshift sample j sits at n = (j + 256) mod 512; the DC of the periodic part is the sum over n >= 256,
  // i.e. over j < 256 (lanes 0..15).
  float dsum = 0.0f;
  if (lane < 16) {
#pragma unroll
    for (int k2a = 0; k2a < 16; ++k2a) dsum += v[k2a].x;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) dsum += __shfl_xor_sync(0xffffffffu, dsum, o);
  const float sq = sqrtf(static_cast<float>(nsz));
  float* resp = reinterpret_cast<float*>(S);
  __syncwarp();
#pragma unroll
  for (int k2a = 0; k2a < 16; ++k2a) {
    const int j = out_bin(lane, k2a);
    const int n = (j + kHalf) & (kN - 1);
    float hv = 0.0f;
    if (periodic) hv = (n < kHalf ? 0.0f : v[k2a].x) - dsum * dcr[n];
    resp[n] = (hv * sq - v[k2a].y) * (1.0f / kN);
  }
  __syncwarp();
}

__global__ void __launch_bounds__(kSynThreads)
world_synth_kernel(const SynthParams P) {
  extern __shared__ __align__(16) uint8_t syn_smem[];
  cpx* tw = reinterpret_cast<cpx*>(syn_smem);                                    // [512] W512^m
  float* dcr = reinterpret_cast<float*>(tw + kN);                                // [512] DC remover
  int* list = reinterpret_cast<int*>(dcr + kN);                                  // [kListMax + 1]
  int* wsum = list + kListMax + 1;                                               // [kSynWarps + 1]
  cpx* wbuf = reinterpret_cast<cpx*>(wsum + 16);                                 // [warps][kSBuf + kEBuf]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.y;
  const long long t0 = static_cast<long long>(blockIdx.x) * kTile;

  for (int m = tid; m < kN; m += kSynThreads) {
    float s, c;
    sincospif(-static_cast<float>(m) / static_cast<float>(kHalf), &s, &c);
    tw[m] = cpx{c, s};
    // r[n] = 0.5 - 0.5 cos(2 pi (n + 1) / (N + 1)) for n < N/2, mirrored; sum_{n < N/2} = N/4 + 1/4 in closed form
    const int i = m < kHalf ? m : kN - 1 - m;
    const double r = 0.5 - 0.5 * cos(kTwoPi * (i + 1.0) / (1.0 + kN));
    dcr[m] = static_cast<float>(r / (2.0 * (kN / 4 + 0.25)));
  }
  const int32_t* head = P.ws.head + 4 * b;
  const int st = head[0], y_len = head[1], first = head[2];
  float* out = P.wav + b * P.wav_pitch;
  const long long t_end = min(t0 + kTile, P.wav_pitch);
  if (st != V100_WORLD_OK || t0 >= y_len) {
    for (long long i = t0 + tid; i < t_end; i += kSynThreads) out[i] = 0.0f;
    return;
  }
  const int Tb = y_len / kHop;

  // pulses with position p in [t0 - 256, t0 + 1279) (response covers [p - 255, p + 256]); pulses sit below y_len - 1
  const int lo = static_cast<int>(max(0LL, t0 - kHalf));
  const int hi = static_cast<int>(min(static_cast<long long>(y_len - 1), t0 + kTile + kHalf - 1));
  constexpr int kPer = (kListMax + kSynThreads - 1) / kSynThreads;
  const int32_t* info = P.ws.info + b * P.Yp;
  const int s0 = lo + tid * kPer;
  int mine = 0;
#pragma unroll
  for (int u = 0; u < kPer; ++u) mine += (s0 + u < hi && info[s0 + u] >= 0) ? 1 : 0;
  int incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int up = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += up;
  }
  if (lane == 31) wsum[warp] = incl;
  __syncthreads();
  if (tid == 0) {
    int run = 0;
    for (int w = 0; w < kSynWarps; ++w) {
      const int c = wsum[w];
      wsum[w] = run;
      run += c;
    }
    wsum[kSynWarps] = run;
  }
  __syncthreads();
  int at = wsum[warp] + incl - mine;
#pragma unroll
  for (int u = 0; u < kPer; ++u)
    if (s0 + u < hi && info[s0 + u] >= 0) list[at++] = s0 + u;
  const int npulse = wsum[kSynWarps];
  __syncthreads();

  cpx* S = wbuf + warp * (kSBuf + kEBuf);
  cpx* E = S + kSBuf;
  float acc[kTile / kSynThreads];
#pragma unroll
  for (int u = 0; u < kTile / kSynThreads; ++u) acc[u] = 0.0f;
  for (int base = 0; base < npulse; base += kSynWarps) {
    if (base + warp < npulse) pulse_response(P, b, Tb, first, list[base + warp], S, E, tw, dcr, lane);
    __syncthreads();
    const int nr = min(kSynWarps, npulse - base);
    for (int w = 0; w < nr; ++w) {                          // pulse order
      const int p0 = list[base + w] - (kHalf - 1);
      const float* resp = reinterpret_cast<const float*>(wbuf + w * (kSBuf + kEBuf));
#pragma unroll
      for (int u = 0; u < kTile / kSynThreads; ++u) {
        const int idx = static_cast<int>(t0 + tid + u * kSynThreads - p0);
        if (idx >= 0 && idx < kN) acc[u] += resp[idx];
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int u = 0; u < kTile / kSynThreads; ++u) {
    const long long i = t0 + tid + u * kSynThreads;
    if (i < t_end) out[i] = i < y_len ? acc[u] : 0.0f;
  }
}

constexpr size_t kSynSmem = kN * sizeof(cpx) + kN * sizeof(float) + (kListMax + 1 + 16) * sizeof(int) +
                            static_cast<size_t>(kSynWarps) * (kSBuf + kEBuf) * sizeof(cpx);

int check_in(const WorldIn& in, int B, const char* who) {
  if (in.f0 == nullptr || in.sp == nullptr || in.ap == nullptr) return fail(V100_E_INVALID, "%s: null input", who);
  if (B <= 0 || in.T < 0) return fail(V100_E_INVALID, "%s: B must be positive and T non-negative", who);
  if (static_cast<long long>(in.T) * kHop > (1LL << 30))
    return fail(V100_E_UNSUPPORTED, "%s: T = %d frames is more than 2^30 samples", who, in.T);
  return 0;
}

int launch_timebase(const WorldIn& in, int B, void* workspace, int32_t* wav_len, int32_t* status,
                    cudaStream_t stream) {
  const long long Yp = ws_pitch(in.T);
  const WorldWs ws = ws_carve(workspace, B, Yp);
  world_timebase_kernel<<<dim3(B), dim3(kTbThreads), 0, stream>>>(in, B, ws, Yp, wav_len, status);
  V100_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace

int64_t world_workspace_bytes(int B, int64_t y_len_max) {
  if (B <= 0 || y_len_max < 0) return 0;
  const long long Yp = (y_len_max + 31) / 32 * 32;
  return static_cast<int64_t>(align256(static_cast<size_t>(B) * 16) + align256(static_cast<size_t>(B) * Yp * 4) +
                              static_cast<size_t>(B) * Yp * 8);
}

int world_noise(double* out, int64_t n, cudaStream_t stream) {
  if (out == nullptr || n < 0) return fail(V100_E_INVALID, "world_noise: null output or negative length");
  if (n == 0) return 0;
  world_noise_kernel<<<dim3(1), dim3(32), 0, stream>>>(out, static_cast<long long>(n));
  V100_CUDA(cudaGetLastError());
  return 0;
}

static WorldIn make_in(const float* f0, int64_t f0_sb, int64_t f0_st, const float* logspc, int64_t sp_sb,
                       int64_t sp_st, int64_t sp_sk, const float* codeap, int64_t ap_sb, int64_t ap_st,
                       const int32_t* frame_len, int T) {
  WorldIn in;
  in.f0 = f0;
  in.f0_sb = f0_sb;
  in.f0_st = f0_st;
  in.sp = logspc;
  in.sp_sb = sp_sb;
  in.sp_st = sp_st;
  in.sp_sk = sp_sk;
  in.ap = codeap;
  in.ap_sb = ap_sb;
  in.ap_st = ap_st;
  in.frame_len = frame_len;
  in.T = T;
  return in;
}

int world_timebase(const float* f0, int64_t f0_sb, int64_t f0_st, const float* logspc, int64_t sp_sb, int64_t sp_st,
                   int64_t sp_sk, const float* codeap, int64_t ap_sb, int64_t ap_st, const int32_t* frame_len, int B,
                   int T, void* workspace, int32_t* wav_len, int32_t* status, cudaStream_t stream) {
  const WorldIn in = make_in(f0, f0_sb, f0_st, logspc, sp_sb, sp_st, sp_sk, codeap, ap_sb, ap_st, frame_len, T);
  if (int rc = check_in(in, B, "world_timebase")) return rc;
  if (workspace == nullptr || wav_len == nullptr || status == nullptr)
    return fail(V100_E_INVALID, "world_timebase: null workspace / wav_len / status");
  return launch_timebase(in, B, workspace, wav_len, status, stream);
}

int world_synthesize(const float* f0, int64_t f0_sb, int64_t f0_st, const float* logspc, int64_t sp_sb,
                     int64_t sp_st, int64_t sp_sk, const float* codeap, int64_t ap_sb, int64_t ap_st,
                     const int32_t* frame_len, int B, int T, const double* noise, int64_t noise_len, void* workspace,
                     float* wav, int64_t wav_pitch, int32_t* wav_len, int32_t* status, cudaStream_t stream) {
  const WorldIn in = make_in(f0, f0_sb, f0_st, logspc, sp_sb, sp_st, sp_sk, codeap, ap_sb, ap_st, frame_len, T);
  if (int rc = check_in(in, B, "world_synthesize")) return rc;
  if (workspace == nullptr || wav == nullptr || wav_len == nullptr || status == nullptr || noise == nullptr)
    return fail(V100_E_INVALID, "world_synthesize: null noise / workspace / wav / wav_len / status");
  const long long Yp = ws_pitch(T);
  if (wav_pitch < Yp || wav_pitch <= 0)
    return fail(V100_E_INVALID, "world_synthesize: wav_pitch %lld < 160 T = %lld", (long long)wav_pitch, Yp);
  if (noise_len < Yp)
    return fail(V100_E_INVALID, "world_synthesize: noise table of %lld values < 160 T = %lld", (long long)noise_len, Yp);
  if (int rc = launch_timebase(in, B, workspace, wav_len, status, stream)) return rc;
  V100_CUDA(cudaFuncSetAttribute(world_synth_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSynSmem));
  SynthParams p;
  p.in = in;
  p.ws = ws_carve(workspace, B, Yp);
  p.Yp = Yp;
  p.noise = noise;
  p.wav = wav;
  p.wav_pitch = wav_pitch;
  const long long tiles = (wav_pitch + kTile - 1) / kTile;
  if (tiles > 0x7fffffffLL || B > 65535) return fail(V100_E_UNSUPPORTED, "world_synthesize: grid too large");
  world_synth_kernel<<<dim3(static_cast<unsigned>(tiles), B), dim3(kSynThreads), kSynSmem, stream>>>(p);
  V100_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace v100
