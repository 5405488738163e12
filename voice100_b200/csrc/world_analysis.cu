// WORLD analysis on the device: 16 kHz PCM -> f0 / log-spectrum / coded aperiodicity (v100_world_analyze in
// include/v100.h).  Restates what the reference's WORLDVocoder.encode (voice100/vocoder.py:66-88) runs through pyworld
// one utterance at a time: Dio, StoneMask, CheapTrick (fft_size 512), D4C and CodeAperiodicity.  The contract is
// oracle/world_analysis.py (float64 numpy); parity with pyworld itself is unverified (DESIGN.md section 3.10).
//
// Kernels, in stream order (all float64; no float atomics; every output depends only on its utterance):
//  - wa_prep:     one CTA per utterance: length, status, and the mean as a fixed tree (256 strided partial sums in
//                 sample order, halved to one) -- the restatement's mean_fixed, bit for bit.
//  - wa_lowcut:   one CTA per (1024-sample tile, utterance): the 641-tap low-cut filter over [-160, L + 160).
//  - wa_bands:    one CTA per (1024-sample tile, utterance, band), run twice: pass 0 counts the events of the four
//                 series of the tile, pass 1 recomputes the band and writes the refined crossings at the offsets that
//                 wa_scan derived from the counts, so each series is a sorted list in a workspace sized from shapes.
//  - wa_contour:  one thread per (frame, utterance): interp1 of each series by binary search, the band candidates and
//                 scores, the best band.
//  - wa_fix:      one thread per utterance: FixF0Contour, sequential over frames.
//  - wa_stonemask, wa_cheaptrick, wa_lovetrain, wa_d4c: one CTA per (frame, utterance), radix-2 FFTs of up to 2048
//                 points in shared memory.  wa_draws runs between them: a per-utterance prefix sum of each frame's
//                 dither draws gives its offset into WORLD's randn table (v100_world_noise).
// The DIO filters, crossings and contour use explicit _rn intrinsics (no FMA contraction) in the restatement's order,
// so the raw and fixed f0 contours are bit-identical to it; StoneMask onwards differ from it by float64 rounding only.
#include <math.h>

#include "common.cuh"
#include "host.h"

namespace v100 {

namespace {

constexpr int kFs = 16000;
constexpr int kHop = 160;
constexpr int kBins = 257;
constexpr int kBands = 7;
constexpr int kSeries = 4 * kBands;
constexpr int kLowHalf = 320;                              // low-cut filter: 641 taps
constexpr int kHpExt = 160;                                // hp is kept over [-160, L + 160)
constexpr int kTile = 1024;
constexpr int kThreads = 256;
constexpr int kMinFrames = 4;
constexpr double kPi = 3.1415926535897932384;
constexpr double kEps = 1e-12;
constexpr double kDblEps = 2.220446049250313e-16;
constexpr double kCtFloor = 3.0 * kFs / (512 - 3.0);       // CheapTrick's f0 floor for fft_size 512
constexpr double kCodeapUnvoiced = -8.6856974912498e-12;   // 20 log10(1 - 1e-12)
constexpr int kDrawsPerFrame = 5290;                       // LoveTrain (<= 1201) + D4C (<= 3 * 1363) per frame
__constant__ int kBandHalf[kBands] = {80, 56, 40, 28, 20, 14, 10};   // round(fs / boundary / 2)
__constant__ int kBandOff[kBands] = {641, 961, 1185, 1345, 1457, 1537, 1593};
__constant__ double kBoundary[kBands] = {100.40916292848975, 142.0, 200.8183258569795, 284.0, 401.636651713959,
                                      568.0, 803.273303427918};   // 71 2^((i + 1) / 2), as Python rounds it

__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double ddiv(double a, double b) { return __ddiv_rn(a, b); }
__device__ __forceinline__ int mround(double x) { return x >= 0 ? static_cast<int>(x + 0.5) : static_cast<int>(x - 0.5); }
__device__ __forceinline__ double frame_time(int t) { return ddiv(dmul(static_cast<double>(t), 10.0), 1000.0); }

struct Ws {
  int32_t* head;    // [B][4]: status, L, frames
  double* mean;     // [B]
  double* hp;       // [B][Lh]
  int32_t* cnt;     // [B][28][tiles]   event counts, then exclusive offsets
  int32_t* tot;     // [B][28]
  double* ev;       // [B][28][E]       refined crossings
  double* cand;     // [B][7][Tw]
  double* best;     // [B][Tw]
  double* fix;      // [B][2][Tw]
  double* f0d;      // [B][Tw]          DIO's fixed contour
  double* f0s;      // [B][Tw]          StoneMask
  double* ratio;    // [B][Tw]          LoveTrain
  int64_t* ct_off;  // [B][Tw]
  int64_t* lt_off;  // [B][Tw]
  int64_t* d4_off;  // [B][Tw]          -1: not analysed
};

struct Dims {
  int B, T, Tw, tiles;
  long long Lmax, Lh, E;
};

__host__ __device__ inline size_t al(size_t x) { return (x + 255) & ~static_cast<size_t>(255); }

__host__ __device__ inline Dims make_dims(int B, long long Lmax, int T) {
  Dims d;
  d.B = B;
  d.T = T;
  d.Lmax = Lmax;
  d.Tw = static_cast<int>(Lmax / kHop + 1);
  d.tiles = static_cast<int>((Lmax + kTile - 1) / kTile);
  d.Lh = Lmax + 2 * kHpExt;
  d.E = Lmax / 2 + 1;
  return d;
}

__host__ __device__ inline size_t carve(void* base, const Dims& d, Ws* w) {
  uint8_t* p = static_cast<uint8_t*>(base);
  size_t o = 0;
  const size_t B = d.B, Tw = d.Tw;
  auto take = [&](size_t bytes) {
    uint8_t* r = p == nullptr ? nullptr : p + o;
    o += al(bytes);
    return r;
  };
  w->head = reinterpret_cast<int32_t*>(take(B * 16));
  w->mean = reinterpret_cast<double*>(take(B * 8));
  w->hp = reinterpret_cast<double*>(take(B * d.Lh * 8));
  w->cnt = reinterpret_cast<int32_t*>(take(B * kSeries * static_cast<size_t>(d.tiles) * 4));
  w->tot = reinterpret_cast<int32_t*>(take(B * kSeries * 4));
  w->ev = reinterpret_cast<double*>(take(B * kSeries * static_cast<size_t>(d.E) * 8));
  w->cand = reinterpret_cast<double*>(take(B * kBands * Tw * 8));
  w->best = reinterpret_cast<double*>(take(B * Tw * 8));
  w->fix = reinterpret_cast<double*>(take(B * 2 * Tw * 8));
  w->f0d = reinterpret_cast<double*>(take(B * Tw * 8));
  w->f0s = reinterpret_cast<double*>(take(B * Tw * 8));
  w->ratio = reinterpret_cast<double*>(take(B * Tw * 8));
  w->ct_off = reinterpret_cast<int64_t*>(take(B * Tw * 8));
  w->lt_off = reinterpret_cast<int64_t*>(take(B * Tw * 8));
  w->d4_off = reinterpret_cast<int64_t*>(take(B * Tw * 8));
  return o;
}

struct In {
  const void* wav;
  int i16;
  long long pitch;
  const int32_t* len;
  const double* taps;
  const double* noise;
};

struct Out {
  float* f0;
  float* sp;
  float* ap;
  int32_t* frame_len;
  int32_t* status;
};

__device__ __forceinline__ double sample(const In& in, int b, long long i) {
  return in.i16 ? static_cast<double>(static_cast<const int16_t*>(in.wav)[b * in.pitch + i]) / 32768.0
                : static_cast<double>(static_cast<const float*>(in.wav)[b * in.pitch + i]);
}

// ------------------------------------------------------------------------------------------------ block helpers

__device__ double block_sum(double v, double* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double s = 0.0;
  for (int w = 0; w < kThreads / 32; ++w) s += red[w];
  return s;
}

struct dc {
  double x, y;
};
__device__ __forceinline__ dc cmul(dc a, dc b) { return dc{a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x}; }

// tw[k] = exp(-2 pi i k / n), k < n / 2
__device__ void make_twiddles(dc* tw, int logn) {
  const int n = 1 << logn;
  for (int k = threadIdx.x; k < n / 2; k += kThreads) {
    double s, c;
    sincospi(-2.0 * k / n, &s, &c);
    tw[k] = dc{c, s};
  }
}

// in-place forward complex DFT of a[0, 2^logn) by the CTA (iterative radix 2)
__device__ void fft(dc* a, const dc* tw, int logn) {
  const int n = 1 << logn;
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += kThreads) {
    const int j = static_cast<int>(__brev(static_cast<unsigned>(i)) >> (32 - logn));
    if (i < j) {
      const dc t = a[i];
      a[i] = a[j];
      a[j] = t;
    }
  }
  __syncthreads();
  for (int s = 1; s <= logn; ++s) {
    const int half = 1 << (s - 1);
    for (int k = threadIdx.x; k < n / 2; k += kThreads) {
      const int pos = k & (half - 1);
      const int i = ((k >> (s - 1)) << s) + pos, j = i + half;
      const dc t = cmul(tw[pos << (logn - s)], a[j]);
      const dc u = a[i];
      a[i] = dc{u.x + t.x, u.y + t.y};
      a[j] = dc{u.x - t.x, u.y - t.y};
    }
    __syncthreads();
  }
}

// WORLD's DCCorrection, in place on p[0, n / 2]
__device__ void dc_correction(double* p, double f0, int n) {
  const int upper = 2 + static_cast<int>(f0 * n / kFs);
  const double df = static_cast<double>(kFs) / n;
  double v = 0.0;
  const int i = threadIdx.x;
  if (i < upper - 1) {
    const double q = (static_cast<double>(i) * kFs / n - f0) / (-df);
    const int k = static_cast<int>(q);
    v = p[i] + (p[k] + (p[k + 1] - p[k]) * (q - k));
  }
  __syncthreads();
  if (i < upper - 1) p[i] = v;
  __syncthreads();
}

// WORLD's LinearSmoothing of p[0, n / 2] into out (may alias p); seg: scratch of n / 2 + 2 bnd + 1 doubles
__device__ void linear_smoothing(const double* p, double width, int n, double* seg, double* out) {
  const int half = n / 2;
  const int bnd = static_cast<int>(width * n / kFs) + 1;
  const int nm = half + 2 * bnd + 1;
  for (int i = threadIdx.x; i < nm; i += kThreads) {
    const double m = i < bnd ? p[bnd - i] : (i < half + bnd ? p[i - bnd] : p[half - (i - (half + bnd))]);
    seg[i] = m * kFs / n;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double run = seg[0];
    for (int i = 1; i < nm; ++i) {
      run = run + seg[i];
      seg[i] = run;
    }
  }
  __syncthreads();
  const double df = static_cast<double>(kFs) / n;
  const double origin = -(bnd - 0.5) * kFs / n;
  for (int i = threadIdx.x; i <= half; i += kThreads) {
    const double fa = static_cast<double>(i) / n * kFs - width / 2.0;
    double lv[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const double q = ((u ? fa + width : fa) - origin) / df;
      const int k = static_cast<int>(q);
      const double dy = k < nm - 1 ? seg[k + 1] - seg[k] : 0.0;
      lv[u] = seg[k] + dy * (q - k);
    }
    out[i] = (lv[1] - lv[0]) / width;
  }
  __syncthreads();
}

// WORLD's GetWindowedWaveform (D4C): ratio periods of a Blackman or Hann window around t, dither added, windowed DC
// removed -> wf[0, 2 h + 1); returns h
__device__ int windowed(const In& in, int b, int L, double t, double f0, double ratio, bool blackman,
                        const double* dither, double* wf, double* red) {
  const int h = mround(ratio * kFs / f0 / 2.0);
  const int origin = mround(t * kFs + 0.001);
  double s1 = 0.0, s2 = 0.0;
  for (int i = threadIdx.x; i <= 2 * h; i += kThreads) {
    const int bi = i - h;
    const double pos = (2.0 * bi / ratio) / kFs;
    const double w = blackman ? 0.42 + 0.5 * cos(kPi * pos * f0) + 0.08 * cos(kPi * pos * f0 * 2)
                              : 0.5 * cos(kPi * pos * f0) + 0.5;
    const int si = min(L - 1, max(0, origin + bi));
    const double v = sample(in, b, si) * w + dither[i] * kEps;
    wf[i] = v;
    s1 += v;
    s2 += w;
  }
  const double coef = block_sum(s1, red) / block_sum(s2, red);
  for (int i = threadIdx.x; i <= 2 * h; i += kThreads) {
    const int bi = i - h;
    const double pos = (2.0 * bi / ratio) / kFs;
    const double w = blackman ? 0.42 + 0.5 * cos(kPi * pos * f0) + 0.08 * cos(kPi * pos * f0 * 2)
                              : 0.5 * cos(kPi * pos * f0) + 0.5;
    wf[i] -= w * coef;
  }
  __syncthreads();
  return h;
}

// ------------------------------------------------------------------------------------------------ DIO

__global__ void __launch_bounds__(kThreads) wa_prep(const In in, Dims d, Ws ws, Out out) {
  __shared__ double part[kThreads];
  __shared__ int bad;
  const int b = blockIdx.x, tid = threadIdx.x;
  long long L = __ldg(in.len + b);
  L = L < 0 ? 0 : (L > d.Lmax ? d.Lmax : L);
  const int frames = static_cast<int>(L / kHop + 1);
  if (tid == 0) bad = 0;
  __syncthreads();
  double s = 0.0;
  bool nf = false;
  for (long long i = tid; i < L; i += kThreads) {
    const double v = sample(in, b, i);
    nf |= !isfinite(v);
    s = dadd(s, v);
  }
  if (nf) bad = 1;
  part[tid] = s;
  __syncthreads();
  for (int o = kThreads / 2; o > 0; o >>= 1) {
    if (tid < o) part[tid] = dadd(part[tid], part[tid + o]);
    __syncthreads();
  }
  if (tid == 0) {
    const int st = frames < kMinFrames ? V100_WORLD_SHORT : (bad ? V100_WORLD_NONFINITE : V100_WORLD_OK);
    ws.head[4 * b] = st;
    ws.head[4 * b + 1] = static_cast<int32_t>(L);
    ws.head[4 * b + 2] = st == V100_WORLD_OK ? frames : 0;
    ws.mean[b] = st == V100_WORLD_OK ? ddiv(part[0], static_cast<double>(L)) : 0.0;
    out.frame_len[b] = st == V100_WORLD_OK ? frames : 0;
    out.status[b] = st;
  }
}

// hp[m] = sum_j h[j] y[m - 160 + 320 - j], y = x - mean inside [0, L), 0 outside
__global__ void __launch_bounds__(kThreads) wa_lowcut(const In in, Dims d, Ws ws) {
  __shared__ double taps[2 * kLowHalf + 1];
  __shared__ double ys[kTile + 4 * kLowHalf];
  const int b = blockIdx.y, tid = threadIdx.x;
  if (ws.head[4 * b] != V100_WORLD_OK) return;
  const long long L = ws.head[4 * b + 1];
  const long long m0 = static_cast<long long>(blockIdx.x) * kTile;
  if (m0 >= L + 2 * kHpExt) return;
  const double mean = ws.mean[b];
  for (int j = tid; j < 2 * kLowHalf + 1; j += kThreads) taps[j] = in.taps[j];
  // ys[k] = y[m0 - 160 - 320 + k]
  const long long y0 = m0 - kHpExt - kLowHalf;
  for (int k = tid; k < kTile + 4 * kLowHalf; k += kThreads) {
    const long long n = y0 + k;
    ys[k] = (n >= 0 && n < L) ? dsub(sample(in, b, n), mean) : 0.0;
  }
  __syncthreads();
  double* hp = ws.hp + b * d.Lh;
  for (int r = tid; r < kTile; r += kThreads) {
    const long long m = m0 + r;
    if (m >= L + 2 * kHpExt) break;
    // y index n - 160 + 320 - j relative to y0: r + 640 - j
    double acc = 0.0;
    for (int j = 0; j <= 2 * kLowHalf; ++j) acc = dadd(acc, dmul(taps[j], ys[r + 2 * kLowHalf - j]));
    hp[m] = acc;
  }
}

// Events of one band in one tile.  PASS 0 writes counts, PASS 1 the refined crossings at their offsets.
template <int PASS>
__global__ void __launch_bounds__(kThreads) wa_bands(const In in, Dims d, Ws ws) {
  __shared__ double taps[4 * 80];
  __shared__ double hs[kTile + 2 + 4 * 80 + 2];
  __shared__ double xs[kTile + 2];
  __shared__ int wsum[kThreads / 32][4];
  const int b = blockIdx.y, band = blockIdx.z, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (ws.head[4 * b] != V100_WORLD_OK) return;
  const long long L = ws.head[4 * b + 1];
  const long long t0 = static_cast<long long>(blockIdx.x) * kTile;
  int32_t* cnt = ws.cnt + (static_cast<long long>(b) * kSeries + 4 * band) * d.tiles + blockIdx.x;
  if (t0 >= L) {
    if (PASS == 0 && tid < 4) cnt[tid * d.tiles] = 0;
    return;
  }
  const int hh = kBandHalf[band], M = 4 * hh;
  for (int j = tid; j < M; j += kThreads) taps[j] = in.taps[kBandOff[band] + j];
  // band[i] = sum_j w[j] hp(i + 2 hh - j); xs[k] = band[t0 - 1 + k]; hs[k] = hp(t0 - 1 - 2 hh + 1 + k)
  const long long h0 = t0 - 2 * hh;
  const int nh = kTile + 2 + M;
  const double* hp = ws.hp + b * d.Lh;
  for (int k = tid; k < nh; k += kThreads) {
    const long long n = h0 + k;                            // hp sample n lives at n + 160
    hs[k] = (n >= -kHpExt && n < L + kHpExt) ? hp[n + kHpExt] : 0.0;
  }
  __syncthreads();
  for (int k = tid; k < kTile + 2; k += kThreads) {
    const long long i = t0 - 1 + k;
    double acc = 0.0;
    if (i >= 0 && i < L) {
      // hp(i + 2 hh - j) = hs[i + 2 hh - j - h0] = hs[k - 1 + 4 hh - j]
      for (int j = 0; j < M; ++j) acc = dadd(acc, dmul(taps[j], hs[k - 1 + M - j]));
    }
    xs[k] = acc;
  }
  __syncthreads();
  // thread owns e = t0 + 4 tid + u
  double fe[4][4];
  int c[4] = {0, 0, 0, 0};
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const long long e = t0 + 4 * tid + u;
    if (e < 1 || e >= L || e >= t0 + kTile) continue;
    const int k = static_cast<int>(e - t0) + 1;             // xs index of e
    const double a = xs[k - 1], x = xs[k];
    if (0.0 < a && x <= 0.0) fe[0][c[0]++] = dsub(static_cast<double>(e), ddiv(a, dsub(x, a)));
    const double na = -a, nx = -x;
    if (0.0 < na && nx <= 0.0) fe[1][c[1]++] = dsub(static_cast<double>(e), ddiv(na, dsub(nx, na)));
    if (e <= L - 2) {
      const double xn = xs[k + 1];
      const double d0 = dsub(-xs[k - 1], -x), d1 = dsub(-x, -xn);
      if (0.0 < d0 && d1 <= 0.0) fe[2][c[2]++] = dsub(static_cast<double>(e), ddiv(d0, dsub(d1, d0)));
      const double m0 = -d0, m1 = -d1;
      if (0.0 < m0 && m1 <= 0.0) fe[3][c[3]++] = dsub(static_cast<double>(e), ddiv(m0, dsub(m1, m0)));
    }
  }
  int incl[4];
#pragma unroll
  for (int s = 0; s < 4; ++s) {
    incl[s] = c[s];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int up = __shfl_up_sync(0xffffffffu, incl[s], o);
      if (lane >= o) incl[s] += up;
    }
    if (lane == 31) wsum[warp][s] = incl[s];
  }
  __syncthreads();
  if (PASS == 0) {
    if (tid < 4) {
      int t = 0;
      for (int w = 0; w < kThreads / 32; ++w) t += wsum[w][tid];
      cnt[tid * d.tiles] = t;
    }
    return;
  }
#pragma unroll
  for (int s = 0; s < 4; ++s) {
    int base = cnt[s * d.tiles];
    for (int w = 0; w < warp; ++w) base += wsum[w][s];
    base += incl[s] - c[s];
    double* ev = ws.ev + (static_cast<long long>(b) * kSeries + 4 * band + s) * d.E;
    for (int q = 0; q < c[s]; ++q) ev[base + q] = fe[s][q];
  }
}

// counts -> exclusive offsets and totals, per (utterance, series)
__global__ void wa_scan(Dims d, Ws ws) {
  const int b = blockIdx.x, s = threadIdx.x;
  if (s >= kSeries || ws.head[4 * b] != V100_WORLD_OK) return;
  int32_t* c = ws.cnt + (static_cast<long long>(b) * kSeries + s) * d.tiles;
  int run = 0;
  for (int i = 0; i < d.tiles; ++i) {
    const int v = c[i];
    c[i] = run;
    run += v;
  }
  ws.tot[b * kSeries + s] = run;
}

__device__ __forceinline__ double ev_loc(const double* e, long long k) {
  return ddiv(ddiv(dadd(e[k], e[k + 1]), 2.0), static_cast<double>(kFs));
}

// interp1 (histc) of one series' intervals at xi
__device__ double series_at(const double* e, int nev, double xi) {
  const int n = nev - 1;                                     // knots
  int lo = 0, hi = n;                                        // first knot with loc > xi
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (ev_loc(e, mid) <= xi) lo = mid + 1;
    else hi = mid;
  }
  int k = lo - 1;
  k = k < 0 ? 0 : (k > n - 2 ? n - 2 : k);
  const double xk = ev_loc(e, k), xk1 = ev_loc(e, k + 1);
  const double yk = ddiv(static_cast<double>(kFs), dsub(e[k + 1], e[k]));
  const double yk1 = ddiv(static_cast<double>(kFs), dsub(e[k + 2], e[k + 1]));
  const double s = ddiv(dsub(xi, xk), dsub(xk1, xk));
  return dadd(yk, dmul(s, dsub(yk1, yk)));
}

__global__ void __launch_bounds__(128) wa_contour(Dims d, Ws ws) {
  const int b = blockIdx.y;
  const int t = blockIdx.x * 128 + threadIdx.x;
  if (ws.head[4 * b] != V100_WORLD_OK) return;
  const int T = ws.head[4 * b + 2];
  if (t >= T) return;
  const double xi = frame_time(t);
  double best = 0.0, bscore = 0.0;
  for (int band = 0; band < kBands; ++band) {
    const int32_t* tot = ws.tot + b * kSeries + 4 * band;
    double c = 0.0, score = 100000.0;
    if (tot[0] - 1 >= 3 && tot[1] - 1 >= 3 && tot[2] - 1 >= 3 && tot[3] - 1 >= 3) {
      double v[4];
#pragma unroll
      for (int s = 0; s < 4; ++s)
        v[s] = series_at(ws.ev + (static_cast<long long>(b) * kSeries + 4 * band + s) * d.E, tot[s], xi);
      c = ddiv(dadd(dadd(dadd(v[0], v[1]), v[2]), v[3]), 4.0);
      const double q0 = dsub(v[0], c), q1 = dsub(v[1], c), q2 = dsub(v[2], c), q3 = dsub(v[3], c);
      const double sd = __dsqrt_rn(ddiv(dadd(dadd(dadd(dmul(q0, q0), dmul(q1, q1)), dmul(q2, q2)), dmul(q3, q3)), 3.0));
      score = ddiv(sd, c);
      const double bd = kBoundary[band];
      if (c > bd || c < ddiv(bd, 2.0) || c > 800.0 || c < 71.0) {
        c = 0.0;
        score = 100000.0;
      }
    }
    ws.cand[(static_cast<long long>(b) * kBands + band) * d.Tw + t] = c;
    if (band == 0 || bscore > score) {
      bscore = score;
      best = c;
    }
  }
  ws.best[static_cast<long long>(b) * d.Tw + t] = best;
}

__device__ double select_best(double cur, double past, const double* cand, long long Tw, int idx) {
  const double ref = ddiv(dsub(dmul(cur, 3.0), past), 2.0);
  double best = cand[idx], err = fabs(dsub(ref, best));
  for (int i = 1; i < kBands; ++i) {
    const double c = cand[i * Tw + idx], e = fabs(dsub(ref, c));
    if (e < err) {
      err = e;
      best = c;
    }
  }
  return fabs(dsub(1.0, ddiv(best, ref))) > 0.1 ? 0.0 : best;
}

// FixF0Contour, one thread per utterance
__global__ void wa_fix(Dims d, Ws ws) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= d.B || ws.head[4 * b] != V100_WORLD_OK) return;
  const int T = ws.head[4 * b + 2];
  const long long Tw = d.Tw;
  const double* best = ws.best + b * Tw;
  const double* cand = ws.cand + b * kBands * Tw;
  double* s1 = ws.fix + 2 * b * Tw;
  double* s2 = s1 + Tw;
  double* q = ws.f0d + b * Tw;
  constexpr int v = 3;
  auto base = [&](int i) { return (i < v || i >= T - v) ? 0.0 : best[i]; };
  for (int i = 0; i < T; ++i) {
    if (i < v) {
      s1[i] = 0.0;
      continue;
    }
    const double f = base(i), p = base(i - 1);
    s1[i] = fabs(ddiv(dsub(f, p), dadd(kEps, f))) < 0.1 ? f : 0.0;
  }
  for (int i = 0; i < T; ++i) {
    double r = s1[i];
    if (i >= 1 && i < T - 1 && (s1[i - 1] == 0.0 || s1[i] == 0.0 || s1[i + 1] == 0.0)) r = 0.0;
    s2[i] = r;
    q[i] = r;
  }
  auto find_neg = [&](int i0) {
    for (int i = i0; i < T; ++i)
      if (s2[i] == 0.0 && s2[i - 1] != 0.0) return i - 1;
    return -1;
  };
  auto find_pos = [&](int i0) {
    for (int i = i0; i >= 1; --i)
      if (s2[i - 1] == 0.0 && s2[i] != 0.0) return i;
    return -1;
  };
  for (int start = find_neg(1); start >= 0;) {
    const int nxt = find_neg(start + 2);
    const int limit = nxt < 0 ? T - 1 : nxt;
    for (int j = start; j < limit; ++j) {
      q[j + 1] = select_best(q[j], q[j - 1], cand, Tw, j + 1);
      if (q[j + 1] == 0.0) break;
    }
    start = nxt;
  }
  for (int p = find_pos(T - 1); p >= 0;) {
    const int prv = find_pos(p - 1);
    const int limit = prv < 0 ? 1 : prv;
    for (int j = p; j > limit; --j) {
      q[j - 1] = select_best(q[j], q[j + 1], cand, Tw, j - 1);
      if (q[j - 1] == 0.0) break;
    }
    p = prv;
  }
}

// ------------------------------------------------------------------------------------------------ StoneMask

__device__ double fix_f0(const double* pw, const double* num, int nfft, double f, int nh) {
  double n = 0.0, dd = 0.0;
  for (int k = 0; k < nh; ++k) {
    const int idx = mround(f * nfft / kFs * (k + 1));
    const double ifr = pw[idx] == 0.0 ? 0.0 : static_cast<double>(idx) * kFs / nfft + num[idx] / pw[idx] * kFs / 2.0 / kPi;
    const double amp = sqrt(pw[idx]);
    n += amp * ifr;
    dd += amp * (k + 1.0);
  }
  return n / (dd + kEps);
}

__global__ void __launch_bounds__(kThreads) wa_stonemask(const In in, Dims d, Ws ws, Out out) {
  extern __shared__ __align__(16) uint8_t smem[];
  dc* a = reinterpret_cast<dc*>(smem);                  // [2048]
  dc* tw = a + 2048;                                    // [1024]
  double* win = reinterpret_cast<double*>(tw + 1024);   // [2048]: window, then power spectrum
  double* num = win + 2048;                             // [1025]
  const int t = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const bool ok = ws.head[4 * b] == V100_WORLD_OK && t < ws.head[4 * b + 2];
  const double f0 = ok ? ws.f0d[static_cast<long long>(b) * d.Tw + t] : 0.0;
  float* fo = out.f0 + static_cast<long long>(b) * d.T + t;
  if (f0 <= 40.0 || f0 > kFs / 12.0) {
    if (tid == 0) {
      *fo = 0.0f;
      if (ok) ws.f0s[static_cast<long long>(b) * d.Tw + t] = 0.0;
    }
    return;
  }
  const int L = ws.head[4 * b + 1];
  const double tt = frame_time(t);
  const int h = static_cast<int>(1.5 * kFs / f0 + 1.0);
  const int n = 2 * h + 1;
  const double wlen = (2.0 * h + 1.0) / kFs;
  const int logn = 2 + static_cast<int>(log(2.0 * h + 1.0) / log(2.0));
  const int nfft = 1 << logn;
  const int base = mround((tt + (-h) / static_cast<double>(kFs)) * kFs + 0.001);
  make_twiddles(tw, logn);
  for (int i = tid; i < n; i += kThreads) {
    const double tmp = (base + i - 1.0) / kFs - tt;
    win[i] = 0.42 + 0.5 * cos(2.0 * kPi * tmp / wlen) + 0.08 * cos(4.0 * kPi * tmp / wlen);
  }
  __syncthreads();
  for (int i = tid; i < nfft; i += kThreads) {
    dc v{0.0, 0.0};
    if (i < n) {
      const double dw = i == 0 ? -win[1] / 2.0 : (i == n - 1 ? win[n - 2] / 2.0 : -(win[i + 1] - win[i - 1]) / 2.0);
      const double x = sample(in, b, min(L - 1, max(0, base + i - 1)));
      v = dc{x * win[i], x * dw};
    }
    a[i] = v;
  }
  fft(a, tw, logn);
  for (int k = tid; k <= nfft / 2; k += kThreads) {
    const dc z = a[k], zn = a[(nfft - k) & (nfft - 1)];
    const dc m{0.5 * (z.x + zn.x), 0.5 * (z.y - zn.y)};
    const dc w{0.5 * (z.y + zn.y), -0.5 * (z.x - zn.x)};
    num[k] = m.x * w.y - m.y * w.x;
    win[k] = m.x * m.x + m.y * m.y;
  }
  __syncthreads();
  if (tid == 0) {
    const double f1 = fix_f0(win, num, nfft, f0, 2);
    double f = (f1 <= 0.0 || f1 > 2.0 * f0) ? 0.0 : fix_f0(win, num, nfft, f1, min(static_cast<int>(kFs / 2.0 / f1), 6));
    if (fabs(f - f0) > f0 * 0.2) f = f0;
    ws.f0s[static_cast<long long>(b) * d.Tw + t] = f;
    *fo = static_cast<float>(f);
  }
}

// ------------------------------------------------------------------------------------------------ dither offsets

__device__ __forceinline__ int ct_draws(double f0) {
  const double f = f0 <= kCtFloor ? 500.0 : f0;
  return 2 * mround(1.5 * kFs / f) + 1 + kBins;
}
__device__ __forceinline__ int d4c_draws(double f0) { return 3 * (2 * mround(2.0 * kFs / fmax(47.0, f0)) + 1); }

// PHASE 0: CheapTrick and LoveTrain offsets; PHASE 1: D4C offsets (after LoveTrain), -1 for frames not analysed
template <int PHASE>
__global__ void wa_draws(Dims d, Ws ws) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= d.B || ws.head[4 * b] != V100_WORLD_OK) return;
  const int T = ws.head[4 * b + 2];
  const long long o = static_cast<long long>(b) * d.Tw;
  const double* f0 = ws.f0s + o;
  if (PHASE == 0) {
    long long ct = 0, lt = 0;
    for (int t = 0; t < T; ++t) {
      ws.ct_off[o + t] = ct;
      ws.lt_off[o + t] = lt;
      ct += ct_draws(f0[t]);
      if (f0[t] != 0.0) lt += 2 * mround(1.5 * kFs / fmax(f0[t], 40.0)) + 1;
    }
    ws.d4_off[o] = lt;                                    // where D4C's own draws start (read back by PHASE 1)
  } else {
    long long at = ws.d4_off[o];
    for (int t = 0; t < T; ++t) {
      const bool live = f0[t] != 0.0 && ws.ratio[o + t] > 0.85;
      ws.d4_off[o + t] = live ? at : -1;
      if (live) at += d4c_draws(f0[t]);
    }
  }
}

// ------------------------------------------------------------------------------------------------ CheapTrick

__global__ void __launch_bounds__(kThreads) wa_cheaptrick(const In in, Dims d, Ws ws, Out out) {
  __shared__ dc a[512];
  __shared__ dc tw[256];
  __shared__ double p[kBins];
  __shared__ double seg[kBins + 2 * 64 + 8];
  __shared__ double red[kThreads / 32];
  const int t = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  float* row = out.sp + (static_cast<long long>(b) * d.T + t) * kBins;
  const bool ok = ws.head[4 * b] == V100_WORLD_OK && t < ws.head[4 * b + 2];
  if (!ok) {
    for (int k = tid; k < kBins; k += kThreads) row[k] = 0.0f;
    return;
  }
  const int L = ws.head[4 * b + 1];
  const long long o = static_cast<long long>(b) * d.Tw + t;
  const double f0 = ws.f0s[o];
  const double fc = f0 <= kCtFloor ? 500.0 : f0;
  const double* dither = in.noise + ws.ct_off[o];
  const double tt = frame_time(t);
  const int h = mround(1.5 * kFs / fc);
  const int origin = mround(tt * kFs + 0.001);
  make_twiddles(tw, 9);
  double ww = 0.0;
  for (int i = tid; i <= 2 * h; i += kThreads) {
    const double w = 0.5 * cos(kPi * ((i - h) / 1.5 / kFs) * fc) + 0.5;
    ww += w * w;
  }
  const double norm = sqrt(block_sum(ww, red));
  double s1 = 0.0, s2 = 0.0;
  for (int i = tid; i < 512; i += kThreads) {
    double v = 0.0;
    if (i <= 2 * h) {
      const double w = (0.5 * cos(kPi * ((i - h) / 1.5 / kFs) * fc) + 0.5) / norm;
      v = sample(in, b, min(L - 1, max(0, origin + i - h))) * w + dither[i] * kEps;
      s1 += v;
      s2 += w;
    }
    a[i] = dc{v, 0.0};
  }
  const double coef = block_sum(s1, red) / block_sum(s2, red);
  for (int i = tid; i <= 2 * h; i += kThreads) {
    const double w = (0.5 * cos(kPi * ((i - h) / 1.5 / kFs) * fc) + 0.5) / norm;
    a[i].x -= w * coef;
  }
  fft(a, tw, 9);
  for (int k = tid; k < kBins; k += kThreads) p[k] = a[k].x * a[k].x + a[k].y * a[k].y;
  __syncthreads();
  dc_correction(p, fc, 512);
  linear_smoothing(p, fc * 2.0 / 3.0, 512, seg, p);
  const double q1 = -0.15;
  for (int k = tid; k < 512; k += kThreads) {
    const int m = k <= 256 ? k : 512 - k;
    a[k] = dc{log(p[m] + fabs(dither[2 * h + 1 + m]) * kDblEps), 0.0};
  }
  fft(a, tw, 9);
  for (int k = tid; k <= 256; k += kThreads) {
    const int m = k;
    const double qf = static_cast<double>(m) / kFs;
    const double sl = m == 0 ? 1.0 : sin(kPi * fc * qf) / (kPi * fc * qf);
    const double cl = m == 0 ? (1.0 - 2.0 * q1) + 2.0 * q1 : (1.0 - 2.0 * q1) + 2.0 * q1 * cos(2.0 * kPi * qf * fc);
    if (k <= 256) p[k] = a[k].x * sl * cl;
  }
  __syncthreads();
  for (int k = tid; k < 512; k += kThreads) a[k] = dc{p[k <= 256 ? k : 512 - k], 0.0};
  fft(a, tw, 9);
  for (int k = tid; k < kBins; k += kThreads) row[k] = static_cast<float>(log(exp(a[k].x / 512.0) + 1e-15));
}

// ------------------------------------------------------------------------------------------------ D4C

__global__ void __launch_bounds__(kThreads) wa_lovetrain(const In in, Dims d, Ws ws) {
  extern __shared__ __align__(16) uint8_t smem[];
  dc* a = reinterpret_cast<dc*>(smem);
  dc* tw = a + 2048;
  double* wf = reinterpret_cast<double*>(tw + 1024);
  __shared__ double red[kThreads / 32];
  const int t = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  if (ws.head[4 * b] != V100_WORLD_OK || t >= ws.head[4 * b + 2]) return;
  const long long o = static_cast<long long>(b) * d.Tw + t;
  const double f0 = ws.f0s[o];
  if (f0 == 0.0) {
    if (tid == 0) ws.ratio[o] = 0.0;
    return;
  }
  make_twiddles(tw, 11);
  const int h = windowed(in, b, ws.head[4 * b + 1], frame_time(t), fmax(f0, 40.0), 3.0, true, in.noise + ws.lt_off[o],
                         wf, red);
  for (int i = tid; i < 2048; i += kThreads) a[i] = dc{i <= 2 * h ? wf[i] : 0.0, 0.0};
  fft(a, tw, 11);
  double s1 = 0.0, s2 = 0.0;
  for (int k = 14 + tid; k <= 1012; k += kThreads) {
    const double pw = a[k].x * a[k].x + a[k].y * a[k].y;
    if (k <= 512) s1 += pw;
    s2 += pw;
  }
  const double c1 = block_sum(s1, red), c2 = block_sum(s2, red);
  if (tid == 0) ws.ratio[o] = c1 / c2;
}

constexpr int kD4Seg = 1025 + 2 * 128;            // LinearSmoothing at widths up to 960 Hz (f0 <= 800 + 20 %)

// the centroid of one 4-period Blackman window (GetCentroid), accumulated into acc[0, 1024]
__device__ void centroid(const In& in, int b, int L, double t, double f0, const double* dither, dc* a, const dc* tw,
                         double* wf, double* acc, double* red, bool first) {
  const int h = windowed(in, b, L, t, f0, 4.0, true, dither, wf, red);
  double pw = 0.0;
  for (int i = threadIdx.x; i <= 2 * h; i += kThreads) pw += wf[i] * wf[i];
  const double s = sqrt(block_sum(pw, red));
  for (int i = threadIdx.x; i < 2048; i += kThreads) {
    const double v = i <= 2 * h ? wf[i] / s : 0.0;
    a[i] = dc{v, v * (i + 1.0)};
  }
  fft(a, tw, 11);
  for (int k = threadIdx.x; k <= 1024; k += kThreads) {
    const dc z = a[k], zn = a[(2048 - k) & 2047];
    const dc A{0.5 * (z.x + zn.x), 0.5 * (z.y - zn.y)};
    const dc Bq{0.5 * (z.y + zn.y), -0.5 * (z.x - zn.x)};
    const double c = Bq.x * A.x + A.y * Bq.y;
    acc[k] = first ? c : acc[k] + c;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kThreads) wa_d4c(const In in, Dims d, Ws ws, Out out) {
  extern __shared__ __align__(16) uint8_t smem[];
  dc* a = reinterpret_cast<dc*>(smem);                     // [2048]
  dc* tw = a + 2048;                                       // [1024]
  double* wf = reinterpret_cast<double*>(tw + 1024);       // [2048]
  double* sc = wf + 2048;                                  // [1025]
  double* sp = sc + 1025;                                  // [1025]
  double* seg = sp + 1025;                                 // [kD4Seg]
  __shared__ double red[kThreads / 32];
  __shared__ int top[kThreads];
  const int t = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  float* ap = out.ap + static_cast<long long>(b) * d.T + t;
  const bool ok = ws.head[4 * b] == V100_WORLD_OK && t < ws.head[4 * b + 2];
  if (!ok) {
    if (tid == 0) *ap = 0.0f;
    return;
  }
  const long long o = static_cast<long long>(b) * d.Tw + t;
  const long long off = ws.d4_off[o];
  if (off < 0) {
    if (tid == 0) *ap = static_cast<float>(kCodeapUnvoiced);
    return;
  }
  const int L = ws.head[4 * b + 1];
  const double f0 = fmax(47.0, ws.f0s[o]);
  const double tt = frame_time(t);
  const int n = 2 * mround(2.0 * kFs / f0) + 1;
  const double* dither = in.noise + off;
  make_twiddles(tw, 11);
  centroid(in, b, L, tt - 0.25 / f0, f0, dither, a, tw, wf, sc, red, true);
  centroid(in, b, L, tt + 0.25 / f0, f0, dither + n, a, tw, wf, sc, red, false);
  dc_correction(sc, f0, 2048);
  const int h = windowed(in, b, L, tt, f0, 4.0, false, dither + 2 * n, wf, red);
  for (int i = tid; i < 2048; i += kThreads) a[i] = dc{i <= 2 * h ? wf[i] : 0.0, 0.0};
  fft(a, tw, 11);
  for (int k = tid; k <= 1024; k += kThreads) sp[k] = a[k].x * a[k].x + a[k].y * a[k].y;
  __syncthreads();
  dc_correction(sp, f0, 2048);
  linear_smoothing(sp, f0, 2048, seg, sp);
  for (int k = tid; k <= 1024; k += kThreads) sc[k] = sc[k] / sp[k];
  __syncthreads();
  linear_smoothing(sc, f0 / 2.0, 2048, seg, sc);           // static group delay
  linear_smoothing(sc, f0, 2048, seg, sp);                 // its smoothed version
  for (int k = tid; k <= 1024; k += kThreads) sc[k] -= sp[k];
  __syncthreads();
  for (int j = tid; j < 2048; j += kThreads) {
    double v = 0.0;
    if (j < 769) {
      const double q = j / 768.0;
      const double w = 0.355768 - 0.487396 * cos(2.0 * kPi * q) + 0.144232 * cos(4.0 * kPi * q) -
                       0.012604 * cos(6.0 * kPi * q);
      v = sc[j] * w;                                       // bins 384 - 384 + j
    }
    a[j] = dc{v, 0.0};
  }
  fft(a, tw, 11);
  for (int k = tid; k <= 1024; k += kThreads) sp[k] = a[k].x * a[k].x + a[k].y * a[k].y;
  __syncthreads();
  // sorted ascending and cumulated, cum[1002] / cum[1024]: the 22 largest of the 1025 powers are left out
  for (int r = 0; r < 22; ++r) {
    double mv = -1.0;
    int mi = -1;
    for (int k = tid; k <= 1024; k += kThreads)
      if (sp[k] > mv) {
        mv = sp[k];
        mi = k;
      }
    top[tid] = mi;
    seg[tid] = mv;
    __syncthreads();
    for (int s = kThreads / 2; s > 0; s >>= 1) {
      if (tid < s && (seg[tid + s] > seg[tid] || (seg[tid + s] == seg[tid] && top[tid + s] < top[tid]))) {
        seg[tid] = seg[tid + s];
        top[tid] = top[tid + s];
      }
      __syncthreads();
    }
    if (tid == 0) sp[top[0]] = -1.0;                        // removed from the sum below
    __syncthreads();
  }
  double all = 0.0, kept = 0.0;
  for (int k = tid; k <= 1024; k += kThreads) {
    const double v = sp[k];
    if (v >= 0.0) kept += v;
  }
  // the total is the kept sum plus the 22 removed powers: recompute them from the spectrum
  for (int k = tid; k <= 1024; k += kThreads) all += a[k].x * a[k].x + a[k].y * a[k].y;
  const double c_kept = block_sum(kept, red), c_all = block_sum(all, red);
  if (tid == 0) {
    const double v = fmin(0.0, 10.0 * log10(c_kept / c_all) + (f0 - 100.0) / 50.0);
    *ap = static_cast<float>(20.0 * log10(pow(10.0, v / 20.0)));
  }
}

constexpr size_t kSmSmem = (2048 + 1024) * sizeof(dc) + (2048 + 1025) * sizeof(double);
constexpr size_t kLtSmem = (2048 + 1024) * sizeof(dc) + 2048 * sizeof(double);
constexpr size_t kD4Smem = (2048 + 1024) * sizeof(dc) + (2048 + 1025 + 1025 + kD4Seg) * sizeof(double);

}  // namespace

int64_t world_analysis_workspace_bytes(int B, int64_t L_max) {
  if (B <= 0 || L_max < 0) return 0;
  Ws w;
  return static_cast<int64_t>(carve(nullptr, make_dims(B, L_max, 0), &w));
}

int64_t world_analysis_noise_values(int64_t L_max) { return (L_max / kHop + 1) * kDrawsPerFrame; }

int world_analyze(const void* wav, int wav_dtype, int64_t wav_pitch, const int32_t* len, int B, int64_t L_max,
                  const double* taps, const double* noise, int64_t noise_len, void* workspace, int T, float* f0,
                  float* logspc, float* codeap, int32_t* frame_len, int32_t* status, cudaStream_t stream) {
  if (wav == nullptr || len == nullptr || taps == nullptr || noise == nullptr || workspace == nullptr ||
      f0 == nullptr || logspc == nullptr || codeap == nullptr || frame_len == nullptr || status == nullptr)
    return fail(V100_E_INVALID, "world_analyze: null pointer");
  if (wav_dtype != 0 && wav_dtype != 1) return fail(V100_E_INVALID, "world_analyze: wav_dtype must be 0 or 1");
  if (B <= 0 || L_max < 0 || wav_pitch < L_max)
    return fail(V100_E_INVALID, "world_analyze: B must be positive, L_max non-negative and wav_pitch >= L_max");
  if (T < L_max / kHop + 1)
    return fail(V100_E_INVALID, "world_analyze: T = %d < L_max / 160 + 1 = %lld", T, (long long)(L_max / kHop + 1));
  if (noise_len < world_analysis_noise_values(L_max))
    return fail(V100_E_INVALID, "world_analyze: noise table of %lld values < %lld", (long long)noise_len,
                (long long)world_analysis_noise_values(L_max));
  if (L_max > (1LL << 30) || B > 65535 || T > 65535)
    return fail(V100_E_UNSUPPORTED, "world_analyze: L_max above 2^30 samples, or B or T above 65535");
  const Dims d = make_dims(B, L_max, T);
  Ws w;
  carve(workspace, d, &w);
  In in{wav, wav_dtype, wav_pitch, len, taps, noise};
  Out o{f0, logspc, codeap, frame_len, status};
  V100_CUDA(cudaFuncSetAttribute(wa_stonemask, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmSmem));
  V100_CUDA(cudaFuncSetAttribute(wa_lovetrain, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLtSmem));
  V100_CUDA(cudaFuncSetAttribute(wa_d4c, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kD4Smem));
  const unsigned hp_tiles = static_cast<unsigned>((d.Lh + kTile - 1) / kTile);
  const unsigned ut = static_cast<unsigned>((B + 31) / 32);
  wa_prep<<<B, kThreads, 0, stream>>>(in, d, w, o);
  if (L_max > 0) {
    wa_lowcut<<<dim3(hp_tiles, B), kThreads, 0, stream>>>(in, d, w);
    wa_bands<0><<<dim3(d.tiles, B, kBands), kThreads, 0, stream>>>(in, d, w);
    wa_scan<<<B, 32, 0, stream>>>(d, w);
    wa_bands<1><<<dim3(d.tiles, B, kBands), kThreads, 0, stream>>>(in, d, w);
    wa_contour<<<dim3((d.Tw + 127) / 128, B), 128, 0, stream>>>(d, w);
    wa_fix<<<ut, 32, 0, stream>>>(d, w);
  }
  wa_stonemask<<<dim3(T, B), kThreads, kSmSmem, stream>>>(in, d, w, o);
  wa_draws<0><<<ut, 32, 0, stream>>>(d, w);
  wa_cheaptrick<<<dim3(T, B), kThreads, 0, stream>>>(in, d, w, o);
  wa_lovetrain<<<dim3(d.Tw, B), kThreads, kLtSmem, stream>>>(in, d, w);
  wa_draws<1><<<ut, 32, 0, stream>>>(d, w);
  wa_d4c<<<dim3(T, B), kThreads, kD4Smem, stream>>>(in, d, w, o);
  V100_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace v100
