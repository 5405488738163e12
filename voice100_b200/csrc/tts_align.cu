// Text alignment for TTS: per-token (gap, duration) pairs -> the aligned-text frame sequence that the audio models
// embed (v100_tts_align in include/v100.h).
//
// Replaces the host loops TextToAlignTextModel.align (voice100/models/tts.py:89-110, rule 1) and
// TextToAlignText.align (voice100/models/_align_v2.py:54-82, rule 2), bit for bit:
//  - one CTA per utterance.  The running frame position is a float64 sum of the float32 entries, taken by ONE thread
//    strictly in token order, because the reference does `t += a` on a Python float: a parallel scan would change
//    how t rounds.  Only the loads and the fill are parallel.
//  - rule 1: s = rint(t + gap), e = rint(t + gap + dur) (rint = round half to even = Python round()); s == e gives
//    e = max(0, e + 1); frame j < 0 wraps to total + j; j outside [-total, total) is the reference's IndexError.
//  - rule 2: the first token's gap is skipped; s = max(trunc(t), u), u = s + 1, e = max(trunc(t + dur), u), u = e;
//    frames at or past total are dropped (the slice assignment of the reference).
//  - the total length is head + int(fp32 sum) + tail (rule 2: int(fp32 sum - a[0][0]), the subtraction in fp32).
//    The reference takes torch.sum on the CPU, whose reduction order depends on the CPU's vector width; here the
//    fp32 sum is the float32 rounding of the sequential float64 sum.  The two can differ only when the sum lies
//    within a few float32 ulps of an integer.
//  - overlapping tokens resolve last-writer-wins, as in the loop: every frame takes the largest index of the tokens
//    that cover it (an atomicMax over token indices, staged in the output row itself), so negative entries,
//    wrapped indices and non-monotone starts take the same path as the ordinary case.
#include <math.h>

#include "common.cuh"
#include "host.h"

namespace v100 {

namespace {

constexpr int kAlignThreads = 256;
constexpr int kAlignMaxTokens = 4096;   // the per-token arrays live in shared memory: 8 bytes a token

__global__ void __launch_bounds__(kAlignThreads)
tts_align_kernel(const float* __restrict__ dur, long long sb, long long sl, long long sc, int log1p_input,
                 float* __restrict__ dur_out, const int64_t* __restrict__ text, long long text_stride,
                 const int32_t* __restrict__ text_len, int L, int rule, int head, int tail,
                 int64_t* __restrict__ aligntext, int T_cap, int32_t* __restrict__ aligntext_len,
                 int32_t* __restrict__ status, int32_t* __restrict__ filled_len, int32_t* __restrict__ frame_len) {
  __shared__ float2 a[kAlignMaxTokens];     // (gap, dur) of token i, then its frame range [s, e) as int2
  __shared__ int s_status, s_total, s_fill;
  pdl_trigger();
  pdl_wait();
  const int b = blockIdx.x;
  int n = text_len == nullptr ? L : __ldg(text_len + b);
  n = n < 0 ? 0 : (n > L ? L : n);
  const float* db = dur + b * sb;
  for (int i = threadIdx.x; i < L; i += kAlignThreads) {
    float g = db[i * sl], d = db[i * sl + sc];
    if (log1p_input) {                      // exp(pred) - 1: rounded twice, never contracted into an fma
      g = __fsub_rn(expf(g), 1.0f);
      d = __fsub_rn(expf(d), 1.0f);
    }
    if (dur_out != nullptr) {
      float* o = dur_out + (static_cast<long long>(b) * L + i) * 2;
      o[0] = g;
      o[1] = d;
    }
    if (i < n) a[i] = make_float2(g, d);
  }
  __syncthreads();

  if (threadIdx.x == 0) {
    // the sum that sizes the output, and its failure modes, come first (the reference computes total before it loops)
    double sum = 0.0;
    for (int i = 0; i < n; ++i) {
      sum += static_cast<double>(a[i].x);
      sum += static_cast<double>(a[i].y);
    }
    float fsum = static_cast<float>(sum);
    if (rule == 2 && n > 0) fsum = __fsub_rn(fsum, a[0].x);
    int st = V100_ALIGN_OK;
    long long total = 0;
    if (isnan(fsum)) {
      st = V100_ALIGN_NAN;                  // int(nan): ValueError
    } else if (isinf(fsum)) {
      st = V100_ALIGN_INF;                  // int(inf): OverflowError
    } else {
      const double tot = static_cast<double>(head) + trunc(static_cast<double>(fsum)) + static_cast<double>(tail);
      if (tot < 0.0) st = V100_ALIGN_NEGATIVE;                       // torch.zeros(total): RuntimeError
      else if (tot > 2147483647.0) st = V100_ALIGN_TOO_LONG;         // frame indices are int32
      else total = static_cast<long long>(tot);
    }
    const double dtotal = static_cast<double>(total);
    if (st == V100_ALIGN_OK && rule == 1) {
      double t = head;
      for (int i = 0; i < n; ++i) {
        t += static_cast<double>(a[i].x);
        double s = rint(t);
        t += static_cast<double>(a[i].y);
        double e = rint(t);
        // range(s, e) frame by frame; s == e writes [s, max(0, s + 1)), which is never empty
        const bool one = s == e;
        const bool empty = !one && e <= s;
        const bool bad = !empty && (s < -dtotal || (one ? s >= dtotal : e > dtotal));
        if (bad) {
          st = V100_ALIGN_INDEX;
          break;
        }
        int2 r = make_int2(0, 0);
        if (!empty) {
          r.x = static_cast<int>(s);
          r.y = one ? max(0, r.x + 1) : static_cast<int>(e);
        }
        reinterpret_cast<int2*>(a)[i] = r;
      }
    } else if (st == V100_ALIGN_OK) {
      // s and e never decrease and start at 0, so everything from 2^40 on lies past any int32 total: clamping there
      // keeps the int64 arithmetic exact and drops the same frames
      const double cap = 1099511627776.0;
      double t = head;
      long long u = 0;
      for (int i = 0; i < n; ++i) {
        if (i > 0) t += static_cast<double>(a[i].x);
        long long s = static_cast<long long>(fmax(fmin(trunc(t), cap), -cap));
        s = s > u ? s : u;
        u = s + 1;
        t += static_cast<double>(a[i].y);
        long long e = static_cast<long long>(fmax(fmin(trunc(t), cap), -cap));
        e = e > u ? e : u;
        u = e;
        const long long lo = s < total ? s : total, hi = e < total ? e : total;
        reinterpret_cast<int2*>(a)[i] = make_int2(static_cast<int>(lo), static_cast<int>(hi));
      }
    }
    int fill = 0;
    if (st == V100_ALIGN_OK) {
      fill = static_cast<int>(total);
      if (aligntext != nullptr && total > T_cap) {
        st = V100_ALIGN_CAPACITY;
        fill = T_cap;
      }
    }
    s_status = st;
    s_total = (st == V100_ALIGN_OK || st == V100_ALIGN_CAPACITY || st == V100_ALIGN_INDEX) ? static_cast<int>(total) : 0;
    s_fill = fill;
    aligntext_len[b] = s_total;
    status[b] = st;
    if (filled_len != nullptr) filled_len[b] = fill;
    if (frame_len != nullptr) frame_len[b] = fill > 0 ? 2 * fill - 1 : 0;
  }
  __syncthreads();
  if (aligntext == nullptr) return;

  const int st = s_status, total = s_total, fill = s_fill;
  int64_t* row = aligntext + static_cast<long long>(b) * T_cap;
  const bool ok = st == V100_ALIGN_OK || st == V100_ALIGN_CAPACITY;
  for (int f = threadIdx.x; f < T_cap; f += kAlignThreads) row[f] = 0;
  if (!ok) return;
  __syncthreads();
  // owner of frame f = 1 + the last token whose range covers it (frame j, or total + j for a wrapped j < 0); 0 = none
  unsigned long long* owner = reinterpret_cast<unsigned long long*>(row);
  for (int i = threadIdx.x; i < n; i += kAlignThreads) {
    const int2 r = reinterpret_cast<const int2*>(a)[i];
    for (int j = r.x; j < r.y; ++j) {
      const int f = j < 0 ? j + total : j;
      if (f < fill) atomicMax(owner + f, static_cast<unsigned long long>(i) + 1ULL);
    }
  }
  __syncthreads();
  const int64_t* tb = text + static_cast<long long>(b) * text_stride;
  for (int f = threadIdx.x; f < fill; f += kAlignThreads) {
    const unsigned long long o = owner[f];
    row[f] = o == 0 ? 0 : tb[o - 1];
  }
}

}  // namespace

int tts_align(const float* durations, int64_t stride_b, int64_t stride_l, int64_t stride_c, int log1p_input,
              float* durations_out, const int64_t* text, int64_t text_stride, const int32_t* text_len, int B, int L,
              int rule, int head, int tail, int64_t* aligntext, int T_cap, int32_t* aligntext_len, int32_t* status,
              int32_t* filled_len, int32_t* frame_len, cudaStream_t stream) {
  if (durations == nullptr || text == nullptr || aligntext_len == nullptr || status == nullptr)
    return fail(V100_E_INVALID, "tts_align: null pointer");
  if (B <= 0 || L < 0) return fail(V100_E_INVALID, "tts_align: B must be positive and L non-negative");
  if (rule != 1 && rule != 2) return fail(V100_E_INVALID, "tts_align: rule must be 1 or 2 (got %d)", rule);
  if (aligntext != nullptr && T_cap < 0) return fail(V100_E_INVALID, "tts_align: negative T_cap");
  if (L > kAlignMaxTokens)
    return fail(V100_E_UNSUPPORTED, "tts_align: L = %d tokens > %d (per-utterance token arrays in shared memory)", L,
                kAlignMaxTokens);
  V100_CUDA(launch_pdl(tts_align_kernel, dim3(B), dim3(kAlignThreads), 0, stream, durations, (long long)stride_b,
                       (long long)stride_l, (long long)stride_c, log1p_input, durations_out, text,
                       (long long)text_stride, text_len, L, rule, head, tail, aligntext, T_cap, aligntext_len, status,
                       filled_len, frame_len));
  return 0;
}

}  // namespace v100
