// ASR evaluation on the device: the CTC forward algorithm (nn.CTCLoss, reduction "none") and the Levenshtein
// distance between id sequences.  Both are small dynamic programs over data the ASR pipelines already hold on the
// device (the head logits and the collapsed greedy ids), so an evaluation pass needs no host round trip.
#include "common.cuh"
#include "host.h"

#include <algorithm>

namespace v100 {

constexpr int kCtcThreads = 256;
constexpr int kCtcMaxTarget = V100_CTC_MAX_TARGET;
constexpr int kCtcMaxVocab = 8192;
constexpr int kCtcStageFloats = 8192;     // frames of scores staged per chunk: F * V <= this (32 KB)
constexpr int kSkip = 1 << 30;            // state code bit: the skip transition s-2 -> s is allowed

__device__ __forceinline__ double ctc_neg_inf() { return __longlong_as_double(0xfff0000000000000LL); }

// One CTA per utterance.  alpha_t(s) over the 2l+1 blank-expanded states is kept in log space, in float64, in two
// shared-memory buffers; every time step is one sweep over the states that can still lie on a complete path
// (s <= 2t+1 and s >= S - 2(n-t)), one barrier per step.  The per-state update is the one torch's CPU kernel uses
// (LossCTC.cpp): m = max of the 2 or 3 predecessors (0 if all are -inf), alpha = log(sum exp(a_i - m)) + m + lp.
// The scores of F frames at a time are staged in shared memory; with `normalize` the kernel also computes each
// frame's log_softmax constants there in float64 (max, then log of the sum of exp(x - max) in a fixed lane order).
__global__ void __launch_bounds__(kCtcThreads, 1)
ctc_loss_kernel(const float* __restrict__ x, long long stride_t, long long stride_b, int T, int V,
                const int32_t* __restrict__ input_len, const int64_t* __restrict__ targets, long long target_stride,
                const int64_t* __restrict__ target_off, long long targets_numel, const int32_t* __restrict__ target_len,
                int L_max, int blank, int normalize, int zero_infinity, int F, float* __restrict__ loss,
                int32_t* __restrict__ status) {
  extern __shared__ __align__(16) unsigned char ctc_smem[];
  const int S_max = 2 * L_max + 1;
  double* buf0 = reinterpret_cast<double*>(ctc_smem);
  double* buf1 = buf0 + S_max;
  double* fconst = buf1 + S_max;                                    // [F][2]: max, log(sum exp(x - max))
  int* code = reinterpret_cast<int*>(fconst + 2 * F);               // [S_max]: label | kSkip
  float* stage = reinterpret_cast<float*>(code + S_max);            // [F][V]
  __shared__ int bad;
  const int b = blockIdx.x, tid = threadIdx.x;
  const double NEG_INF = ctc_neg_inf();

  const int n = input_len[b];
  const int l = target_len[b];
  const long long off = target_off ? target_off[b] : static_cast<long long>(b) * target_stride;
  if (tid == 0) bad = 0;
  __syncthreads();
  const bool bad_len = n < 0 || n > T || l < 0 || l > L_max || off < 0 || off + l > targets_numel;
  if (bad_len) {
    if (tid == 0) {
      loss[b] = __int_as_float(0x7fc00000);
      if (status) status[b] = V100_CTC_BAD_LENGTH;
    }
    return;
  }
  const int S = 2 * l + 1;
  for (int s = tid; s < S; s += kCtcThreads) {
    int c = blank;
    if (s & 1) {
      const long long lab = targets[off + (s >> 1)];
      if (lab < 0 || lab >= V) bad = 1;
      c = (lab < 0 || lab >= V) ? 0 : static_cast<int>(lab);
      if (s >= 3 && targets[off + (s >> 1) - 1] != lab) c |= kSkip;
    }
    code[s] = c;
    buf0[s] = NEG_INF;
    buf1[s] = NEG_INF;
  }
  __syncthreads();
  if (bad) {
    if (tid == 0) {
      loss[b] = __int_as_float(0x7fc00000);
      if (status) status[b] = V100_CTC_BAD_LABEL;
    }
    return;
  }
  const float* xb = x + static_cast<long long>(b) * stride_b;
  const int warp = tid >> 5, lane = tid & 31;
  double* prev = buf0;
  double* next = buf1;
  for (int t0 = 0; t0 < n; t0 += F) {
    const int nf = min(F, n - t0);
    // stage frames [t0, t0 + nf) (coalesced along V) and, with normalize, their log_softmax constants
    for (int i = tid; i < nf * V; i += kCtcThreads) {
      const int f = i / V, v = i - f * V;
      stage[i] = xb[static_cast<long long>(t0 + f) * stride_t + v];
    }
    __syncthreads();
    if (normalize) {
      for (int f = warp; f < nf; f += kCtcThreads / 32) {
        const float* row = stage + f * V;
        float mx = -__int_as_float(0x7f800000);
        for (int v = lane; v < V; v += 32) mx = fmaxf(mx, row[v]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        double sum = 0.0;
        for (int v = lane; v < V; v += 32) sum += exp(static_cast<double>(row[v]) - static_cast<double>(mx));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        if (lane == 0) { fconst[2 * f] = mx; fconst[2 * f + 1] = log(sum); }
      }
      __syncthreads();
    }
    for (int f = 0; f < nf; ++f) {
      const int t = t0 + f;
      const float* row = stage + f * V;
      const double mx = normalize ? fconst[2 * f] : 0.0, ls = normalize ? fconst[2 * f + 1] : 0.0;
      if (t == 0) {
        // alpha_0: the blank and the first label; every other state is -inf
        for (int s = tid; s < min(S, 2); s += kCtcThreads) {
          const double xv = row[code[s] & (kSkip - 1)];
          next[s] = normalize ? (xv - mx) - ls : xv;
        }
      } else {
        const int lo = max(0, S - 2 * (n - t)), hi = min(S, 2 * t + 2);
        for (int s = lo + tid; s < hi; s += kCtcThreads) {
          const int c = code[s];
          const double a0 = prev[s];
          const double a1 = s >= 1 ? prev[s - 1] : NEG_INF;
          const double a2 = (c & kSkip) ? prev[s - 2] : NEG_INF;
          double m = fmax(fmax(a0, a1), a2);
          if (m == NEG_INF) m = 0.0;
          const double xv = row[c & (kSkip - 1)];
          const double lp = normalize ? (xv - mx) - ls : xv;
          next[s] = log(exp(a0 - m) + exp(a1 - m) + exp(a2 - m)) + m + lp;
        }
      }
      __syncthreads();
      double* tmp = prev; prev = next; next = tmp;
    }
  }
  if (tid == 0) {
    double ll;
    if (n == 0) {
      ll = l == 0 ? 0.0 : NEG_INF;
    } else if (S == 1) {
      ll = prev[0];
    } else {
      const double l1 = prev[S - 1], l2 = prev[S - 2];
      double m = fmax(l1, l2);
      if (m == NEG_INF) m = 0.0;
      ll = log(exp(l1 - m) + exp(l2 - m)) + m;
    }
    float r = static_cast<float>(-ll);
    if (zero_infinity && isinf(r)) r = 0.0f;
    loss[b] = r;
    if (status) status[b] = V100_CTC_OK;
  }
}

int ctc_loss(const float* x, int64_t stride_t, int64_t stride_b, int T, int B, int V, const int32_t* input_len,
             const int64_t* targets, int64_t target_stride, const int64_t* target_off, int64_t targets_numel,
             const int32_t* target_len, int L_max, int blank, int normalize, int zero_infinity, float* loss,
             int32_t* status, cudaStream_t stream) {
  if (x == nullptr || input_len == nullptr || target_len == nullptr || loss == nullptr ||
      (targets == nullptr && targets_numel > 0))
    return fail(V100_E_INVALID, "ctc_loss: null pointer");
  if (B <= 0 || T <= 0 || V <= 0 || L_max < 0 || targets_numel < 0 || stride_t < 0 || stride_b < 0)
    return fail(V100_E_INVALID, "ctc_loss: bad sizes");
  if (blank < 0 || blank >= V) return fail(V100_E_INVALID, "ctc_loss: blank %d must be in [0, %d)", blank, V);
  if (L_max > kCtcMaxTarget)
    return fail(V100_E_UNSUPPORTED, "ctc_loss: target length limit %d exceeds %d tokens", L_max, kCtcMaxTarget);
  if (V > kCtcMaxVocab) return fail(V100_E_UNSUPPORTED, "ctc_loss: V = %d exceeds %d classes", V, kCtcMaxVocab);
  const int F = std::max(1, std::min(32, kCtcStageFloats / V));
  const int S_max = 2 * L_max + 1;
  const size_t smem = size_t(2) * S_max * 8 + size_t(2) * F * 8 + size_t(S_max) * 4 + size_t(F) * V * 4;
  static thread_local int configured_dev = -1;
  int dev = 0;
  V100_CUDA(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    V100_CUDA(cudaFuncSetAttribute(ctc_loss_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    configured_dev = dev;
  }
  ctc_loss_kernel<<<B, kCtcThreads, smem, stream>>>(x, stride_t, stride_b, T, V, input_len, targets, target_stride,
                                                   target_off, targets_numel, target_len, L_max, blank, normalize,
                                                   zero_infinity, F, loss, status);
  V100_CUDA(cudaGetLastError());
  return 0;
}

// Levenshtein distance with unit costs, one CTA per pair, along anti-diagonals d = i + j of the (n+1) x (m+1) table.
// i runs over the shorter sequence, so a diagonal has at most min(n, m) + 1 cells; three int32 diagonals live in
// shared memory and each diagonal is one parallel sweep followed by one barrier.  Integer arithmetic: exact.
__global__ void __launch_bounds__(1024)
edit_distance_kernel(const int64_t* __restrict__ hyp, long long hyp_stride, const int32_t* __restrict__ hyp_len,
                     int hyp_width, const int64_t* __restrict__ ref, long long ref_stride,
                     const int32_t* __restrict__ ref_len, int ref_width, int32_t* __restrict__ dist) {
  extern __shared__ int ed_smem[];
  const int b = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
  const int D = min(hyp_width, ref_width) + 1;                      // diagonal buffer size
  int* d0 = ed_smem;                                                // diagonal d - 2
  int* d1 = ed_smem + D;                                            // diagonal d - 1
  int* d2 = ed_smem + 2 * D;                                        // diagonal d
  int nh = hyp_len ? hyp_len[b] : hyp_width, nr = ref_len ? ref_len[b] : ref_width;
  nh = min(max(nh, 0), hyp_width);
  nr = min(max(nr, 0), ref_width);
  const int64_t* a = hyp + static_cast<long long>(b) * hyp_stride;  // indexed by i (the shorter side)
  const int64_t* c = ref + static_cast<long long>(b) * ref_stride;  // indexed by j
  int n = nh, m = nr;
  if (nh > nr) { const int64_t* p = a; a = c; c = p; n = nr; m = nh; }
  if (n == 0) {
    if (tid == 0) dist[b] = m;
    return;
  }
  // diagonal 0 = {D[0][0] = 0}, diagonal 1 = {D[0][1] = 1, D[1][0] = 1}
  if (tid == 0) { d0[0] = 0; d1[0] = 1; d1[1] = 1; }
  __syncthreads();
  for (int d = 2; d <= n + m; ++d) {
    const int i_lo = max(0, d - m), i_hi = min(n, d);
    for (int i = i_lo + tid; i <= i_hi; i += nt) {
      const int j = d - i;
      int v;
      if (i == 0) v = j;
      else if (j == 0) v = i;
      else {
        const int sub = d0[i - 1] + (__ldg(a + i - 1) != __ldg(c + j - 1));
        v = min(min(d1[i - 1], d1[i]) + 1, sub);
      }
      d2[i] = v;
    }
    __syncthreads();
    int* tmp = d0; d0 = d1; d1 = d2; d2 = tmp;
  }
  if (tid == 0) dist[b] = d1[n];
}

int edit_distance(const int64_t* hyp, int64_t hyp_stride, const int32_t* hyp_len, int hyp_width, const int64_t* ref,
                  int64_t ref_stride, const int32_t* ref_len, int ref_width, int B, int32_t* dist,
                  cudaStream_t stream) {
  if (dist == nullptr || (hyp == nullptr && hyp_width > 0) || (ref == nullptr && ref_width > 0))
    return fail(V100_E_INVALID, "edit_distance: null pointer");
  if (B <= 0 || hyp_width < 0 || ref_width < 0 || hyp_stride < 0 || ref_stride < 0)
    return fail(V100_E_INVALID, "edit_distance: bad sizes");
  if (hyp_width > V100_EDIT_MAX_LEN || ref_width > V100_EDIT_MAX_LEN)
    return fail(V100_E_UNSUPPORTED, "edit_distance: widths %d / %d exceed %d tokens", hyp_width, ref_width,
                V100_EDIT_MAX_LEN);
  const int D = std::min(hyp_width, ref_width) + 1;
  const int threads = std::min(1024, std::max(32, (D + 31) / 32 * 32));
  const size_t smem = size_t(3) * D * 4;
  static thread_local int configured_dev = -1;
  int dev = 0;
  V100_CUDA(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    V100_CUDA(cudaFuncSetAttribute(edit_distance_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    configured_dev = dev;
  }
  edit_distance_kernel<<<B, threads, smem, stream>>>(hyp, hyp_stride, hyp_len, hyp_width, ref, ref_stride, ref_len,
                                                     ref_width, dist);
  V100_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace v100
