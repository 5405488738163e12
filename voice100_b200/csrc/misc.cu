// Small layout / head-tail kernels around the GEMMs (all HBM-trivial next to the conv stack).
#include "common.cuh"
#include "host.h"

#include <algorithm>

namespace v100 {

// fp32 [B][T][C] -> bf16 NCW [B][C][pitch] through a 32x32 shared tile (AudioToTextCTC.forward's transpose).
template <int DT>
__global__ void __launch_bounds__(256)
ntc_to_ncw_kernel(const float* __restrict__ x, unsigned short* __restrict__ y, int T, int C, long long y_pitch) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) {
    const int t = t0 + r, c = c0 + tx;
    tile[r][tx] = (t < T && c < C) ? x[(static_cast<long long>(b) * T + t) * C + c] : 0.0f;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int c = c0 + r, t = t0 + tx;
    if (c < C && t < T) y[(static_cast<long long>(b) * C + c) * y_pitch + t] = f2h<DT>(tile[tx][r]);
  }
}

static int check_dt(int dtype, const char* what) {
  if (dtype != DT_BF16 && dtype != DT_F16) return fail(V100_E_INVALID, "%s: dtype must be V100_DTYPE_BF16 or V100_DTYPE_F16", what);
  return 0;
}

int ntc_f32_to_ncw16(const float* x, void* y, int B, int T, int C, int64_t y_pitch, int dtype, cudaStream_t stream) {
  if (int e = check_dt(dtype, "ntc_to_ncw")) return e;
  if (x == nullptr || y == nullptr) return fail(V100_E_INVALID, "ntc_to_ncw: null pointer");
  if (B <= 0 || T <= 0 || C <= 0 || B > 65535 || y_pitch < T) return fail(V100_E_INVALID, "ntc_to_ncw: bad sizes");
  dim3 grid((T + 31) / 32, (C + 31) / 32, B);
  if (dtype == DT_F16) ntc_to_ncw_kernel<DT_F16><<<grid, 256, 0, stream>>>(x, static_cast<unsigned short*>(y), T, C, y_pitch);
  else ntc_to_ncw_kernel<DT_BF16><<<grid, 256, 0, stream>>>(x, static_cast<unsigned short*>(y), T, C, y_pitch);
  V100_CUDA(cudaGetLastError());
  return 0;
}

// Dense NCW casts between the caller's fp32 [B][C][T] tensors and the pitched bf16 working layout
// (entry/exit of ConvVoiceEncoder.forward / VoiceDecoder.forward when used as stand-alone modules).
template <int DT>
__global__ void __launch_bounds__(256)
ncw_cast_kernel(const float* __restrict__ xf, const unsigned short* __restrict__ xb, float* __restrict__ yf,
                unsigned short* __restrict__ yb, long long rows, int T, long long pitch) {
  const long long total = rows * T;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < total; i += gridDim.x * 256LL) {
    const long long r = i / T;
    const int t = int(i - r * T);
    if (yb) yb[r * pitch + t] = f2h<DT>(xf[i]);
    else yf[i] = h2f<DT>(xb[r * pitch + t]);
  }
}

int ncw_f32_to_16(const float* x, void* y, int64_t y_pitch, int B, int C, int T, int dtype, cudaStream_t stream) {
  if (int e = check_dt(dtype, "ncw_f32_to_16")) return e;
  if (x == nullptr || y == nullptr || B <= 0 || C <= 0 || T <= 0 || y_pitch < T)
    return fail(V100_E_INVALID, "ncw_f32_to_16: bad arguments");
  const long long rows = static_cast<long long>(B) * C;
  const int grid = int(std::min<long long>((rows * T + 255) / 256, 148LL * 16));
  if (dtype == DT_F16) ncw_cast_kernel<DT_F16><<<grid, 256, 0, stream>>>(x, nullptr, nullptr, static_cast<unsigned short*>(y), rows, T, y_pitch);
  else ncw_cast_kernel<DT_BF16><<<grid, 256, 0, stream>>>(x, nullptr, nullptr, static_cast<unsigned short*>(y), rows, T, y_pitch);
  V100_CUDA(cudaGetLastError());
  return 0;
}

int ncw_16_to_f32(const void* x, int64_t x_pitch, float* y, int B, int C, int T, int dtype, cudaStream_t stream) {
  if (int e = check_dt(dtype, "ncw_16_to_f32")) return e;
  if (x == nullptr || y == nullptr || B <= 0 || C <= 0 || T <= 0 || x_pitch < T)
    return fail(V100_E_INVALID, "ncw_16_to_f32: bad arguments");
  const long long rows = static_cast<long long>(B) * C;
  const int grid = int(std::min<long long>((rows * T + 255) / 256, 148LL * 16));
  if (dtype == DT_F16) ncw_cast_kernel<DT_F16><<<grid, 256, 0, stream>>>(nullptr, static_cast<const unsigned short*>(x), y, nullptr, rows, T, x_pitch);
  else ncw_cast_kernel<DT_BF16><<<grid, 256, 0, stream>>>(nullptr, static_cast<const unsigned short*>(x), y, nullptr, rows, T, x_pitch);
  V100_CUDA(cudaGetLastError());
  return 0;
}

// y[b][c][t] = table[ids[b][t]][c]; one thread = one channel x 8 time steps (16-byte store).
__global__ void __launch_bounds__(256)
embedding_kernel(const int64_t* __restrict__ ids, const unsigned short* __restrict__ table,
                 unsigned short* __restrict__ y, long long y_pitch, int T, int V, int C, int32_t* __restrict__ status) {
  const int b = blockIdx.z;
  const int c = blockIdx.y * 8 + (threadIdx.x >> 5);
  const int t0 = (blockIdx.x * 32 + (threadIdx.x & 31)) * 8;
  if (c >= C || t0 >= T) return;
  const unsigned short* tab = table;
  uint32_t o[4];
#pragma unroll
  for (int i = 0; i < 8; i += 2) {
    unsigned short v[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int t = t0 + i + h;
      const long long id = t < T ? ids[static_cast<long long>(b) * T + t] : 0;
      const bool ok = id >= 0 && id < V;
      // nn.Embedding raises IndexError for such an id; a kernel cannot, so the row is zero and the flag is set
      if (!ok && status != nullptr && c == 0) atomicOr(status, V100_STATUS_BAD_INDEX);
      v[h] = (t < T && ok) ? tab[id * C + c] : 0;
    }
    o[i >> 1] = uint32_t(v[0]) | (uint32_t(v[1]) << 16);
  }
  *reinterpret_cast<uint4*>(y + (static_cast<long long>(b) * C + c) * y_pitch + t0) = make_uint4(o[0], o[1], o[2], o[3]);
}

// Same gather with the table slice and the row's ids staged in shared memory: one CTA = one utterance x 64 channels.
// (The kernel above gathers 2-byte elements from global memory, eight per thread, and re-reads the ids once per
// channel: 158 us for the 76 MB output of 256 x 512 x 292, 0.48 TB/s.)  Work items are (channel, group of 8 steps),
// consecutive threads taking consecutive groups of one channel, so every thread stores 16 bytes next to its neighbour's.
constexpr int kEmbCh = 64;
constexpr int kEmbRow = kEmbCh + 2;   // staged row pitch: 33 words, so that different ids of one channel fall into different banks
__global__ void __launch_bounds__(256)
embedding_smem_kernel(const int64_t* __restrict__ ids, const unsigned short* __restrict__ table,
                      unsigned short* __restrict__ y, long long y_pitch, int T, int V, int C, int32_t* __restrict__ status) {
  extern __shared__ __align__(16) unsigned char emb_smem[];
  unsigned short* tab = reinterpret_cast<unsigned short*>(emb_smem);            // [V][66]
  int* sid = reinterpret_cast<int*>(emb_smem + ((size_t(V) * kEmbRow * 2 + 15) & ~size_t(15)));   // [T8]: id or -1
  const int b = blockIdx.y, c0 = blockIdx.x * kEmbCh;
  const int groups = (T + 7) / 8, T8 = groups * 8;
  for (int i = threadIdx.x; i < V * (kEmbCh / 2); i += 256) {                   // 32-bit pieces of the table slice (C % 2 == 0)
    const int v = i / (kEmbCh / 2), j = i % (kEmbCh / 2);
    uint32_t w = 0u;
    if (c0 + 2 * j + 2 <= C) w = *reinterpret_cast<const uint32_t*>(table + static_cast<long long>(v) * C + c0 + 2 * j);
    *reinterpret_cast<uint32_t*>(tab + v * kEmbRow + 2 * j) = w;
  }
  bool bad = false;
  for (int t = threadIdx.x; t < T8; t += 256) {
    const long long id = t < T ? ids[static_cast<long long>(b) * T + t] : -1;
    const bool ok = id >= 0 && id < V;
    bad |= t < T && !ok;
    sid[t] = ok ? int(id) : -1;
  }
  // nn.Embedding raises IndexError for an id outside the table; a kernel cannot, so the row is zero and the flag is set
  if (bad && status != nullptr && blockIdx.x == 0) atomicOr(status, V100_STATUS_BAD_INDEX);
  __syncthreads();
  const int nch = min(kEmbCh, C - c0);
  for (int i = threadIdx.x; i < nch * groups; i += 256) {
    const int c = i / groups, g = i - c * groups;
    uint32_t o[4];
#pragma unroll
    for (int e = 0; e < 8; e += 2) {
      const int i0 = sid[8 * g + e], i1 = sid[8 * g + e + 1];
      const uint32_t v0 = i0 >= 0 ? tab[i0 * kEmbRow + c] : 0u, v1 = i1 >= 0 ? tab[i1 * kEmbRow + c] : 0u;
      o[e >> 1] = v0 | (v1 << 16);
    }
    *reinterpret_cast<uint4*>(y + (static_cast<long long>(b) * C + c0 + c) * y_pitch + 8 * g) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

int embedding_ncw16(const int64_t* ids, const void* table, void* y, int64_t y_pitch, int B, int T, int V, int C,
                    int32_t* status, cudaStream_t stream) {
  if (ids == nullptr || table == nullptr || y == nullptr) return fail(V100_E_INVALID, "embedding: null pointer");
  if (B <= 0 || T <= 0 || V <= 0 || C <= 0 || B > 65535) return fail(V100_E_INVALID, "embedding: bad sizes");
  if (y_pitch < T || (y_pitch & 7) || (reinterpret_cast<uintptr_t>(y) & 15))
    return fail(V100_E_INVALID, "embedding: pitch must be >= T and a multiple of 8, base 16B aligned");
  const size_t smem = ((size_t(V) * kEmbRow * 2 + 15) & ~size_t(15)) + size_t((T + 7) / 8) * 8 * 4;
  if (smem <= 96 * 1024 && (C % 2) == 0 && (reinterpret_cast<uintptr_t>(table) & 3) == 0) {
    static thread_local int configured_dev = -1;
    int dev = 0;
    V100_CUDA(cudaGetDevice(&dev));
    if (configured_dev != dev) {
      V100_CUDA(cudaFuncSetAttribute(embedding_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
      configured_dev = dev;
    }
    dim3 grid((C + kEmbCh - 1) / kEmbCh, B);
    embedding_smem_kernel<<<grid, 256, smem, stream>>>(ids, static_cast<const unsigned short*>(table),
                                                       static_cast<unsigned short*>(y), y_pitch, T, V, C, status);
    V100_CUDA(cudaGetLastError());
    return 0;
  }
  dim3 grid((T + 255) / 256, (C + 7) / 8, B);   // large vocabularies / long rows: gather from global memory
  embedding_kernel<<<grid, 256, 0, stream>>>(ids, static_cast<const unsigned short*>(table),
                                             static_cast<unsigned short*>(y), y_pitch, T, V, C, status);
  V100_CUDA(cudaGetLastError());
  return 0;
}

// fp32 NCW [B][V][pitch] -> logits [B][T][V] (optional) + greedy tokens (first maximal index).
__global__ void __launch_bounds__(128)
ctc_finalize_kernel(const float* __restrict__ y, long long pitch, float* __restrict__ logits,
                    int64_t* __restrict__ tokens, int V, int T, const int32_t* __restrict__ audio_len,
                    int32_t* __restrict__ out_len) {
  const int b = blockIdx.y;
  const int t = blockIdx.x * 128 + threadIdx.x;
  // ConvVoiceEncoder.output_length (asr.py:81-82): (audio_len + 1) // 2, emitted here so the pipeline needs no
  // separate element-wise launch
  if (out_len != nullptr && blockIdx.x == 0 && threadIdx.x == 0) out_len[b] = (audio_len[b] + 1) / 2;
  if (t >= T) return;
  const float* col = y + static_cast<long long>(b) * V * pitch + t;
  float best = col[0];
  int arg = 0;
  float* lrow = logits ? logits + (static_cast<long long>(b) * T + t) * V : nullptr;
  if (lrow) lrow[0] = best;
  for (int v = 1; v < V; ++v) {
    const float x = col[static_cast<long long>(v) * pitch];
    if (lrow) lrow[v] = x;
    if (x > best) { best = x; arg = v; }
  }
  tokens[static_cast<long long>(b) * T + t] = arg;
}

int ctc_finalize(const float* y_ncw, int64_t y_pitch, float* logits, int64_t* tokens, int B, int V, int T,
                 const int32_t* audio_len, int32_t* out_len, cudaStream_t stream) {
  if (y_ncw == nullptr || tokens == nullptr) return fail(V100_E_INVALID, "ctc_finalize: null pointer");
  if ((audio_len == nullptr) != (out_len == nullptr)) return fail(V100_E_INVALID, "ctc_finalize: audio_len and out_len go together");
  if (B <= 0 || V <= 0 || T <= 0 || B > 65535 || y_pitch < T) return fail(V100_E_INVALID, "ctc_finalize: bad sizes");
  dim3 grid((T + 127) / 128, B);
  ctc_finalize_kernel<<<grid, dim3(128), 0, stream>>>(y_ncw, static_cast<long long>(y_pitch), logits, tokens, V, T,
                                                      audio_len, out_len);
  V100_CUDA(cudaGetLastError());
  return 0;
}

// CTC collapse on the device (voice100/text.py:99-104 merge_repeated, minus the string handling): within the
// valid prefix of each row drop a token equal to its predecessor, then drop blanks (id 0).  One warp per row:
// keep-flags -> ballot -> prefix popcount gives each survivor its output slot, order preserved.
__global__ void __launch_bounds__(128)
ctc_collapse_kernel(const int64_t* __restrict__ tokens, const int64_t* __restrict__ valid_len,
                    int64_t* __restrict__ out, int32_t* __restrict__ out_len, int B, int T, int blank) {
  const int row = blockIdx.x * 4 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= B) return;
  const int64_t* in = tokens + static_cast<long long>(row) * T;
  int64_t* o = out + static_cast<long long>(row) * T;
  int n = valid_len ? static_cast<int>(valid_len[row]) : T;
  n = n < 0 ? 0 : (n > T ? T : n);
  int written = 0;
  for (int t0 = 0; t0 < n; t0 += 32) {
    const int t = t0 + lane;
    const int64_t cur = t < n ? in[t] : blank;
    const int64_t prev = (t > 0 && t < n) ? in[t - 1] : -1;
    const bool keep = t < n && cur != prev && cur != blank;
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (keep) o[written + __popc(m & ((1u << lane) - 1u))] = cur;
    written += __popc(m);
  }
  for (int t = written + lane; t < T; t += 32) o[t] = blank;   // pad the tail with blanks
  if (lane == 0) out_len[row] = written;
}

int ctc_collapse(const int64_t* tokens, const int64_t* valid_len, int64_t* out, int32_t* out_len, int B, int T,
                 int blank, cudaStream_t stream) {
  if (tokens == nullptr || out == nullptr || out_len == nullptr) return fail(V100_E_INVALID, "ctc_collapse: null pointer");
  if (B <= 0 || T <= 0) return fail(V100_E_INVALID, "ctc_collapse: bad sizes");
  if (tokens == out) return fail(V100_E_INVALID, "ctc_collapse: in-place collapse is not supported");
  ctc_collapse_kernel<<<(B + 3) / 4, 128, 0, stream>>>(tokens, valid_len, out, out_len, B, T, blank);
  V100_CUDA(cudaGetLastError());
  return 0;
}

// Batched CTC forced alignment (Viterbi best path), voice100/models/align.py:18-66 (`ctc_best_path`, called per
// utterance through .cpu().numpy() by the v2 aligner, _asr_v2.py:100-119).  One CTA per utterance; the state
// vector (expanded labels: blank, l0, blank, l1, ... = S = 2L+1 states) lives in shared memory, every time step
// is one parallel sweep over the states, back-pointers go to a caller-provided workspace.  Arithmetic is the
// reference's: fp32 `score[k] + logprob[i][label[v]]`, candidates j = 0,1,2 (stay / advance / skip, the skip
// never lands on a blank), first maximum wins, the active prefix grows by two states per step.
// With `normalize` the input is raw logits and the kernel applies log_softmax itself (_asr_v2.py:95):
// lse[i] = max + log(sum exp(x - max)) per frame, one warp per frame, kept in shared memory.
__global__ void __launch_bounds__(256)
ctc_best_path_kernel(const float* __restrict__ logprob, const int32_t* __restrict__ logit_len,
                     const int64_t* __restrict__ text, const int32_t* __restrict__ text_len,
                     uint8_t* __restrict__ back, float* __restrict__ score, int32_t* __restrict__ path,
                     int64_t* __restrict__ path_labels, int T, int V, int L, int normalize) {
  extern __shared__ float vit_smem[];
  const int b = blockIdx.x;
  const int S_max = 2 * L + 1;
  float* sc0 = vit_smem;
  float* sc1 = vit_smem + S_max;
  int* lab = reinterpret_cast<int*>(vit_smem + 2 * S_max);
  float* lse = vit_smem + 3 * S_max;                 // [T] when normalize
  __shared__ int bad_label;
  const int n = min(max(logit_len[b], 0), T);
  const int l = min(max(text_len[b], 0), L);
  const int S = 2 * l + 1;
  const float* lp = logprob + static_cast<long long>(b) * T * V;
  uint8_t* bk = back + static_cast<long long>(b) * T * S_max;
  const float NEG_INF = __int_as_float(0xff800000);
  const float NAN_F = __int_as_float(0x7fc00000);

  if (threadIdx.x == 0) bad_label = 0;
  __syncthreads();
  for (int v = threadIdx.x; v < S; v += blockDim.x) {
    long long lb = (v & 1) ? text[static_cast<long long>(b) * L + (v >> 1)] : 0;
    if (lb < 0 || lb >= V) { bad_label = 1; lb = 0; }   // numpy would raise IndexError: reject the utterance
    lab[v] = static_cast<int>(lb);
    sc0[v] = NEG_INF;
  }
  if (normalize) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = warp; i < n; i += 8) {
      const float* row = lp + static_cast<long long>(i) * V;
      float mx = NEG_INF;
      for (int v = lane; v < V; v += 32) mx = fmaxf(mx, row[v]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      float sum = 0.0f;
      for (int v = lane; v < V; v += 32) sum += expf(row[v] - mx);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      if (lane == 0) { lse[2 * i] = mx; lse[2 * i + 1] = logf(sum); }
    }
  }
  __syncthreads();
  auto fail_row = [&]() {
    if (threadIdx.x == 0) score[b] = NAN_F;
    for (int i = threadIdx.x; i < T; i += blockDim.x) {
      path[static_cast<long long>(b) * T + i] = -1;
      path_labels[static_cast<long long>(b) * T + i] = 0;
    }
  };
  if (n == 0 || bad_label) { fail_row(); return; }
  // log_softmax(x) = (x - max) - log(sum exp(x - max)), the order torch evaluates it in
  auto emit = [&](int i, int v) -> float {
    const float x = lp[static_cast<long long>(i) * V + lab[v]];
    return normalize ? (x - lse[2 * i]) - lse[2 * i + 1] : x;
  };
  if (threadIdx.x < 2 && threadIdx.x < S) sc0[threadIdx.x] = emit(0, threadIdx.x);
  __syncthreads();
  int len = min(2, S);
  float* prev = sc0;
  float* next = sc1;
  for (int i = 1; i < n; ++i) {
    const int len_next = min(len + 2, S);
    for (int v = threadIdx.x; v < len_next; v += blockDim.x) {
      const float e = emit(i, v);
      float best = NEG_INF;
      int best_j = 0;
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const int k = v - j;
        float c = NEG_INF;
        if (k >= 0 && k < len && !(j == 2 && lab[v] == 0)) c = prev[k] + e;
        if (c > best) { best = c; best_j = j; }       // strict: the first maximum wins, like np.argmax
      }
      const int kb = v - best_j;
      next[v] = best;
      // back-pointer code: 0..2 = came from v - code; 3 = the reference's uninitialised 0 (no valid predecessor)
      bk[static_cast<long long>(i) * S_max + v] = (kb >= 0 && kb < len) ? static_cast<uint8_t>(best_j) : static_cast<uint8_t>(3);
    }
    __syncthreads();
    float* t = prev; prev = next; next = t;
    len = len_next;
  }
  // the reference ends with  j = labels_len + (-1 if scores[-1] > scores[-2] else -2); best = scores[j]  on the
  // `len` live scores: IndexError when len < 2 (empty text) or j >= len -- i.e. always when fewer than S - 1 states
  // were reached, and for len == S - 1 only when the last live score is the larger one (align.py:57-58)
  int j = (len >= 2) ? S + ((prev[len - 1] > prev[len - 2]) ? -1 : -2) : S;
  if (j >= len) { fail_row(); return; }
  if (threadIdx.x == 0) {
    score[b] = prev[j];
    for (int i = n - 1; i >= 0; --i) {
      path[static_cast<long long>(b) * T + i] = j;
      path_labels[static_cast<long long>(b) * T + i] = lab[j];
      if (i > 0) {
        const uint8_t code = bk[static_cast<long long>(i) * S_max + j];
        j = code == 3 ? 0 : j - code;
      }
    }
    for (int i = n; i < T; ++i) { path[static_cast<long long>(b) * T + i] = 0; path_labels[static_cast<long long>(b) * T + i] = 0; }
  }
}

int ctc_best_path(const float* logprob, const int32_t* logit_len, const int64_t* text, const int32_t* text_len,
                  uint8_t* workspace, float* score, int32_t* path, int64_t* path_labels, int B, int T, int V, int L,
                  int normalize, cudaStream_t stream) {
  if (logprob == nullptr || logit_len == nullptr || text == nullptr || text_len == nullptr || workspace == nullptr ||
      score == nullptr || path == nullptr || path_labels == nullptr)
    return fail(V100_E_INVALID, "ctc_best_path: null pointer");
  if (B <= 0 || T <= 0 || V <= 0 || L <= 0) return fail(V100_E_INVALID, "ctc_best_path: bad sizes");
  const size_t smem = size_t(3) * (2 * L + 1) * 4 + (normalize ? size_t(2) * T * 4 : 0);
  if (smem > 200 * 1024) return fail(V100_E_UNSUPPORTED, "ctc_best_path: text length %d / %d frames too long for shared memory", L, T);
  static thread_local int configured_dev = -1;
  int dev = 0;
  V100_CUDA(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    V100_CUDA(cudaFuncSetAttribute(ctc_best_path_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    configured_dev = dev;
  }
  ctc_best_path_kernel<<<B, 256, smem, stream>>>(logprob, logit_len, text, text_len, workspace, score, path,
                                                 path_labels, T, V, L, normalize);
  V100_CUDA(cudaGetLastError());
  return 0;
}

// fp32 NCW [B][C][pitch] -> [B][T][C] through a 32x32 tile.
__global__ void __launch_bounds__(256)
ncw_to_ntc_kernel(const float* __restrict__ y, long long pitch, float* __restrict__ out, int C, int T) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) {
    const int c = c0 + r, t = t0 + tx;
    tile[r][tx] = (c < C && t < T) ? y[(static_cast<long long>(b) * C + c) * pitch + t] : 0.0f;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int t = t0 + r, c = c0 + tx;
    if (t < T && c < C) out[(static_cast<long long>(b) * T + t) * C + c] = tile[tx][r];
  }
}

int ncw_f32_to_ntc(const float* y_ncw, int64_t y_pitch, float* out, int B, int C, int T, cudaStream_t stream) {
  if (y_ncw == nullptr || out == nullptr) return fail(V100_E_INVALID, "ncw_to_ntc: null pointer");
  if (B <= 0 || C <= 0 || T <= 0 || B > 65535 || y_pitch < T) return fail(V100_E_INVALID, "ncw_to_ntc: bad sizes");
  dim3 grid((T + 31) / 32, (C + 31) / 32, B);
  ncw_to_ntc_kernel<<<grid, 256, 0, stream>>>(y_ncw, y_pitch, out, C, T);
  V100_CUDA(cudaGetLastError());
  return 0;
}

// BatchSpectrogramAugumentation.maskaudio (voice100/audio.py:106-108): log(clamp(exp(audio) * mask, min = log_offset)) with
// mask = t < audio_len[b].  One thread per element; expf / logf (not the fast intrinsics) so that valid frames come back
// within an ulp or two of the reference's exp -> log round trip.
__global__ void __launch_bounds__(256)
maskaudio_kernel(const float* __restrict__ audio, const int32_t* __restrict__ audio_len, float* __restrict__ out,
                 long long n, int T, int C, float log_offset) {
  const long long tc = static_cast<long long>(T) * C;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += gridDim.x * 256LL) {
    const long long b = i / tc;
    const int t = int((i - b * tc) / C);
    const float m = t < __ldg(audio_len + b) ? 1.0f : 0.0f;
    out[i] = logf(fmaxf(expf(audio[i]) * m, log_offset));
  }
}

int maskaudio(const float* audio, const int32_t* audio_len, float* out, int B, int T, int C, float log_offset,
              cudaStream_t stream) {
  if (audio == nullptr || audio_len == nullptr || out == nullptr) return fail(V100_E_INVALID, "maskaudio: null pointer");
  if (B <= 0 || T <= 0 || C <= 0) return fail(V100_E_INVALID, "maskaudio: non-positive size");
  if (!(log_offset > 0.0f)) return fail(V100_E_INVALID, "maskaudio: log_offset must be positive");
  const long long n = static_cast<long long>(B) * T * C;
  long long blocks = (n + 255) / 256;
  const long long cap = 32LL * num_sms();
  if (blocks > cap) blocks = cap;
  maskaudio_kernel<<<dim3((unsigned)blocks), dim3(256), 0, stream>>>(audio, audio_len, out, n, T, C, log_offset);
  V100_CUDA(cudaGetLastError());
  return 0;
}

// WORLD head tail: split the decoder output into its parameter groups, un-normalise (WORLDNorm.unnormalize,
// _layers_v1.py:131-138) and apply the presence gates, transposing NCW -> [B][T][.] on the way.
//   layout 1 (AlignTextToAudioModel, tts.py:160-167,181-190):  [hasf0 | f0 | logspc(S) | codeap(A)]
//   layout 2 (AlignTextToAudio, _tts_v2.py:65-71,80-91):       [hasf0 | f0 | logspc(S) | hascodeap(A) | codeap(A)]
// S = logspc_size (257 bins, or 25 mel-cepstra with use_mcep), A = codeap_size.
// mean/std index: 0 = f0, 1..S = logspc, S+1..S+A = codeap.  With `unnormalize`: v = std*v + mean, f0 = 0 where
// hasf0 < 0, and (layout 2) codeap = 0 where hascodeap < 0.
__global__ void __launch_bounds__(256)
world_finalize_kernel(const float* __restrict__ y, long long pitch, const float* __restrict__ mean,
                      const float* __restrict__ stdv, float* __restrict__ hasf0, float* __restrict__ f0,
                      float* __restrict__ logspc, float* __restrict__ hascodeap, float* __restrict__ codeap, int T,
                      int S, int A, int layout, int unnormalize) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int i_hc = 2 + S;                               // first hascodeap channel (layout 2)
  const int i_ap = layout == 2 ? 2 + S + A : 2 + S;     // first codeap channel
  const int C = i_ap + A;
  const float* yb = y + static_cast<long long>(b) * C * pitch;
  for (int r = ty; r < 32; r += 8) {
    const int c = c0 + r, t = t0 + tx;
    float v = 0.0f;
    if (c < C && t < T) {
      v = yb[static_cast<long long>(c) * pitch + t];
      if (unnormalize) {
        if (c >= 1 && c < i_hc) v = fmaf(stdv[c - 1], v, mean[c - 1]);
        else if (c >= i_ap) v = fmaf(stdv[1 + S + (c - i_ap)], v, mean[1 + S + (c - i_ap)]);
        if (c == 1 && yb[t] < 0.0f) v = 0.0f;
        if (layout == 2 && c >= i_ap && yb[static_cast<long long>(i_hc + (c - i_ap)) * pitch + t] < 0.0f) v = 0.0f;
      }
    }
    tile[r][tx] = v;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int t = t0 + r, c = c0 + tx;
    if (t >= T || c >= C) continue;
    const float v = tile[tx][r];
    const long long bt = static_cast<long long>(b) * T + t;
    if (c == 0) { if (hasf0) hasf0[bt] = v; }
    else if (c == 1) f0[bt] = v;
    else if (c < i_hc) logspc[bt * S + (c - 2)] = v;
    else if (c < i_ap) { if (hascodeap) hascodeap[bt * A + (c - i_hc)] = v; }
    else codeap[bt * A + (c - i_ap)] = v;
  }
}

// Same operation with one CTA = one utterance x 32 steps x ALL channels (dynamic shared tile [C][33]): the 32 x 32 tiles
// above make 43,776 CTAs of 8 KB each for [256, 260, 583] and reach 1.7 TB/s; here every channel row is read in 128-byte
// pieces, the gates come from the tile itself, and a step's S log-spectrum bins are written as one contiguous run.
__global__ void __launch_bounds__(256)
world_finalize_wide_kernel(const float* __restrict__ y, long long pitch, const float* __restrict__ mean,
                           const float* __restrict__ stdv, float* __restrict__ hasf0, float* __restrict__ f0,
                           float* __restrict__ logspc, float* __restrict__ hascodeap, float* __restrict__ codeap, int T,
                           int S, int A, int layout, int unnormalize) {
  extern __shared__ float wf_tile[];                    // [C][33]
  const int b = blockIdx.y, t0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int i_hc = 2 + S;                               // first hascodeap channel (layout 2)
  const int i_ap = layout == 2 ? 2 + S + A : 2 + S;     // first codeap channel
  const int C = i_ap + A;
  const float* yb = y + static_cast<long long>(b) * C * pitch;
  const int t = t0 + tx;
  for (int cb = ty; cb < C; cb += 64) {      // eight independent 128-byte row pieces in flight per warp
    float v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int c = cb + 8 * u;
      v[u] = (c < C && t < T) ? __ldg(yb + static_cast<long long>(c) * pitch + t) : 0.0f;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int c = cb + 8 * u;
      if (c >= C) break;
      float w = v[u];
      if (unnormalize && t < T) {
        if (c >= 1 && c < i_hc) w = fmaf(__ldg(stdv + c - 1), w, __ldg(mean + c - 1));
        else if (c >= i_ap) w = fmaf(__ldg(stdv + 1 + S + (c - i_ap)), w, __ldg(mean + 1 + S + (c - i_ap)));
      }
      wf_tile[c * 33 + tx] = w;
    }
  }
  __syncthreads();
  int c = threadIdx.x % C, tl = threadIdx.x / C;         // flat walk over [32 steps][C channels], channel fastest
  const int dc = 256 % C, dt = 256 / C;
  while (tl < 32 && t0 + tl < T) {
    float v = wf_tile[c * 33 + tl];
    if (unnormalize) {
      if (c == 1 && wf_tile[tl] < 0.0f) v = 0.0f;                                          // hasf0 gate
      if (layout == 2 && c >= i_ap && wf_tile[(i_hc + (c - i_ap)) * 33 + tl] < 0.0f) v = 0.0f;   // hascodeap gate
    }
    const long long bt = static_cast<long long>(b) * T + t0 + tl;
    if (c == 0) { if (hasf0) hasf0[bt] = v; }
    else if (c == 1) f0[bt] = v;
    else if (c < i_hc) logspc[bt * S + (c - 2)] = v;
    else if (c < i_ap) { if (hascodeap) hascodeap[bt * A + (c - i_hc)] = v; }
    else codeap[bt * A + (c - i_ap)] = v;
    c += dc; tl += dt;
    if (c >= C) { c -= C; ++tl; }
  }
}

int world_finalize(const float* y_ncw, int64_t y_pitch, const float* mean, const float* stdv, float* hasf0, float* f0,
                   float* logspc, float* hascodeap, float* codeap, int B, int T, int logspc_size, int codeap_size,
                   int layout, int unnormalize, cudaStream_t stream) {
  if (y_ncw == nullptr || f0 == nullptr || logspc == nullptr || codeap == nullptr)
    return fail(V100_E_INVALID, "world_finalize: null pointer");
  if (layout != 1 && layout != 2) return fail(V100_E_INVALID, "world_finalize: layout must be 1 (v1) or 2 (v2)");
  if (logspc_size <= 0 || codeap_size <= 0) return fail(V100_E_INVALID, "world_finalize: bad logspc/codeap size");
  if (unnormalize && (mean == nullptr || stdv == nullptr)) return fail(V100_E_INVALID, "world_finalize: null mean/std");
  if (B <= 0 || T <= 0 || B > 65535 || y_pitch < T) return fail(V100_E_INVALID, "world_finalize: bad sizes");
  const int C = 2 + logspc_size + (layout == 2 ? 2 : 1) * codeap_size;
  const size_t smem = size_t(C) * 33 * sizeof(float);
  if (smem <= 96 * 1024) {
    static thread_local int configured_dev = -1;
    int dev = 0;
    V100_CUDA(cudaGetDevice(&dev));
    if (configured_dev != dev) {
      V100_CUDA(cudaFuncSetAttribute(world_finalize_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
      configured_dev = dev;
    }
    dim3 grid((T + 31) / 32, B);
    world_finalize_wide_kernel<<<grid, 256, smem, stream>>>(y_ncw, y_pitch, mean, stdv, hasf0, f0, logspc, hascodeap, codeap,
                                                            T, logspc_size, codeap_size, layout, unnormalize);
    V100_CUDA(cudaGetLastError());
    return 0;
  }
  dim3 grid((T + 31) / 32, (C + 31) / 32, B);
  world_finalize_kernel<<<grid, 256, 0, stream>>>(y_ncw, y_pitch, mean, stdv, hasf0, f0, logspc, hascodeap, codeap, T,
                                                  logspc_size, codeap_size, layout, unnormalize);
  V100_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace v100
