// One bidirectional LSTM layer (voice100/models/_asr_v2.py:33-35,46 and the other v2 models) as persistent
// tcgen05 kernels.  Activations are time-major (seq.cu): x[c][t * Bp + b].
//
// Per direction the batch is cut into groups of 64 utterances and the hidden units into blocks of 64; a CTA pair
// owns (direction, group, unit block) for the whole sequence and the H/64 pairs of a (direction, group) exchange
// h_t through a small L2-resident buffer, synchronising once per step on a counter in global memory (release add /
// acquire poll).  All CTAs of a launch are co-resident (one CTA per SM), which is what makes the spin wait safe;
// the wait is bounded and traps on a protocol bug instead of hanging.
#include "common.cuh"
#include "host.h"

namespace v100 {

// ------------------------------------------------------------------------------------------------
// helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float tanh_fast(float x) {
  float r;
  asm("tanh.approx.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float sigmoid_fast(float x) { return fmaf(tanh_fast(0.5f * x), 0.5f, 0.5f); }

__device__ __forceinline__ unsigned int ld_acquire_u32(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_add_u32(unsigned int* p, unsigned int v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// generic-proxy global writes <-> async-proxy (TMA) global reads
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }

#ifdef V100_LSTM_PROF
// profiling build only (tools/lstm_prof.py): globaltimer stamps of block 0 for a few steps
__device__ unsigned long long g_lstm_prof[64 * 12];
__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define LSTM_STAMP(step, slot) \
  do { if (blockIdx.x == 0 && (step) >= 100 && (step) < 164) g_lstm_prof[((step) - 100) * 12 + (slot)] = gtime(); } while (0)
#else
#define LSTM_STAMP(step, slot) do {} while (0)
#endif

// ================================================================================================
// The kernel.  W_hh is the UMMA "A" operand (M = 256 gate rows per CTA pair = 64 hidden units).  It never changes,
// so each CTA keeps its 128 rows in TENSOR MEMORY for the whole sequence (tcgen05.mma with A from TMEM: 256 of the
// 512 columns for H = 512) and the tensor core fetches only the small B operand from shared memory every step.
// h_{t-1} of a 64-utterance group is that "B" operand (N = 64); with cta_group::2 each CTA stages only its 32 rows
// of it (32 KB per step by TMA).  The accumulator comes out as [gate row][utterance], so a thread owns one gate of
// one unit: it adds the input projection (read straight from global memory, one step ahead), applies its
// non-linearity, and the four gates of a unit meet through a 32 KB shared-memory exchange; the cell update then
// runs with thread = (unit, 8 utterances), cell state in registers.  Eight gate warps (two per TMEM lane quadrant,
// 32 utterances each) halve the serial gate work of a step compared with four.
//
// History (profiles/r01_v2.md): a first version gave one CTA a 16-unit slice of W_hh in shared memory and made 128
// utterances the M dimension: 5.3 us per step, bound by every SM pulling the whole [128 x H] h tile (128 KB at
// ~57 GB/s).  Swapping the operand roles and sharing the tile between two SMs: 5.2 us (now the 32 MMAs took 1.28
// us, issued one by one behind R2UR waterfalls); W in TMEM + the whole warp walking the MMA loop with one elected
// issuer: 4.6 us; eight gate warps: 4.25 us.  What is left is signalling through L2: release 0.64 + visibility 0.9
// + TMA latency 0.65 us of every step.
// ================================================================================================
constexpr int kPairUnits = 32;     // hidden units per CTA (64 per pair)
constexpr int kPairBatch = 64;     // utterances per group (UMMA N)
constexpr int kPairThreads = 288;  // warps 0-7: gate = warp & 3, lane = unit, utterance half = warp >> 2; warp 8: TMA + MMA issue
constexpr int kPairCtl = 8;        // control warp

struct LstmPairParams {
  int H, T, B, Bp;
  int pairs;         // H / 64
  int groups_total;  // ceil(B / 64)
  int group0, groups;
  long long n_cols;  // T * Bp
  const int32_t* lengths;
  const unsigned short* gx;  // [8H][n_cols]
  const unsigned short* w_hh;  // [2][4H][H]
  unsigned short* y;         // [2H][n_cols]
  unsigned short* hx;        // exchange buffer [2 dirs][groups_total][2][H/64][64 rows][64]
  unsigned int* counters;    // [2 dirs][groups_total]
};

template <int DT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kPairThreads, 1)
lstm_pair_kernel(const __grid_constant__ CUtensorMap tm_h, const LstmPairParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int KB = p.H / 64;
  uint8_t* sH = smem;                                       // KB x [32 utterances x 64 k] (4 KB each)
  float* sX = reinterpret_cast<float*>(sH + KB * 4096);     // [4 gates][64 utterances][32 units]
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(sX) + 4 * kPairBatch * kPairUnits * 4);
  uint64_t* h_full = bars;        // leader's copy collects both CTAs' bytes
  uint64_t* acc_full = bars + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);
  // TMEM columns: [0, 64) accumulator, [64, 64 + H/2) this CTA's 128 rows of W_hh
  const uint32_t tmem_cols = p.H > 384 ? 512u : (p.H > 128 ? 256u : 128u);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pi = blockIdx.x >> 1;
  const int pair = pi % p.pairs;
  const int gl = (pi / p.pairs) % p.groups;
  const int dir = pi / (p.pairs * p.groups);
  const int grp = p.group0 + gl;
  const int dg = dir * p.groups_total + grp;
  unsigned int* counter = p.counters + dg;
  const int unit0 = pair * 64 + int(rank) * kPairUnits;

  if (warp == kPairCtl && lane == 0) {
    tma_prefetch_desc(&tm_h);
    mbar_init(h_full, 1);
    mbar_init(acc_full, 1);
    fence_mbar_init();
  }
  if (warp == kPairCtl) {
    tmem_alloc_cg2(tmem_slot, tmem_cols);
    tmem_relinquish_cg2();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kPairCtl) {
    // ===================== control warp =====================
    cluster_sync_all();  // both CTAs' gate warps have written their half of W to tensor memory
    tc_fence_after();
    const uint32_t fmt = DT == DT_F16 ? 0u : 1u;
    // kind::f16, D = f32, A and B K-major, M = 256 (pair), N = 64
    const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | (uint32_t(kPairBatch >> 3) << 17) |
                           (uint32_t(256 >> 4) << 24);
    const uint32_t h_addr = smem_u32(sH);
    const uint32_t tmem_w = tmem_base + kPairBatch;
    const uint32_t h_full_leader = mapa_u32(smem_u32(h_full), 0);
    const unsigned int per_step = 2u * p.pairs;
    for (int k = 1; k < p.T; ++k) {
      if (lane == 0) {
        if (leader) mbar_expect_tx(h_full, 2u * KB * 4096);
        const unsigned int need = unsigned(k) * per_step;
        LSTM_STAMP(k, 0);
        if (ld_acquire_u32(counter) < need) {
          const long long t_start = clock64();
          while (ld_acquire_u32(counter) < need) {
            if (clock64() - t_start > 8000000000LL) {
              printf("libv100: lstm step wait timed out (block %d step %d have %u need %u)\n", blockIdx.x, k,
                     ld_acquire_u32(counter), need);
              __trap();
            }
          }
        }
      }
      if (lane == 0) LSTM_STAMP(k, 1);
      __syncwarp();
      if (lane < KB) {  // this CTA's 32 rows of h_{k-1}, one 4 KB box per k block, credited to the leader's barrier
        fence_proxy_async_global();
        const int hrow = ((dg * 2 + ((k - 1) & 1)) * KB + lane) * kPairBatch + int(rank) * 32;
        tma_load_2d_cg2(sH + lane * 4096, &tm_h, h_full_leader, 0, hrow);
      }
      if (leader) {  // the whole warp walks the MMA loop (uniform operands), one elected lane issues
        if (lane == 0) LSTM_STAMP(k, 8);
        mbar_wait(h_full, (k - 1) & 1);
        if (lane == 0) LSTM_STAMP(k, 10);
        __syncwarp();
        tc_fence_after();
        const bool issuer = elect_one();
        for (int kb = 0; kb < KB; ++kb) {
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            const uint64_t db = umma_desc(h_addr + kb * 4096 + kk * 32, 16, 1024);
            if (issuer) umma_ts_cg2(tmem_base, tmem_w + kb * 32 + kk * 8, db, idesc, (kb | kk) ? 1u : 0u);
          }
        }
        if (issuer) umma_commit_cg2(acc_full);
        if (lane == 0) LSTM_STAMP(k, 2);
      }
      __syncwarp();
    }
  } else {
    // ===================== gate warps =====================
    const int g = warp & 3;                               // 0 = input, 1 = forget, 2 = cell candidate, 3 = output
    const int half = warp >> 2;                           // utterances [32 half, 32 half + 32) of the group
    const uint32_t lane_addr = tmem_base + (uint32_t(g * 32) << 16);
    {
      // row (gate g, unit lane) of W_hh -> TMEM lane 32 g + lane, straight from global memory: the row-major bf16
      // row is already "two K elements per 32-bit column"
      const uint4* wrow = reinterpret_cast<const uint4*>(
          p.w_hh + (static_cast<long long>(dir) * 4 * p.H + g * p.H + unit0 + lane) * p.H);
      for (int c0 = half * 32; c0 < p.H / 2; c0 += 64) {  // the two warps of a quadrant alternate 32-column blocks
        uint32_t r[32];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const uint4 v = __ldg(wrow + (c0 >> 2) + i);
          r[4 * i] = v.x; r[4 * i + 1] = v.y; r[4 * i + 2] = v.z; r[4 * i + 3] = v.w;
        }
        tmem_st32(lane_addr + kPairBatch + c0, r);
      }
      tmem_st_wait();
      tc_fence_before();
    }
    cluster_sync_all();  // matches the control warp's second cluster barrier (.aligned: every warp takes part)
    const long long col_grp = static_cast<long long>(grp) * kPairBatch;
    const unsigned short* gx_row = p.gx + (static_cast<long long>(dir) * 4 * p.H + g * p.H + unit0 + lane) * p.n_cols;
    int len[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int b = grp * kPairBatch + warp * 8 + j;
      len[j] = b < p.B ? __ldg(p.lengths + b) : 0;
    }
    float c[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) c[j] = 0.0f;
    auto load_gx = [&](int k, uint4 (&dst)[4]) {
      const int t = dir ? p.T - 1 - k : k;
      const long long col0 = static_cast<long long>(t) * p.Bp + col_grp + half * 32;
#pragma unroll
      for (int i = 0; i < 4; ++i)
        dst[i] = col0 + 8 * i + 8 <= p.n_cols ? __ldg(reinterpret_cast<const uint4*>(gx_row + col0) + i)
                                               : make_uint4(0u, 0u, 0u, 0u);
    };
    uint4 gx_cur[4], gx_next[4];
    load_gx(0, gx_cur);
    unsigned short* hx_col = p.hx + int(rank) * 32 + lane;  // column of this unit inside its k block
    for (int k = 0; k < p.T; ++k) {
      const int t = dir ? p.T - 1 - k : k;
      if (k + 1 < p.T) load_gx(k + 1, gx_next);
      uint32_t acc[32];
      if (k > 0) {
        mbar_wait(acc_full, (k - 1) & 1);
        tc_fence_after();
        tmem_ld32(lane_addr + half * 32, acc);
        tmem_ld_wait();
        tc_fence_before();
        if (threadIdx.x == 0) LSTM_STAMP(k, 3);
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) acc[i] = 0u;
      }
      // this thread's gate of this unit for its 32 utterances -> exchange buffer [gate][utterance][unit]
      float* xw = sX + (g * kPairBatch + half * 32) * kPairUnits + lane;
      const uint32_t* gxw = reinterpret_cast<const uint32_t*>(gx_cur);
#pragma unroll
      for (int j = 0; j < 32; j += 2) {
        const uint32_t pk = gxw[j >> 1];
        const float a0 = __uint_as_float(acc[j]) + unpack_lo<DT>(pk);
        const float a1 = __uint_as_float(acc[j + 1]) + unpack_hi<DT>(pk);
        xw[j * kPairUnits] = g == 2 ? tanh_fast(a0) : sigmoid_fast(a0);
        xw[(j + 1) * kPairUnits] = g == 2 ? tanh_fast(a1) : sigmoid_fast(a1);
      }
      if (threadIdx.x == 0) LSTM_STAMP(k, 9);
      named_bar_sync(1, 256);
      if (threadIdx.x == 0) LSTM_STAMP(k, 11);
      // cell update: this thread = unit `lane`, utterances warp*8 .. warp*8+7
      const float* xr = sX + (warp * 8) * kPairUnits + lane;
      uint32_t hw[4];
      float hprev = 0.0f;
      unsigned short* hx_row = hx_col + (static_cast<long long>((dg * 2 + (k & 1)) * KB + pair) * kPairBatch + warp * 8) * 64;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float gi = xr[(0 * kPairBatch + j) * kPairUnits], gf = xr[(1 * kPairBatch + j) * kPairUnits];
        const float gg = xr[(2 * kPairBatch + j) * kPairUnits], go = xr[(3 * kPairBatch + j) * kPairUnits];
        const float cn = fmaf(gf, c[j], gi * gg);
        const float hn = go * tanh_fast(cn);
        const bool live = t < len[j];
        c[j] = live ? cn : 0.0f;
        const float h = live ? hn : 0.0f;
        hx_row[j * 64] = f2h<DT>(h);  // h_t for the next step's MMA: row = utterance, 32 lanes = 64 contiguous bytes
        if (j & 1) hw[j >> 1] = pack2<DT>(hprev, h);
        else hprev = h;
      }
      if (threadIdx.x == 0) LSTM_STAMP(k, 4);
      fence_proxy_async_global();
      if (threadIdx.x == 0) LSTM_STAMP(k, 5);
      named_bar_sync(1, 256);  // also: every thread is done reading the gate exchange buffer
      if (threadIdx.x == 0) LSTM_STAMP(k, 6);
      if (threadIdx.x == 0) red_release_add_u32(counter, 1u);
      if (threadIdx.x == 0) LSTM_STAMP(k, 7);
      // layer output (off the critical path): y[dir*H + unit][t*Bp + utterance], 8 utterances = 16 bytes
      if (col_grp + warp * 8 < p.Bp) {
        const long long col0 = static_cast<long long>(t) * p.Bp + col_grp + warp * 8;
        *reinterpret_cast<uint4*>(p.y + (static_cast<long long>(dir) * p.H + unit0 + lane) * p.n_cols + col0) =
            make_uint4(hw[0], hw[1], hw[2], hw[3]);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) gx_cur[i] = gx_next[i];
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == kPairCtl) {
    tc_fence_after();
    tmem_dealloc_cg2(tmem_base, tmem_cols);
  }
}

static int lstm_layer_pair(const void* gx, const void* w_hh, const int32_t* lengths, void* y, void* workspace, int B,
                           int Bp, int T, int H, int dtype, cudaStream_t stream) {
  const CUtensorMapDataType tt = dtype == DT_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  LstmPairParams p{};
  p.H = H; p.T = T; p.B = B; p.Bp = Bp;
  p.pairs = H / 64;
  p.groups_total = (B + kPairBatch - 1) / kPairBatch;
  p.n_cols = static_cast<long long>(T) * Bp;
  p.lengths = lengths;
  p.gx = static_cast<const unsigned short*>(gx);
  p.w_hh = static_cast<const unsigned short*>(w_hh);
  p.y = static_cast<unsigned short*>(y);
  p.hx = static_cast<unsigned short*>(workspace);
  const size_t hx_bytes = size_t(2) * p.groups_total * 2 * kPairBatch * H * 2;
  p.counters = reinterpret_cast<unsigned int*>(static_cast<uint8_t*>(workspace) + hx_bytes);
  V100_CUDA(cudaMemsetAsync(p.counters, 0, 2 * p.groups_total * sizeof(unsigned int), stream));
  const int KB = H / 64;
  CUtensorMap tm_h;
  if (int e = make_tmap_2d(&tm_h, tt, workspace, 64, int64_t(2) * p.groups_total * 2 * KB * kPairBatch, 128, 64, 32)) return e;
  const size_t smem = 1024 + size_t(KB) * 4096 + 4 * kPairBatch * kPairUnits * 4 + 64;
  auto kern = dtype == DT_F16 ? lstm_pair_kernel<DT_F16> : lstm_pair_kernel<DT_BF16>;
  V100_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  // Every CTA pair of a launch must be co-resident: the chain of a (direction, group) hands h_t from pair to pair
  // through a global counter.  Two guards: (1) the launch is sized from what the occupancy calculator says fits on
  // this device (one CTA per SM, clusters of two), and refused if not even one group fits; (2) it is a COOPERATIVE
  // launch, so the hardware starts it only when all of its CTAs can be resident -- a concurrent kernel or MPS
  // client that holds SMs delays the launch instead of leaving half a chain spinning until the poll traps.
  cudaLaunchConfig_t cfg{};
  cfg.blockDim = dim3(kPairThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cfg.gridDim = dim3(2 * p.pairs * 2);          // one group: 2 directions x pairs clusters x 2 CTAs
  int max_clusters = 0;
  V100_CUDA(cudaOccupancyMaxActiveClusters(&max_clusters, kern, &cfg));
  const int max_groups = max_clusters / (2 * p.pairs);
  if (max_groups < 1)
    return fail(V100_E_UNSUPPORTED, "lstm_layer: H=%d needs %d co-resident CTA pairs, this device fits %d", H, 2 * p.pairs, max_clusters);
  cudaLaunchAttribute attrs[1];                 // (the cluster shape is the kernel's compile-time __cluster_dims__)
  attrs[0].id = cudaLaunchAttributeCooperative;
  attrs[0].val.cooperative = 1;
  cfg.attrs = attrs;
  cfg.numAttrs = 1;
  for (int g0 = 0; g0 < p.groups_total; g0 += max_groups) {
    p.group0 = g0;
    p.groups = p.groups_total - g0 < max_groups ? p.groups_total - g0 : max_groups;
    cfg.gridDim = dim3(2 * p.groups * p.pairs * 2);
    V100_CUDA(cudaLaunchKernelEx(&cfg, kern, tm_h, p));
  }
  return 0;
}

#ifdef V100_LSTM_PROF
extern "C" int v100_debug_lstm_prof(unsigned long long* out) {
  return static_cast<int>(cudaMemcpyFromSymbol(out, g_lstm_prof, sizeof(g_lstm_prof)));
}
#endif

size_t lstm_workspace_bytes(int B, int H) {
  // h exchange buffers [2 directions][groups of 64][2 parities][64 x H] + per-(direction, group) step counters
  const size_t groups = (size_t(B) + kPairBatch - 1) / kPairBatch;
  return 2 * groups * 2 * kPairBatch * size_t(H) * 2 + 256 + 2 * groups * sizeof(unsigned int);
}

int lstm_layer(const void* gx, const void* w_hh, const int32_t* lengths, void* y, void* workspace, int B, int Bp,
               int T, int H, int dtype, cudaStream_t stream) {
  if (gx == nullptr || w_hh == nullptr || lengths == nullptr || y == nullptr || workspace == nullptr)
    return fail(V100_E_INVALID, "lstm_layer: null pointer");
  if (dtype != DT_BF16 && dtype != DT_F16) return fail(V100_E_INVALID, "lstm_layer: bad dtype");
  if (B <= 0 || T <= 0 || Bp < B || (Bp & 7) != 0) return fail(V100_E_INVALID, "lstm_layer: bad sizes (Bp must be a multiple of 8, >= B)");
  if (H < 64 || H % 64 != 0 || H > 512) return fail(V100_E_UNSUPPORTED, "lstm_layer: hidden size %d (supported: multiples of 64 up to 512)", H);
  if ((reinterpret_cast<uintptr_t>(workspace) & 1023) != 0) return fail(V100_E_INVALID, "lstm_layer: workspace must be 1024-byte aligned");
  if ((reinterpret_cast<uintptr_t>(gx) & 15) != 0 || (reinterpret_cast<uintptr_t>(w_hh) & 15) != 0 || (reinterpret_cast<uintptr_t>(y) & 15) != 0)
    return fail(V100_E_INVALID, "lstm_layer: gx, w_hh and y must be 16-byte aligned");
  if (static_cast<long long>(T) * Bp > 2147483647LL - 256) return fail(V100_E_UNSUPPORTED, "lstm_layer: T*Bp too large");
  return lstm_layer_pair(gx, w_hh, lengths, y, workspace, B, Bp, T, H, dtype, stream);
}

}  // namespace v100
