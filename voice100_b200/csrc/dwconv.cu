// Depthwise Conv1d + folded BatchNorm + ReLU6 on NCW bf16 / fp16 activations.
//
// With k up to 83 taps the depthwise stage of ConvVoiceEncoder costs 72 MFLOP per audio-second -- on fp32 CUDA cores
// that is ~2.5x MORE time than its HBM traffic, so the FIR runs on the tensor cores as a Toeplitz matrix product.
//  * dw_tc_kernel (stride 1, the hot one): per channel, the 128 x K_w Toeplitz matrix of the filter is a tcgen05 A
//    operand resident in tensor memory and the utterances of the batch are the N axis; data by TMA boxes.
//  * dw_bulk_kernel (stride 1, filters of up to 33 taps on rows of 512 steps or more): mma.sync with register-resident
//    Toeplitz fragments, each row staged by one bulk copy.
//  * dw_s2_mma_kernel / dw_s2_kernel: stride 2 (the first encoder block) as two polyphase FIRs on mma.sync, and a
//    CUDA-core kernel for filters longer than 59 taps.
//  * dw_simt_kernel: any stride / any k, plain CUDA cores; last resort and exported for cross-checking.
#include "common.cuh"
#include "host.h"

namespace v100 {

constexpr int kDwChunk = 1024;            // outputs per CTA along time (4 double-tiles of 256)
// The staged row is kept as two arrays, even and odd 16-sample blocks: up to 5 double tiles of 16 blocks + Q blocks of
// halo = 87 blocks (44 even, 43 odd).  The odd array starts 736 samples = 1472 B = 64 (mod 128) bytes in, so that the
// 16-byte cp.async chunks of one quarter-warp (two even-block halves, two odd-block halves, ...) fall into distinct
// banks: with the arrays a multiple of 128 bytes apart ncu showed the staging copies costing 2.3x the wavefronts of the
// FIR's own data reads.
constexpr int kDwHalf = 736;
constexpr int kDwRow = kDwHalf + 43 * 16; // 1424 samples staged per row
constexpr int kDwWarps = 8;

template <int DT>
__device__ __forceinline__ void mma_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                          uint32_t b0, uint32_t b1) {
  if constexpr (DT == DT_F16) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
  } else {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
  }
}

constexpr int kDwRowsPerWarp = 8;   // batch rows a warp walks through with one set of Toeplitz fragments
// dw_bulk_kernel's staged rows start p rounded up to a multiple of 16 samples before the chunk: 32 bytes, so a staged
// row starts on a sector boundary (with 8-sample rounding the filters whose rounded half-width was an odd multiple of
// 8 samples ran 16-22 % slower).
constexpr int kDwPad = 15;

// ------------------------------------------------------------------------------------------------------------------
// dw_tc_kernel: the stride-1 FIR as a batched Toeplitz GEMM on tcgen05.  For one channel and a tile of 128 outputs
//   out[b][t0 + m] = sum_s Toep[m][s] * x[b][t0 - P + s],     m < 128, s < K_w = 128 + 2 P,
//   Toep[m][s]     = w[s - m - (P - p)]   (zero outside the filter),   P = 16 NP >= p = (k - 1) / 2
// is ONE UMMA of M = 128 steps x N utterances x K = K_w.  The Toeplitz matrix is the same for every tile and every
// utterance of the channel, so it is the A operand resident in TENSOR MEMORY, written once per channel by the epilogue
// warps with tcgen05.st into the idle one of two buffers while the other channel's MMAs run.  B is the data: x seen as a
// (T, C, B) tensor, 128B-swizzled TMA boxes of [64 steps x 1 channel x N utterances] -- the canonical K-major B layout, a
// 16-step K slice is +32 bytes.  Boxes sit on a grid of 64 steps anchored at -P and tile j reads boxes 2j .. 2j + NCH - 1,
// so consecutive tiles share NCH - 2 boxes and each input sample crosses HBM once.  The out-of-bounds zero fill supplies
// the halo on both sides, the clip tail and the rows of a partial batch block; the pitch padding is never read.
// The mma.sync kernels this replaces were bound by the SM (fragment loads through shared memory, HMMA issue); here the
// data fragments never pass through registers and shared memory is read by the tensor core alone.
// Work unit = (channel, block of N <= 128 utterances); a CTA takes every batch block of its channels back to back.
// Warps: 0 = TMA producer, 1 = MMA issuer, 2 = TMEM allocator, 3 idle, 4..11 = epilogue (TMEM lane quadrant warp & 3 =
// 32 time steps, two groups of 64 utterances): scale * acc + shift, ReLU6, rounding -> a 128B-swizzled [utterance][64
// steps] shared-memory tile -> coalesced 16-byte stores of whole 256-byte row pieces.
// TMEM (512 columns): two fp32 accumulators [128 steps][N <= 128 utterances] and two 128-column Toeplitz buffers
// (K_w <= 224 16-bit elements packed two per column).
// ------------------------------------------------------------------------------------------------------------------
constexpr int kTcStages = 8;                                 // input ring, one box per stage
constexpr int kTcBoxBytes = 128 * 128;                       // [N <= 128 utterances][64 steps]
constexpr int kTcOutBytes = 2 * kTcBoxBytes;                 // one output tile: two halves of 64 steps
constexpr int kTcSmem = 1024 + kTcStages * kTcBoxBytes + 2 * kTcOutBytes + 256;
constexpr int kTcWz = 384;                                   // zero-extended taps staged per epilogue warp

template <int NP, bool RELU6, int DT>
__global__ void __launch_bounds__(384, 1)
dw_tc_kernel(const __grid_constant__ CUtensorMap tm_x, const unsigned short* __restrict__ w, const float* __restrict__ scale,
             const float* __restrict__ shift, unsigned short* __restrict__ y, long long y_pitch, int B, int C, int T,
             int k, int N) {
  constexpr int P = 16 * NP;
  constexpr int KS = (128 + 2 * P) / 16;   // K = 16 slices per tile
  constexpr int NCH = (KS + 3) / 4;        // 64-step boxes per tile
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(16) unsigned short wz_all[8][kTcWz];
  uint8_t* ring = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* outs = ring + kTcStages * kTcBoxBytes;                          // [2 buffers][2 halves][128 rows][128 B]
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(outs + 2 * kTcOutBytes);   // [kTcStages]
  uint64_t* empty_bar = full_bar + kTcStages;                              // [kTcStages]
  uint64_t* acc_full = empty_bar + kTcStages;                              // [2]
  uint64_t* acc_empty = acc_full + 2;                                      // [2]
  uint64_t* a_full = acc_full + 4;                                         // [2] Toeplitz buffers
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 6);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int n_bb = (B + N - 1) / N;                // batch blocks per channel
  const int n_t = (T + 127) / 128;                 // time tiles per row
  const int n_box = 2 * (n_t - 1) + NCH;           // boxes per work unit
  constexpr uint32_t kAcc0 = 0, kA0 = 256;         // TMEM columns: accumulators 0 / 128, Toeplitz buffers 256 / 384

  pdl_trigger();
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_x);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kTcStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&acc_full[a], 1);
      mbar_init(&acc_empty[a], 8);
      mbar_init(&a_full[a], 8);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();      // (x is the previous kernel's output)

  if (warp == 0) {
    // ===================== TMA producer =====================
    const bool issuer = elect_one();
    const uint32_t box_bytes = uint32_t(N) * 128u;   // out-of-bounds (zero-filled) elements count too
    uint32_t seq = 0;
    for (int c = blockIdx.x; c < C; c += gridDim.x)
      for (int bb = 0; bb < n_bb; ++bb)
        for (int g = 0; g < n_box; ++g, ++seq) {
          const uint32_t s = seq % kTcStages;
          mbar_wait(&empty_bar[s], ((seq / kTcStages) & 1) ^ 1);
          if (issuer) {
            mbar_expect_tx(&full_bar[s], box_bytes);
            tma_load_3d(ring + s * kTcBoxBytes, &tm_x, &full_bar[s], 64 * g - P, c, bb * N);
          }
          __syncwarp();
        }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const bool issuer = elect_one();
    // kind::f16 instruction descriptor: D = f32, A (TMEM) and B (smem) K-major, M = 128, N = utterances
    // (format code: 1 = bf16, 0 = fp16)
    const uint32_t fmt = DT == DT_F16 ? 0u : 1u;
    const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | (uint32_t(N >> 3) << 17) | (uint32_t(128 >> 4) << 24);
    const uint32_t ring_addr = smem_u32(ring);
    uint32_t seq0 = 0;   // ring sequence number of the work unit's first box
    int it = 0;          // tiles issued
    int u = 0;           // channels issued
    for (int c = blockIdx.x; c < C; c += gridDim.x, ++u) {
      mbar_wait(&a_full[u & 1], (u >> 1) & 1);
      tc_fence_after();
      const uint32_t a_tmem = tmem_base + kA0 + 128 * (u & 1);
      for (int bb = 0; bb < n_bb; ++bb, seq0 += n_box) {
        for (int j = 0; j < n_t; ++j, ++it) {
          const int acc = it & 1;
          mbar_wait(&acc_empty[acc], ((it >> 1) & 1) ^ 1);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + kAcc0 + 128 * acc;
#pragma unroll
          for (int cc = 0; cc < NCH; ++cc) {
            const uint32_t sq = seq0 + 2 * j + cc;
            const uint32_t s = sq % kTcStages;
            mbar_wait(&full_bar[s], (sq / kTcStages) & 1);
            tc_fence_after();
#pragma unroll
            for (int kk = 4 * cc; kk < 4 * cc + 4 && kk < KS; ++kk) {
              // B: K-major SW128, rows of 128 B (one utterance's 64 steps), 8-row groups 1024 B apart
              const uint64_t db = umma_desc(ring_addr + s * kTcBoxBytes + (kk & 3) * 32, 16, 1024);
              if (issuer) umma_ts(d_tmem, a_tmem + kk * 8, db, idesc, kk > 0 ? 1u : 0u);
            }
          }
          if (issuer) {
            // free the boxes no later tile of the unit reads (2j and 2j + 1; all of them after the last tile) once
            // these MMAs have read them, then hand the accumulator to the epilogue
            const int n_rel = j + 1 < n_t ? 2 : NCH;
            for (int r = 0; r < n_rel; ++r) umma_commit(&empty_bar[(seq0 + 2 * j + r) % kTcStages]);
            umma_commit(&acc_full[acc]);
          }
          __syncwarp();
        }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (+ Toeplitz builder) =====================
    // Two groups of four warps; group g drains accumulator columns (utterances) 64 g .. 64 g + 63 and writes the
    // Toeplitz columns 32 b .. 32 b + 31 for b = g (mod 2).
    const int q = warp & 3;                          // TMEM lane quadrant: time steps 32 q .. 32 q + 31 of a tile
    const int g = (warp - 4) >> 2;
    const uint32_t lane_addr = tmem_base + (uint32_t(32 * q) << 16);
    unsigned short* wz = wz_all[warp - 4];
    const int m = 32 * q + lane;                     // this lane's Toeplitz row
    const int off = P - ((k - 1) >> 1);
    // Toeplitz matrix of channel c -> buffer `buf`: wz[i] = w[i - 127 - off], so Toep[m][s] = wz[s - m + 127]
    auto build = [&](int c, int buf) {
      for (int i = lane; i < kTcWz; i += 32) {
        const int j = i - 127 - off;
        wz[i] = (j >= 0 && j < k) ? w[static_cast<long long>(c) * k + j] : static_cast<unsigned short>(0);
      }
      __syncwarp();
#pragma unroll 1
      for (int c0 = 32 * g; c0 < 32 * NCH; c0 += 64) {
        uint32_t r[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const int s = 2 * (c0 + i) - m + 127;
          r[i] = uint32_t(wz[s]) | (uint32_t(wz[s + 1]) << 16);
        }
        tmem_st32(lane_addr + kA0 + 128 * buf + c0, r);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();   // (also: every lane is done reading wz before the next build rewrites it)
      if (lane == 0) mbar_arrive(&a_full[buf]);
    };
    // Output tile staging: half h = steps 64 h .. 64 h + 63 is [utterance n][128 B], 16-byte chunk cidx of row n at
    // (cidx ^ (n & 7)).  Lanes 2a and 2a + 1 own steps (t, t + 1) = (32 q + 2a, 32 q + 2a + 1) and trade one value per
    // utterance pair so that each stores one 32-bit (t, t + 1) word: the even lane for utterance 2i, the odd lane for
    // utterance 2 (i ^ 2) + 1.  The two rows then differ in bit 2 of n & 7, which puts the even and the odd lanes'
    // words into disjoint banks (with rows 2i / 2i + 1 they collide two ways).
    const bool odd = lane & 1;
    const uint32_t wofs = ((uint32_t(4 * (q & 1) + (lane >> 3))) << 4) + (uint32_t((lane >> 1) & 3) << 2);   // chunk, word
    // Write-out: one warp instruction = rows n, n + 1 (256 contiguous bytes of y each), lane = (row, half, chunk).
    // The TMA tensor store of the same tile (256 rows of 128 B per tile on top of the 256 rows loaded) left the kernel
    // at 384 us for the k = 83 layer against 240 us of HBM time, flat in k.
    const int rl = lane >> 4, hl = (lane >> 3) & 1, cl = lane & 7;
    int it = 0;
    if (int(blockIdx.x) < C) build(blockIdx.x, 0);
    if (int(blockIdx.x + gridDim.x) < C) build(blockIdx.x + gridDim.x, 1);
    int u = 0;
    for (int c = blockIdx.x; c < C; c += gridDim.x, ++u) {
      const float sc = scale ? __ldg(scale + c) : 1.0f;
      const float sh = __ldg(shift + c);
      for (int bb = 0; bb < n_bb; ++bb) {
        for (int j = 0; j < n_t; ++j, ++it) {
          const int acc = it & 1;
          uint8_t* obuf = outs + acc * kTcOutBytes;
          mbar_wait(&acc_full[acc], (it >> 1) & 1);
          tc_fence_after();
          const uint32_t obase = smem_u32(obuf + (q >> 1) * kTcBoxBytes);
          for (int n0 = 64 * g; n0 < min(N, 64 * g + 64); n0 += 32) {
            uint32_t v[32];
            tmem_ld32(lane_addr + kAcc0 + 128 * acc + n0, v);
            tmem_ld_wait();
            tmem_ld_fence(v);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const int ne = 2 * i, no = 2 * (i ^ 2) + 1;
              const float fe = fmaf(__uint_as_float(v[ne]), sc, sh);
              const float fo = fmaf(__uint_as_float(v[no]), sc, sh);
              const float recv = __shfl_xor_sync(0xffffffffu, odd ? fe : fo, 1);
              const float lo = odd ? recv : fe, hi = odd ? fo : recv;
              const uint32_t o = RELU6 ? pack2_relu6<DT>(lo, hi) : pack2<DT>(lo, hi);
              const uint32_t n = uint32_t(n0 + (odd ? no : ne));
              const uint32_t addr = obase + n * 128u + (wofs ^ ((n & 7u) << 4));
              asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(o) : "memory");
            }
          }
          // the accumulator is drained: the MMAs of tile it + 2 may overwrite it
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&acc_empty[acc]);
          // the tile is staged (and, by program order, every warp is done writing out tile it - 1 -- the buffer
          // tile it + 1 fills)
          named_bar_sync(1, 256);
          const int t = 128 * j + 64 * hl + 8 * cl;
          if (t < T) {
            // t < T <= pitch, both multiples of 8: the 16 bytes stay inside the row (past T they land in its padding)
            for (int n = 2 * (warp - 4) + rl; n < N && bb * N + n < B; n += 16) {
              uint4 val;
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                           : "=r"(val.x), "=r"(val.y), "=r"(val.z), "=r"(val.w)
                           : "r"(smem_u32(obuf + hl * kTcBoxBytes + n * 128 + ((cl ^ (n & 7)) << 4))));
              *reinterpret_cast<uint4*>(y + (static_cast<long long>(bb * N + n) * C + c) * y_pitch + t) = val;
            }
          }
        }
      }
      // every MMA of channel u has completed (its last accumulator was waited for): its Toeplitz buffer is free
      if (c + 2 * int(gridDim.x) < C) build(c + 2 * gridDim.x, u & 1);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// dw_bulk_kernel: short filters (k <= 33) on long rows.  The FIR runs on mma.sync.m16n8k16 as Toeplitz blocks of the
// filter (register-resident "A" fragments, W_q[m][kk] = wz[16 q + kk - m], wz = the filter zero-extended by e1 on the
// left) times 16-sample columns of the row, each warp walking 8 batch rows of its channel; the row is staged by ONE bulk
// copy (cp.async.bulk global -> shared, mbarrier completion).  The two accumulators of a 256-output double tile are its
// two HALVES:
//   A[m][n] = out[tau + m + 16 n],   B[m][n] = out[tau + 128 + m + 16 n],          m < 16, n < 8
//   A = sum_c W_c * X_c,  X_c[kk][n] = xs[16 (n + c) + kk]:  a lane's (b0, b1) is the aligned 64-bit word lane + 4 c
// (consecutive lanes, consecutive words: conflict-free), 2 Q fragment loads per double tile.  Everything outside the copied span is zeroed once per buffer -- every row of a CTA has the same span.
// The copy moves whole 16-byte groups up to T & ~7; the last T & 7 samples of a clip come by plain loads one row ahead
// (generic-proxy stores into bytes no bulk copy ever writes, so the row loop needs no proxy fence).
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

template <int Q, bool RELU6, int DT>
__global__ void __launch_bounds__(kDwWarps * 32, 4)
dw_bulk_kernel(const unsigned short* __restrict__ x, long long x_pitch, const unsigned short* __restrict__ w,
               const float* __restrict__ scale, const float* __restrict__ shift, unsigned short* __restrict__ y,
               long long y_pitch, int B, int C, int T, int k) {
  __shared__ __align__(128) unsigned short xs_all[kDwWarps][2][kDwRow];
  __shared__ __align__(16) unsigned short ws_all[kDwWarps][16 * Q + 16];
  __shared__ __align__(8) uint64_t bars[kDwWarps][2];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.y * kDwWarps + warp;
  const int b0 = blockIdx.z * kDwRowsPerWarp;
  const int nb = min(kDwRowsPerWarp, B - b0);
  const int tc0 = blockIdx.x * kDwChunk;
  const int p = (k - 1) >> 1;
  const int pl8 = (p + kDwPad) & ~kDwPad;   // the staged row starts at x[tc0 - pl8], a multiple of 16 samples
  const int e = pl8 - p;
  const int e1 = e & 1;           // folded into the zero-extended filter
  const int s = e - e1;           // tiles start s outputs before tc0
  const int tcA = tc0 - pl8;
  unsigned short* ws = ws_all[warp];
  const unsigned short* xbase = x + static_cast<long long>(c) * x_pitch;
  const long long xbstride = static_cast<long long>(C) * x_pitch;

  const int len = min(kDwChunk, T - tc0);            // outputs this CTA owns: [tc0, tc0 + len)
  const int n_dt = (len + s + 255) / 256;            // double tiles
  const int need = 16 * (16 * n_dt + Q - 1);         // staged samples the tiles read
  const int T8 = T & ~7;                             // rows are copied in whole 16-byte groups
  const int cs = max(tcA, 0), ce = max(min(tcA + need, T8), cs);
  const uint32_t bytes = uint32_t(ce - cs) * 2u;
  const int dst_off = cs - tcA;
  pdl_trigger();

  // zero both buffers once (halo left of the clip, everything right of the copied span), barriers
  for (int i = lane; i < 2 * kDwRow / 8; i += 32)
    reinterpret_cast<uint4*>(xs_all[warp][0])[i] = make_uint4(0u, 0u, 0u, 0u);
  if (lane == 0) {
    mbar_init(&bars[warp][0], 1);
    mbar_init(&bars[warp][1], 1);
    fence_mbar_init();
  }
  fence_proxy_async();     // the zeros (generic proxy) are ordered before the bulk copies (async proxy) into the same rows
  __syncwarp();
  pdl_wait();              // (x is the previous kernel's output)
  // the clip's last T & 7 samples (staged index tail0 + lane), when the tiles read them
  const int tail0 = T8 - tcA;
  const bool has_tail = lane < (T & 7) && tail0 >= 0 && tail0 + lane < need;
  if (lane == 0 && bytes > 0) {
    mbar_expect_tx(&bars[warp][0], bytes);
    bulk_load(xs_all[warp][0] + dst_off, xbase + b0 * xbstride + cs, bytes, &bars[warp][0]);
  }
  if (has_tail) xs_all[warp][0][tail0 + lane] = xbase[b0 * xbstride + T8 + lane];

  // zero-extended filter: ws[16 + i] = w[i - e1] for 0 <= i - e1 < k; Toeplitz fragments stay in registers
  for (int i = lane; i < 16 * Q + 16; i += 32) {
    const int j = i - 16 - e1;
    ws[i] = (j >= 0 && j < k) ? w[static_cast<long long>(c) * k + j] : static_cast<unsigned short>(0);
  }
  __syncwarp();
  const int g = lane >> 2, tg = lane & 3;
  uint32_t af[Q][4];
  {
    const unsigned short* wsu = ws;
#pragma unroll
    for (int q = 0; q < Q; ++q) {
      const int i0 = 16 + 16 * q + 4 * tg - g;   // wz[16q + kk - m] at m = g, kk = 4 tg
      af[q][0] = uint32_t(wsu[i0]) | (uint32_t(wsu[i0 + 1]) << 16);          // (m = g    , kk = 4tg, 4tg+1)
      af[q][1] = uint32_t(wsu[i0 - 8]) | (uint32_t(wsu[i0 - 7]) << 16);      // (m = g + 8, kk = 4tg, 4tg+1)
      af[q][2] = uint32_t(wsu[i0 + 2]) | (uint32_t(wsu[i0 + 3]) << 16);      // (m = g    , kk = 4tg+2, 4tg+3)
      af[q][3] = uint32_t(wsu[i0 - 6]) | (uint32_t(wsu[i0 - 5]) << 16);      // (m = g + 8, kk = 4tg+2, 4tg+3)
    }
  }
  const float sc = scale ? scale[c] : 1.0f;
  const float sh = shift[c];
  const bool even = (g & 1) == 0;
  // after the pair exchange this lane stores outputs (t, t+1) and (t+16, t+17) of an accumulator, t relative to tc0:
  const int pos0 = 32 * tg + (even ? g : g + 7) - s;

  for (int r = 0; r < nb; ++r) {
    unsigned short* xs = xs_all[warp][r & 1];
    unsigned short tail_next = 0;
    if (r + 1 < nb) {   // the other buffer was last read in iteration r - 1, which ended with __syncwarp
      if (lane == 0 && bytes > 0) {
        mbar_expect_tx(&bars[warp][(r + 1) & 1], bytes);
        bulk_load(xs_all[warp][(r + 1) & 1] + dst_off, xbase + (b0 + r + 1) * xbstride + cs, bytes, &bars[warp][(r + 1) & 1]);
      }
      if (has_tail) tail_next = xbase[(b0 + r + 1) * xbstride + T8 + lane];   // stored after this row's tiles
    }
    if (bytes > 0) {
      const uint32_t parity = (r >> 1) & 1;
      int spins = 0;
      while (!mbar_try_wait(&bars[warp][r & 1], parity))
        if (++spins > (1 << 28)) __trap();   // a protocol bug must fail the launch, not hang the GPU
    }
    __syncwarp();
    const uint2* x2 = reinterpret_cast<const uint2*>(xs) + lane;
    unsigned short* yp = y + (static_cast<long long>(b0 + r) * C + c) * y_pitch + tc0 + pos0;
    int pos = pos0;
    auto finish = [&](float (&acc)[4], unsigned short* yq, int posq) {
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[i] = fmaf(acc[i], sc, sh);
      // acc = out[tau + g + 32 tg + {0, 16}], out[tau + g + 8 + 32 tg + {0, 16}]; trade with lane g^1 so that even
      // g holds (g, g+1) of the first pair of rows and odd g holds (g-1+8, g+8) of the second
      const float r0 = __shfl_xor_sync(0xffffffffu, even ? acc[2] : acc[0], 4);
      const float r1 = __shfl_xor_sync(0xffffffffu, even ? acc[3] : acc[1], 4);
      const float lo0 = even ? acc[0] : r0, hi0 = even ? r0 : acc[2];
      const float lo1 = even ? acc[1] : r1, hi1 = even ? r1 : acc[3];
      uint32_t o0, o1;
      if (RELU6) {
        o0 = pack2_relu6<DT>(lo0, hi0);
        o1 = pack2_relu6<DT>(lo1, hi1);
      } else {
        o0 = pack2<DT>(lo0, hi0);
        o1 = pack2<DT>(lo1, hi1);
      }
      if (posq >= 0 && posq < len) *reinterpret_cast<uint32_t*>(yq) = o0;
      if (posq + 16 >= 0 && posq + 16 < len) *reinterpret_cast<uint32_t*>(yq + 16) = o1;
    };
#pragma unroll 1
    for (int d = 0; d < n_dt; ++d) {
      float accA[4] = {0.0f, 0.0f, 0.0f, 0.0f}, accB[4] = {0.0f, 0.0f, 0.0f, 0.0f};
      if (256 * d + 128 - s < len) {
#pragma unroll
        for (int cq = 0; cq < Q; ++cq) {
          const uint2 fa = x2[4 * cq], fb = x2[4 * cq + 32];
          mma_16816<DT>(accA, af[cq][0], af[cq][1], af[cq][2], af[cq][3], fa.x, fa.y);
          mma_16816<DT>(accB, af[cq][0], af[cq][1], af[cq][2], af[cq][3], fb.x, fb.y);
        }
        finish(accA, yp, pos);
        finish(accB, yp + 128, pos + 128);
      } else {   // the row ends in the first half of this double tile (short rows: T = 100 text tokens, ...)
#pragma unroll
        for (int cq = 0; cq < Q; ++cq) {
          const uint2 fa = x2[4 * cq];
          mma_16816<DT>(accA, af[cq][0], af[cq][1], af[cq][2], af[cq][3], fa.x, fa.y);
        }
        finish(accA, yp, pos);
      }
      x2 += 64;      // sixteen blocks per double tile
      yp += 256;
      pos += 256;
    }
    if (has_tail && r + 1 < nb) xs_all[warp][(r + 1) & 1][tail0 + lane] = tail_next;
    __syncwarp();   // everyone is done reading xs before it is refilled two rows from now
  }
}

// Stride-2 depthwise conv on the same tensor-core FIR (the first encoder block, asr.py:68), as two polyphase
// stride-1 filters:   out[o] = sum_j w[j] x[2 o + j - p]
//                            = sum_a w_e[a] x_e[o + a - p_e]  +  sum_a w_o[a] x_o[o + a - p_o],
// x_e[i] = x[2 i], x_o[i] = x[2 i + 1];  w_e = the taps j = p (mod 2) (they meet even samples), w_o = the others;
// p_e = floor(p / 2), p_o = ceil(p / 2).  The row is staged de-interleaved twice over -- by sample parity (a PRMT pair
// per 32-bit word on the way from the 16-byte global loads to shared memory) and by 16-sample block parity: block i >> 4
// of a phase row lives in the even-block array xs[0 .. kDwHalf) or the odd-block array xs[kDwHalf .. kDwRow), so eight
// blocks of one parity are 256 contiguous bytes
// (sample i at ((i >> 4) & 1) * kDwHalf + ((i >> 5) << 4) + (i & 15)).  Both filters accumulate into the same two accumulators of a
// 256-output double tile, A taking its even 16-output blocks and B its odd ones:
//   A[m][n] = out[tau + m + 32 n],   B[m][n] = out[tau + 16 + m + 32 n],   A = sum_c W_c X_c,   B = sum_c W_(c-1) X_c,
// X_c[kk][n] = xs[16 (2 n + c) + kk]: one data fragment feeds both accumulators (Q + 1 fragment loads for 2 Q MMAs);
// with the mma's kk axis permuted a lane's (b0, b1) pair is one aligned 64-bit load.  The zero extensions
// z_e = z + (p & 1), z_o = z give both filters the same delay D = z_o + p_o (even); tiles start s = P2 - D outputs early.
// The CUDA-core version of this kernel (dw_s2_kernel below, kept for long filters) ran at 0.30 of the HBM roofline with
// the issue slots 88 % busy on fp32 FMAs and bf16 unpacking.
template <int Q, int DT, int NV>
__global__ void __launch_bounds__(kDwWarps * 32, NV <= 7 ? 3 : 2)
dw_s2_mma_kernel(const unsigned short* __restrict__ x, long long x_pitch, const unsigned short* __restrict__ w,
                 const float* __restrict__ scale, const float* __restrict__ shift, unsigned short* __restrict__ y,
                 long long y_pitch, int B, int C, int T_in, int T_out, int k, int act) {
  __shared__ __align__(128) unsigned short xs_all[kDwWarps][2][kDwRow];     // [phase e / o][block-parity layout]
  __shared__ __align__(16) unsigned short ws_all[kDwWarps][2][16 * Q + 16];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.y * kDwWarps + warp;
  const int b0 = blockIdx.z * kDwRowsPerWarp;
  const int nb = min(kDwRowsPerWarp, B - b0);
  const int oc0 = blockIdx.x * kDwChunk;          // first output of this CTA
  const int p = (k - 1) >> 1;
  const int p_o = (p + 1) >> 1;                   // taps of the odd-phase filter before its centre
  const int z = p_o & 1;                          // makes the common delay D even
  const int D = z + p_o;
  const int P2 = (D + 7) & ~7;                    // the staged phase arrays start at x_e / x_o index oc0 - P2
  const int s = P2 - D;                           // tiles start s outputs before oc0 (even)
  const int iA = oc0 - P2;                        // phase index of staged sample 0 (x index 2 iA, a multiple of 16)
  pdl_trigger();
  if (c >= C) return;

  const int len = min(kDwChunk, T_out - oc0);
  const int n_dt = (len + s + 255) / 256;
  const int n_vec = min(4 * 87, 4 * (16 * n_dt + Q));   // 16-byte global loads per row: 8 samples = 4 per phase each

  // zero-extended polyphase filters: ws[ph][16 + z_ph + a] = w_ph[a]
  for (int i = lane; i < 2 * (16 * Q + 16); i += 32) {
    const int ph = i / (16 * Q + 16), ii = i - ph * (16 * Q + 16);
    const int first = ph == 0 ? (p & 1) : 1 - (p & 1);           // w_e takes taps j = p (mod 2)
    const int a = ii - 16 - (ph == 0 ? z + (p & 1) : z);
    const int j = first + 2 * a;
    ws_all[warp][ph][ii] = (a >= 0 && j < k) ? w[static_cast<long long>(c) * k + j] : static_cast<unsigned short>(0);
  }
  __syncwarp();
  const int g = lane >> 2, tg = lane & 3;
  uint32_t af[2][Q][4];
#pragma unroll
  for (int ph = 0; ph < 2; ++ph) {
    const unsigned short* wsu = ws_all[warp][ph];
#pragma unroll
    for (int q = 0; q < Q; ++q) {
      const int i0 = 16 + 16 * q + 4 * tg - g;
      af[ph][q][0] = uint32_t(wsu[i0]) | (uint32_t(wsu[i0 + 1]) << 16);
      af[ph][q][1] = uint32_t(wsu[i0 - 8]) | (uint32_t(wsu[i0 - 7]) << 16);
      af[ph][q][2] = uint32_t(wsu[i0 + 2]) | (uint32_t(wsu[i0 + 3]) << 16);
      af[ph][q][3] = uint32_t(wsu[i0 - 6]) | (uint32_t(wsu[i0 - 5]) << 16);
    }
  }
  const float sc = scale ? scale[c] : 1.0f;
  const float sh = shift[c];
  const bool even = (g & 1) == 0;
  const int pos0 = 64 * tg + (even ? g : g + 7) - s;
  const bool relu6 = act == V100_ACT_RELU6;
  unsigned short* xs_e = xs_all[warp][0];
  unsigned short* xs_o = xs_all[warp][1];
  pdl_wait();

  // The row passes through registers on its way to shared memory (cp.async cannot split 16-bit samples by parity), so
  // the NEXT row's 16-byte loads are issued before this row's MMAs and are in flight while they run: with the loads
  // issued and consumed back to back the kernel sat at 0.44 of the HBM roofline waiting on them.
  constexpr int kS2Vec = NV;   // 16-byte loads per lane and row: 11 covers a full 1024-output chunk, 7 three double tiles
  uint4 pre[kS2Vec];
  // Load i of a lane is vector v = 32 i + lane: x index t = t_lane + 256 i, staged word d = d_lane + 64 i (the staged index
  // of phase sample 4 v with the lane part taken out: block parity = bit 2 of the lane, block pair = 4 i + lane / 8, word in block = lane & 3), so the
  // loop below is immediate offsets from two per-lane constants (the generic form cost ~25 integer instructions per load).
  const int t_lane = 2 * iA + 8 * lane;
  const int d_lane = ((lane >> 2) & 1) * kDwHalf + ((lane >> 3) << 4) + 4 * (lane & 3);
  auto load_row = [&](int r) {
    const unsigned short* xrow = x + (static_cast<long long>(b0 + r) * C + c) * x_pitch + t_lane;
#pragma unroll
    for (int i = 0; i < kS2Vec; ++i) {
      const int t = t_lane + 256 * i;                               // x index of the first sample (a multiple of 8)
      pre[i] = make_uint4(0u, 0u, 0u, 0u);
      if (32 * i + lane < n_vec && t >= 0 && t < T_in) pre[i] = __ldg(reinterpret_cast<const uint4*>(xrow + 256 * i));
    }
  };
  load_row(0);
  for (int r = 0; r < nb; ++r) {
    // ---- stage: 8 consecutive samples -> 4 even-phase + 4 odd-phase samples ----
#pragma unroll
    for (int i = 0; i < kS2Vec; ++i) {
      if (32 * i + lane < n_vec) {
        uint4 val = pre[i];
        const int nvalid = T_in - (t_lane + 256 * i);               // samples of this vector inside the clip
        if (nvalid > 0 && nvalid < 8) {                             // the one vector that straddles the end of the clip
          uint32_t* u = reinterpret_cast<uint32_t*>(&val);
#pragma unroll
          for (int wd = 0; wd < 4; ++wd) {
            const int cnt = nvalid - 2 * wd;
            u[wd] &= cnt >= 2 ? 0xFFFFFFFFu : (cnt == 1 ? 0x0000FFFFu : 0u);
          }
        }
        const uint2 ev = make_uint2(__byte_perm(val.x, val.y, 0x5410), __byte_perm(val.z, val.w, 0x5410));
        const uint2 od = make_uint2(__byte_perm(val.x, val.y, 0x7632), __byte_perm(val.z, val.w, 0x7632));
        *reinterpret_cast<uint2*>(xs_e + d_lane + 64 * i) = ev;     // phase samples 4v .. 4v+3: one 8-byte word
        *reinterpret_cast<uint2*>(xs_o + d_lane + 64 * i) = od;
      }
    }
    __syncwarp();
    if (r + 1 < nb) load_row(r + 1);
    unsigned short* yp = y + (static_cast<long long>(b0 + r) * C + c) * y_pitch + oc0 + pos0;
    int pos = pos0;
    auto finish = [&](float (&acc)[4], unsigned short* yq, int posq) {
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[i] = fmaf(acc[i], sc, sh);
      const float r0 = __shfl_xor_sync(0xffffffffu, even ? acc[2] : acc[0], 4);
      const float r1 = __shfl_xor_sync(0xffffffffu, even ? acc[3] : acc[1], 4);
      const float lo0 = even ? acc[0] : r0, hi0 = even ? r0 : acc[2];
      const float lo1 = even ? acc[1] : r1, hi1 = even ? r1 : acc[3];
      const uint32_t o0 = relu6 ? pack2_relu6<DT>(lo0, hi0) : pack2<DT>(lo0, hi0);
      const uint32_t o1 = relu6 ? pack2_relu6<DT>(lo1, hi1) : pack2<DT>(lo1, hi1);
      // (a pair that starts on the row's last column also writes the pitch padding next to it: posq is even, so that
      //  column exists whenever the row length is odd -- the pitch is a multiple of 8)
      if (posq >= 0 && posq < len) *reinterpret_cast<uint32_t*>(yq) = o0;
      if (posq + 32 >= 0 && posq + 32 < len) *reinterpret_cast<uint32_t*>(yq + 32) = o1;
    };
#pragma unroll 1
    for (int d = 0; d < n_dt; ++d) {
      float accA[4] = {0.0f, 0.0f, 0.0f, 0.0f}, accB[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
      for (int ph = 0; ph < 2; ++ph) {
        const uint2* xe = reinterpret_cast<const uint2*>(ph == 0 ? xs_e : xs_o) + 32 * d + lane;
        const uint2* xo = reinterpret_cast<const uint2*>((ph == 0 ? xs_e : xs_o) + kDwHalf) + 32 * d + lane;
#pragma unroll
        for (int cq = 0; cq <= Q; ++cq) {
          const uint2 f = (cq & 1) ? xo[4 * (cq >> 1)] : xe[4 * (cq >> 1)];
          if (cq < Q) mma_16816<DT>(accA, af[ph][cq][0], af[ph][cq][1], af[ph][cq][2], af[ph][cq][3], f.x, f.y);
          if (cq > 0) mma_16816<DT>(accB, af[ph][cq - 1][0], af[ph][cq - 1][1], af[ph][cq - 1][2], af[ph][cq - 1][3], f.x, f.y);
        }
      }
      finish(accA, yp, pos);
      finish(accB, yp + 16, pos + 16);
      yp += 256;
      pos += 256;
    }
    __syncwarp();   // everyone is done reading the staged row before the next one overwrites it
  }
}

// Stride-2 depthwise conv (the first encoder block, asr.py:68): one warp per (batch, channel) row,
// the row segment staged in shared memory with coalesced 16-byte loads, each lane producing outputs
// o = oc0 + 32 r + lane so that the 32-bit input words (x[2o+2m], x[2o+2m+1]) are consecutive across lanes.
constexpr int kS2Chunk = 512;                 // outputs per CTA pass
constexpr int kS2Row = 2 * kS2Chunk + 96;     // staged inputs (halo <= 48 each side)
constexpr int kS2MaxWords = 48;               // (k + 1) / 2 + 1 <= 48  ->  k <= 93

template <int DT>
__global__ void __launch_bounds__(kDwWarps * 32)
dw_s2_kernel(const unsigned short* __restrict__ x, long long x_pitch, const unsigned short* __restrict__ w,
             const float* __restrict__ scale, const float* __restrict__ shift, unsigned short* __restrict__ y,
             long long y_pitch, int C, int T_in, int T_out, int k, int act) {
  __shared__ __align__(16) unsigned short xs_all[kDwWarps][kS2Row];
  __shared__ __align__(8) float ws_all[kDwWarps][2 * kS2MaxWords];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.y * kDwWarps + warp;
  pdl_trigger();
  if (c >= C) return;
  const int b = blockIdx.z;
  const int oc0 = blockIdx.x * kS2Chunk;
  const int p = (k - 1) >> 1;
  const int p8 = (p + 7) & ~7;
  const int e = p8 - p;                       // xs[2*ol + j + e] = x[2*(oc0+ol) + j - p]
  unsigned short* xs = xs_all[warp];
  float* ws = ws_all[warp];
  pdl_wait();
  const unsigned short* xrow = x + (static_cast<long long>(b) * C + c) * x_pitch;
  const int ia = 2 * oc0 - p8;
  for (int v = lane; v < kS2Row / 8; v += 32) {
    const int t = ia + v * 8;
    uint4 val = make_uint4(0u, 0u, 0u, 0u);
    if (t >= 0 && t < T_in) {
      val = *reinterpret_cast<const uint4*>(xrow + t);
      if (t + 8 > T_in) {
        uint32_t* u = reinterpret_cast<uint32_t*>(&val);
#pragma unroll
        for (int i = 0; i < 8; ++i)
          if (t + i >= T_in) u[i >> 1] &= (i & 1) ? 0x0000FFFFu : 0xFFFF0000u;
      }
    }
    *reinterpret_cast<uint4*>(xs + v * 8) = val;
  }
  const int n_words = (k + e + 1) >> 1;       // taps j' = j + e in [e, k+e) -> words [0, n_words)
  for (int i = lane; i < 2 * n_words; i += 32) {
    const int j = i - e;
    ws[i] = (j >= 0 && j < k) ? h2f<DT>(w[static_cast<long long>(c) * k + j]) : 0.0f;
  }
  __syncwarp();
  const float sc = scale ? scale[c] : 1.0f, sh = shift[c];
  const uint32_t* xw = reinterpret_cast<const uint32_t*>(xs);
  const float2* w2 = reinterpret_cast<const float2*>(ws);
  unsigned short* yrow = y + (static_cast<long long>(b) * C + c) * y_pitch;
  for (int r0 = 0; r0 < kS2Chunk / 32 && oc0 + r0 * 32 < T_out; r0 += 4) {
    float acc[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    for (int m = 0; m < n_words; ++m) {
      const float2 wm = w2[m];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t v = xw[(r0 + u) * 32 + lane + m];
        acc[u] = fmaf(wm.x, unpack_lo<DT>(v), acc[u]);
        acc[u] = fmaf(wm.y, unpack_hi<DT>(v), acc[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int o = oc0 + (r0 + u) * 32 + lane;
      float v = fmaf(acc[u], sc, sh);
      if (act == V100_ACT_RELU6) v = fminf(fmaxf(v, 0.0f), 6.0f);
      if (o < T_out) yrow[o] = f2h<DT>(v);
    }
  }
}

template <int DT>
__global__ void __launch_bounds__(128)
dw_simt_kernel(const unsigned short* __restrict__ x, long long x_pitch, const unsigned short* __restrict__ w,
               const float* __restrict__ scale, const float* __restrict__ shift, unsigned short* __restrict__ y,
               long long y_pitch, int C, int T_in, int T_out, int k, int stride, int act) {
  const int c = blockIdx.y, b = blockIdx.z;
  const int o0 = (blockIdx.x * 128 + threadIdx.x) * 8;
  pdl_trigger();
  pdl_wait();
  if (o0 >= T_out) return;
  const int p = (k - 1) >> 1;
  const unsigned short* xrow = x + (static_cast<long long>(b) * C + c) * x_pitch;
  const unsigned short* wrow = w + static_cast<long long>(c) * k;
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int j = 0; j < k; ++j) {
    const float wj = h2f<DT>(wrow[j]);
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const int i = (o0 + r) * stride + j - p;
      if (i >= 0 && i < T_in) acc[r] = fmaf(wj, h2f<DT>(xrow[i]), acc[r]);
    }
  }
  const float sc = scale ? scale[c] : 1.0f, sh = shift[c];
  uint32_t o[4];
#pragma unroll
  for (int r = 0; r < 8; r += 2) {
    float v0 = fmaf(acc[r], sc, sh), v1 = fmaf(acc[r + 1], sc, sh);
    if (act == V100_ACT_RELU6) {
      v0 = fminf(fmaxf(v0, 0.0f), 6.0f);
      v1 = fminf(fmaxf(v1, 0.0f), 6.0f);
    }
    o[r >> 1] = pack2<DT>(v0, v1);
  }
  // o0 % 8 == 0 and pitch % 8 == 0, so the 16-byte store stays inside the row's pitch
  *reinterpret_cast<uint4*>(y + (static_cast<long long>(b) * C + c) * y_pitch + o0) = make_uint4(o[0], o[1], o[2], o[3]);
}
template <int NP, bool RELU6, int DT>
static int launch_dw_tc_k(const CUtensorMap& tx, const unsigned short* w, const float* scale, const float* shift,
                          unsigned short* y, long long y_pitch, int B, int C, int T, int k, int N, cudaStream_t stream) {
  auto kern = dw_tc_kernel<NP, RELU6, DT>;
  V100_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmem));
  const int grid = C < num_sms() ? C : num_sms();
  V100_CUDA(launch_pdl(kern, dim3(grid), dim3(384), kTcSmem, stream, tx, w, scale, shift, y, y_pitch, B, C, T, k, N));
  return 0;
}

template <int NP>
static int launch_dw_tc(const CUtensorMap& tx, const unsigned short* w, const float* scale, const float* shift,
                        unsigned short* y, long long y_pitch, int B, int C, int T, int k, int N, int act, int dtype,
                        cudaStream_t stream) {
  if (dtype == DT_F16)
    return act == V100_ACT_RELU6 ? launch_dw_tc_k<NP, true, DT_F16>(tx, w, scale, shift, y, y_pitch, B, C, T, k, N, stream)
                                 : launch_dw_tc_k<NP, false, DT_F16>(tx, w, scale, shift, y, y_pitch, B, C, T, k, N, stream);
  return act == V100_ACT_RELU6 ? launch_dw_tc_k<NP, true, DT_BF16>(tx, w, scale, shift, y, y_pitch, B, C, T, k, N, stream)
                               : launch_dw_tc_k<NP, false, DT_BF16>(tx, w, scale, shift, y, y_pitch, B, C, T, k, N, stream);
}


int dwconv1d(const void* x, int64_t x_pitch, const void* w, const float* scale, const float* shift, void* y,
             int64_t y_pitch, int B, int C, int T_in, int k, int stride, int act, int dtype, int force_simt,
             cudaStream_t stream) {
  if (dtype != DT_BF16 && dtype != DT_F16) return fail(V100_E_INVALID, "dwconv: dtype must be V100_DTYPE_BF16 or V100_DTYPE_F16");
  if (B <= 0 || C <= 0 || T_in <= 0 || k <= 0 || stride <= 0) return fail(V100_E_INVALID, "dwconv: non-positive size");
  if ((k & 1) == 0) return fail(V100_E_UNSUPPORTED, "dwconv: kernel size %d must be odd", k);
  if (x == nullptr || w == nullptr || shift == nullptr || y == nullptr) return fail(V100_E_INVALID, "dwconv: null pointer");
  const int T_out = (T_in - 1) / stride + 1;
  if (x_pitch < T_in || (x_pitch & 7) || y_pitch < T_out || (y_pitch & 7) ||
      (reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(y) & 15))
    return fail(V100_E_INVALID, "dwconv: pitches must be multiples of 8 and >= T, bases 16-byte aligned");
  if (B > 65535 || C > 65535 * kDwWarps) return fail(V100_E_UNSUPPORTED, "dwconv: B or C too large for the grid");
  const int p = (k - 1) / 2;
  const int e1 = (((p + kDwPad) & ~kDwPad) - p) & 1;
  const int Q = (k + 15 + e1 + 15) / 16;
  auto xp = static_cast<const unsigned short*>(x);
  auto wp = static_cast<const unsigned short*>(w);
  auto yp = static_cast<unsigned short*>(y);
  // Stride 1.  Same-box A/B (B = 256, CUDA events): dw_tc_kernel is flat in k (293 us at C = 2048, 153 us at C = 1024,
  // T = 751) and wins from k = 35 up and on the TTS short rows (T = 100 / 292); dw_bulk_kernel, whose cost grows with
  // the filter, still wins for k <= 33 on long rows (k = 19 / 27: 142-147 us, T = 583, k = 7 / 11: 115-119 us vs 126).
  if (!force_simt && stride == 1 && k <= 33 && T_in >= 512 && (C % kDwWarps) == 0) {
    dim3 grid((T_in + kDwChunk - 1) / kDwChunk, C / kDwWarps, (B + kDwRowsPerWarp - 1) / kDwRowsPerWarp);
    const long long xpl = x_pitch, ypl = y_pitch;
#define V100_BULK(QQ, RL, DTT) \
    launch_pdl(dw_bulk_kernel<QQ, RL, DTT>, grid, dim3(kDwWarps * 32), 0, stream, xp, xpl, wp, scale, shift, yp, ypl, B, C, T_in, k)
#define V100_BULK_Q(QQ)                                                                                                   \
    do {                                                                                                                  \
      if (dtype == DT_F16) { if (act == V100_ACT_RELU6) V100_BULK(QQ, true, DT_F16); else V100_BULK(QQ, false, DT_F16); } \
      else { if (act == V100_ACT_RELU6) V100_BULK(QQ, true, DT_BF16); else V100_BULK(QQ, false, DT_BF16); }               \
    } while (0)
    switch (Q) {
      case 1: V100_BULK_Q(1); break;
      case 2: V100_BULK_Q(2); break;
      default: V100_BULK_Q(3); break;
    }
#undef V100_BULK_Q
#undef V100_BULK
  } else if (!force_simt && stride == 1 && p <= 48) {
    // every other stride-1 call: the Toeplitz GEMM on tcgen05 (dw_tc_kernel), N = the utterances of a batch block
    const int N = B >= 128 ? 128 : (B + 15) & ~15;
    const CUtensorMapDataType tt = dtype == DT_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    CUtensorMap tx;
    if (int e = make_tmap_rows(&tx, tt, x, T_in, C, B, x_pitch * 2, 64, N, CU_TENSOR_MAP_SWIZZLE_128B)) return e;
    const long long ypl = y_pitch;
    if (p <= 16) return launch_dw_tc<1>(tx, wp, scale, shift, yp, ypl, B, C, T_in, k, N, act, dtype, stream);
    if (p <= 32) return launch_dw_tc<2>(tx, wp, scale, shift, yp, ypl, B, C, T_in, k, N, act, dtype, stream);
    return launch_dw_tc<3>(tx, wp, scale, shift, yp, ypl, B, C, T_in, k, N, act, dtype, stream);
  } else if (!force_simt && stride == 2 && k <= 59) {
    // polyphase tensor-core kernel: each phase filter has <= 30 taps -> Q <= 3
    const int pp = (k - 1) / 2, p_o = (pp + 1) / 2, zz = p_o & 1;
    const int ke = (k - (pp & 1) + 1) / 2, ko = (k - (1 - (pp & 1)) + 1) / 2;
    const int q_e = (ke + 15 + zz + (pp & 1) + 15) / 16, q_o = (ko + 15 + zz + 15) / 16;
    const int Qs = q_e > q_o ? q_e : q_o;
    dim3 grid((T_out + kDwChunk - 1) / kDwChunk, (C + kDwWarps - 1) / kDwWarps, (B + kDwRowsPerWarp - 1) / kDwRowsPerWarp);
    const long long xpl = x_pitch, ypl = y_pitch;
    // 16-byte loads per row of the longest chunk (the kernel's n_vec), which sizes the register prefetch
    const int len0 = T_out < kDwChunk ? T_out : kDwChunk;
    const bool small = 4 * (16 * ((len0 + 14 + 255) / 256) + 3) <= 7 * 32;
#define V100_S2(QQ, NV)                                                                                                     \
    do {                                                                                                                    \
      if (dtype == DT_F16)                                                                                                  \
        launch_pdl(dw_s2_mma_kernel<QQ, DT_F16, NV>, grid, dim3(kDwWarps * 32), 0, stream, xp, xpl, wp, scale, shift, yp, ypl, B, C, T_in, T_out, k, act); \
      else                                                                                                                  \
        launch_pdl(dw_s2_mma_kernel<QQ, DT_BF16, NV>, grid, dim3(kDwWarps * 32), 0, stream, xp, xpl, wp, scale, shift, yp, ypl, B, C, T_in, T_out, k, act); \
    } while (0)
    if (Qs <= 2) { if (small) V100_S2(2, 7); else V100_S2(2, 11); }
    else { if (small) V100_S2(3, 7); else V100_S2(3, 11); }
#undef V100_S2
  } else if (!force_simt && stride == 2 && k <= 2 * kS2MaxWords - 3) {
    dim3 grid((T_out + kS2Chunk - 1) / kS2Chunk, (C + kDwWarps - 1) / kDwWarps, B);
    const long long xpl = x_pitch, ypl = y_pitch;
    if (dtype == DT_F16)
      launch_pdl(dw_s2_kernel<DT_F16>, grid, dim3(kDwWarps * 32), 0, stream, xp, xpl, wp, scale, shift, yp, ypl, C, T_in, T_out, k, act);
    else
      launch_pdl(dw_s2_kernel<DT_BF16>, grid, dim3(kDwWarps * 32), 0, stream, xp, xpl, wp, scale, shift, yp, ypl, C, T_in, T_out, k, act);
  } else {
    dim3 grid((T_out + 1023) / 1024, C, B);
    const long long xpl = x_pitch, ypl = y_pitch;
    if (dtype == DT_F16)
      launch_pdl(dw_simt_kernel<DT_F16>, grid, dim3(128), 0, stream, xp, xpl, wp, scale, shift, yp, ypl, C, T_in, T_out, k, stride, act);
    else
      launch_pdl(dw_simt_kernel<DT_BF16>, grid, dim3(128), 0, stream, xp, xpl, wp, scale, shift, yp, ypl, C, T_in, T_out, k, stride, act);
  }
  V100_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace v100
