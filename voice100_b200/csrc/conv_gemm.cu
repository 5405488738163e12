// Pointwise / multi-tap Conv1d as a persistent, warp-specialised tcgen05 GEMM (sm_100a).
//
//   D[acc(tap)][co][t] += sum_ci  W[co][tap*C_in + ci] * X[b][xrow(tap) + ci][t]
// (1x1 conv: one tap; ConvTranspose1d k5/s2: five taps over a [x(t+1) | x(t) | x(t-1)] channel stack --
//  TMA needs 16-byte aligned inner coordinates, so +-1 time shifts cannot be expressed as box offsets.)
//
// Operand roles: the WEIGHTS are the UMMA "A" operand (M = 128 output channels, K-major, 128B swizzle),
// the ACTIVATIONS are the "B" operand (N = 128/256 time steps, MN-major because NCW keeps time
// contiguous, 128B swizzle).  Accumulators live in TMEM (lane = output channel, column = time), double
// buffered so the epilogue of tile i overlaps the MMAs of tile i+1.
//
// CG == 2 (cta_group::2): a CTA pair computes a 256-channel x 256-step tile.  Each CTA stages its own 128
// weight rows and its own 128 time columns, the pair's leader issues one 256-row UMMA that reads both
// CTAs' shared memory, and each CTA drains its own 128 accumulator rows.  Per output element this moves
// 1.5x fewer operand bytes from L2 to shared memory than the single-CTA tile -- the first working
// version of this kernel measured ~10.7 TB/s of L2->SM operand traffic, i.e. it was L2-bound.
//
// WRES (weights resident): for C_in <= 512 a CTA pair keeps its 256 x C_in weight block in TENSOR MEMORY for the whole
// kernel (tcgen05.mma with the A operand from TMEM, 16-bit elements packed two per column) and works only on tiles of
// that channel block; the ring then carries activations only.  ncu on the plain pair kernel (profiles/r02_gemm_stalls.md):
// the MMA warp spends 55 % of its time waiting for operand bytes while the producer waits for free slots -- a 256 x 256
// tile needs 64 B/clk/SM of operands (32 KB per 512 clk k-block) and gets 52-58.  Without the weights a k-block moves
// half the bytes through L2, the TMA unit and shared memory, so the same ring covers twice the MMA time (ncu: -23 %
// cycles, tensor pipe 91 % busy; the wall-clock gain is 10 % because the full chip is then held back by the power limit).
// Tiles are 256 channels x 128 steps (two 128-column accumulators + C_in/2 weight columns = 512 TMEM columns at C_in = 512).
//
// Warp roles (384 threads): warp 0 = TMA producer, warp 1 = MMA issuer (one thread), warp 2 = TMEM
// allocator, warp 3 = idle, warps 4..11 = epilogue (two groups of four warps; warp%4 selects the TMEM
// lane quadrant it is allowed to read).
//
// Epilogues:
//   OUT_BF16: y = act(scale*acc + shift) (+ residual) -> bf16.  Each epilogue warp stages its own
//             [32 channels x 64 steps] sub-tiles in 128B-swizzled smem and TMA-stores them; the residual
//             sub-tile is TMA-loaded into the same slot one chunk ahead.  With N_ACC == 2 (ConvTranspose1d k5 s2) the even/odd output phases are two
//             accumulators interleaved here.
//   OUT_F32 : y = acc + bias -> fp32 NCW, direct 16-byte stores (the small biased heads).
#include "common.cuh"
#include "host.h"

namespace v100 {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;
constexpr int kATileBytes = kBlockM * kBlockK * 2;  // 16 KB
constexpr int kBAtomBytes = kBlockK * 64 * 2;       // 8 KB: 64 k-rows x 64 time steps
constexpr int kChunkBytes = kBlockM * 64 * 2;       // 16 KB: 128 channels x 64 time steps
constexpr int kWarpChunkBytes = 32 * 64 * 2;        // 4 KB: one epilogue warp's 32 channels x 64 time steps
constexpr int kMaxTaps = 5;
constexpr int kGemmThreads = 384;
constexpr int kEpiWarps = 8;

enum { OUT_BF16 = 0, OUT_F32 = 1 };

struct GemmParams {
  int C_out, C_in, B;
  int m_tiles, t_tiles, num_tiles, k_blocks;
  int n_taps;
  int tap_xrow[kMaxTaps];   // first X channel row of the tap
  int tap_col[kMaxTaps];    // column (time) offset of the tap; must keep the box 16-byte aligned
  int tap_acc[kMaxTaps];
  const float* scale;
  const float* shift;
  int act;
  int has_res;
  int dtype;                // DT_BF16 / DT_F16: storage type of x, W, y, res
  float* y32;
  long long y32_pitch;
  const unsigned short* w_raw;  // WRES: the row-major [C_out][C_in] weights themselves
};

// Walks this CTA's tiles (tile, tile + step, ...) keeping tile = (b * t_tiles + t) * m_tiles + m decomposed, so the
// per-tile divisions (two in the producer, three per epilogue chunk: ~50 SASS instructions each time) are done once.
struct TileWalk {
  int m, t, b;      // current tile
  int sm, st, sb;   // the step in the mixed radix (m_tiles, t_tiles)
  __device__ __forceinline__ void init(int tile, int step, int m_tiles, int t_tiles) {
    m = tile % m_tiles; int r = tile / m_tiles; t = r % t_tiles; b = r / t_tiles;
    sm = step % m_tiles; r = step / m_tiles; st = r % t_tiles; sb = r / t_tiles;
  }
  __device__ __forceinline__ void next(int m_tiles, int t_tiles) {
    m += sm;
    int c = m >= m_tiles ? 1 : 0;
    m -= c ? m_tiles : 0;
    t += st + c;
    c = t >= t_tiles ? 1 : 0;
    t -= c ? t_tiles : 0;
    b += sb + c;
  }
};

// epilogue variant bits (compile time: the generic epilogue was ~2000 SASS instructions of run-time branches and the
// epilogue warps spent 28 % of their samples on instruction fetch)
enum { EPI_RELU6 = 1, EPI_RES = 2, EPI_F16 = 4 };

template <int BLOCK_N, int N_ACC, int OUT_MODE, int STAGES, int CG = 1, bool WRES = false>
struct GemmCfg {
  static constexpr int kBCols = BLOCK_N / CG;  // time columns this CTA stages per k-block
  static constexpr int kStageK = WRES ? 128 : kBlockK;  // K extent of one ring stage
  static constexpr int kStageBytes = WRES ? kStageK * 64 * 2 * (kBCols / 64) : kATileBytes + (kBCols / 64) * kBAtomBytes;
  static constexpr int kWCol0 = 2 * N_ACC * BLOCK_N;  // WRES: first TMEM column of the resident weights
  static constexpr int kStagingBytes = OUT_MODE == OUT_BF16 ? 4 * kChunkBytes : 0;
  // mbarriers: full/empty per stage, 2 + 2 for the accumulators, 2 per epilogue warp for the residual tiles, + the TMEM slot
  static constexpr int kBarBytes = ((2 * STAGES + 4 + 2 * kEpiWarps) * 8 + 8 + 127) & ~127;
  static constexpr int kSmemBytes = 1024 + STAGES * kStageBytes + kStagingBytes + kBarBytes;
  static constexpr int kTmemCols = WRES ? 512 : 2 * N_ACC * BLOCK_N;
  static_assert(!WRES || (CG == 2 && BLOCK_N == 128 && N_ACC == 1), "WRES: CTA pairs, 128-column tiles");
  static constexpr int kOutCols = N_ACC * BLOCK_N;       // output time steps per tile
  static constexpr int kChunksPerGroup = kOutCols / 128;  // 64-column chunks per epilogue group per tile
  static_assert(kTmemCols == 512 || kTmemCols == 256, "TMEM allocation must be a power of two");
  static_assert(kSmemBytes <= 232448, "exceeds 227 KB of shared memory");
};

template <int BLOCK_N, int N_ACC, int OUT_MODE, int STAGES, int CG, int EPI, bool WRES>
__device__ __forceinline__ void conv_gemm_body(const CUtensorMap& tm_w, const CUtensorMap& tm_x,
                                               const CUtensorMap& tm_y, const CUtensorMap& tm_res,
                                               const GemmParams& p) {
  using Cfg = GemmCfg<BLOCK_N, N_ACC, OUT_MODE, STAGES, CG, WRES>;
  static_assert(CG == 1 || (N_ACC == 1 && OUT_MODE == OUT_BF16), "the CTA-pair path serves the plain bf16 conv");
  constexpr bool kRelu6 = (EPI & EPI_RELU6) != 0, kRes = (EPI & EPI_RES) != 0;
  constexpr int DT = (EPI & EPI_F16) ? DT_F16 : DT_BF16;
  const uint32_t cta_rank = CG == 2 ? cluster_ctarank() : 0u;
  const bool leader = cta_rank == 0;
  // WRES: gridDim.x / CG is a multiple of m_tiles, so `tile % m_tiles` is the same for every tile of this CTA
  const int tile0 = blockIdx.x / CG, tile_step = gridDim.x / CG;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* staging = smem + STAGES * Cfg::kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + Cfg::kStagingBytes);
  uint64_t* full_bar = bars;                    // [STAGES]
  uint64_t* empty_bar = bars + STAGES;          // [STAGES]
  uint64_t* tmem_full = bars + 2 * STAGES;      // [2]
  uint64_t* tmem_empty = bars + 2 * STAGES + 2; // [2]
  uint64_t* res_bar = bars + 2 * STAGES + 4;    // [8 epilogue warps][2 buffers]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4 + 2 * kEpiWarps);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);  // provably warp-uniform for the compiler
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    if (!WRES) tma_prefetch_desc(&tm_w);
    tma_prefetch_desc(&tm_x);
    if (OUT_MODE == OUT_BF16) {
      tma_prefetch_desc(&tm_y);
      if (kRes) tma_prefetch_desc(&tm_res);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], kEpiWarps * CG);  // the leader's copy collects both CTAs' epilogue warps
    }
    for (int i = 0; i < 2 * kEpiWarps; ++i) mbar_init(&res_bar[i], 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    if constexpr (CG == 2) {
      tmem_alloc_cg2(tmem_slot, Cfg::kTmemCols);
      tmem_relinquish_cg2();
    } else {
      tmem_alloc(tmem_slot, Cfg::kTmemCols);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if constexpr (WRES) {
    // This CTA's 128 weight rows -> tensor memory, straight from global memory: TMEM lane = output channel, and a
    // row-major 16-bit row already is "two K elements per 32-bit column".  The two epilogue warps of a lane quadrant
    // alternate 32-column blocks.
    if (warp >= 4) {
      const int q = warp & 3, g = (warp - 4) >> 2;
      const int ch = ((tile0 % p.m_tiles) * CG + int(cta_rank)) * kBlockM + q * 32 + lane;
      const uint4* wrow = reinterpret_cast<const uint4*>(p.w_raw + static_cast<long long>(ch) * p.C_in);
      for (int c0 = g * 32; c0 < p.C_in / 2; c0 += 64) {
        uint32_t r[32];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const uint4 v = __ldg(wrow + (c0 >> 2) + i);
          r[4 * i] = v.x; r[4 * i + 1] = v.y; r[4 * i + 2] = v.z; r[4 * i + 3] = v.w;
        }
        tmem_st32(tmem_base + (uint32_t(q * 32) << 16) + Cfg::kWCol0 + c0, r);
      }
      tmem_st_wait();
    }
    tc_fence_before();
    cluster_sync_all();   // the leader's MMAs read both CTAs' halves
    tc_fence_after();
  }

  if (warp == 0) {
    // ===================== TMA producer =====================
    // The whole warp walks the loop and one elected lane issues: the coordinates and descriptors stay
    // warp-uniform (uniform registers) instead of being moved there lane by lane in front of every TMA/MMA
    // instruction (measured on the LSTM kernel: 37 ns per MMA issued from a single divergent lane).
    const bool issuer = elect_one();
    {
      int stage = 0;
      uint32_t phase = 0;
      TileWalk tw;
      tw.init(tile0, tile_step, p.m_tiles, p.t_tiles);
      for (int tile = tile0; tile < p.num_tiles; tile += tile_step, tw.next(p.m_tiles, p.t_tiles)) {
        const int t_tile = tw.t, b = tw.b;
        const int m0 = (tw.m * CG + int(cta_rank)) * kBlockM;
        for (int tap = 0; tap < p.n_taps; ++tap) {
          const int t_in0 = t_tile * BLOCK_N + int(cta_rank) * Cfg::kBCols + p.tap_col[tap];
          const int xrow0 = p.tap_xrow[tap];
          for (int kb = 0; kb < p.k_blocks; ++kb) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* sa = smem + stage * Cfg::kStageBytes;
            if (issuer) {
              if constexpr (WRES) {
                // activations only: one [128 k rows x 64 steps] box per CTA, credited to the leader's barrier
                if (leader) mbar_expect_tx(&full_bar[stage], 2 * Cfg::kStageBytes);
                const uint32_t fb = mapa_u32(smem_u32(&full_bar[stage]), 0);
                tma_load_3d_cg2(sa, &tm_x, fb, t_in0, xrow0 + kb * Cfg::kStageK, b);
              } else if constexpr (CG == 2) {
                uint8_t* sb = sa + kATileBytes;
                // both CTAs' bytes are credited to the LEADER's full barrier (the MMA issuer waits there)
                if (leader) mbar_expect_tx(&full_bar[stage], 2 * Cfg::kStageBytes);
                const uint32_t fb = mapa_u32(smem_u32(&full_bar[stage]), 0);
                tma_load_2d_cg2(sa, &tm_w, fb, tap * p.C_in + kb * kBlockK, m0);
#pragma unroll
                for (int a = 0; a < Cfg::kBCols / 64; ++a)
                  tma_load_3d_cg2(sb + a * kBAtomBytes, &tm_x, fb, t_in0 + a * 64, xrow0 + kb * kBlockK, b);
              } else {
                uint8_t* sb = sa + kATileBytes;
                mbar_expect_tx(&full_bar[stage], Cfg::kStageBytes);
                tma_load_2d(sa, &tm_w, &full_bar[stage], tap * p.C_in + kb * kBlockK, m0);
#pragma unroll
                for (int a = 0; a < Cfg::kBCols / 64; ++a)
                  tma_load_3d(sb + a * kBAtomBytes, &tm_x, &full_bar[stage], t_in0 + a * 64, xrow0 + kb * kBlockK, b);
              }
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (leader) {
      // ===================== MMA issuer (the pair's leader only; whole warp, one elected lane) =====================
      const bool issuer = elect_one();
      // kind::f16 instruction descriptor: D=f32, A=B=bf16, A K-major, B MN-major, M=128*CG, N=BLOCK_N
      // (format code: 1 = bf16, 0 = fp16)
      const uint32_t fmt = p.dtype == DT_F16 ? 0u : 1u;
      const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | (0u << 15) | (1u << 16) |
                             (uint32_t(BLOCK_N >> 3) << 17) | (uint32_t((kBlockM * CG) >> 4) << 24);
      int stage = 0;
      uint32_t phase = 0;
      int iter = 0;
      for (int tile = tile0; tile < p.num_tiles; tile += tile_step, ++iter) {
        const int accbuf = iter & 1;
        const uint32_t acc_phase = (iter >> 1) & 1;
        mbar_wait(&tmem_empty[accbuf], acc_phase ^ 1);
        tc_fence_after();
        uint32_t used = 0;
        for (int tap = 0; tap < p.n_taps; ++tap) {
          const int acc = p.tap_acc[tap];
          const uint32_t d_tmem = tmem_base + accbuf * (N_ACC * BLOCK_N) + acc * BLOCK_N;
          for (int kb = 0; kb < p.k_blocks; ++kb) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            const uint32_t a_addr = smem_u32(smem + stage * Cfg::kStageBytes);
            if constexpr (WRES) {
              // A from tensor memory: 8 columns per K = 16 step; B: MN-major SW128, 16 k rows = 2048 B per K step
              const uint32_t a_tmem = tmem_base + Cfg::kWCol0 + kb * (Cfg::kStageK / 2);
#pragma unroll
              for (int k = 0; k < Cfg::kStageK / 16; ++k) {
                const uint64_t db = umma_desc(a_addr + k * 2048, kBAtomBytes, 1024);
                if (issuer) umma_ts_cg2(d_tmem, a_tmem + k * 8, db, idesc, ((used >> acc) & 1u) | (k > 0 ? 1u : 0u));
              }
            } else {
              const uint32_t b_addr = a_addr + kATileBytes;
#pragma unroll
              for (int k = 0; k < kBlockK / 16; ++k) {
                // A: K-major SW128 (8-row groups 1024 B apart; +32 B per 16-element K step inside the atom)
                const uint64_t da = umma_desc(a_addr + k * 32, 16, 1024);
                // B: MN-major SW128 (64-time atoms 8 KB apart = LBO; 8-k-row groups 1024 B apart = SBO;
                //    16 k rows = 2048 B per K step)
                const uint64_t db = umma_desc(b_addr + k * 2048, kBAtomBytes, 1024);
                if (issuer) {
                  if constexpr (CG == 2) umma_bf16_cg2(d_tmem, da, db, idesc, ((used >> acc) & 1u) | (k > 0 ? 1u : 0u));
                  else umma_bf16(d_tmem, da, db, idesc, ((used >> acc) & 1u) | (k > 0 ? 1u : 0u));
                }
              }
            }
            used |= 1u << acc;
            // frees the smem slot (in both CTAs of a pair) once these MMAs have read it
            if (issuer) {
              if constexpr (CG == 2) umma_commit_cg2(&empty_bar[stage]); else umma_commit(&empty_bar[stage]);
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
        if (issuer) {
          if constexpr (CG == 2) umma_commit_cg2(&tmem_full[accbuf]); else umma_commit(&tmem_full[accbuf]);
        }
        __syncwarp();
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue =====================
    const int q = warp & 3;             // TMEM lane quadrant this warp may access
    const int g = (warp - 4) >> 2;      // epilogue group
    const int row = q * 32 + lane;      // accumulator row == output channel within the tile
    const uint32_t lane_addr = tmem_base + (uint32_t(q * 32) << 16);

    if constexpr (OUT_MODE == OUT_BF16) {
      // Every epilogue warp is its own pipeline: it owns 32 accumulator rows (its TMEM lane quadrant) and
      // the 64-column chunks c = h, h+2, ... of the tile; it stages each [32 x 64] bf16 sub-tile in its
      // private, 128B-swizzled, double-buffered 4 KB smem slot and TMA-stores it.  No cross-warp barriers.
      constexpr int CPG = Cfg::kChunksPerGroup;
      const int h = g;                                   // which half of the tile's chunks
      uint8_t* stg = staging + (warp - 4) * 2 * kWarpChunkBytes;
      uint64_t* rbar = res_bar + (warp - 4) * 2;
      // this lane's staged row (128 bytes) with the 128B-swizzle term folded in: 16-byte piece k16 lives at row ^ (k16 << 4)
      const uint32_t row_s = smem_u32(stg) + uint32_t(lane) * 128u + (uint32_t(lane & 7) << 4);
      const uint32_t tmem_empty_leader = CG == 2 ? mapa_u32(smem_u32(&tmem_empty[0]), 0) : 0u;

      // one elected lane of the (converged) warp issues every TMA operation of this warp; bulk async-groups are
      // per thread, so the same lane also commits and waits
      const bool issuer = elect_one();
      TileWalk tw;
      tw.init(tile0, tile_step, p.m_tiles, p.t_tiles);
      if (kRes && issuer && tile0 < p.num_tiles) {
        mbar_expect_tx(&rbar[0], kWarpChunkBytes);
        tma_load_3d(stg, &tm_res, &rbar[0], tw.t * Cfg::kOutCols + h * 64,
                    (tw.m * CG + int(cta_rank)) * kBlockM + q * 32, tw.b);
      }
      // per-channel BN scalars of a tile; loaded one tile ahead so their L2 latency is off the critical
      // path (ncu: the wait for these two loads was 16 % of the kernel's stall samples on the expand layers)
      auto load_scalars = [&](bool in_range, int m_tile, float& sc_o, float& sh_o) {
        const int ch_t = (m_tile * CG + int(cta_rank)) * kBlockM + q * 32 + lane;
        const bool live = in_range && ch_t < p.C_out;
        sc_o = (live && p.scale != nullptr) ? __ldg(p.scale + ch_t) : 1.0f;
        sh_o = live ? __ldg(p.shift + ch_t) : 0.0f;
      };
      // eight accumulator columns -> one 16-byte piece of this lane's staged row (shared-space accesses: the generic
      // form cost a 64-bit address and an address-space check per store)
      auto emit8 = [&](const float (&a)[8], uint32_t dst) {
        float o[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) o[e] = a[e];
        uint4 w;
        if constexpr (!kRes) {
          if constexpr (kRelu6) {
            w.x = pack2_relu6<DT>(o[0], o[1]); w.y = pack2_relu6<DT>(o[2], o[3]);
            w.z = pack2_relu6<DT>(o[4], o[5]); w.w = pack2_relu6<DT>(o[6], o[7]);
          } else {
            w.x = pack2<DT>(o[0], o[1]); w.y = pack2<DT>(o[2], o[3]);
            w.z = pack2<DT>(o[4], o[5]); w.w = pack2<DT>(o[6], o[7]);
          }
        } else {
          if constexpr (kRelu6) {
#pragma unroll
            for (int e = 0; e < 8; ++e) o[e] = fminf(fmaxf(o[e], 0.0f), 6.0f);
          }
          uint4 rr;
          asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(rr.x), "=r"(rr.y), "=r"(rr.z), "=r"(rr.w) : "r"(dst) : "memory");
          o[0] += unpack_lo<DT>(rr.x); o[1] += unpack_hi<DT>(rr.x);
          o[2] += unpack_lo<DT>(rr.y); o[3] += unpack_hi<DT>(rr.y);
          o[4] += unpack_lo<DT>(rr.z); o[5] += unpack_hi<DT>(rr.z);
          o[6] += unpack_lo<DT>(rr.w); o[7] += unpack_hi<DT>(rr.w);
          w.x = pack2<DT>(o[0], o[1]); w.y = pack2<DT>(o[2], o[3]);
          w.z = pack2<DT>(o[4], o[5]); w.w = pack2<DT>(o[6], o[7]);
        }
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(w.x), "r"(w.y), "r"(w.z), "r"(w.w) : "memory");
      };
      float sc, sh;
      load_scalars(tile0 < p.num_tiles, tw.m, sc, sh);
      int iter = 0;
      uint32_t n = 0;  // chunk sequence number of this warp
      for (int tile = tile0; tile < p.num_tiles; tile += tile_step, ++iter) {
        const int t_tile = tw.t, b = tw.b;
        const int accbuf = iter & 1;
        const int m0 = (tw.m * CG + int(cta_rank)) * kBlockM + q * 32;
        tw.next(p.m_tiles, p.t_tiles);               // tw now describes the NEXT tile of this CTA
        float sc_next, sh_next;
        load_scalars(tile + tile_step < p.num_tiles, tw.m, sc_next, sh_next);
        mbar_wait(&tmem_full[accbuf], (iter >> 1) & 1);
        tc_fence_after();
#pragma unroll
        for (int i = 0; i < CPG; ++i, ++n) {
          const int c = h + 2 * i;  // 64-column output chunk of this tile
          const int buf = n & 1;
          uint32_t v0[32], v1[32];
          const uint32_t col0 = accbuf * (N_ACC * BLOCK_N);
          const uint32_t rowp = row_s + uint32_t(buf) * kWarpChunkBytes;
          auto release_acc = [&]() {
            if (i == CPG - 1) {  // this warp is done reading the accumulator buffer
              tc_fence_before();
              __syncwarp();
              if (lane == 0) {
                if constexpr (CG == 2) mbar_arrive_cluster(tmem_empty_leader + accbuf * 8);
                else mbar_arrive(&tmem_empty[accbuf]);
              }
            }
          };
          if constexpr (N_ACC == 1) {
            // the second half of the chunk is in flight while the first half is converted and staged
            tmem_ld32(lane_addr + col0 + c * 64, v0);
            tmem_ld_wait();
            tmem_ld_fence(v0);
            tmem_ld32(lane_addr + col0 + c * 64 + 32, v1);
            // slot `buf` is free: lane 0 waited for its previous TMA store before the __syncwarp that ended
            // the previous chunk.  With a residual it now holds this chunk's residual sub-tile.
            if constexpr (kRes) mbar_wait(&rbar[buf], (n >> 1) & 1);
#pragma unroll
            for (int k16 = 0; k16 < 4; ++k16) {
              float a[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) a[e] = fmaf(__uint_as_float(v0[k16 * 8 + e]), sc, sh);
              emit8(a, rowp ^ (uint32_t(k16) << 4));
            }
            tmem_ld_wait();
            tmem_ld_fence(v1);
            release_acc();
#pragma unroll
            for (int k16 = 4; k16 < 8; ++k16) {
              float a[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) a[e] = fmaf(__uint_as_float(v1[(k16 - 4) * 8 + e]), sc, sh);
              emit8(a, rowp ^ (uint32_t(k16) << 4));
            }
          } else {
            tmem_ld32(lane_addr + col0 + c * 32, v0);            // even output phase
            tmem_ld32(lane_addr + col0 + BLOCK_N + c * 32, v1);  // odd output phase
            tmem_ld_wait();
            release_acc();
            if constexpr (kRes) mbar_wait(&rbar[buf], (n >> 1) & 1);
#pragma unroll
            for (int k16 = 0; k16 < 8; ++k16) {
              float a[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const int j = k16 * 4 + (e >> 1);
                a[e] = fmaf(__uint_as_float((e & 1) ? v1[j] : v0[j]), sc, sh);
              }
              emit8(a, rowp ^ (uint32_t(k16) << 4));
            }
          }
          fence_proxy_async();
          __syncwarp();
          if (issuer) {
            tma_store_3d(&tm_y, stg + buf * kWarpChunkBytes, t_tile * Cfg::kOutCols + c * 64, m0, b);
            tma_store_commit();
            tma_store_wait_read<1>();  // every store but the newest has finished reading smem: buf^1 is free
            if constexpr (kRes) {
              if (i < CPG - 1) {                      // next chunk of this tile
                mbar_expect_tx(&rbar[buf ^ 1], kWarpChunkBytes);
                tma_load_3d(stg + (buf ^ 1) * kWarpChunkBytes, &tm_res, &rbar[buf ^ 1],
                            t_tile * Cfg::kOutCols + (c + 2) * 64, m0, b);
              } else if (tile + tile_step < p.num_tiles) {   // first chunk of the next tile (tw already points at it)
                mbar_expect_tx(&rbar[buf ^ 1], kWarpChunkBytes);
                tma_load_3d(stg + (buf ^ 1) * kWarpChunkBytes, &tm_res, &rbar[buf ^ 1],
                            tw.t * Cfg::kOutCols + h * 64, (tw.m * CG + int(cta_rank)) * kBlockM + q * 32, tw.b);
              }
            }
          }
          __syncwarp();
        }
        sc = sc_next;
        sh = sh_next;
      }
      if (issuer) tma_store_wait_all<0>();
    } else {
      // fp32 NCW direct store, bias only; group g owns columns [g*BLOCK_N/2, (g+1)*BLOCK_N/2)
      int iter = 0;
      for (int tile = tile0; tile < p.num_tiles; tile += tile_step, ++iter) {
        const int m_tile = tile % p.m_tiles;
        const int r = tile / p.m_tiles;
        const int t_tile = r % p.t_tiles;
        const int b = r / p.t_tiles;
        const int accbuf = iter & 1;
        const int ch = m_tile * kBlockM + row;
        const bool live = ch < p.C_out;
        const float bias = live ? __ldg(p.shift + ch) : 0.0f;
        float* yrow = p.y32 + (static_cast<long long>(b) * p.C_out + (live ? ch : 0)) * p.y32_pitch;
        mbar_wait(&tmem_full[accbuf], (iter >> 1) & 1);
        tc_fence_after();
#pragma unroll
        for (int cc = 0; cc < BLOCK_N / 64; ++cc) {
          const int col = g * (BLOCK_N / 2) + cc * 32;
          uint32_t v[32];
          tmem_ld32(lane_addr + accbuf * (N_ACC * BLOCK_N) + col, v);
          tmem_ld_wait();
          if (cc == BLOCK_N / 64 - 1) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[accbuf]);
          }
          if (live) {
            const long long t0 = static_cast<long long>(t_tile) * BLOCK_N + col;
#pragma unroll
            for (int k4 = 0; k4 < 8; ++k4) {
              if (t0 + 4 * k4 < p.y32_pitch) {
                float4 o;
                o.x = __uint_as_float(v[4 * k4 + 0]) + bias;
                o.y = __uint_as_float(v[4 * k4 + 1]) + bias;
                o.z = __uint_as_float(v[4 * k4 + 2]) + bias;
                o.w = __uint_as_float(v[4 * k4 + 3]) + bias;
                *reinterpret_cast<float4*>(yrow + t0 + 4 * k4) = o;
              }
            }
          }
        }
      }
    }
  }

  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    if constexpr (CG == 2) tmem_dealloc_cg2(tmem_base, Cfg::kTmemCols); else tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

template <int BLOCK_N, int N_ACC, int OUT_MODE, int STAGES, int EPI>
__global__ void __launch_bounds__(kGemmThreads, 1)
conv_gemm_kernel(const __grid_constant__ CUtensorMap tm_w, const __grid_constant__ CUtensorMap tm_x,
                 const __grid_constant__ CUtensorMap tm_y, const __grid_constant__ CUtensorMap tm_res,
                 const GemmParams p) {
  conv_gemm_body<BLOCK_N, N_ACC, OUT_MODE, STAGES, 1, EPI, false>(tm_w, tm_x, tm_y, tm_res, p);
}

// CTA-pair variant: 256 output channels x BLOCK_N (256, or 128 for short rows) time steps per cluster of two CTAs
template <int BLOCK_N, int STAGES, int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemmThreads, 1)
conv_gemm_pair_kernel(const __grid_constant__ CUtensorMap tm_w, const __grid_constant__ CUtensorMap tm_x,
                      const __grid_constant__ CUtensorMap tm_y, const __grid_constant__ CUtensorMap tm_res,
                      const GemmParams p) {
  conv_gemm_body<BLOCK_N, 1, OUT_BF16, STAGES, 2, EPI, false>(tm_w, tm_x, tm_y, tm_res, p);
}

// CTA-pair variant with the pair's weight block resident in tensor memory: 256 channels x 128 steps per tile
template <int STAGES, int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemmThreads, 1)
conv_gemm_wres_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_y,
                      const __grid_constant__ CUtensorMap tm_res, const GemmParams p) {
  conv_gemm_body<128, 1, OUT_BF16, STAGES, 2, EPI, true>(tm_x, tm_x, tm_y, tm_res, p);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------

static int epi_of(const GemmParams& p) {
  return (p.act == V100_ACT_RELU6 ? EPI_RELU6 : 0) | (p.has_res ? EPI_RES : 0) | (p.dtype == DT_F16 ? EPI_F16 : 0);
}

template <int BLOCK_N, int N_ACC, int OUT_MODE, int STAGES, int EPI>
static int launch_gemm_e(const CUtensorMap& tw, const CUtensorMap& tx, const CUtensorMap& ty, const CUtensorMap& tr,
                         const GemmParams& p, cudaStream_t stream) {
  using Cfg = GemmCfg<BLOCK_N, N_ACC, OUT_MODE, STAGES>;
  auto kern = conv_gemm_kernel<BLOCK_N, N_ACC, OUT_MODE, STAGES, EPI>;
  static thread_local int configured_dev = -1;
  int dev = 0;
  V100_CUDA(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    V100_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    configured_dev = dev;
  }
  const int grid = p.num_tiles < num_sms() ? p.num_tiles : num_sms();
  kern<<<dim3(grid), dim3(kGemmThreads), Cfg::kSmemBytes, stream>>>(tw, tx, ty, tr, p);
  V100_CUDA(cudaGetLastError());
  return 0;
}

// run-time epilogue flags -> the compile-time variant
#define V100_EPI_DISPATCH(FN, ...)                      \
  switch (epi_of(p)) {                                  \
    case 0: return FN<__VA_ARGS__, 0>(V100_EPI_ARGS);   \
    case 1: return FN<__VA_ARGS__, 1>(V100_EPI_ARGS);   \
    case 2: return FN<__VA_ARGS__, 2>(V100_EPI_ARGS);   \
    case 3: return FN<__VA_ARGS__, 3>(V100_EPI_ARGS);   \
    case 4: return FN<__VA_ARGS__, 4>(V100_EPI_ARGS);   \
    case 5: return FN<__VA_ARGS__, 5>(V100_EPI_ARGS);   \
    case 6: return FN<__VA_ARGS__, 6>(V100_EPI_ARGS);   \
    default: return FN<__VA_ARGS__, 7>(V100_EPI_ARGS);  \
  }

template <int BLOCK_N, int N_ACC, int OUT_MODE, int STAGES>
static int launch_gemm(const CUtensorMap& tw, const CUtensorMap& tx, const CUtensorMap& ty, const CUtensorMap& tr,
                       const GemmParams& p, cudaStream_t stream) {
#define V100_EPI_ARGS tw, tx, ty, tr, p, stream
  if constexpr (OUT_MODE == OUT_F32) {
    return launch_gemm_e<BLOCK_N, N_ACC, OUT_MODE, STAGES, 0>(V100_EPI_ARGS);
  } else if constexpr (N_ACC == 2) {  // transposed conv: bias only
    if (p.act != V100_ACT_NONE || p.has_res) return fail(V100_E_UNSUPPORTED, "two-phase GEMM: bias-only epilogue");
    if (p.dtype == DT_F16) return launch_gemm_e<BLOCK_N, N_ACC, OUT_MODE, STAGES, EPI_F16>(V100_EPI_ARGS);
    return launch_gemm_e<BLOCK_N, N_ACC, OUT_MODE, STAGES, 0>(V100_EPI_ARGS);
  } else {
    V100_EPI_DISPATCH(launch_gemm_e, BLOCK_N, N_ACC, OUT_MODE, STAGES)
  }
#undef V100_EPI_ARGS
}

constexpr int kPairStages = 5;      // 256-column tiles: 32 KB per stage
constexpr int kPairStages128 = 6;   // 128-column tiles: 24 KB per stage

template <int BLOCK_N, int STAGES, int EPI>
static int launch_gemm_pair_e(const CUtensorMap& tw, const CUtensorMap& tx, const CUtensorMap& ty,
                              const CUtensorMap& tr, const GemmParams& p, cudaStream_t stream) {
  using Cfg = GemmCfg<BLOCK_N, 1, OUT_BF16, STAGES, 2>;
  auto kern = conv_gemm_pair_kernel<BLOCK_N, STAGES, EPI>;
  static thread_local int configured_dev = -1;
  int dev = 0;
  V100_CUDA(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    V100_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    configured_dev = dev;
  }
  int pairs = num_sms() / 2;
  if (p.num_tiles < pairs) pairs = p.num_tiles;
  kern<<<dim3(2 * pairs), dim3(kGemmThreads), Cfg::kSmemBytes, stream>>>(tw, tx, ty, tr, p);
  V100_CUDA(cudaGetLastError());
  return 0;
}

static int launch_gemm_pair(const CUtensorMap& tw, const CUtensorMap& tx, const CUtensorMap& ty, const CUtensorMap& tr,
                            const GemmParams& p, int block_n, cudaStream_t stream) {
#define V100_EPI_ARGS tw, tx, ty, tr, p, stream
  if (block_n == 128) {
    V100_EPI_DISPATCH(launch_gemm_pair_e, 128, kPairStages128)
  }
  V100_EPI_DISPATCH(launch_gemm_pair_e, 256, kPairStages)
#undef V100_EPI_ARGS
}

// Weights-resident pair kernel (WRES).  Each pair serves ONE 256-channel block for the whole launch, so the number of
// pairs is rounded down to a multiple of the number of channel blocks (72 of 74 pairs for 4 or 8 blocks).
constexpr int kWresStages = 9;

template <int STAGES, int EPI>
static int launch_gemm_wres_e(const CUtensorMap& tx, const CUtensorMap& ty, const CUtensorMap& tr, const GemmParams& p,
                              int pairs, cudaStream_t stream) {
  using Cfg = GemmCfg<128, 1, OUT_BF16, STAGES, 2, true>;
  auto kern = conv_gemm_wres_kernel<STAGES, EPI>;
  static thread_local int configured_dev = -1;
  int dev = 0;
  V100_CUDA(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    V100_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    configured_dev = dev;
  }
  kern<<<dim3(2 * pairs), dim3(kGemmThreads), Cfg::kSmemBytes, stream>>>(tx, ty, tr, p);
  V100_CUDA(cudaGetLastError());
  return 0;
}

static int launch_gemm_wres(const CUtensorMap& tx, const CUtensorMap& ty, const CUtensorMap& tr, const GemmParams& p,
                            int pairs, cudaStream_t stream) {
#define V100_EPI_ARGS tx, ty, tr, p, pairs, stream
  V100_EPI_DISPATCH(launch_gemm_wres_e, kWresStages)
#undef V100_EPI_ARGS
}

// WRES applies when the pair's weight block fits in tensor memory next to two 128-column accumulators and the
// channel blocks divide the device's pairs without leaving more than ~5 % of them idle.
static int wres_pairs(int C_in, int C_out, int B, int T) {
  if (C_in > 512 || C_in % 128 != 0 || C_out % (2 * kBlockM) != 0) return 0;
  const int m_tiles = C_out / (2 * kBlockM), all = num_sms() / 2;
  const int slots = all / m_tiles;
  if (slots < 1 || slots * m_tiles * 20 < all * 19) return 0;
  const long long units = static_cast<long long>((T + 127) / 128) * B;
  if (units < 4LL * slots) return 0;   // too little work per pair to pay for loading the weights
  return slots * m_tiles;
}

static int pick_block_n(int T) {
  const int pad256 = (T + 255) / 256 * 256, pad128 = (T + 127) / 128 * 128;
  return pad128 < pad256 ? 128 : 256;
}

static int check_ncw(const void* p, int64_t pitch, int T, const char* what) {
  if (p == nullptr) return fail(V100_E_INVALID, "%s: null pointer", what);
  if ((reinterpret_cast<uintptr_t>(p) & 15) != 0) return fail(V100_E_INVALID, "%s: base not 16-byte aligned", what);
  if (pitch < T || (pitch & 7) != 0) return fail(V100_E_INVALID, "%s: pitch %lld must be >= T=%d and a multiple of 8", what, (long long)pitch, T);
  return 0;
}

static int check_dtype(int dtype, const char* what) {
  if (dtype != DT_BF16 && dtype != DT_F16) return fail(V100_E_INVALID, "%s: dtype must be V100_DTYPE_BF16 or V100_DTYPE_F16", what);
  return 0;
}

static CUtensorMapDataType tmap_type(int dtype) {
  return dtype == DT_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
}

int conv1x1(const void* x, int64_t x_pitch, const void* W, const float* scale, const float* shift,
            const void* res, void* y, int64_t y_pitch, int B, int C_in, int C_out, int T, int act, int dtype,
            cudaStream_t stream) {
  if (int e = check_dtype(dtype, "conv1x1")) return e;
  if (B <= 0 || C_in <= 0 || C_out <= 0 || T <= 0) return fail(V100_E_INVALID, "conv1x1: non-positive size");
  if (C_in % 8 != 0) return fail(V100_E_UNSUPPORTED, "conv1x1: C_in=%d must be a multiple of 8", C_in);
  if (shift == nullptr || W == nullptr) return fail(V100_E_INVALID, "conv1x1: null W/shift");
  if (int e = check_ncw(x, x_pitch, T, "conv1x1 x")) return e;
  if (int e = check_ncw(y, y_pitch, T, "conv1x1 y")) return e;
  if (res != nullptr) if (int e = check_ncw(res, y_pitch, T, "conv1x1 res")) return e;
  const int bn = pick_block_n(T);
  CUtensorMap tw, tx, ty, tr;
  if (int e = make_tmap_2d(&tw, tmap_type(dtype), W, C_in, C_out, int64_t(C_in) * 2, 64, 128)) return e;
  if (int e = make_tmap_3d(&tx, tmap_type(dtype), x, T, C_in, B, x_pitch * 2, int64_t(C_in) * x_pitch * 2, 64, 64)) return e;
  if (int e = make_tmap_3d(&ty, tmap_type(dtype), y, T, C_out, B, y_pitch * 2, int64_t(C_out) * y_pitch * 2, 64, 32)) return e;
  if (int e = make_tmap_3d(&tr, tmap_type(dtype), res ? res : y, T, C_out, B, y_pitch * 2, int64_t(C_out) * y_pitch * 2, 64, 32)) return e;
  GemmParams p{};
  p.C_out = C_out; p.C_in = C_in; p.B = B;
  p.k_blocks = (C_in + kBlockK - 1) / kBlockK;
  p.n_taps = 1; p.tap_xrow[0] = 0; p.tap_acc[0] = 0;
  p.scale = scale; p.shift = shift; p.act = act; p.has_res = res != nullptr; p.dtype = dtype;
  p.t_tiles = (T + bn - 1) / bn;
  if (const int pairs = wres_pairs(C_in, C_out, B, T)) {
    CUtensorMap txw;   // [64 steps x 128 k rows] boxes: one per ring stage and CTA
    if (int e = make_tmap_3d(&txw, tmap_type(dtype), x, T, C_in, B, x_pitch * 2, int64_t(C_in) * x_pitch * 2, 64, 128)) return e;
    p.w_raw = static_cast<const unsigned short*>(W);
    p.k_blocks = C_in / 128;
    p.t_tiles = (T + 127) / 128;
    p.m_tiles = C_out / (2 * kBlockM);
    p.num_tiles = p.m_tiles * p.t_tiles * B;
    return launch_gemm_wres(txw, ty, tr, p, pairs, stream);
  }
  if (C_out % (2 * kBlockM) == 0) {   // CTA pairs; 128-column tiles where they pad the row less
    p.m_tiles = C_out / (2 * kBlockM);
    p.num_tiles = p.m_tiles * p.t_tiles * B;
    return launch_gemm_pair(tw, tx, ty, tr, p, bn, stream);
  }
  p.m_tiles = (C_out + kBlockM - 1) / kBlockM;
  p.num_tiles = p.m_tiles * p.t_tiles * B;
  if (bn == 256) return launch_gemm<256, 1, OUT_BF16, 3>(tw, tx, ty, tr, p, stream);
  return launch_gemm<128, 1, OUT_BF16, 4>(tw, tx, ty, tr, p, stream);
}

int conv1x1_f32out(const void* x, int64_t x_pitch, const void* W, const float* bias, float* y, int64_t y_pitch,
                   int B, int C_in, int C_out, int T, int dtype, cudaStream_t stream) {
  if (int e = check_dtype(dtype, "conv1x1_f32out")) return e;
  if (B <= 0 || C_in <= 0 || C_out <= 0 || T <= 0) return fail(V100_E_INVALID, "conv1x1_f32out: non-positive size");
  if (C_in % 8 != 0) return fail(V100_E_UNSUPPORTED, "conv1x1_f32out: C_in=%d must be a multiple of 8", C_in);
  if (bias == nullptr || W == nullptr || y == nullptr) return fail(V100_E_INVALID, "conv1x1_f32out: null pointer");
  if (int e = check_ncw(x, x_pitch, T, "conv1x1_f32out x")) return e;
  if (y_pitch < T || (y_pitch & 3) != 0 || (reinterpret_cast<uintptr_t>(y) & 15) != 0)
    return fail(V100_E_INVALID, "conv1x1_f32out: y pitch must be >= T and a multiple of 4, base 16B aligned");
  const int bn = pick_block_n(T);
  CUtensorMap tw, tx;
  if (int e = make_tmap_2d(&tw, tmap_type(dtype), W, C_in, C_out, int64_t(C_in) * 2, 64, 128)) return e;
  if (int e = make_tmap_3d(&tx, tmap_type(dtype), x, T, C_in, B, x_pitch * 2, int64_t(C_in) * x_pitch * 2, 64, 64)) return e;
  GemmParams p{};
  p.C_out = C_out; p.C_in = C_in; p.B = B;
  p.m_tiles = (C_out + kBlockM - 1) / kBlockM;
  p.t_tiles = (T + bn - 1) / bn;
  p.num_tiles = p.m_tiles * p.t_tiles * B;
  p.k_blocks = (C_in + kBlockK - 1) / kBlockK;
  p.n_taps = 1; p.tap_xrow[0] = 0; p.tap_acc[0] = 0;
  p.scale = nullptr; p.shift = bias; p.act = V100_ACT_NONE; p.has_res = 0; p.dtype = dtype;
  p.y32 = y; p.y32_pitch = y_pitch;
  if (bn == 256) return launch_gemm<256, 1, OUT_F32, 4>(tw, tx, tx, tx, p, stream);
  return launch_gemm<128, 1, OUT_F32, 4>(tw, tx, tx, tx, p, stream);
}

// Dense Conv1d, stride 1, "same" padding, on the TIME-MAJOR layout x[c][t*Bp + b] (seq.cu): a tap is a shift by a
// whole number of Bp-column groups, i.e. a 16-byte aligned column offset of the TMA box, and what falls off either
// end of the tensor is exactly the conv's zero padding -- k taps accumulate into one tile with no data movement.
int conv1d_tm(const void* x, const void* Wp, const float* bias, void* y, int C_in, int C_out, int T, int Bp, int k,
              int dtype, cudaStream_t stream) {
  if (int e = check_dtype(dtype, "conv1d_tm")) return e;
  if (C_in <= 0 || C_out <= 0 || T <= 0 || Bp <= 0) return fail(V100_E_INVALID, "conv1d_tm: non-positive size");
  if (k < 1 || k > kMaxTaps || (k & 1) == 0) return fail(V100_E_UNSUPPORTED, "conv1d_tm: kernel size %d (odd, <= %d)", k, kMaxTaps);
  if (C_in % 64 != 0) return fail(V100_E_UNSUPPORTED, "conv1d_tm: C_in=%d must be a multiple of 64", C_in);
  if ((Bp & 7) != 0) return fail(V100_E_INVALID, "conv1d_tm: Bp must be a multiple of 8");
  if (bias == nullptr || Wp == nullptr) return fail(V100_E_INVALID, "conv1d_tm: null W/bias");
  const long long N = static_cast<long long>(T) * Bp;
  if (N > 2147483647LL - 512) return fail(V100_E_UNSUPPORTED, "conv1d_tm: T*Bp too large");
  if (int e = check_ncw(x, N, int(N), "conv1d_tm x")) return e;
  if (int e = check_ncw(y, N, int(N), "conv1d_tm y")) return e;
  const int bn = pick_block_n(int(N));
  CUtensorMap tw, tx, ty;
  if (int e = make_tmap_2d(&tw, tmap_type(dtype), Wp, int64_t(C_in) * k, C_out, int64_t(C_in) * k * 2, 64, 128)) return e;
  if (int e = make_tmap_3d(&tx, tmap_type(dtype), x, N, C_in, 1, N * 2, int64_t(C_in) * N * 2, 64, 64)) return e;
  if (int e = make_tmap_3d(&ty, tmap_type(dtype), y, N, C_out, 1, N * 2, int64_t(C_out) * N * 2, 64, 32)) return e;
  GemmParams p{};
  p.C_out = C_out; p.C_in = C_in; p.B = 1;
  p.k_blocks = C_in / kBlockK;
  p.n_taps = k;
  for (int j = 0; j < k; ++j) { p.tap_xrow[j] = 0; p.tap_col[j] = (j - (k - 1) / 2) * Bp; p.tap_acc[j] = 0; }
  p.scale = nullptr; p.shift = bias; p.act = V100_ACT_NONE; p.has_res = 0; p.dtype = dtype;
  p.t_tiles = int((N + bn - 1) / bn);
  if (bn == 256 && C_out % (2 * kBlockM) == 0) {
    p.m_tiles = C_out / (2 * kBlockM);
    p.num_tiles = p.m_tiles * p.t_tiles;
    return launch_gemm_pair(tw, tx, ty, ty, p, 256, stream);
  }
  p.m_tiles = (C_out + kBlockM - 1) / kBlockM;
  p.num_tiles = p.m_tiles * p.t_tiles;
  if (bn == 256) return launch_gemm<256, 1, OUT_BF16, 3>(tw, tx, ty, ty, p, stream);
  return launch_gemm<128, 1, OUT_BF16, 4>(tw, tx, ty, ty, p, stream);
}

// xs[b][s*C + c][t] = x[b][c][t + 1 - s], s = 0,1,2, zero outside [0,T): the three time-shifted views the
// transposed conv needs, stacked along channels so they become plain K offsets of one GEMM.
__global__ void __launch_bounds__(256)
shift_stack3_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ xs, int C, int T, long long pitch) {
  const int b = blockIdx.z, c = blockIdx.y;
  const int t0 = (blockIdx.x * 256 + threadIdx.x) * 8;
  if (t0 >= pitch) return;
  const unsigned short* row = reinterpret_cast<const unsigned short*>(x) + (static_cast<long long>(b) * C + c) * pitch;
  unsigned short v[10];
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const int t = t0 - 1 + i;
    v[i] = (t >= 0 && t < T) ? row[t] : 0;
  }
#pragma unroll
  for (int s = 0; s < 3; ++s) {
    uint4 o;
    uint32_t* ow = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
    for (int i = 0; i < 4; ++i) ow[i] = uint32_t(v[2 * i + 2 - s]) | (uint32_t(v[2 * i + 3 - s]) << 16);
    *reinterpret_cast<uint4*>(xs + ((static_cast<long long>(b) * 3 + s) * C + c) * pitch + t0) = o;
  }
}

int convtranspose1d_k5s2(const void* x, int64_t x_pitch, const void* Wp, const float* bias, void* workspace,
                         void* y, int64_t y_pitch, int B, int C_in, int C_out, int T, int dtype, cudaStream_t stream) {
  if (int e = check_dtype(dtype, "convtranspose")) return e;
  if (B <= 0 || C_in <= 0 || C_out <= 0 || T <= 0) return fail(V100_E_INVALID, "convtranspose: non-positive size");
  if (C_in % 64 != 0) return fail(V100_E_UNSUPPORTED, "convtranspose: C_in=%d must be a multiple of 64", C_in);
  if (bias == nullptr || Wp == nullptr) return fail(V100_E_INVALID, "convtranspose: null W/bias");
  if (B > 65535 || C_in > 65535) return fail(V100_E_UNSUPPORTED, "convtranspose: B or C_in too large for the grid");
  const int T_out = 2 * T - 1;
  if (int e = check_ncw(x, x_pitch, T, "convtranspose x")) return e;
  if (int e = check_ncw(workspace, x_pitch, T, "convtranspose workspace")) return e;
  if (int e = check_ncw(y, y_pitch, T_out, "convtranspose y")) return e;
  {
    dim3 grid((unsigned)((x_pitch / 8 + 255) / 256), C_in, B);
    shift_stack3_kernel<<<grid, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(x),
                                                  static_cast<__nv_bfloat16*>(workspace), C_in, T, x_pitch);
    V100_CUDA(cudaGetLastError());
  }
  CUtensorMap tw, tx, ty;
  if (int e = make_tmap_2d(&tw, tmap_type(dtype), Wp, int64_t(C_in) * 5, C_out, int64_t(C_in) * 5 * 2, 64, 128)) return e;
  if (int e = make_tmap_3d(&tx, tmap_type(dtype), workspace, T, int64_t(C_in) * 3, B, x_pitch * 2, int64_t(C_in) * 3 * x_pitch * 2, 64, 64)) return e;
  if (int e = make_tmap_3d(&ty, tmap_type(dtype), y, T_out, C_out, B, y_pitch * 2, int64_t(C_out) * y_pitch * 2, 64, 32)) return e;
  GemmParams p{};
  p.C_out = C_out; p.C_in = C_in; p.B = B;
  p.m_tiles = (C_out + kBlockM - 1) / kBlockM;
  p.t_tiles = (T + 127) / 128;
  p.num_tiles = p.m_tiles * p.t_tiles * B;
  p.k_blocks = C_in / kBlockK;
  // y[co][o] = b[co] + sum_{ci,k,t: o = 2t - 2 + k} x[ci][t] W[ci][co][k]   (tts.py:22, stride 2, padding 2)
  //   o = 2j   : (k,t) = (0,j+1) (2,j) (4,j-1)   -> accumulator 0
  //   o = 2j+1 : (k,t) = (1,j+1) (3,j)           -> accumulator 1
  // x(t+1), x(t), x(t-1) are channel blocks 0, 1, 2 of the workspace.
  p.n_taps = 5;
  const int blocks[5] = {0, 0, 1, 1, 2};
  const int accs[5] = {0, 1, 0, 1, 0};
  for (int i = 0; i < 5; ++i) { p.tap_xrow[i] = blocks[i] * C_in; p.tap_acc[i] = accs[i]; }
  p.scale = nullptr; p.shift = bias; p.act = V100_ACT_NONE; p.has_res = 0; p.dtype = dtype;
  return launch_gemm<128, 2, OUT_BF16, 4>(tw, tx, ty, ty, p, stream);
}

}  // namespace v100
