// tcgen05 / TMEM / TMA tap-GEMM for sm_100a.
//
//   D[b,t,n] = sum_seg sum_k  A_seg[b, t+shift_seg, c_off_seg+k] * W[n, koff_seg+k]
//
// A (activations) and W (packed weights) are stored as 16-bit split planes (see fd_common.cuh).
// One persistent CTA per SM, warp-specialised:
//   warp 0      : TMA producer  (cp.async.bulk.tensor, 128B/64B/32B swizzle, OOB rows zero-filled: that is how the
//                 conv zero padding and the time shift of each tap are realised; the hi and lo planes of an operand
//                 arrive in one box)
//   warp 1      : MMA issuer    (one elected lane issues tcgen05.mma kind::f16; three products per k16 step
//                 -- lo*hi + hi*lo + hi*hi -- or one in single-product mode; fp32 accumulation in TMEM)
//   warp 2      : TMEM allocator
//   warps 4..   : epilogue      (8 warps; 16 for tiles of <= 32 columns): tcgen05.ld 32x32b -> registers -> fused
//                 epilogue -> global.  256-column tiles: the two warps of a TMEM lane quadrant split the columns;
//                 narrower tiles: groups of 4 warps take alternate tiles.
// Pipelines: smem full/empty ring between TMA and MMA; 2 (256 columns) or 4 TMEM accumulator stages between MMA and
// epilogue, so the epilogue of tile i overlaps the mainloop of the following tiles.
#include <cuda.h>
#include "fd_common.cuh"
#include "fd_host.h"
#include "fd_tc_ptx.cuh"

namespace {

constexpr int BLOCK_M = 128;
constexpr int EPI_WARP0 = 4;

// NPL = operand planes staged per k-block: 2 (hi + lo, three products) or 1 (hi only, one product: 11-bit (f16) /
// 8-bit (bf16) operand mantissas, the arithmetic of a plain half-precision tensor-core GEMM with fp32 accumulation).
template <int BLOCK_N, int BLOCK_K, int EPI, int NPL>
struct Cfg {
  static constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;
  static constexpr int W_BYTES = BLOCK_N * BLOCK_K * 2;
  // One pipeline stage holds GROUP consecutive k-blocks (64 K-elements worth): with narrow channel counts a k-block
  // is a single conv tap of 16 or 32 channels, and one barrier round trip per tap is what bounds the small-channel
  // vocoder stages.  hi and lo planes of an operand arrive in ONE TMA box (plane dimension = 2).
  static constexpr int GROUP = BLOCK_K >= 64 ? 1 : 64 / BLOCK_K;
  static constexpr int SUB_BYTES = NPL * (A_BYTES + W_BYTES);           // multiple of 1024 for every instantiation
  static constexpr int STAGE_BYTES = GROUP * SUB_BYTES;
  static constexpr int TX_BYTES = SUB_BYTES;                            // per k-block
  // BLOCK_N = 256: the two epilogue warps of a TMEM lane quadrant split the columns of one tile (2 accumulator
  // stages fill the 512 TMEM columns).  Narrower tiles: the two groups of 4 epilogue warps take ALTERNATE tiles and
  // 4 accumulator stages keep the MMA warp ahead -- the per-tile epilogue latency chain (bias, TMEM load, global
  // read-modify-write) of one group overlaps the other group's.
  // The epilogue of such tiles is bound by the latency of its global operands, i.e. by how many tiles are in flight per
  // SM: tiles of <= 32 columns (small per-thread state) run FOUR groups of 4 warps, one accumulator stage each; 64 / 128
  // columns keep two groups (the coalescing epilogue needs more than the 96 registers a 640-thread CTA leaves).
  static constexpr bool SPLIT_COLS = BLOCK_N >= 256;
  static constexpr int ACC_STAGES = SPLIT_COLS ? 2 : 4;
  static constexpr int EPI_GROUPS = SPLIT_COLS ? 1 : (BLOCK_N <= 32 ? 4 : 2);
  static constexpr int EPI_THREADS = SPLIT_COLS ? 256 : 128 * EPI_GROUPS;
  static constexpr int NUM_THREADS = EPI_WARP0 * 32 + EPI_THREADS;
  static constexpr int TMEM_COLS_RAW = ACC_STAGES * BLOCK_N;
  static constexpr int TMEM_COLS = TMEM_COLS_RAW <= 32 ? 32 : TMEM_COLS_RAW <= 64 ? 64 : TMEM_COLS_RAW <= 128 ? 128
                                   : TMEM_COLS_RAW <= 256 ? 256 : 512;
  static constexpr int SWIZZLE_BYTES = BLOCK_K * 2;                       // 128 / 64 / 32
  static constexpr uint32_t LAYOUT_TYPE = BLOCK_K == 64 ? 2u : BLOCK_K == 32 ? 4u : 6u;
  static constexpr uint32_t SBO = 8 * SWIZZLE_BYTES;
  static constexpr int BIAS_FLOATS = (EPI == FD_EPI_GATE ? 3 : 1) * BLOCK_N * EPI_GROUPS;
  // coalescing epilogue (LINEAR / RES_SKIP with >= 32 columns per warp): a 32x32 fp32 transpose scratch per warp
  static constexpr bool COALESCED = (EPI == FD_EPI_LINEAR || EPI == FD_EPI_RES_SKIP || EPI == FD_EPI_GATE_BWD) && BLOCK_N >= 64;
  static constexpr int SCRATCH_BYTES = COALESCED ? (EPI_THREADS / 32) * 4096 : 0;
  static constexpr int FIXED_BYTES = 1024 /*align slack*/ + BIAS_FLOATS * 4 + (2 * 8 + 2 * ACC_STAGES) * 8 + 16 + SCRATCH_BYTES;
  static constexpr int RAW_STAGES = (227 * 1024 - 512 - FIXED_BYTES) / STAGE_BYTES;
  static constexpr int NUM_STAGES = RAW_STAGES > 8 ? 8 : RAW_STAGES;
  static constexpr int SMEM_BYTES = 1024 /*align slack*/ + NUM_STAGES * STAGE_BYTES + BIAS_FLOATS * 4 +
                                    (2 * NUM_STAGES + 2 * ACC_STAGES) * 8 + 16 + SCRATCH_BYTES;
  static_assert(NUM_STAGES >= 2, "pipeline needs at least two stages");
};

template <int BLOCK_N, int BLOCK_K, int EPI, int PREC, int NPL>
__global__ void __launch_bounds__((Cfg<BLOCK_N, BLOCK_K, EPI, NPL>::NUM_THREADS), 1)
fd_tapgemm_tc_kernel(const __grid_constant__ CUtensorMap tm_src0, const __grid_constant__ CUtensorMap tm_src1,
                     const __grid_constant__ CUtensorMap tm_w, const FdTapGemm p) {
  using C = Cfg<BLOCK_N, BLOCK_K, EPI, NPL>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* stage_base = smem;
  float* bias_s = reinterpret_cast<float*>(smem + C::NUM_STAGES * C::STAGE_BYTES);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(bias_s + C::BIAS_FLOATS);
  uint64_t* empty_bar = full_bar + C::NUM_STAGES;
  uint64_t* tfull_bar = empty_bar + C::NUM_STAGES;
  uint64_t* tempty_bar = tfull_bar + C::ACC_STAGES;
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(tempty_bar + C::ACC_STAGES);
  float* scratch_s = reinterpret_cast<float*>(tmem_ptr_s + 4);   // 16-byte aligned (all preceding sizes are)

  const int warp = threadIdx.x / 32;
  const int lane = threadIdx.x % 32;

  const int tiles_t = (p.T + BLOCK_M - 1) / BLOCK_M;
  const int num_m_tiles = p.B * tiles_t;
  const int num_n_tiles = p.n_total / BLOCK_N;
  const int num_tiles = num_m_tiles * num_n_tiles;
  int total_k_blocks = 0;
  for (int sI = 0; sI < p.num_seg; ++sI) total_k_blocks += p.seg[sI].k_len / BLOCK_K;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_src0);
    prefetch_tmap(&tm_src1);
    prefetch_tmap(&tm_w);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < C::NUM_STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < C::ACC_STAGES; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], C::EPI_THREADS / 32 / C::EPI_GROUPS); }
    fence_barrier_init();
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_s)),
                 "r"((uint32_t)C::TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;

  if (warp == 0) {
    // =========================================================== TMA producer
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m_tile = tile / num_n_tiles;
        // rotate the column tile with the row tile: with a grid that is a multiple of num_n_tiles every CTA would
        // otherwise see the same n-tile forever, and epilogue costs differ per n-tile (residual vs skip columns)
        const int n_tile = (tile % num_n_tiles + m_tile) % num_n_tiles;
        const int b = m_tile / tiles_t, t0 = (m_tile % tiles_t) * BLOCK_M;
        const int n0 = n_tile * BLOCK_N;
        int s = 0, k0 = 0, koff = 0;                 // flattened (segment, k offset) iterator
        for (int kb = 0; kb < total_k_blocks; kb += C::GROUP) {
          const int nb = min(C::GROUP, total_k_blocks - kb);
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* st = stage_base + stage * C::STAGE_BYTES;
          mbar_expect_tx(&full_bar[stage], nb * C::TX_BYTES);
          for (int g = 0; g < nb; ++g) {
            const FdSeg sg = p.seg[s];
            const CUtensorMap* tm = sg.src == 0 ? &tm_src0 : &tm_src1;
            uint8_t* sub = st + g * C::SUB_BYTES;
            tma_load_4d(sub, tm, &full_bar[stage], sg.c_off + k0, t0 + sg.shift, b, 0);          // hi + lo planes
            const int kw = koff + k0 + p.w_kshift + (int)(b * p.w_bstride_k);
            tma_load_3d(sub + NPL * C::A_BYTES, &tm_w, &full_bar[stage], kw, n0, 0);               // hi + lo planes
            k0 += BLOCK_K;
            if (k0 >= sg.k_len) { koff += sg.k_len; k0 = 0; ++s; }
          }
          if (++stage == C::NUM_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // =========================================================== MMA issuer
    if (lane == 0) {
      const uint32_t fmt = PREC == FD_F16 ? 0u : 1u;
      const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(BLOCK_N >> 3) << 17) |
                             ((uint32_t)(BLOCK_M >> 4) << 24);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
        for (int kb = 0; kb < total_k_blocks; kb += C::GROUP) {
          const int nb = min(C::GROUP, total_k_blocks - kb);
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          for (int g = 0; g < nb; ++g) {
            const uint32_t st = smem_u32(stage_base + stage * C::STAGE_BYTES + g * C::SUB_BYTES);
            const uint64_t a_hi = make_kmajor_desc(st, C::SBO, C::LAYOUT_TYPE);
            const uint64_t a_lo = make_kmajor_desc(st + C::A_BYTES, C::SBO, C::LAYOUT_TYPE);
            const uint64_t w_hi = make_kmajor_desc(st + NPL * C::A_BYTES, C::SBO, C::LAYOUT_TYPE);
            const uint64_t w_lo = make_kmajor_desc(st + NPL * C::A_BYTES + C::W_BYTES, C::SBO, C::LAYOUT_TYPE);
#pragma unroll
            for (int k = 0; k < BLOCK_K / 16; ++k) {
              const uint64_t adv = (uint64_t)((k * 32) >> 4);   // 16 elements * 2 B along K inside the swizzle row
              if (NPL == 2) {
                // small terms first, the dominant hi*hi product last
                umma_f16(d_tmem, a_lo + adv, w_hi + adv, idesc, (kb | g | k) != 0 ? 1u : 0u);
                umma_f16(d_tmem, a_hi + adv, w_lo + adv, idesc, 1u);
                umma_f16(d_tmem, a_hi + adv, w_hi + adv, idesc, 1u);
              } else {
                umma_f16(d_tmem, a_hi + adv, w_hi + adv, idesc, (kb | g | k) != 0 ? 1u : 0u);
              }
            }
          }
          umma_commit(&empty_bar[stage]);
          if (++stage == C::NUM_STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tfull_bar[acc]);
        if (++acc == C::ACC_STAGES) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= EPI_WARP0) {
    // =========================================================== epilogue (8 warps)
    // warp w may access TMEM lanes [32*(w%4), +32); the two warps of a lane quadrant split the columns.
    const int q = warp % 4;
    const int wgrp = (warp - EPI_WARP0) / 4;                 // which set of four epilogue warps
    const int half = C::SPLIT_COLS ? wgrp : 0;               // column half handled inside a shared tile
    const int group = C::SPLIT_COLS ? 0 : wgrp;              // alternate-tile group
    constexpr int GTHREADS = C::EPI_THREADS / C::EPI_GROUPS; // threads cooperating on one tile
    const int row = q * 32 + lane;
    const int etid = (threadIdx.x - EPI_WARP0 * 32) % GTHREADS;
    constexpr int HALVES = C::SPLIT_COLS ? 2 : 1;
    float* const bias_g = bias_s + group * (C::BIAS_FLOATS / C::EPI_GROUPS);
    int acc = 0; uint32_t acc_phase = 0;
    int it = 0;
    long long staged_key = -1;                               // which bias vectors this group holds in shared memory
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      if (C::EPI_GROUPS > 1 && (it % C::EPI_GROUPS) != group) {   // another group's tile: just keep the stage counters
        if (++acc == C::ACC_STAGES) { acc = 0; acc_phase ^= 1; }
        continue;
      }
      const int m_tile = tile / num_n_tiles;
        // rotate the column tile with the row tile: with a grid that is a multiple of num_n_tiles every CTA would
        // otherwise see the same n-tile forever, and epilogue costs differ per n-tile (residual vs skip columns)
        const int n_tile = (tile % num_n_tiles + m_tile) % num_n_tiles;
      const int b = m_tile / tiles_t, t0 = (m_tile % tiles_t) * BLOCK_M;
      const int n0 = n_tile * BLOCK_N;
      const int t = t0 + row;
      const bool valid = t < p.T;

      // stage the per-column bias vectors of this tile in shared memory (named barrier of this tile's warps); skipped
      // while the group keeps seeing the same columns / item -- with a single column tile that is once per launch, which
      // takes a dependent global load and two barriers out of every tile's latency chain
      const long long bias_key = EPI == FD_EPI_GATE ? (long long)b * p.gbias_bstride + n0
                                                    : (long long)b * p.bias_bstride + n0;
      if (EPI != FD_EPI_MAG && EPI != FD_EPI_GATE_BWD && bias_key != staged_key) {
        staged_key = bias_key;
        asm volatile("bar.sync %0, %1;" ::"r"(1 + group), "r"(GTHREADS) : "memory");
        if (EPI == FD_EPI_GATE) {
          const size_t bo = (size_t)b * p.gbias_bstride + n0;
          for (int i = etid; i < BLOCK_N; i += GTHREADS) {
            bias_g[i] = p.gbias_full[bo + i];
            bias_g[BLOCK_N + i] = p.gbias_lo[bo + i];
            bias_g[2 * BLOCK_N + i] = p.gbias_hi[bo + i];
          }
        } else {
          for (int i = etid; i < BLOCK_N; i += GTHREADS)
            bias_g[i] = p.bias ? p.bias[(size_t)b * p.bias_bstride + n0 + i] : 0.f;
        }
        asm volatile("bar.sync %0, %1;" ::"r"(1 + group), "r"(GTHREADS) : "memory");
      }

      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + acc * BLOCK_N + ((uint32_t)(q * 32) << 16);

      if (EPI == FD_EPI_GATE || EPI == FD_EPI_MAG) {
        constexpr int HALF = BLOCK_N / 2;       // gate columns | filter columns
        constexpr int PER = HALF / HALVES;      // gate columns handled by this warp
        const int cb = half * PER;
        // GATE: the bias vectors are read with shared-space loads (through the generic pointers of fd_epi_gate every one of
        // them was a generic LD and a long-scoreboard stall) and the zero-padding corrections of the first / last `dilation`
        // rows are skipped by a warp vote where no lane needs them: 81 -> ~60 instructions per element.  Same-box A/B of the
        // one-product training step: 12.77 / 13.04 -> 12.71 / 12.75 ms, i.e. within noise -- in that mode the kernel is bound by
        // its operand stream (each 256-column tile re-reads 0.9 MB of weights from L2; 4 ring stages of 48 KB), not by this
        // epilogue; in the three-product mode the epilogue hides under the MMAs either way.
        const uint32_t sb = smem_u32(bias_g);
        const bool e_lo = t < p.dil, e_hi = t + p.dil >= p.T;
        const bool edge_any = __any_sync(0xffffffffu, valid && (e_lo || e_hi));
        const size_t zplane = (size_t)p.B * p.T * p.C, zrow = ((size_t)b * p.T + t) * p.C + (size_t)n_tile * HALF;
        const size_t yplane = (size_t)p.B * p.T * p.n_total, yrow = ((size_t)b * p.T + t) * p.n_total;
        const int halfg = p.gate_tile / 2;
        // conditioner term of the hoisted sampler path (fp32, packed column order like the accumulator tile)
        const bool has_add = EPI == FD_EPI_GATE && p.addend != nullptr && valid;
        const float* const add_row = has_add ? p.addend + yrow + n0 : nullptr;
        for (int c = 0; c < PER; c += 16) {
          const int c0 = cb + c;
          float g[16], f[16];
          // this row's 2 x 64 bytes of the addend are requested before the TMEM wait, so their latency overlaps it
          float4 ag[4], af[4];
          if (has_add) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              ag[i] = __ldg(reinterpret_cast<const float4*>(add_row + c0) + i);
              af[i] = __ldg(reinterpret_cast<const float4*>(add_row + HALF + c0) + i);
            }
          }
          tmem_ld16_nowait(taddr + c0, g);
          tmem_ld16_nowait(taddr + HALF + c0, f);
          tmem_wait16(g);
          tmem_wait16(f);
          if (valid) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int cc = c0 + h * 8;
              if (EPI == FD_EPI_MAG) {
                float g8[8], f8[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) { g8[i] = g[h * 8 + i]; f8[i] = f[h * 8 + i]; }
                fd_epi_mag<8, PREC>(p, b, t, n_tile * HALF + cc, g8, f8);
              } else {
                float yg[8], yf[8], z[8];
                {
                  const float4 a0 = lds128(sb + 4u * cc), a1 = lds128(sb + 4u * cc + 16u);
                  const float4 b0 = lds128(sb + 4u * (HALF + cc)), b1 = lds128(sb + 4u * (HALF + cc) + 16u);
                  const float bg[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
                  const float bf[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                  for (int i = 0; i < 8; ++i) {
                    yg[i] = g[h * 8 + i] * p.acc_scale + bg[i];
                    yf[i] = f[h * 8 + i] * p.acc_scale + bf[i];
                  }
                }
                if (edge_any) {
#pragma unroll
                  for (int e = 0; e < 2; ++e) {
                    if (e == 0 ? e_lo : e_hi) {
                      const uint32_t eb = sb + 4u * ((1 + e) * BLOCK_N + cc);
                      const float4 a0 = lds128(eb), a1 = lds128(eb + 16u);
                      const float4 b0 = lds128(eb + 4u * HALF), b1 = lds128(eb + 4u * HALF + 16u);
                      const float eg[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
                      const float ef[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                      for (int i = 0; i < 8; ++i) { yg[i] -= eg[i]; yf[i] -= ef[i]; }
                    }
                  }
                }
                if (has_add) {
                  const float4 a0 = ag[2 * h], a1 = ag[2 * h + 1], b0 = af[2 * h], b1 = af[2 * h + 1];
                  const float eg[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
                  const float ef[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                  for (int i = 0; i < 8; ++i) { yg[i] += eg[i]; yf[i] += ef[i]; }
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) z[i] = fd_sigmoid(yg[i]) * fd_tanh(yf[i]);
                if (p.y_planes != nullptr) {   // training: keep the pre-activations (packed column order: gates | filters per tile)
                  const int zc0 = n_tile * HALF + cc;
                  const int ng = p.gate_tile == BLOCK_N ? n_tile * BLOCK_N + cc : (zc0 / halfg) * p.gate_tile + (zc0 % halfg);
                  fd_store_planes<8>(p.y_planes, yplane, yrow + ng, yg, PREC);
                  fd_store_planes<8>(p.y_planes, yplane, yrow + ng + halfg, yf, PREC);
                }
                fd_store_planes<8>(p.out_planes, zplane, zrow + cc, z, PREC);
              }
            }
          }
        }
      } else if (C::COALESCED) {
        // ---- LINEAR / RES_SKIP, coalescing epilogue: 32-column chunks, accumulators transposed through a warp-private
        //      smem scratch so that 8 lanes cover one 128-byte row segment; all global loads of a half-chunk are issued
        //      before the TMEM wait (latency overlap); per-item math is the shared V=4 epilogue of fd_common.cuh order.
        constexpr int PER = BLOCK_N / HALVES;
        const uint32_t my_scratch = smem_u32(scratch_s) + (warp - EPI_WARP0) * 4096;
        const uint32_t bias_addr = smem_u32(bias_g);
        const int j4 = (lane & 7) * 4, rsub = lane >> 3;
        const int rbase = t0 + q * 32 + rsub;            // time index of pass 0
#pragma unroll 1
        for (int c = 0; c < PER; c += 32) {
          const int col = half * PER + c + j4;           // first of this lane's 4 columns inside the tile
          const int n = n0 + col;                        // global packed column
          float v[32];
          constexpr bool LATE_TMEM_LD = EPI == FD_EPI_LINEAR || EPI == FD_EPI_GATE_BWD;   // see the LINEAR branch below
          if (!LATE_TMEM_LD) {
            tmem_ld16_nowait(taddr + half * PER + c, *reinterpret_cast<float(*)[16]>(&v[0]));
            tmem_ld16_nowait(taddr + half * PER + c + 16, *reinterpret_cast<float(*)[16]>(&v[16]));
          }
          const float4 bias4 = EPI == FD_EPI_GATE_BWD ? make_float4(0.f, 0.f, 0.f, 0.f) : lds128(bias_addr + 4u * col);
          if (EPI == FD_EPI_GATE_BWD) {
            // backward of z = sigmoid(g) tanh(f) fused into the dz GEMM (training): this lane's 4 channels n..n+3 of 8 rows
            const int half_g = p.gate_tile / 2;
            const uint32_t pg = (uint32_t)((n / half_g) * p.gate_tile + (n % half_g));     // packed gate column
            const uint32_t rowbase = (uint32_t)b * (uint32_t)p.T;
            const int nrows = rbase < p.T ? min(8, (p.T - rbase + 3) / 4) : 0;
            const uint32_t W2 = 2u * (uint32_t)p.C;
            const size_t yplane = (size_t)p.B * p.T * W2;
            const uint16_t* const y_lo = p.y_planes + yplane;
            uint16_t* const o_lo = p.out_planes + yplane;
            tmem_ld16_nowait(taddr + half * PER + c, *reinterpret_cast<float(*)[16]>(&v[0]));
            tmem_ld16_nowait(taddr + half * PER + c + 16, *reinterpret_cast<float(*)[16]>(&v[16]));
            tmem_wait16(*reinterpret_cast<float(*)[16]>(&v[0]));
            tmem_wait16(*reinterpret_cast<float(*)[16]>(&v[16]));
            float4 a[8];
            warp_transpose_32x32(my_scratch, lane, v, a);
            float sg4[4] = {0.f, 0.f, 0.f, 0.f}, sf4[4] = {0.f, 0.f, 0.f, 0.f};          // column sums over this lane's rows
            float e0g[4] = {0.f, 0.f, 0.f, 0.f}, e0f[4] = {0.f, 0.f, 0.f, 0.f}, e1g[4] = {0.f, 0.f, 0.f, 0.f}, e1f[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int hb = 0; hb < 2; ++hb) {           // two batches of 4 rows: 16 plane words in flight per batch
              uint2 gh[4], gl[4], fh[4], fl[4];
              uint32_t eo4[4];
#pragma unroll
              for (int q4 = 0; q4 < 4; ++q4) {
                const int pp = hb * 4 + q4;
                eo4[q4] = (rowbase + (uint32_t)min(rbase + pp * 4, p.T - 1)) * W2 + pg;
                gh[q4] = *reinterpret_cast<const uint2*>(p.y_planes + eo4[q4]);
                gl[q4] = *reinterpret_cast<const uint2*>(y_lo + eo4[q4]);
                fh[q4] = *reinterpret_cast<const uint2*>(p.y_planes + eo4[q4] + half_g);
                fl[q4] = *reinterpret_cast<const uint2*>(y_lo + eo4[q4] + half_g);
              }
#pragma unroll
              for (int q4 = 0; q4 < 4; ++q4) {
                const int pp = hb * 4 + q4;
                if (pp >= nrows) break;
                float g[4], f[4];
                fd_combine2(gh[q4].x, gl[q4].x, PREC, g[0], g[1]);
                fd_combine2(gh[q4].y, gl[q4].y, PREC, g[2], g[3]);
                fd_combine2(fh[q4].x, fl[q4].x, PREC, f[0], f[1]);
                fd_combine2(fh[q4].y, fl[q4].y, PREC, f[2], f[3]);
                const float dzv[4] = {a[pp].x * p.acc_scale, a[pp].y * p.acc_scale, a[pp].z * p.acc_scale, a[pp].w * p.acc_scale};
                float dg[4], df[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                  const float sg = fd_sigmoid(g[i]), th = fd_tanh(f[i]);
                  dg[i] = dzv[i] * th * sg * (1.f - sg);
                  df[i] = dzv[i] * sg * (1.f - th * th);
                }
                uint32_t h0, l0, h1, l1;
                fd_split2(dg[0], dg[1], PREC, h0, l0);
                fd_split2(dg[2], dg[3], PREC, h1, l1);
                *reinterpret_cast<uint2*>(p.out_planes + eo4[q4]) = make_uint2(h0, h1);
                *reinterpret_cast<uint2*>(o_lo + eo4[q4]) = make_uint2(l0, l1);
                fd_split2(df[0], df[1], PREC, h0, l0);
                fd_split2(df[2], df[3], PREC, h1, l1);
                *reinterpret_cast<uint2*>(p.out_planes + eo4[q4] + half_g) = make_uint2(h0, h1);
                *reinterpret_cast<uint2*>(o_lo + eo4[q4] + half_g) = make_uint2(l0, l1);
                if (p.cs != nullptr) {
                  const int tt = rbase + pp * 4;
                  const bool in0 = tt < p.dil, in1 = tt + p.dil >= p.T;
#pragma unroll
                  for (int i = 0; i < 4; ++i) {
                    sg4[i] += dg[i]; sf4[i] += df[i];
                    if (in0) { e0g[i] += dg[i]; e0f[i] += df[i]; }
                    if (in1) { e1g[i] += dg[i]; e1f[i] += df[i]; }
                  }
                }
              }
            }
            if (p.cs != nullptr) {
              // rows of the 4 lanes that share these columns (lane bits 3,4), then one atomic per column and warp
              const bool edge0 = t0 + q * 32 < p.dil, edge1 = t0 + q * 32 + 32 + p.dil > p.T;     // warp-uniform
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                sg4[i] += __shfl_xor_sync(0xffffffffu, sg4[i], 8); sg4[i] += __shfl_xor_sync(0xffffffffu, sg4[i], 16);
                sf4[i] += __shfl_xor_sync(0xffffffffu, sf4[i], 8); sf4[i] += __shfl_xor_sync(0xffffffffu, sf4[i], 16);
                if (edge0) {
                  e0g[i] += __shfl_xor_sync(0xffffffffu, e0g[i], 8); e0g[i] += __shfl_xor_sync(0xffffffffu, e0g[i], 16);
                  e0f[i] += __shfl_xor_sync(0xffffffffu, e0f[i], 8); e0f[i] += __shfl_xor_sync(0xffffffffu, e0f[i], 16);
                }
                if (edge1) {
                  e1g[i] += __shfl_xor_sync(0xffffffffu, e1g[i], 8); e1g[i] += __shfl_xor_sync(0xffffffffu, e1g[i], 16);
                  e1f[i] += __shfl_xor_sync(0xffffffffu, e1f[i], 8); e1f[i] += __shfl_xor_sync(0xffffffffu, e1f[i], 16);
                }
              }
              if (rsub == 0) {
                float* const csb = p.cs + (size_t)b * W2 + pg;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                  atomicAdd(csb + i, sg4[i] * p.cs_scale);
                  atomicAdd(csb + half_g + i, sf4[i] * p.cs_scale);
                }
                if (p.cs_edge != nullptr && (edge0 || edge1)) {
                  float* const ce0 = p.cs_edge + (size_t)b * W2 + pg;
                  float* const ce1 = ce0 + (size_t)p.B * W2;
#pragma unroll
                  for (int i = 0; i < 4; ++i) {
                    if (edge0) { atomicAdd(ce0 + i, e0g[i] * p.cs_scale); atomicAdd(ce0 + half_g + i, e0f[i] * p.cs_scale); }
                    if (edge1) { atomicAdd(ce1 + i, e1g[i] * p.cs_scale); atomicAdd(ce1 + half_g + i, e1f[i] * p.cs_scale); }
                  }
                }
              }
            }
          } else if (EPI == FD_EPI_RES_SKIP) {
            // residual columns: x' = (x + y)/sqrt2 on the split planes; skip columns: fp32 accumulation.  32-bit element
            // offsets (checked on the host), rows past T clamped for the loads and skipped for the stores.
            // Tried and dropped (round 2, same-box A/B, B=32 x T=4000): fetching these read-modify-write operands one
            // chunk ahead (next 32 columns, or the first chunk of the group's next tile) -- 0.408 -> 0.517 ms per launch:
            // the second operand set pushes the kernel over its 168 registers (104 bytes of spills inside the chunk loop)
            // and the epilogue is not latency-bound enough to pay for that.
            const bool is_res = n0 < p.C;
            const uint32_t rowbase = (uint32_t)b * (uint32_t)p.T;
            const uint32_t cn = (uint32_t)(is_res ? n : n - p.C);
            const int nrows = rbase < p.T ? min(8, (p.T - rbase + 3) / 4) : 0;
            const size_t plane = (size_t)p.B * p.T * p.C;
            uint32_t eo[8];
#pragma unroll
            for (int pp = 0; pp < 8; ++pp)
              eo[pp] = (rowbase + (uint32_t)min(rbase + pp * 4, p.T - 1)) * (uint32_t)p.C + cn;
            uint4 op[8];     // residual tile: .xy = hi-plane words, .zw = lo-plane words; skip tile: 4 floats
            if (is_res) {
              if (!p.last_layer) {
                const uint16_t* const xlo = p.x_planes + plane;
#pragma unroll
                for (int pp = 0; pp < 8; ++pp) {
                  const uint2 h2 = *reinterpret_cast<const uint2*>(p.x_planes + eo[pp]);
                  const uint2 l2 = *reinterpret_cast<const uint2*>(xlo + eo[pp]);
                  op[pp] = make_uint4(h2.x, h2.y, l2.x, l2.y);
                }
              }
            } else if (!p.first_layer) {
#pragma unroll
              for (int pp = 0; pp < 8; ++pp) op[pp] = *reinterpret_cast<const uint4*>(p.skip_f32 + eo[pp]);
            }
            tmem_wait16(*reinterpret_cast<float(*)[16]>(&v[0]));
            tmem_wait16(*reinterpret_cast<float(*)[16]>(&v[16]));
            float4 a[8];
            warp_transpose_32x32(my_scratch, lane, v, a);
            if (is_res) {
              if (!p.last_layer) {
                uint16_t* const xo = p.x_out_planes != nullptr ? p.x_out_planes : p.x_planes;
                uint16_t* const xo_lo = xo + plane;
#pragma unroll
                for (int pp = 0; pp < 8; ++pp) {
                  if (pp >= nrows) break;
                  float x0, x1, x2, x3;
                  fd_combine2(op[pp].x, op[pp].z, PREC, x0, x1);
                  fd_combine2(op[pp].y, op[pp].w, PREC, x2, x3);
                  x0 = (x0 + (a[pp].x * p.acc_scale + bias4.x)) * 0.70710678118654752440f;
                  x1 = (x1 + (a[pp].y * p.acc_scale + bias4.y)) * 0.70710678118654752440f;
                  x2 = (x2 + (a[pp].z * p.acc_scale + bias4.z)) * 0.70710678118654752440f;
                  x3 = (x3 + (a[pp].w * p.acc_scale + bias4.w)) * 0.70710678118654752440f;
                  uint32_t h0, l0, h1, l1;
                  fd_split2(x0, x1, PREC, h0, l0);
                  fd_split2(x2, x3, PREC, h1, l1);
                  *reinterpret_cast<uint2*>(xo + eo[pp]) = make_uint2(h0, h1);
                  *reinterpret_cast<uint2*>(xo_lo + eo[pp]) = make_uint2(l0, l1);
                }
              }
            } else {
              uint16_t* const sk_lo = p.skip_planes + plane;
#pragma unroll
              for (int pp = 0; pp < 8; ++pp) {
                if (pp >= nrows) break;
                float y0 = a[pp].x * p.acc_scale + bias4.x, y1 = a[pp].y * p.acc_scale + bias4.y;
                float y2 = a[pp].z * p.acc_scale + bias4.z, y3 = a[pp].w * p.acc_scale + bias4.w;
                if (!p.first_layer) {
                  y0 += __uint_as_float(op[pp].x); y1 += __uint_as_float(op[pp].y);
                  y2 += __uint_as_float(op[pp].z); y3 += __uint_as_float(op[pp].w);
                }
                if (p.last_layer) {
                  uint32_t h0, l0, h1, l1;
                  fd_split2(y0 * p.skip_scale, y1 * p.skip_scale, PREC, h0, l0);
                  fd_split2(y2 * p.skip_scale, y3 * p.skip_scale, PREC, h1, l1);
                  *reinterpret_cast<uint2*>(p.skip_planes + eo[pp]) = make_uint2(h0, h1);
                  *reinterpret_cast<uint2*>(sk_lo + eo[pp]) = make_uint2(l0, l1);
                } else {
                  *reinterpret_cast<float4*>(p.skip_f32 + eo[pp]) = make_float4(y0, y1, y2, y3);
                }
              }
            }
          } else {
            // LINEAR (vocoder convs, WaveNet head / tail, data gradients).  This epilogue is bound by the latency of its global
            // operands and by its own instruction count, so: ALL of a chunk's operand loads (8 rows x 16 bytes per lane
            // and operand kind) are issued up front and folded kind by kind into one pre-sum (register cost = one kind
            // in flight); the accumulators are fetched from TMEM only afterwards; element offsets are 32-bit (checked on
            // the host) and rows past T are clamped for the loads / skipped for the stores.
            const uint32_t rowbase = (uint32_t)b * (uint32_t)p.T;
            const int nrows = rbase < p.T ? min(8, (p.T - rbase + 3) / 4) : 0;  // rows rbase + 4*pp < T
            uint32_t eo[8];                                                     // element offset of this lane's 4 columns
#pragma unroll
            for (int pp = 0; pp < 8; ++pp)
              eo[pp] = (rowbase + (uint32_t)min(rbase + pp * 4, p.T - 1)) * (uint32_t)p.n_total + (uint32_t)n;
            float4 pre[8];
#pragma unroll
            for (int pp = 0; pp < 8; ++pp) pre[pp] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p.addend != nullptr) {
              float4 t4[8];
#pragma unroll
              for (int pp = 0; pp < 8; ++pp) t4[pp] = *reinterpret_cast<const float4*>(p.addend + eo[pp]);
#pragma unroll
              for (int pp = 0; pp < 8; ++pp) { pre[pp].x += t4[pp].x; pre[pp].y += t4[pp].y; pre[pp].z += t4[pp].z; pre[pp].w += t4[pp].w; }
            }
            asm volatile("" ::: "memory");     // one operand kind in flight at a time (register budget)
            if (p.res_f32 != nullptr) {
              float4 t4[8];
#pragma unroll
              for (int pp = 0; pp < 8; ++pp) t4[pp] = *reinterpret_cast<const float4*>(p.res_f32 + eo[pp]);
#pragma unroll
              for (int pp = 0; pp < 8; ++pp) { pre[pp].x += t4[pp].x; pre[pp].y += t4[pp].y; pre[pp].z += t4[pp].z; pre[pp].w += t4[pp].w; }
            }
            asm volatile("" ::: "memory");
            if (p.res_planes != nullptr) {
              const uint16_t* const lo_base = p.res_planes + (size_t)p.B * p.T * p.n_total;
              uint2 h2[8], l2[8];
#pragma unroll
              for (int pp = 0; pp < 8; ++pp) {
                h2[pp] = *reinterpret_cast<const uint2*>(p.res_planes + eo[pp]);
                l2[pp] = *reinterpret_cast<const uint2*>(lo_base + eo[pp]);
              }
#pragma unroll
              for (int pp = 0; pp < 8; ++pp) {
                float r0, r1, r2, r3;
                fd_combine2(h2[pp].x, l2[pp].x, PREC, r0, r1);
                fd_combine2(h2[pp].y, l2[pp].y, PREC, r2, r3);
                pre[pp].x += p.res_scale * r0; pre[pp].y += p.res_scale * r1;
                pre[pp].z += p.res_scale * r2; pre[pp].w += p.res_scale * r3;
              }
            }
            asm volatile("" ::: "memory");
            uint32_t mkbits = 0;
            if (p.row_mask != nullptr) {
#pragma unroll
              for (int pp = 0; pp < 8; ++pp)
                if (p.row_mask[rowbase + (uint32_t)min(rbase + pp * 4, p.T - 1)] != 0) mkbits |= 1u << pp;
            }
            // the accumulators are fetched only now: keeping them out of the registers while the operand loads are in
            // flight is what lets 8 rows per lane be outstanding
            tmem_ld16_nowait(taddr + half * PER + c, *reinterpret_cast<float(*)[16]>(&v[0]));
            tmem_ld16_nowait(taddr + half * PER + c + 16, *reinterpret_cast<float(*)[16]>(&v[16]));
            tmem_wait16(*reinterpret_cast<float(*)[16]>(&v[0]));
            tmem_wait16(*reinterpret_cast<float(*)[16]>(&v[16]));
            float4 a[8];
            warp_transpose_32x32(my_scratch, lane, v, a);
#pragma unroll
            for (int pp = 0; pp < 8; ++pp) {
              a[pp].x = (a[pp].x * p.acc_scale + bias4.x + pre[pp].x) * p.post_scale;
              a[pp].y = (a[pp].y * p.acc_scale + bias4.y + pre[pp].y) * p.post_scale;
              a[pp].z = (a[pp].z * p.acc_scale + bias4.z + pre[pp].z) * p.post_scale;
              a[pp].w = (a[pp].w * p.acc_scale + bias4.w + pre[pp].w) * p.post_scale;
            }
            if (p.out_f32 != nullptr && p.out_accum) {       // accumulate launches: one more batch of 8 loads
#pragma unroll
              for (int pp = 0; pp < 8; ++pp) pre[pp] = *reinterpret_cast<const float4*>(p.out_f32 + eo[pp]);
#pragma unroll
              for (int pp = 0; pp < 8; ++pp) { a[pp].x += pre[pp].x; a[pp].y += pre[pp].y; a[pp].z += pre[pp].z; a[pp].w += pre[pp].w; }
            }
            const float slope = p.act == FD_ACT_NONE ? 1.f : p.act == FD_ACT_RELU ? 0.f : p.act_slope;
            uint16_t* const out_lo = p.out_planes + (size_t)p.B * p.T * p.n_total;
#pragma unroll
            for (int pp = 0; pp < 8; ++pp) {
              if (pp >= nrows) break;
              if ((mkbits >> pp) & 1u) a[pp] = make_float4(0.f, 0.f, 0.f, 0.f);      // masked row: zeros everywhere
              if (p.out_f32 != nullptr) *reinterpret_cast<float4*>(p.out_f32 + eo[pp]) = a[pp];
              if (p.out_planes != nullptr) {
                uint32_t h0, l0, h1, l1;
                fd_split2(fd_act(a[pp].x * p.planes_scale, slope), fd_act(a[pp].y * p.planes_scale, slope), PREC, h0, l0);
                fd_split2(fd_act(a[pp].z * p.planes_scale, slope), fd_act(a[pp].w * p.planes_scale, slope), PREC, h1, l1);
                *reinterpret_cast<uint2*>(p.out_planes + eo[pp]) = make_uint2(h0, h1);
                *reinterpret_cast<uint2*>(out_lo + eo[pp]) = make_uint2(l0, l1);
              }
            }
          }
        }
      } else {
        // ---- LINEAR / RES_SKIP with narrow tiles (BLOCK_N <= 32): row-owner epilogue, 16-column chunks
        constexpr int PER = BLOCK_N / HALVES;
        if (half < HALVES) {
          for (int c = 0; c < PER; c += 16) {
            const int col = half * PER + c;
            float v[16];
            tmem_ld16_nowait(taddr + col, v);
            tmem_wait16(v);
            if (valid) {
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                float v8[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) v8[i] = v[h * 8 + i];
                const int cc = col + h * 8;
                if (EPI == FD_EPI_LINEAR) fd_epi_linear<8, PREC>(p, b, t, n0 + cc, v8, bias_g, n0);
                else fd_epi_res_skip<8, PREC>(p, b, t, n0 + cc, v8, bias_g + cc);
              }
            }
          }
        }
      }
      // release this accumulator stage back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      if (++acc == C::ACC_STAGES) { acc = 0; acc_phase ^= 1; }
    }
  }

  // ---------------------------------------------------------------- teardown
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)C::TMEM_COLS)
                 : "memory");
  }
}

// ------------------------------------------------------------------ host side
CUtensorMapSwizzle swizzle_for(int block_k) {
  return block_k == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : block_k == 32 ? CU_TENSOR_MAP_SWIZZLE_64B
                                                                      : CU_TENSOR_MAP_SWIZZLE_32B;
}

int make_src_map(CUtensorMap* m, const uint16_t* ptr, int B, int T, int C, long long rs, long long bs,
                 long long ps, int block_k, int npl) {
  PFN_tmapEncodeTiled enc = get_encode();
  FD_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled not available from the driver");
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)T, (cuuint64_t)B, 2};
  cuuint64_t strides[3] = {(cuuint64_t)rs * 2, (cuuint64_t)bs * 2, (cuuint64_t)ps * 2};
  cuuint32_t box[4] = {(cuuint32_t)block_k, (cuuint32_t)BLOCK_M, 1, (cuuint32_t)npl};   // planes in one box
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_UINT16, 4, const_cast<uint16_t*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(block_k), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  FD_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(src) failed: %d (B=%d T=%d C=%d bk=%d ptr=%p)", (int)r, B,
             T, C, block_k, (const void*)ptr);
  return 0;
}

int make_w_map(CUtensorMap* m, const uint16_t* ptr, int N, int K, int block_n, int block_k, int npl) {
  PFN_tmapEncodeTiled enc = get_encode();
  FD_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled not available from the driver");
  cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)N, 2};
  cuuint64_t strides[2] = {(cuuint64_t)K * 2, (cuuint64_t)N * K * 2};
  cuuint32_t box[3] = {(cuuint32_t)block_k, (cuuint32_t)block_n, (cuuint32_t)npl};   // planes in one box
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_UINT16, 3, const_cast<uint16_t*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(block_k), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  FD_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(w) failed: %d (N=%d K=%d bn=%d bk=%d)", (int)r, N, K,
             block_n, block_k);
  return 0;
}


template <int BLOCK_N, int BLOCK_K, int EPI, int PREC, int NPL>
int launch_inst(const FdTapGemm& p, cudaStream_t stream) {
  using C = Cfg<BLOCK_N, BLOCK_K, EPI, NPL>;
  CUtensorMap tm0, tm1, tmw;
  int rc = make_src_map(&tm0, p.src[0], p.B, p.T, p.src_C[0], p.src_rs[0], p.src_bs[0], p.src_ps[0], BLOCK_K, NPL);
  if (rc) return rc;
  if (p.src[1] != nullptr) {
    rc = make_src_map(&tm1, p.src[1], p.B, p.T, p.src_C[1], p.src_rs[1], p.src_bs[1], p.src_ps[1], BLOCK_K, NPL);
    if (rc) return rc;
  } else {
    tm1 = tm0;
  }
  rc = make_w_map(&tmw, p.w, p.n_total, p.k_total, BLOCK_N, BLOCK_K, NPL);
  if (rc) return rc;

  auto kern = fd_tapgemm_tc_kernel<BLOCK_N, BLOCK_K, EPI, PREC, NPL>;
  static bool attr_set[FD_MAX_DEVICES] = {false};   // the max-dynamic-smem attribute is per device
  const int dev = fd_current_device();
  if (!attr_set[dev]) {
    FD_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    attr_set[dev] = true;
  }
  const int g_num_sms = fd_device_sms(dev);
  const int tiles_t = (p.T + BLOCK_M - 1) / BLOCK_M;
  const int num_tiles = p.B * tiles_t * (p.n_total / BLOCK_N);
  const int grid = num_tiles < g_num_sms ? num_tiles : g_num_sms;
  kern<<<grid, C::NUM_THREADS, C::SMEM_BYTES, stream>>>(tm0, tm1, tmw, p);
  FD_CHECK_CUDA(cudaGetLastError());
  return 0;
}

template <int BLOCK_N, int BLOCK_K, int EPI>
int launch_cfg(const FdTapGemm& p, cudaStream_t stream) {
  if (p.single) {
    return p.prec == FD_F16 ? launch_inst<BLOCK_N, BLOCK_K, EPI, FD_F16, 1>(p, stream)
                            : launch_inst<BLOCK_N, BLOCK_K, EPI, FD_BF16, 1>(p, stream);
  }
  return p.prec == FD_F16 ? launch_inst<BLOCK_N, BLOCK_K, EPI, FD_F16, 2>(p, stream)
                          : launch_inst<BLOCK_N, BLOCK_K, EPI, FD_BF16, 2>(p, stream);
}

template <int BLOCK_N, int BLOCK_K>
int launch_epi(const FdTapGemm& p, cudaStream_t stream) {
  if (p.epi == FD_EPI_GATE) return launch_cfg<BLOCK_N, BLOCK_K, FD_EPI_GATE>(p, stream);
  if (p.epi == FD_EPI_MAG) return launch_cfg<BLOCK_N, BLOCK_K, FD_EPI_MAG>(p, stream);
  if (p.epi == FD_EPI_RES_SKIP) return launch_cfg<BLOCK_N, BLOCK_K, FD_EPI_RES_SKIP>(p, stream);
  if (p.epi == FD_EPI_GATE_BWD) return launch_cfg<BLOCK_N, BLOCK_K, FD_EPI_GATE_BWD>(p, stream);
  return launch_cfg<BLOCK_N, BLOCK_K, FD_EPI_LINEAR>(p, stream);
}

// choose (BLOCK_N, BLOCK_K) for a problem; bn = 0 if no tensor-core instantiation fits
void pick_cfg(const FdTapGemm& p, int* bn, int* bk) {
  *bn = 0; *bk = 0;
  bool all64 = true, all32 = true, all16 = true;
  for (int s = 0; s < p.num_seg; ++s) {
    if (p.seg[s].c_off % 16 != 0) return;
    all64 &= p.seg[s].k_len % 64 == 0;
    all32 &= p.seg[s].k_len % 32 == 0;
    all16 &= p.seg[s].k_len % 16 == 0;
  }
  const int k = all64 ? 64 : all32 ? 32 : all16 ? 16 : 0;
  if (k == 0) return;
  if (p.epi == FD_EPI_GATE || p.epi == FD_EPI_MAG) {
    const int n = p.gate_tile;
    if ((n != 256 && n != 128) || p.n_total % n != 0 || k != 64) return;
    *bn = n; *bk = 64;
    return;
  }
  int n = 256;
  // (GEMM2 with narrower column tiles was measured in round 2: 256 -> 0.406 ms, 128 -> 0.426 ms, 64 -> 0.667 ms per launch)
  while (n >= 16 && (p.n_total % n != 0 || (p.epi == FD_EPI_RES_SKIP && p.C % n != 0))) n >>= 1;
  if (n < 16) return;
  if (k == 64) {
    if (n < 64) return;
    // Wave quantisation (a persistent grid runs ceil(tiles / SMs) tile times; at the training shape, 157 row tiles, an N = 512
    // GEMM is 314 tiles of 256 columns = 3 waves for 2.12 waves of work) was tried against 128-column tiles for LINEAR /
    // GATE_BWD whenever the quantised time came out > 5 % better: same-box A/B of the training step 12.87 / 12.81 -> 12.81 /
    // 12.80 ms (one product), 19.84 / 20.07 -> 19.87 / 19.66 ms (three products) -- noise; left out.
    *bn = n; *bk = 64;
  } else if (k == 32) {
    if (p.epi != FD_EPI_LINEAR || n < 32) return;   // (GATE_BWD: BLOCK_K 64 only)
    *bn = n > 64 ? 64 : n; *bk = 32;
  } else {
    if (p.epi != FD_EPI_LINEAR) return;
    *bn = n > 32 ? 32 : n; *bk = 16;
  }
}

}  // namespace

int fd_tapgemm_tc_supported(const FdTapGemm& p) {
  int bn, bk;
  pick_cfg(p, &bn, &bk);
  if (bn == 0) return 0;
  for (int s = 0; s < 2; ++s)
    if (p.src[s] != nullptr && (p.src_rs[s] % 8 != 0 || p.src_bs[s] % 8 != 0 || p.src_ps[s] % 8 != 0)) return 0;
  if (p.k_total % 8 != 0) return 0;
  return 1;
}

int fd_tapgemm_tc_launch(const FdTapGemm& p, cudaStream_t stream) {
  int bn, bk;
  pick_cfg(p, &bn, &bk);
  FD_REQUIRE((long long)p.B * p.T * p.n_total < (1ll << 32),
             "tapgemm(tc): B*T*n_total = %lld exceeds the 32-bit element offsets of the epilogue",
             (long long)p.B * p.T * p.n_total);
  FD_REQUIRE(bn != 0 && fd_tapgemm_tc_supported(p),
             "tapgemm(tc): no tensor-core instantiation for n_total=%d k_total=%d epi=%d", p.n_total, p.k_total,
             p.epi);
  if (bk == 64) {
    if (bn == 256) return launch_epi<256, 64>(p, stream);
    if (bn == 128) return launch_epi<128, 64>(p, stream);
    if (p.epi == FD_EPI_GATE_BWD) return launch_cfg<64, 64, FD_EPI_GATE_BWD>(p, stream);
    if (p.epi == FD_EPI_RES_SKIP) return launch_cfg<64, 64, FD_EPI_RES_SKIP>(p, stream);
    return launch_cfg<64, 64, FD_EPI_LINEAR>(p, stream);
  }
  if (bk == 32) {
    FD_REQUIRE(p.epi == FD_EPI_LINEAR, "tapgemm(tc): BLOCK_K=32 only instantiated for the linear epilogue");
    if (bn == 64) return launch_cfg<64, 32, FD_EPI_LINEAR>(p, stream);
    return launch_cfg<32, 32, FD_EPI_LINEAR>(p, stream);
  }
  FD_REQUIRE(p.epi == FD_EPI_LINEAR, "tapgemm(tc): BLOCK_K=16 only instantiated for the linear epilogue");
  if (bn == 32) return launch_cfg<32, 16, FD_EPI_LINEAR>(p, stream);
  return launch_cfg<16, 16, FD_EPI_LINEAR>(p, stream);
}
