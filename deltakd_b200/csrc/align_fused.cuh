// Fused forward + dgrad of the hidden-state matching loss (CurKD early / mid, ViTKD mimicking; model/loss.py:376-393,
// 277-289) for one Linear(192 -> Dt) head, Dt = 384 (DeiT-Small teacher) or 768 (DeiT-Base teacher):
//     Y = S W^T + b ;  d = Y - t ;  loss += sum d^2 ;  G = gscale * d (bf16 planes, kept for the weight-gradient GEMM) ;
//     g_s = G W
// in ONE persistent tcgen05 kernel per layer.
//
// Per 128-row tile:
//   * the S tile (student rows as bf16 hi / lo planes) is the A operand of the forward MMA and lives in TENSOR MEMORY
//     (tcgen05.st by the epilogue threads, lane = row, a column = two consecutive K elements; tcgen05.mma reads A from TMEM):
//     no shared memory and no shared-memory bandwidth for it — with S in shared memory (96 KB in the fp32 mode) only two W
//     ring slots fit and every chunk exposed a full TMA round trip, and the 64-wide forward MMAs re-read the 4 KB A slice
//     from shared memory per instruction (192 B/clk against the 128 B/clk the SM has);
//   * W streams through a 4-slot ring in 64-row chunks of the teacher width (Dt), and the SAME chunk is used twice: K-major
//     as the B operand of the forward MMA (Y_c = S W_c^T, K = Ds) and MN-major as the B operand of the dgrad MMA
//     (g_s += d_c W_c, K = the chunk's 64 teacher channels);
//   * the residual chunk d_c goes TMEM -> registers (teacher subtracted, loss accumulated) -> a 128-byte-swizzled K-major
//     shared-memory tile that is both the A operand of dgrad and the source of ONE tensor store per plane into the G planes
//     (no per-thread global stores for G); the g_s accumulator (128 x 192 fp32) stays in TMEM across the Dt / 64 chunks
//     (6 at Dt = 384, 12 at Dt = 768).
// Compared with the three-launch form (forward, dgrad, wgrad) the dgrad kernel's read of G (154 MB per layer in the fp32
// mode) and one pass over the S planes are gone.
//
// Warp roles (352 threads): warp 0 TMA producer (W ring), warp 1 MMA issuer (forward chunk c, then dgrad of chunk c-1),
// warps 2-9 epilogue (two groups of four: group g owns columns [32g, 32g+32) of every chunk,
// its share of the S tile, and alternate 32-column pieces of g_s), warp 10 G tensor stores.
// TMEM (512 columns): Y chunk double-buffered (2 x 64) | g_s (192) | S planes (2 x 96).
// Shared memory: W ring 4 x 48 KB + d tile 32 KB = 224 KB (fp32 mode, P = 2 planes); 4 x 24 + 16 = 112 KB (bf16, P = 1).
// Neither depends on the teacher width: a wider teacher only adds chunks to the walk over each row tile.
#pragma once
#include <stdlib.h>

#include "epilogues.cuh"

namespace dkd {

template <int P_, int DT_>
struct AlignFusedCfg {
  static constexpr int P = P_;                        // bf16 planes per operand (1: bf16, 2: bf16x3)
  static constexpr int TERMS = P_ == 2 ? 3 : 1;
  static constexpr int DS = 192, DT = DT_, CH = 64;   // student width, teacher width, teacher channels per chunk
  static constexpr int NCH = DT / CH;                 // 6 (Dt = 384) or 12 (Dt = 768) chunks per tile
  static constexpr int KB = DS / 64;                  // 3 K blocks of the forward GEMM
  static constexpr int WST = 4;                       // W ring slots
  static constexpr int W_PLANE = KB * CH * 128;       // 24 KB: [KB][64 rows][128 B]
  static constexpr int D_PLANE = 128 * 128;           // 16 KB: [128 rows][64 k]
  static constexpr int W_STAGE = P_ * W_PLANE, D_BYTES = P_ * D_PLANE;
  static constexpr int EPI_WARPS = 8;
  static constexpr int THREADS = 64 + 32 * EPI_WARPS + 32;   // + the G-store warp
  static constexpr size_t SMEM = (size_t)WST * W_STAGE + D_BYTES + 1024 + 256;
  static constexpr uint32_t TM_Y = 0, TM_GS = 128, TM_S = 320;   // TMEM column offsets; S plane pl at TM_S + 96 * pl
  static constexpr int S_COLS = DS / 2;               // 96 packed columns per plane
  static_assert(SMEM <= 227 * 1024, "shared memory");
  static_assert(DT % (2 * CH) == 0, "teacher width: whole pairs of 64-channel chunks");
  static_assert(TM_GS == 2 * CH && TM_S == TM_GS + DS && TM_S + 2 * S_COLS == 512, "TMEM column map: Y (2 x 64) | g_s | S planes = 512");
};

struct AlignFusedParams {
  CUtensorMap tmW;        // W planes [P][Dt][192], box {64, 64, 1}
  CUtensorMap tmG;        // G planes [P][M][Dt], box {64, 128, 1} (stores)
  const __nv_bfloat16* S; // student planes [P][M][192]
  const void* t;          // teacher [B, Tt, Dt]
  const float* bias;      // [Dt] or null
  void* g_s;              // [B, Ts, 192] dtype, or null
  double* partials;       // [gridDim.x]
  int64_t M;
  int n_tok, Tt, t_off, Ts, s_off;
  int t_is_bf16, out_is_bf16;
  float gscale;           // G = gscale * d
  float gs_alpha;         // g_s = gs_alpha * (G W)
  int m_tiles;
};

template <class Cfg>
__global__ void __launch_bounds__(Cfg::THREADS, 1) align_fused_kernel(const __grid_constant__ AlignFusedParams p) {
  using namespace sm100;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sW = smem;
  uint8_t* sD = sW + (size_t)Cfg::WST * Cfg::W_STAGE;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sD + Cfg::D_BYTES);
  uint64_t* s_full = bars;                    // S tile stored to TMEM (8 epilogue warps)
  uint64_t* s_empty = bars + 1;               // last forward MMA of the tile retired
  uint64_t* w_full = bars + 2;
  uint64_t* w_empty = w_full + Cfg::WST;
  uint64_t* y_full = w_empty + Cfg::WST;      // [2]
  uint64_t* y_empty = y_full + 2;             // [2]
  uint64_t* d_full = y_empty + 2;
  uint64_t* d_empty = d_full + 1;
  uint64_t* gs_full = d_empty + 1;
  uint64_t* gs_empty = gs_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(gs_empty + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    mbar_init(s_full, Cfg::EPI_WARPS); mbar_init(s_empty, 1);
    for (int s = 0; s < Cfg::WST; ++s) { mbar_init(&w_full[s], 1); mbar_init(&w_empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&y_full[a], 1); mbar_init(&y_empty[a], Cfg::EPI_WARPS); }
    mbar_init(d_full, Cfg::EPI_WARPS); mbar_init(d_empty, 2);   // d tile free = dgrad MMAs retired + tensor store has read it
    mbar_init(gs_full, 1); mbar_init(gs_empty, Cfg::EPI_WARPS);
    fence_barrier_init();
    tma_prefetch_desc(&p.tmW);
    tma_prefetch_desc(&p.tmG);
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ============================== TMA producer: W chunks ==============================
    if (lane == 0) {
      uint32_t wi = 0;
      for (int tile = blockIdx.x; tile < p.m_tiles; tile += gridDim.x) {
        for (int c = 0; c < Cfg::NCH; ++c, ++wi) {
          const int ws = wi % Cfg::WST;
          mbar_wait(&w_empty[ws], ((wi / Cfg::WST) & 1) ^ 1);
          mbar_expect_tx(&w_full[ws], Cfg::W_STAGE);
          uint8_t* dst = sW + (size_t)ws * Cfg::W_STAGE;
#pragma unroll
          for (int pl = 0; pl < Cfg::P; ++pl)
#pragma unroll
            for (int kb = 0; kb < Cfg::KB; ++kb)
              tma_load_3d(dst + (size_t)pl * Cfg::W_PLANE + (size_t)kb * Cfg::CH * 128, &p.tmW, &w_full[ws], kb * 64, c * Cfg::CH, pl);
        }
      }
    }
  } else if (warp == 1) {
    // ============================== MMA issuer ================================
    // The WHOLE warp runs this loop (barrier waits by all 32 lanes, warp-uniform addresses) and one elected lane issues the
    // tcgen05 instructions: inside an `if (lane == 0)` region every descriptor is a per-thread value and ptxas moves it to
    // the uniform datapath with an ELECT / R2UR / BRA.U.ANY loop per operand (~13 instructions and several dependent
    // uniform-pipe latencies per MMA) — more than the 32 tensor cycles of a 128 x 64 x 16 MMA, i.e. the issue thread, not
    // the tensor pipe, paced the 64-column forward chunks.
    {
      constexpr uint32_t idesc_f = make_idesc_bf16(128, Cfg::CH, MAJOR_K, MAJOR_K);     // Y_c[128, 64] = S[128, 192] W_c[64, 192]^T
      constexpr uint32_t idesc_d = make_idesc_bf16(128, Cfg::DS, MAJOR_K, MAJOR_MN);    // g_s[128, 192] += d_c[128, 64] W_c[64, 192]
      uint32_t ti = 0, ci = 0;     // tiles / chunks processed by this CTA
      const uint32_t sW_base = smem_u32(sW), sD_base = smem_u32(sD);
      // dgrad of global chunk `cd` (tile-local index `d`): needs the d tile from the epilogue; chunk 0 also needs the
      // previous tile's g_s rows read out of tensor memory
      auto dgrad = [&](uint32_t cd, int d, uint32_t ti_) {
        const int ws = cd % Cfg::WST;
        mbar_wait(d_full, cd & 1);
        if (d == 0) mbar_wait(gs_empty, (ti_ & 1) ^ 1);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t w_addr = sW_base + ws * Cfg::W_STAGE;
          const uint32_t t_gs = tmem_base + Cfg::TM_GS;
#pragma unroll
          for (int term = 0; term < Cfg::TERMS; ++term) {
            const uint32_t a_pl = sD_base + (Cfg::P == 2 && term == 1 ? Cfg::D_PLANE : 0);
            const uint32_t b_pl = w_addr + (Cfg::P == 2 && term == 0 ? Cfg::W_PLANE : 0);
#pragma unroll
            for (int k = 0; k < Cfg::CH / 16; ++k)
              umma_bf16(t_gs, kmajor_desc(a_pl + k * 32), mnmajor_desc(b_pl + k * 2048, Cfg::CH * 128), idesc_d,
                        (d == 0 && term == 0 && k == 0) ? 0u : 1u);
          }
          umma_commit(d_empty);          // the d tile may be rewritten ...
          umma_commit(&w_empty[ws]);     // ... and the W chunk's ring slot refilled once these MMAs retire
        }
        __syncwarp();
      };
      for (int tile = blockIdx.x; tile < p.m_tiles; tile += gridDim.x, ++ti) {
        mbar_wait(s_full, ti & 1);
        // forward chunk c, then dgrad of chunk c-1 (whose d tile the epilogue produces while forward c runs)
#pragma unroll 1
        for (int c = 0; c < Cfg::NCH; ++c, ++ci) {
          const int ws = ci % Cfg::WST;
          const uint32_t yb = ci & 1;
          mbar_wait(&w_full[ws], (ci / Cfg::WST) & 1);
          mbar_wait(&y_empty[yb], ((ci >> 1) & 1) ^ 1);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t w_addr = sW_base + ws * Cfg::W_STAGE;
            const uint32_t t_y = tmem_base + Cfg::TM_Y + yb * Cfg::CH;
#pragma unroll
            for (int term = 0; term < Cfg::TERMS; ++term) {      // (S plane, W plane): (hi, lo) (lo, hi) (hi, hi)
              const uint32_t a_pl = tmem_base + Cfg::TM_S + (Cfg::P == 2 && term == 1 ? Cfg::S_COLS : 0);
              const uint32_t b_pl = w_addr + (Cfg::P == 2 && term == 0 ? Cfg::W_PLANE : 0);
#pragma unroll
              for (int kb = 0; kb < Cfg::KB; ++kb)
#pragma unroll
                for (int k = 0; k < 4; ++k)      // 16 K elements = 8 packed TMEM columns per instruction
                  umma_bf16_ts(t_y, a_pl + kb * 32 + k * 8, kmajor_desc(b_pl + kb * Cfg::CH * 128 + k * 32), idesc_f,
                               (term | kb | k) != 0 ? 1u : 0u);
            }
            umma_commit(&y_full[yb]);
            if (c == Cfg::NCH - 1) umma_commit(s_empty);    // last forward MMA of the tile: the S planes may be replaced
          }
          __syncwarp();
          if (c >= 1) dgrad(ci - 1, c - 1, ti);
        }
        dgrad(ci - 1, Cfg::NCH - 1, ti);
        if (elect_one()) umma_commit(gs_full);
        __syncwarp();
      }
    }
  } else if (warp == 2 + Cfg::EPI_WARPS) {
    // ============================== G store warp ==============================
    // every finished d tile (= this chunk of G as bf16 planes, already in the swizzled box layout) goes to HBM with one
    // tensor store per plane; rows past M are clipped by the tensor map
    if (lane == 0) {
      uint32_t ci = 0;
      for (int tile = blockIdx.x; tile < p.m_tiles; tile += gridDim.x) {
        for (int c = 0; c < Cfg::NCH; ++c, ++ci) {
          mbar_wait(d_full, ci & 1);
#pragma unroll
          for (int pl = 0; pl < Cfg::P; ++pl) tma_store_3d(&p.tmG, sD + (size_t)pl * Cfg::D_PLANE, c * Cfg::CH, tile * 128, pl);
          tma_store_commit();
          tma_store_wait_read<0>();       // the store has read the tile
          mbar_arrive(d_empty);
        }
      }
      tma_store_wait<0>();
    }
  } else {
    // ============================== epilogue ==================================
    const int quad = warp & 3;                 // TMEM lane quadrant of this warp
    const int group = (warp - 2) >> 2;         // 0 | 1
    const int row_in_tile = quad * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    float acc = 0.f;
    float ta[32], tb[32];
    uint32_t ti = 0, ci = 0;

    // S tile of `tile_` -> tensor memory (lane = row, 96 packed columns per plane).  P = 2: group g stores plane g;
    // P = 1: group 0 stores columns [0, 64), group 1 columns [64, 96).  The row's loads are issued first (one DRAM round
    // trip), then the TMEM stores.
    auto stage_S = [&](int tile_, uint32_t ti_) {
      const int64_t m_ = (int64_t)tile_ * 128 + row_in_tile;
      const bool live_ = m_ < p.M;
      constexpr int NR = Cfg::P == 2 ? 96 : 64;                           // register words (P = 1, group 1 uses the first 32)
      const int plane = Cfg::P == 2 ? group : 0;
      const int col0 = Cfg::P == 2 ? 0 : group * 64;                      // first packed column of this thread's share
      const int nw = Cfg::P == 2 ? 96 : (group ? 32 : 64);
      uint32_t r[NR];
      const uint4* src = reinterpret_cast<const uint4*>(p.S + (int64_t)plane * p.M * Cfg::DS + (live_ ? m_ : 0) * Cfg::DS + 2 * col0);
#pragma unroll
      for (int q = 0; q < NR / 4; ++q) {
        uint4 w = make_uint4(0u, 0u, 0u, 0u);
        if (live_ && 4 * q < nw) w = __ldg(src + q);
        r[4 * q] = w.x; r[4 * q + 1] = w.y; r[4 * q + 2] = w.z; r[4 * q + 3] = w.w;
      }
      mbar_wait(s_empty, (ti_ & 1) ^ 1);      // the previous tile's forward MMAs have retired
      tc_fence_after();
      const uint32_t t_s = tmem_base + lane_base + Cfg::TM_S + plane * Cfg::S_COLS + col0;
      tmem_st32(t_s, *reinterpret_cast<const uint32_t(*)[32]>(&r[0]));
      if (Cfg::P == 2 || group == 0) tmem_st32(t_s + 32, *reinterpret_cast<const uint32_t(*)[32]>(&r[32]));
      if constexpr (Cfg::P == 2) tmem_st32(t_s + 64, *reinterpret_cast<const uint32_t(*)[32]>(&r[64]));
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(s_full);
    };

    if ((int)blockIdx.x < p.m_tiles) stage_S(blockIdx.x, 0);
    for (int tile = blockIdx.x; tile < p.m_tiles; tile += gridDim.x, ++ti) {
      const int64_t m = (int64_t)tile * 128 + row_in_tile;
      const bool live = m < p.M;
      const int64_t b = live ? m / p.n_tok : 0;
      const int64_t tok = live ? m - b * p.n_tok : 0;
      const int64_t trow = b * p.Tt + p.t_off + tok;
      // teacher values: two register buffers used alternately (no copies: a copy would wait for the load it was meant to
      // hide); chunk c+1's values are requested before chunk c is processed, chunk 0 of the NEXT tile before this tile's
      // g_s rows are stored
      auto load_t = [&](int64_t trow_, bool live_, int col, float (&x)[32]) {
        if (!live_) {
#pragma unroll
          for (int j = 0; j < 32; ++j) x[j] = 0.f;
        } else {
          load_act32(p.t, trow_ * Cfg::DT + col, p.t_is_bf16, x);
        }
      };
      auto chunk = [&](int c, const float (&tv)[32]) {
        const uint32_t yb = ci & 1;
        const int col = c * Cfg::CH + group * 32;           // teacher / G column of this thread's 32 values
        float bs[32];
        ldg_vec32(p.bias ? p.bias + col : nullptr, bs);
        mbar_wait(&y_full[yb], (ci >> 1) & 1);
        tc_fence_after();
        float v[32];
        tmem_ld32(tmem_base + lane_base + Cfg::TM_Y + yb * Cfg::CH + group * 32, v);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&y_empty[yb]);           // the accumulator chunk is in registers: the next forward may overwrite it
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          const float d0 = v[j] + bs[j] - tv[j], d1 = v[j + 1] + bs[j + 1] - tv[j + 1];
          if (live) { acc = fmaf(d0, d0, acc); acc = fmaf(d1, d1, acc); }
          const float g0 = live ? p.gscale * d0 : 0.f, g1 = live ? p.gscale * d1 : 0.f;
          const __nv_bfloat162 h = __floats2bfloat162_rn(g0, g1);
          hi[j >> 1] = *reinterpret_cast<const uint32_t*>(&h);
          if (Cfg::P == 2) {
            const __nv_bfloat162 l = __floats2bfloat162_rn(g0 - __low2float(h), g1 - __high2float(h));
            lo[j >> 1] = *reinterpret_cast<const uint32_t*>(&l);
          }
        }
        // d_c into the K-major operand tile — dgrad's A operand AND the source of the G-plane tensor store
        // (128-byte swizzle: 16-byte chunk j of row r sits at chunk j ^ (r & 7))
        mbar_wait(d_empty, (ci & 1) ^ 1);
        {
          uint8_t* drow = sD + row_in_tile * 128;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int phys = (group * 4 + q) ^ (row_in_tile & 7);
            *reinterpret_cast<uint4*>(drow + phys * 16) = make_uint4(hi[4 * q], hi[4 * q + 1], hi[4 * q + 2], hi[4 * q + 3]);
            if (Cfg::P == 2)
              *reinterpret_cast<uint4*>(drow + Cfg::D_PLANE + phys * 16) = make_uint4(lo[4 * q], lo[4 * q + 1], lo[4 * q + 2], lo[4 * q + 3]);
          }
        }
        fence_proxy_async();        // generic-proxy stores -> visible to the tensor core's (async proxy) operand reads
        __syncwarp();
        if (lane == 0) mbar_arrive(d_full);
        ++ci;
      };
      if (ti == 0) load_t(trow, live, group * 32, ta);      // later tiles: requested at the end of the previous tile
      // the next tile's row (for its chunk-0 prefetch)
      const int tile_n = tile + (int)gridDim.x;
      const int64_t m_n = (int64_t)tile_n * 128 + row_in_tile;
      const bool live_n = tile_n < p.m_tiles && m_n < p.M;
      const int64_t b_n = live_n ? m_n / p.n_tok : 0;
      const int64_t trow_n = b_n * p.Tt + p.t_off + (live_n ? m_n - b_n * p.n_tok : 0);
      static_assert(Cfg::NCH % 2 == 0, "chunks are processed in pairs");
#pragma unroll 1
      for (int c = 0; c < Cfg::NCH; c += 2) {
        load_t(trow, live, (c + 1) * Cfg::CH + group * 32, tb);
        chunk(c, ta);
        if (c + 2 < Cfg::NCH) load_t(trow, live, (c + 2) * Cfg::CH + group * 32, ta);
        else load_t(trow_n, live_n, group * 32, ta);
        chunk(c + 1, tb);
      }
      // the next tile's S planes go to tensor memory BEFORE this tile's g_s rows are read out: its forward MMAs then run
      // under the g_s stores (the last forward of this tile retired before y_full of its last chunk, so s_empty has completed)
      if (tile_n < p.m_tiles) stage_S(tile_n, ti + 1);
      // ---- g_s rows of this tile: 6 pieces of 32 columns, alternating between the two groups
      mbar_wait(gs_full, ti & 1);
      tc_fence_after();
      const int64_t orow = b * p.Ts + p.s_off + tok;
#pragma unroll 1
      for (int c0 = group * 32; c0 < Cfg::DS; c0 += 64) {
        float v[32];
        tmem_ld32(tmem_base + lane_base + Cfg::TM_GS + c0, v);
        tmem_ld_wait();
        if (!live || p.g_s == nullptr) continue;
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] *= p.gs_alpha;
        float z8[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) z8[j] = 0.f;
        if (p.out_is_bf16) {
          __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(p.g_s) + orow * Cfg::DS + c0;
          stg256(op, *reinterpret_cast<float(*)[16]>(&v[0]));
          stg256(op + 16, *reinterpret_cast<float(*)[16]>(&v[16]));
          if (tok == 0)      // the special-token rows in front of this sample's patches get zero gradient
            for (int r = 1; r <= p.s_off; ++r)
#pragma unroll
              for (int j = 0; j < 4; ++j) Vec<__nv_bfloat16, 8>::store(op - (int64_t)r * Cfg::DS + 8 * j, z8);
        } else {
          float* op = reinterpret_cast<float*>(p.g_s) + orow * Cfg::DS + c0;
#pragma unroll
          for (int j = 0; j < 4; ++j) stg256(op + 8 * j, *reinterpret_cast<float(*)[8]>(&v[8 * j]));
          if (tok == 0)
            for (int r = 1; r <= p.s_off; ++r)
#pragma unroll
              for (int j = 0; j < 4; ++j) stg256(op - (int64_t)r * Cfg::DS + 8 * j, z8);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(gs_empty);
    }
    epilogue_block_partial<Cfg::EPI_WARPS>(acc, threadIdx.x - 64, p.partials);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// host: forward + dgrad of one layer.  `grid_out` = number of loss partials written.
template <int P, int DT>
inline int align_fused_fwd_dgrad_t(const __nv_bfloat16* S, const __nv_bfloat16* Wp, const float* bias, const void* t, int t_is_bf16, int Tt,
                                   int t_off, int n_tok, __nv_bfloat16* G, double* partials, float gscale, void* g_s, int Ts, int s_off,
                                   int out_is_bf16, float gs_alpha, int64_t M, cudaStream_t st, int* grid_out, const char* what) {
  using Cfg = AlignFusedCfg<P, DT>;
  AlignFusedParams p;
  int rc = make_plane_tmap(&p.tmW, Wp, P, Cfg::DT, Cfg::DS, Cfg::DS, (int64_t)Cfg::DT * Cfg::DS, Cfg::CH, what);
  if (rc != DKD_OK) return rc;
  rc = make_plane_tmap(&p.tmG, G, P, M, Cfg::DT, Cfg::DT, M * Cfg::DT, 128, what);
  if (rc != DKD_OK) return rc;
  p.S = S; p.t = t; p.bias = bias; p.g_s = g_s; p.partials = partials; p.M = M; p.n_tok = n_tok; p.Tt = Tt; p.t_off = t_off;
  p.Ts = Ts; p.s_off = s_off; p.t_is_bf16 = t_is_bf16; p.out_is_bf16 = out_is_bf16; p.gscale = gscale; p.gs_alpha = gs_alpha;
  p.m_tiles = (int)((M + 127) / 128);
  const int grid = p.m_tiles < kNumSMs ? p.m_tiles : kNumSMs;
  auto kern = align_fused_kernel<Cfg>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
  kern<<<grid, Cfg::THREADS, Cfg::SMEM, st>>>(p);
  *grid_out = grid;
  return check_launch(what);
}

// host: the instantiation for (P, Dt); Dt in {384, 768} (the caller has checked it)
inline int align_fused_fwd_dgrad(int P, int Dt, const __nv_bfloat16* S, const __nv_bfloat16* Wp, const float* bias, const void* t,
                                 int t_is_bf16, int Tt, int t_off, int n_tok, __nv_bfloat16* G, double* partials, float gscale, void* g_s,
                                 int Ts, int s_off, int out_is_bf16, float gs_alpha, int64_t M, cudaStream_t st, int* grid_out,
                                 const char* what) {
  auto run = [&](auto kern) {
    return kern(S, Wp, bias, t, t_is_bf16, Tt, t_off, n_tok, G, partials, gscale, g_s, Ts, s_off, out_is_bf16, gs_alpha, M, st, grid_out, what);
  };
  if (Dt == 768) return P == 2 ? run(align_fused_fwd_dgrad_t<2, 768>) : run(align_fused_fwd_dgrad_t<1, 768>);
  return P == 2 ? run(align_fused_fwd_dgrad_t<2, 384>) : run(align_fused_fwd_dgrad_t<1, 384>);
}

}  // namespace dkd
