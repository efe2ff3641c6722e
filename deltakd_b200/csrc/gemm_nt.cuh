// Split-K "contract over rows" tcgen05 GEMM for sm_100a:   D[NA, NB] += sum_r A[r, NA] * B[r, NB]
// (weight gradients and Gram-type products).  Both operands are row-major bf16 plane tensors whose
// contraction index is the ROW, so they are consumed as MN-major UMMA operands: a TMA box
// {64 cols, KROWS rows} (128-byte swizzle) is one 64(mn) x KROWS(k) operand block.
//
// Work item = (output tile, row split); the Loader policy decodes it.  Each CTA loops over its items;
// per item it accumulates over the split's row blocks in TMEM (one 128 x NB fp32 tile) and the epilogue
// adds the tile into fp32 D with red.global.add (D is zeroed by the host wrapper), or, with `store` and `split_stride`,
// writes it with plain stores into the split's own slot of a partial buffer that fold_splits_kernel then reduces in split
// order (the deterministic mode: no float add depends on CTA timing).  Warp roles as in
// gemm_tn.cuh: warp 0 TMA producer, warp 1 MMA issuer, warps 2-5 epilogue.
//
// The B operand may carry one extra box from a constant "ones" tile (column 0 = 1): its first 16
// columns extend N by 16 and column NB_DATA of the result is then sum_r A[r, :] (a bias gradient).
#pragma once
#include "umma.cuh"

namespace dkd {

// PLANES_ = 2: a stage holds both bf16 planes of the A and B blocks and the three bf16x3 products are issued from it
// (each operand byte is fetched once instead of 1.5 times); the caller passes nterms = 3.
// CLUSTER_ > 1: clusters of CLUSTER_ CTAs work on items that share the B operand (same contraction rows, same B columns,
// different A column tile): each CTA fetches 1/CLUSTER_ of every B block and multicasts it to the cluster (Loader::issue_cluster).
template <int NB_BOXES_, bool ONES_, int N0_, int N1_, int STAGES_, int KROWS_ = 64, bool A_KMAJOR_ = false, int PLANES_ = 1,
          int CLUSTER_ = 1>
struct GemmNtCfg {
  static constexpr int CLUSTER = CLUSTER_;
  static constexpr int PLANES = PLANES_;
  static constexpr bool A_KMAJOR = A_KMAJOR_;       // A tile is [128 rows x 64 k] K-major (one box) instead of two MN-major boxes
  static constexpr int NA = 128;                      // UMMA M
  static constexpr int NB_BOXES = NB_BOXES_;          // 64-column boxes of B data
  static constexpr bool ONES = ONES_;
  static constexpr int NB_DATA = 64 * NB_BOXES_;
  static constexpr int NB = NB_DATA + (ONES_ ? 16 : 0);
  static constexpr int N0 = N0_, N1 = N1_;            // N of the one or two MMA instructions per K step
  static constexpr int KROWS = KROWS_;                // contraction rows per stage (multiple of 16)
  static constexpr int KSTEPS = KROWS_ / 16;
  static constexpr int BOX_BYTES = KROWS_ * 128;
  static constexpr int A_BYTES = 2 * BOX_BYTES;
  static constexpr int B_BYTES = (NB_BOXES_ + (ONES_ ? 1 : 0)) * BOX_BYTES;
  static constexpr int STAGE_BYTES = PLANES_ * (A_BYTES + B_BYTES);
  static constexpr int STAGES = STAGES_;
  static constexpr int TMEM_COLS = NB <= 32 ? 32 : NB <= 64 ? 64 : NB <= 128 ? 128 : NB <= 256 ? 256 : 512;
  static constexpr int THREADS = 192;
  static constexpr size_t SMEM = (size_t)STAGES_ * STAGE_BYTES + 1024 + 256;
  static_assert(N0_ + N1_ == NB, "instruction N split must cover NB");
  static_assert(N0_ % 16 == 0 && N0_ <= 256 && N1_ % 16 == 0 && N1_ <= 256 && (N1_ == 0 || N0_ % 64 == 0), "UMMA N split");
  static_assert(KROWS_ % 16 == 0 && BOX_BYTES % 1024 == 0, "K rows per stage");
  static_assert(NB <= 512 && SMEM <= 227 * 1024, "resources");
  static_assert(!A_KMAJOR_ || KROWS_ == 64, "K-major A tiles are 128 x 64");
};

struct NtEpilogueParams {
  float* D = nullptr;     // fp32, += via red.add (or plain stores when `store`)
  float* Dcol = nullptr;  // += column NB_DATA of the tile (ones trick), or null; plain stores when `store`
  int ldd = 0;
  float alpha = 1.f;
  int store = 0;          // 1: the tile is written with plain stores (each item owns its output, e.g. per-split partials)
  int64_t split_stride = 0;  // elements between the per-split slots of D and Dcol (items carry their split index)
  int rows_valid = 128;   // output rows of the 128-row tile that exist (A narrower than 128 columns)
  __nv_bfloat16* Dplanes = nullptr;  // if set: the tile is written as bf16 hi(/lo) planes here instead of fp32 D
  int64_t plane_stride = 0;
  int n_planes = 0;
};

// Loader policy interface:
//   Params; num_items(p); decode(p, item, Item&); row_blocks(p, item_info) -> [rb0, rb1);
//   issue(p, info, term, rb, sA, sB, bar); out_ptr(p, info) -> float* of the tile's (row 0, col 0); col_ptr
template <class Cfg, class Loader>
struct GemmNtParamsT {
  typename Loader::Params ld;
  NtEpilogueParams ep;
  int nterms;
  int a_lo_zero = 0;   // PLANES == 2: A's lo plane is identically zero: not fetched, (A lo, B hi) product skipped
};

template <class Cfg, class Loader>
__global__ void __launch_bounds__(Cfg::THREADS, 1) gemm_nt_kernel(const __grid_constant__ GemmNtParamsT<Cfg, Loader> p) {
  using namespace sm100;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;
  constexpr int A_STAGE = Cfg::PLANES * Cfg::A_BYTES, B_STAGE = Cfg::PLANES * Cfg::B_BYTES;
  uint8_t* sB = smem + (size_t)Cfg::STAGES * A_STAGE;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)Cfg::STAGES * Cfg::STAGE_BYTES);
  uint64_t* empty = full + Cfg::STAGES;
  uint64_t* acc_full = empty + Cfg::STAGES;
  uint64_t* acc_empty = acc_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_items = Loader::num_items(p.ld);
  // cluster form: the CTAs of a cluster take the same item (the loader maps the rank to the A column tile)
  const int crank = Cfg::CLUSTER > 1 ? (int)cluster_ctarank() : 0;
  const int item0 = (int)blockIdx.x / Cfg::CLUSTER, item_step = (int)gridDim.x / Cfg::CLUSTER;
  constexpr uint16_t kClusterMask = (uint16_t)((1u << Cfg::CLUSTER) - 1u);

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < Cfg::STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], Cfg::CLUSTER); }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, 4);
    fence_barrier_init();
    Loader::prefetch(p.ld);
  }
  if (warp == 1) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  if constexpr (Cfg::CLUSTER > 1) cluster_sync();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int s = 0; uint32_t ph = 0;
      for (int item = item0; item < num_items; item += item_step) {
        typename Loader::Item it;
        if constexpr (Cfg::CLUSTER > 1) Loader::decode_cluster(p.ld, item, crank, it);
        else Loader::decode(p.ld, item, it);
        if constexpr (Cfg::PLANES == 2) {
          for (int rb = it.rb0; rb < it.rb1; ++rb) {
            mbar_wait(&empty[s], ph ^ 1);
            mbar_expect_tx(&full[s], Loader::TX_BYTES - (p.a_lo_zero ? Cfg::A_BYTES : 0));
            const bool with_a_lo = !p.a_lo_zero;
            if constexpr (Cfg::CLUSTER > 1) {
              Loader::issue_planes_cluster(p.ld, it, 0, 0, rb, sA + (size_t)s * A_STAGE, sB + (size_t)s * B_STAGE, &full[s], crank, true);
              Loader::issue_planes_cluster(p.ld, it, 1, 1, rb, sA + (size_t)s * A_STAGE + Cfg::A_BYTES, sB + (size_t)s * B_STAGE + Cfg::B_BYTES,
                                           &full[s], crank, with_a_lo);
            } else {
              Loader::issue_planes(p.ld, it, 0, 0, rb, sA + (size_t)s * A_STAGE, sB + (size_t)s * B_STAGE, &full[s], true);
              Loader::issue_planes(p.ld, it, 1, 1, rb, sA + (size_t)s * A_STAGE + Cfg::A_BYTES, sB + (size_t)s * B_STAGE + Cfg::B_BYTES, &full[s],
                                   with_a_lo);
            }
            if (++s == Cfg::STAGES) { s = 0; ph ^= 1; }
          }
        } else {
          for (int term = 0; term < p.nterms; ++term) {
            for (int rb = it.rb0; rb < it.rb1; ++rb) {
              mbar_wait(&empty[s], ph ^ 1);
              mbar_expect_tx(&full[s], Loader::TX_BYTES);
              if constexpr (Cfg::CLUSTER > 1)
                Loader::issue_cluster(p.ld, it, term, p.nterms, rb, sA + (size_t)s * A_STAGE, sB + (size_t)s * B_STAGE, &full[s], crank);
              else
                Loader::issue(p.ld, it, term, p.nterms, rb, sA + (size_t)s * A_STAGE, sB + (size_t)s * B_STAGE, &full[s]);
              if (++s == Cfg::STAGES) { s = 0; ph ^= 1; }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    {   // whole warp walks the loop, one elected lane issues (see gemm_tn.cuh)
      constexpr uint32_t a_major = Cfg::A_KMAJOR ? MAJOR_K : MAJOR_MN;
      constexpr uint32_t idesc0 = make_idesc_bf16(128, Cfg::N0, a_major, MAJOR_MN);
      constexpr uint32_t idesc1 = make_idesc_bf16(128, Cfg::N1 > 0 ? Cfg::N1 : 16, a_major, MAJOR_MN);
      int s = 0; uint32_t ph = 0; uint32_t aph = 0;
      for (int item = item0; item < num_items; item += item_step) {
        typename Loader::Item it;
        if constexpr (Cfg::CLUSTER > 1) Loader::decode_cluster(p.ld, item, crank, it);
        else Loader::decode(p.ld, item, it);
        const int nk = (it.rb1 - it.rb0) * (Cfg::PLANES == 2 ? 1 : p.nterms);
        if (nk <= 0) continue;  // (hosts never create empty splits)
        mbar_wait(acc_empty, aph ^ 1);
        tc_fence_after();
        for (int kit = 0; kit < nk; ++kit) {
          mbar_wait(&full[s], ph);
          tc_fence_after();
          const uint32_t a_st = smem_u32(sA + (size_t)s * A_STAGE);
          const uint32_t b_st = smem_u32(sB + (size_t)s * B_STAGE);
          constexpr int TERMS = Cfg::PLANES == 2 ? 3 : 1;     // (A plane, B plane): (hi,lo) (lo,hi) (hi,hi)
          if (elect_one()) {
#pragma unroll
            for (int term = 0; term < TERMS; ++term) {
              if (Cfg::PLANES == 2 && term == 1 && p.a_lo_zero) continue;
              const uint32_t a_addr = a_st + (Cfg::PLANES == 2 && term == 1 ? Cfg::A_BYTES : 0);
              const uint32_t b_addr = b_st + (Cfg::PLANES == 2 && term == 0 ? Cfg::B_BYTES : 0);
#pragma unroll
              for (int k = 0; k < Cfg::KSTEPS; ++k) {  // UMMA_K = 16 rows = 2 groups of 8 rows = 2048 B
                const uint64_t da = Cfg::A_KMAJOR ? kmajor_desc(a_addr + k * 32) : mnmajor_desc(a_addr + k * 2048, Cfg::BOX_BYTES);
                umma_bf16(tmem_base, da, mnmajor_desc(b_addr + k * 2048, Cfg::BOX_BYTES), idesc0, (kit | term | k) != 0 ? 1u : 0u);
                if constexpr (Cfg::N1 > 0)
                  umma_bf16(tmem_base + Cfg::N0, da, mnmajor_desc(b_addr + (Cfg::N0 / 64) * Cfg::BOX_BYTES + k * 2048, Cfg::BOX_BYTES),
                            idesc1, (kit | term | k) != 0 ? 1u : 0u);
              }
            }
            if constexpr (Cfg::CLUSTER > 1) umma_commit_mc(&empty[s], kClusterMask);
            else umma_commit(&empty[s]);
            if (kit == nk - 1) umma_commit(acc_full);
          }
          __syncwarp();
          if (++s == Cfg::STAGES) { s = 0; ph ^= 1; }
        }
        aph ^= 1;
      }
    }
  } else {
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    uint32_t aph = 0;
    for (int item = item0; item < num_items; item += item_step) {
      typename Loader::Item it;
      if constexpr (Cfg::CLUSTER > 1) Loader::decode_cluster(p.ld, item, crank, it);
      else Loader::decode(p.ld, item, it);
      if (it.rb1 <= it.rb0) continue;
      mbar_wait(acc_full, aph);
      tc_fence_after();
      const uint32_t t_acc = tmem_base + ((uint32_t)(quad * 32) << 16);
      const int64_t slot = (int64_t)it.split * p.ep.split_stride;
      float* drow = p.ep.D + slot + it.d_off + (size_t)row * p.ep.ldd;
      const bool row_ok = row < p.ep.rows_valid && row < it.rows;
#pragma unroll 1
      for (int c0 = 0; c0 < Cfg::NB_DATA; c0 += 32) {
        float v[32];
        tmem_ld32(t_acc + c0, v);
        tmem_ld_wait();
        if (!row_ok) continue;
        if (p.ep.Dplanes) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] *= p.ep.alpha;
          store_planes32(p.ep.Dplanes + it.d_off + (size_t)row * p.ep.ldd + c0, p.ep.plane_stride, p.ep.n_planes, v);
        } else if (p.ep.store) {
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            *reinterpret_cast<float4*>(drow + c0 + j) =
                make_float4(v[j] * p.ep.alpha, v[j + 1] * p.ep.alpha, v[j + 2] * p.ep.alpha, v[j + 3] * p.ep.alpha);
        } else {   // split-K reduction: 128-bit vector reductions (REDG.ADD.F32x4): a quarter of the L2 atomic operations
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(drow + c0 + j), "f"(v[j] * p.ep.alpha),
                         "f"(v[j + 1] * p.ep.alpha), "f"(v[j + 2] * p.ep.alpha), "f"(v[j + 3] * p.ep.alpha)
                         : "memory");
        }
      }
      if constexpr (Cfg::ONES) {
        float v[32];
        tmem_ld32(t_acc + Cfg::NB_DATA - 16, v);  // columns NB_DATA-16 .. NB_DATA+15 (inside the allocation)
        tmem_ld_wait();
        if (row_ok && p.ep.Dcol && it.dcol_off >= 0) {
          if (p.ep.store) p.ep.Dcol[slot + it.dcol_off + row] = v[16] * p.ep.alpha;
          else atomicAdd(p.ep.Dcol + it.dcol_off + row, v[16] * p.ep.alpha);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty);
      aph ^= 1;
    }
  }

  tc_fence_before();
  __syncthreads();
  if constexpr (Cfg::CLUSTER > 1) cluster_sync();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// host: launch, as clusters of Cfg::CLUSTER CTAs when asked (`grid` = CTAs, a multiple of the cluster size)
template <class Cfg, class Loader>
inline void launch_gemm_nt(const GemmNtParamsT<Cfg, Loader>& p, int grid, cudaStream_t st) {
  auto kern = gemm_nt_kernel<Cfg, Loader>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
  if constexpr (Cfg::CLUSTER > 1) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(Cfg::THREADS);
    cfg.dynamicSmemBytes = Cfg::SMEM;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = Cfg::CLUSTER;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, kern, p);
  } else {
    kern<<<grid, Cfg::THREADS, Cfg::SMEM, st>>>(p);
  }
}

// host: number of row splits in [lo, hi] that fills whole waves best: maximises items / (ceil(items / slots) * slots)
inline int nt_best_splits(int combos, int slots, int total_row_blocks, int lo, int hi) {
  int best = lo;
  double best_eff = -1.0;
  for (int sp = lo; sp <= hi && sp <= total_row_blocks; ++sp) {
    const int per = (total_row_blocks + sp - 1) / sp;
    const int real = (total_row_blocks + per - 1) / per;         // splits that exist after rounding
    const long items = (long)combos * real;
    const long waves = (items + slots - 1) / slots;
    // ragged last split costs a full `per`: weigh by the work actually done
    const double eff = (double)combos * total_row_blocks / ((double)waves * slots * per);
    if (eff > best_eff + 1e-9) { best_eff = eff; best = sp; }
  }
  return best;
}

struct NtItem {
  int rb0, rb1;      // row blocks [rb0, rb1) of KROWS rows
  int a_col0;        // first A column (output row) of the tile
  int b_col0;        // first B column
  int64_t d_off;     // element offset of the tile's (0,0) in D
  int dcol_off;      // offset into Dcol, or -1
  int aux;           // loader specific (e.g. filter tap)
  int rows = 128;    // output rows of this item's tile that exist (<= 128)
  int split = 0;     // row split: selects the partial slot (NtEpilogueParams::split_stride)
};

// Plain loader: A = planes [P][R][NA_total], B = planes [P][R][NB_total], 3-D maps {cols, rows, planes}, box {64, KROWS, 1}.
// GROUPS_ (cluster form only): the A column tiles are GROUPS_ groups of CLUSTER tiles (na_tiles == GROUPS_ * CLUSTER).
struct NtPlainParams {
  CUtensorMap tmA, tmB, tmOnes;
  int na_tiles, splits, row_blocks_per_split, total_row_blocks, b_col0, ldd;
};
template <class Cfg, int GROUPS_ = 1>
struct NtPlainLoader {
  using Params = NtPlainParams;
  using Item = NtItem;
  static constexpr uint32_t TX_BYTES = Cfg::STAGE_BYTES;
  static_assert(GROUPS_ >= 1 && (GROUPS_ == 1 || Cfg::CLUSTER > 1), "tile groups are a cluster-form schedule");
  static __device__ __forceinline__ int num_items(const Params& p) { return Cfg::CLUSTER > 1 ? GROUPS_ * p.splits : p.na_tiles * p.splits; }
  static __device__ __forceinline__ void prefetch(const Params& p) {
    sm100::tma_prefetch_desc(&p.tmA);
    sm100::tma_prefetch_desc(&p.tmB);
  }
  static __device__ __forceinline__ void decode(const Params& p, int item, Item& it) {
    const int tile = item % p.na_tiles, split = item / p.na_tiles;
    it.split = split;
    it.rb0 = split * p.row_blocks_per_split;
    it.rb1 = min(it.rb0 + p.row_blocks_per_split, p.total_row_blocks);
    it.a_col0 = tile * 128;
    it.b_col0 = p.b_col0;
    it.d_off = (int64_t)tile * 128 * p.ldd;
    it.dcol_off = tile * 128;
    it.aux = 0;
  }
  static __device__ __forceinline__ void issue(const Params& p, const Item& it, int term, int nterms, int rb, uint8_t* a, uint8_t* b, uint64_t* bar) {
    int pa, pb;
    term_planes(term, nterms, pa, pb);
    issue_planes(p, it, pa, pb, rb, a, b, bar);
  }
  static __device__ __forceinline__ void issue_planes(const Params& p, const Item& it, int pa, int pb, int rb, uint8_t* a, uint8_t* b, uint64_t* bar,
                                                      bool with_a = true) {
    if (with_a) {
      sm100::tma_load_3d(a, &p.tmA, bar, it.a_col0, rb * Cfg::KROWS, pa);
      sm100::tma_load_3d(a + Cfg::BOX_BYTES, &p.tmA, bar, it.a_col0 + 64, rb * Cfg::KROWS, pa);
    }
#pragma unroll
    for (int i = 0; i < Cfg::NB_BOXES; ++i)
      sm100::tma_load_3d(b + (size_t)i * Cfg::BOX_BYTES, &p.tmB, bar, it.b_col0 + i * 64, rb * Cfg::KROWS, pb);
    if constexpr (Cfg::ONES)  // plane 0 of the ones tile is {1,0,0,...}; its lo plane is all zero
      sm100::tma_load_3d(b + (size_t)Cfg::NB_BOXES * Cfg::BOX_BYTES, &p.tmOnes, bar, 0, 0, pb);
  }
  // ---- cluster form: a work item is one (tile group, row split) pair, and the CLUSTER CTAs of a cluster are the A column
  // tiles of ONE group (CTA `crank` of group g owns tile g * CLUSTER + crank) over ONE row split: they contract over the
  // same rows of B, so CTA `crank` fetches B box `crank` and multicasts it (NB_BOXES == CLUSTER).  GROUPS_ = 1: the
  // cluster covers all A tiles (na_tiles == CLUSTER) and an item is a row split.
  static __device__ __forceinline__ int num_items_cluster(const Params& p) { return GROUPS_ * p.splits; }
  static __device__ __forceinline__ void decode_cluster(const Params& p, int item, int crank, Item& it) {
    const int group = item % GROUPS_, split = item / GROUPS_;
    const int tile = group * Cfg::CLUSTER + crank;
    it.split = split;
    it.rb0 = split * p.row_blocks_per_split;
    it.rb1 = min(it.rb0 + p.row_blocks_per_split, p.total_row_blocks);
    it.a_col0 = tile * 128;
    it.b_col0 = p.b_col0;
    it.d_off = (int64_t)tile * 128 * p.ldd;
    it.dcol_off = tile * 128;
    it.aux = 0;
  }
  static __device__ __forceinline__ void issue_planes_cluster(const Params& p, const Item& it, int pa, int pb, int rb, uint8_t* a, uint8_t* b,
                                                              uint64_t* bar, int crank, bool with_a = true) {
    static_assert(Cfg::CLUSTER == 1 || Cfg::NB_BOXES == Cfg::CLUSTER, "one B box per CTA of the cluster");
    if (with_a) {
      sm100::tma_load_3d(a, &p.tmA, bar, it.a_col0, rb * Cfg::KROWS, pa);
      sm100::tma_load_3d(a + Cfg::BOX_BYTES, &p.tmA, bar, it.a_col0 + 64, rb * Cfg::KROWS, pa);
    }
    sm100::tma_load_3d_mc(b + (size_t)crank * Cfg::BOX_BYTES, &p.tmB, bar, it.b_col0 + crank * 64, rb * Cfg::KROWS, pb,
                          (uint16_t)((1u << Cfg::CLUSTER) - 1u));
    if constexpr (Cfg::ONES) sm100::tma_load_3d(b + (size_t)Cfg::NB_BOXES * Cfg::BOX_BYTES, &p.tmOnes, bar, 0, 0, pb);
  }
  static __device__ __forceinline__ void issue_cluster(const Params& p, const Item& it, int term, int nterms, int rb, uint8_t* a, uint8_t* b,
                                                       uint64_t* bar, int crank) {
    int pa, pb;
    term_planes(term, nterms, pa, pb);
    issue_planes_cluster(p, it, pa, pb, rb, a, b, bar, crank);
  }
};

// host: elements between the per-split slots of a deterministic-mode partial buffer that holds `n` floats per split.
// The store epilogue writes the tile with 16-byte vector stores from the slot base, so a slot starts on a 128-byte
// boundary (whole L2 sectors) whatever `n` is (e.g. LRKD's rank * (Ds + 1) for an odd rank).
inline int64_t nt_slot_floats(int64_t n) { return (n + 31) / 32 * 32; }

// host: split `total_row_blocks` over about `want` splits with no empty split
inline void nt_make_splits(int total_row_blocks, int want, int* splits, int* per_split) {
  if (want < 1) want = 1;
  *per_split = (total_row_blocks + want - 1) / want;
  if (*per_split < 1) *per_split = 1;
  *splits = (total_row_blocks + *per_split - 1) / *per_split;
}

}  // namespace dkd
