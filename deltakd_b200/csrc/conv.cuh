// 3x3 / pad 1 convolution on the HW x HW token grid (HW = 14: 224-px inputs, HW = 24: 384-px inputs, patch 16) as implicit
// GEMM on tcgen05 (sm_100a).  The [B, HW*HW, C] token layout is NHWC, so no permute is needed (the reference permutes to
// NCHW, model/loss.py:444).  Activations are bf16 plane tensors [P][B*HW*HW][C]; viewed through a 4-D tensor map
// {c, w, hb, plane} (hb = b*HW + h) a TMA box {64, HW, 1, 1} is one image row of 64 channels, and the zero padding comes
// for free: the w coordinate starts at dx-1 (out-of-bounds columns are zero-filled by TMA) and rows that fall outside
// their image are requested at an out-of-bounds hb coordinate.
//
//   forward / dgrad  (gemm_tn): tile = 128 / HW whole image rows (9 x 14 = 126, 5 x 24 = 120 pixels) x 384 channels;
//                     K walks 9 taps x 6 chunks.  Accumulator rows >= TILE_M are dead.
//                     out[m, co] = sum_{tap, ci} X[m + shift(tap), ci] * Wc[co, tap*C + ci]
//   wgrad            (gemm_nt): dW[tap][co][ci] += sum_m G[m, co] * X[m + shift(tap), ci], K block = conv_wgrad_rows(HW)
//                     whole image rows (8 x 14 = 112, 4 x 24 = 96 pixels).
#pragma once
#include "epilogues.cuh"
#include "gemm_nt.cuh"

namespace dkd {

// one image row of 64 bf16 channels in shared memory
template <int HW>
constexpr int conv_row_bytes() { return HW * 128; }

// image rows per forward / dgrad tile: as many whole rows as fit the 128-row UMMA tile
template <int HW>
constexpr int conv_tile_m() { return 128 / HW * HW; }

// image rows per wgrad K block: the most whole rows whose pixel count is a multiple of the UMMA K step (16) and at most
// 112 (the block that keeps three 5-box stages in shared memory).  Whole rows, so the padding test is per TMA box.
template <int HW>
constexpr int conv_wgrad_rows() {
  int best = 0;
  for (int r = 1; r * HW <= 112; ++r)
    if (r * HW % 16 == 0) best = r;
  return best;
}

struct ConvLoaderParams {
  CUtensorMap tmX;   // 4-D {C, HW, B*HW, P}, box {64, HW, 1, 1}
  CUtensorMap tmW;   // 3-D {9*C, C_out, P}, box {64, 192, 1}
  int total_hrows;   // B * HW
  int nterms;        // 1 | 3
};

template <class Cfg, int HW>
struct ConvRowsLoader {
  using Params = ConvLoaderParams;
  static constexpr int kRowBytes = conv_row_bytes<HW>();
  static constexpr int ROWS = Cfg::TILE_M / HW;  // image rows per tile (9 at HW = 14, 5 at HW = 24)
  static constexpr int KB = 54;                  // 9 taps x 6 channel chunks (C = 384)
  static constexpr uint32_t TX_BYTES = ROWS * kRowBytes + Cfg::B_BYTES;
  static_assert(Cfg::TILE_M == conv_tile_m<HW>() && Cfg::BN == 384, "conv tile");
  static __device__ __forceinline__ int num_k_iters(const Params& p) { return KB * p.nterms; }
  static __device__ __forceinline__ void prefetch(const Params& p) {
    sm100::tma_prefetch_desc(&p.tmX);
    sm100::tma_prefetch_desc(&p.tmW);
  }
  // The CTAs of a cluster work on different image rows but need the SAME 384 x 64 weight block at every K iteration —
  // CTA `crank` fetches rows [crank * 384/CL, ...) of it and multicasts them to the whole cluster (tmW's box has
  // 384 / CLUSTER rows).  Weight traffic L2 -> SM drops from 48 KB to 48/CL KB per K block and CTA.
  static constexpr int W_ROWS = 384 / Cfg::CLUSTER;
  static __device__ __forceinline__ void issue_cluster(const Params& p, int kit, int mt, int nt, uint8_t* sA, uint8_t* sB, uint64_t* bar,
                                                       int crank) {
    const int term = kit / KB, r = kit - term * KB;
    const int tap = r / 6, cb = r - tap * 6;
    const int dy = tap / 3, dx = tap - dy * 3;
    int pa, pb;
    term_planes(term, p.nterms, pa, pb);
#pragma unroll
    for (int rr = 0; rr < ROWS; ++rr) {
      const int hb = mt * ROWS + rr;
      const int sh = hb % HW + dy - 1;
      const bool ok = sh >= 0 && sh < HW && hb < p.total_hrows;
      sm100::tma_load_4d(sA + rr * kRowBytes, &p.tmX, bar, cb * 64, dx - 1, ok ? hb + dy - 1 : -4, pa);
    }
    sm100::tma_load_3d_mc(sB + (size_t)crank * W_ROWS * 128, &p.tmW, bar, tap * 384 + cb * 64, nt * Cfg::BN + crank * W_ROWS, pb,
                          (uint16_t)((1u << Cfg::CLUSTER) - 1u));
  }
};

// ---- epilogue of the generator / alignment GEMMs: fp32 accumulator row -> bf16 planes ---------------
enum ConvEpiMode : int {
  EPI_PLAIN = 0,     // out = v
  EPI_RELU = 1,      // out = relu(v + bias)
  EPI_MSE = 2,       // g = v + bias; masked rows: d = g - t, loss += d^2, out = gscale*d; other rows: out = 0
  EPI_DRELU = 3,     // out = act > 0 ? v : 0
  EPI_MASKFILL = 4   // out = mask ? mask_token : v + bias
};

struct ConvEpiParams {
  __nv_bfloat16* out;          // planes [P][M][N]
  const float* bias;           // [N] or null
  const float* mask;           // [M] 0/1 (flattened [B, n_tok]) or null
  const float* mask_token;     // [N]
  const void* t;               // teacher [B, Tt, N]
  const __nv_bfloat16* act;    // hi plane [M][N] of the ReLU output (EPI_DRELU)
  double* partials;
  int64_t M;
  int N, planes, n_tok, Tt, t_off, t_is_bf16;
  float gscale;
};

template <class Cfg, int MODE>
struct ConvEpi {
  using Params = ConvEpiParams;
  struct State { float acc; };
  static __device__ __forceinline__ void init(const Params&, State& st) { st.acc = 0.f; }

  static __device__ __forceinline__ void tile(const Params& p, State& st, int m0, int n0, int row_in_tile, uint32_t t_acc, int group = 0,
                                              int groups = 1) {
    const int64_t m = (int64_t)m0 + row_in_tile;
    const bool live = row_in_tile < Cfg::TILE_M && m < p.M;
    float mk = 0.f;
    int64_t trow = 0;
    if (live && (MODE == EPI_MSE || MODE == EPI_MASKFILL)) mk = __ldg(p.mask + m);
    if (live && MODE == EPI_MSE) {
      const int64_t b = m / p.n_tok;
      trow = b * p.Tt + p.t_off + (m - b * p.n_tok);
    }
#pragma unroll 1
    for (int c0 = group * 32; c0 < Cfg::BN; c0 += 32 * groups) {
      float v[32];
      sm100::tmem_ld32(t_acc + c0, v);
      float aux[32];
      if (live) {
        if (MODE == EPI_MSE && mk != 0.f) load_act32(p.t, trow * p.N + n0 + c0, p.t_is_bf16, aux);
        if (MODE == EPI_DRELU) load_act32(p.act, m * p.N + n0 + c0, 1, aux);
      }
      sm100::tmem_ld_wait();
      if (!live) continue;
      float bs[32];   // bias of this chunk, or the mask token for masked rows of the mask-fill epilogue
      if (MODE == EPI_MASKFILL && mk != 0.f) ldg_vec32(p.mask_token + n0 + c0, bs);
      else if (MODE == EPI_RELU || MODE == EPI_MSE || MODE == EPI_MASKFILL) ldg_vec32(p.bias ? p.bias + n0 + c0 : nullptr, bs);
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        float x = v[j];
        if (MODE == EPI_RELU) x = fmaxf(x + bs[j], 0.f);
        if (MODE == EPI_MASKFILL) x = mk != 0.f ? bs[j] : x + bs[j];
        if (MODE == EPI_DRELU) x = aux[j] > 0.f ? x : 0.f;
        if (MODE == EPI_MSE) {
          if (mk != 0.f) {
            const float d = x + bs[j] - aux[j];
            st.acc = fmaf(d, d, st.acc);
            x = p.gscale * d;
          } else {
            x = 0.f;
          }
        }
        v[j] = x;
      }
      store_planes32(p.out + m * p.N + n0 + c0, p.M * p.N, p.planes, v);
    }
  }

  static __device__ __forceinline__ void finish(const Params& p, State& st, int tid) {
    if (MODE == EPI_MSE) epilogue_block_partial<Cfg::EPI_WARPS>(st.acc, tid, p.partials);
  }
};

// ---- wgrad loader (gemm_nt): A = G planes [P][M][C] (3-D map, box {64, KROWS, 1}), B = shifted X rows ----
struct NtConvParams {
  CUtensorMap tmG;   // 3-D {C, M, P}, box {64, KROWS, 1}
  CUtensorMap tmX;   // 4-D {C, HW, B*HW, P}, box {64, HW, 1, 1}
  int splits, row_blocks_per_split, total_row_blocks, total_hrows;
};
template <class Cfg, int HW>
struct NtConvLoader {
  using Params = NtConvParams;
  using Item = NtItem;
  static constexpr int COMBOS_CLUSTER = 9 * 2;   // tap x ci half (192); the cluster's 3 CTAs are the co tiles (128)
  static constexpr int kRowBytes = conv_row_bytes<HW>();
  static constexpr int RB_ROWS = conv_wgrad_rows<HW>();   // image rows per K block (8 at HW = 14, 4 at HW = 24)
  static constexpr uint32_t TX_BYTES = Cfg::STAGE_BYTES;
  static_assert(Cfg::KROWS == RB_ROWS * HW && Cfg::NB_BOXES == 3 && !Cfg::ONES, "conv wgrad stage = RB_ROWS image rows x 192 channels");
  static_assert(Cfg::CLUSTER == 3, "a cluster = the 3 output-channel tiles");
  static __device__ __forceinline__ int num_items(const Params& p) { return COMBOS_CLUSTER * p.splits; }
  static __device__ __forceinline__ void prefetch(const Params& p) {
    sm100::tma_prefetch_desc(&p.tmG);
    sm100::tma_prefetch_desc(&p.tmX);
  }
  // A cluster's 3 CTAs are the 3 output-channel tiles of one (tap, ci half, row split): same shifted X rows for all
  // three, so CTA `crank` fetches channel box `crank` of every image row and multicasts it: per 16-row K step a CTA pulls
  // 4 KB (its G tile) + 2 KB from L2 instead of 4 + 6 KB.
  static __device__ __forceinline__ int num_items_cluster(const Params& p) { return COMBOS_CLUSTER * p.splits; }
  static __device__ __forceinline__ void decode_cluster(const Params& p, int item, int crank, Item& it) {
    const int combo = item % COMBOS_CLUSTER, split = item / COMBOS_CLUSTER;
    const int tap = combo >> 1, ci_half = combo & 1;
    it.split = split;
    it.rb0 = split * p.row_blocks_per_split;
    it.rb1 = min(it.rb0 + p.row_blocks_per_split, p.total_row_blocks);
    it.a_col0 = crank * 128;
    it.b_col0 = ci_half * 192;
    it.d_off = ((int64_t)tap * 384 + crank * 128) * 384 + ci_half * 192;
    it.dcol_off = -1;
    it.aux = tap;
  }
  static __device__ __forceinline__ void issue_cluster(const Params& p, const Item& it, int term, int nterms, int rb, uint8_t* a, uint8_t* b,
                                                       uint64_t* bar, int crank) {
    int pa, pb;
    term_planes(term, nterms, pa, pb);
    const int dy = it.aux / 3, dx = it.aux - dy * 3;
    sm100::tma_load_3d(a, &p.tmG, bar, it.a_col0, rb * Cfg::KROWS, pa);
    sm100::tma_load_3d(a + Cfg::BOX_BYTES, &p.tmG, bar, it.a_col0 + 64, rb * Cfg::KROWS, pa);
#pragma unroll
    for (int rr = 0; rr < RB_ROWS; ++rr) {
      const int hb = rb * RB_ROWS + rr;
      const int sh = hb % HW + dy - 1;
      const bool ok = sh >= 0 && sh < HW && hb < p.total_hrows;
      const int coord = ok ? hb + dy - 1 : -4;
      sm100::tma_load_4d_mc(b + (size_t)crank * Cfg::BOX_BYTES + rr * kRowBytes, &p.tmX, bar, it.b_col0 + crank * 64, dx - 1, coord, pb,
                            (uint16_t)0x7);
    }
  }
};

// host: 4-D activation map {C, HW, B*HW, P} over planes [P][B*HW*HW][C]
inline int make_image_tmap(CUtensorMap* out, const void* base, int64_t B, int HW, int C, int P, const char* what) {
  const uint64_t dims[4] = {(uint64_t)C, (uint64_t)HW, (uint64_t)(B * HW), (uint64_t)P};
  const uint64_t strides[3] = {(uint64_t)C * 2, (uint64_t)C * HW * 2, (uint64_t)B * HW * HW * C * 2};
  const uint32_t box[4] = {64, (uint32_t)HW, 1, 1};
  return make_tmap_bf16(out, base, 4, dims, strides, box, what);
}

}  // namespace dkd
