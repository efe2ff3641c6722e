// Masked generative distillation core, forward + backward:
//     x   = align(s[:, s_off:])                       Linear(Ds -> Dt)
//     x_m = where(mask, mask_token, x)
//     h   = relu(conv3x3(x_m; W1, b1)) ; g = conv3x3(h; W2, b2)      on the HW x HW token grid, pad 1
//     loss += scale * sum( mask * (g - t[:, t_off:])^2 )
// Reference: mgd_loss (model/loss.py:422-451), saliency_mgd_loss (:335-360), curkd_loss late phase (:394-420)
// and the ViTKD generation term (:291-310) — they differ only in how `mask` is chosen and in `scale`.
// The reference's cat/gather with ids_restore equals where(mask, mask_token, x) (SURVEY.md A.4).
// The grid side HW is 14 (196 patch tokens, 224-px inputs) or 24 (576 tokens, 384-px inputs); it only changes the
// convolutions' tiling (conv.cuh), so each generator convolution is instantiated for both and picked from n_tok.
//
// Every contraction runs on tcgen05 (gemm_tn / gemm_nt skeletons); activations travel between the
// GEMMs as bf16 hi/lo planes.  Launch sequence (one stream, no host sync):
//   prep: S' planes (masked rows dropped), weight planes for align / conv1 / conv2 (forward + flipped)
//   fwd : align GEMM (mask-fill epilogue) -> X ; conv1 (ReLU epilogue) -> H ; conv2 (masked-MSE epilogue) -> G, loss
//   bwd : conv2 wgrad (G^T (*) H) + colsum(G) ; conv2 dgrad (dReLU epilogue) -> DH ; conv1 wgrad + colsum(DH) ;
//         conv1 dgrad -> dXm (into G) ; masked colsum(dXm) -> g_b_align, g_mask_token ;
//         g_s = (1-mask) * dXm W_align (row-masked store) ; g_W_align = dXm^T S'
// Deterministic mode (DKD_PREC_DETERMINISTIC): the two conv wgrads, the align wgrad and the three column sums write
// per-split (per-CTA) fp32 partials with plain stores into one region appended to the workspace (they run one after
// another on the stream, so they share it), and each is folded in a fixed order in fp64: conv_wgrad_transpose_kernel
// for the convolutions, fold_splits_kernel for the align wgrad, fold_rows_kernel for the column sums.  No float atomic
// is left, and every split count is a function of B alone.
#include "conv.cuh"
#include "planes.cuh"

namespace dkd {
namespace {

using AlignCfg = GemmCfg<192, 1, 4, 2, 128, 1, 8>;   // X tile 128 x 192 (K = 192), 8 epilogue warps
// 128 / HW image rows x 384 channels, K = 9 x 384, 8 epilogue warps; clusters of 2 CTAs with the weight block multicast
template <int HW>
using ConvCfg = GemmCfg<384, 2, 3, 1, conv_tile_m<HW>(), 1, 8, 2>;
using DalignCfg = GemmCfg<192, 1, 4, 2, 128, 1, 8>;  // g_s tile 128 x 192 (K = 384)
// dW tile 128(co) x 192(ci), conv_wgrad_rows<HW>() image rows per stage; 3-CTA clusters with the shifted-X block multicast
template <int HW>
using ConvWgradCfg = GemmNtCfg<3, false, 192, 0, 3, conv_wgrad_rows<HW>() * HW, false, 1, 3>;
using AlignWgradCfg = GemmNtCfg<3, false, 192, 0, 4>;      // g_W_align tile 128 x 192

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct Workspace {
  __nv_bfloat16 *S, *X, *H, *G, *DH, *Wa, *Wat, *W1c, *W1d, *W2c, *W2d;
  float *dW1t, *dW2t;
  double* partials;
  float* wpart;   // deterministic mode only: the weight-gradient / column-sum partials, appended last
  size_t bytes;
};

// grid side of a supported patch-token count, 0 for any other
int grid_side(int n_tok) { return n_tok == 14 * 14 ? 14 : n_tok == 24 * 24 ? 24 : 0; }

template <int HW>
int conv_wgrad_splits(int64_t B, int slots);
size_t wpart_bytes(int64_t B, int n_tok, int Ds, int Dt) {
  const int64_t M = B * n_tok;
  const int conv_splits = grid_side(n_tok) == 24 ? conv_wgrad_splits<24>(B, kNumSMs / ConvWgradCfg<24>::CLUSTER)
                                                  : conv_wgrad_splits<14>(B, kNumSMs / ConvWgradCfg<14>::CLUSTER);
  const size_t conv = (size_t)conv_splits * 9 * Dt * Dt * sizeof(float);
  int splits, per;   // as the align wgrad launch below
  nt_make_splits((int)((M + AlignWgradCfg::KROWS - 1) / AlignWgradCfg::KROWS), kNumSMs / (Dt / 128), &splits, &per);
  const size_t align = (size_t)splits * nt_slot_floats((int64_t)Dt * Ds) * sizeof(float), colsum = colsum_planes_part_bytes(Dt);
  const size_t m = conv > align ? conv : align;
  return m > colsum ? m : colsum;
}
Workspace carve(void* base, int64_t B, int n_tok, int Ds, int Dt, int P, bool det) {
  Workspace w;
  const int64_t M = B * n_tok;
  size_t off = 0;
  auto take = [&](size_t n) { size_t o = off; off = align_up(off + n, 1024); return reinterpret_cast<char*>(base) + o; };
  const size_t act = (size_t)P * M * Dt * 2, cw = (size_t)P * Dt * Dt * 9 * 2;
  w.S = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * M * Ds * 2));
  w.X = reinterpret_cast<__nv_bfloat16*>(take(act));
  w.H = reinterpret_cast<__nv_bfloat16*>(take(act));
  w.G = reinterpret_cast<__nv_bfloat16*>(take(act));
  w.DH = reinterpret_cast<__nv_bfloat16*>(take(act));
  w.Wa = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * Dt * Ds * 2));
  w.Wat = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * Dt * Ds * 2));
  w.W1c = reinterpret_cast<__nv_bfloat16*>(take(cw));
  w.W1d = reinterpret_cast<__nv_bfloat16*>(take(cw));
  w.W2c = reinterpret_cast<__nv_bfloat16*>(take(cw));
  w.W2d = reinterpret_cast<__nv_bfloat16*>(take(cw));
  w.dW1t = reinterpret_cast<float*>(take((size_t)9 * Dt * Dt * 4));
  w.dW2t = reinterpret_cast<float*>(take((size_t)9 * Dt * Dt * 4));
  w.partials = reinterpret_cast<double*>(take((size_t)kNumSMs * sizeof(double)));
  w.wpart = det ? reinterpret_cast<float*>(take(wpart_bytes(B, n_tok, Ds, Dt))) : nullptr;
  w.bytes = off;
  return w;
}

template <class Cfg, class L, class E>
int launch_tn(GemmParams<L, E>& p, cudaStream_t st, const char* what, int* grid_out = nullptr) {
  const int grid = gemm_tn_grid<Cfg, L, E>(p.m_tiles * p.n_tiles);
  launch_gemm_tn<Cfg, L, E>(p, grid, st);
  if (grid_out) *grid_out = grid;
  return check_launch(what);
}

// one generator convolution (forward or dgrad) on the HW x HW grid: out planes = epilogue(conv3x3(in planes; w planes))
template <int HW, int MODE>
int run_conv_grid(const __nv_bfloat16* in, const __nv_bfloat16* wplanes, ConvEpiParams ep, int64_t B, int C, int P, cudaStream_t st,
                  const char* what, int* grid_out) {
  using Cfg = ConvCfg<HW>;
  using L = ConvRowsLoader<Cfg, HW>;
  using E = ConvEpi<Cfg, MODE>;
  GemmParams<L, E> p;
  int rc = make_image_tmap(&p.ld.tmX, in, B, HW, C, P, what);
  if (rc != DKD_OK) return rc;
  rc = make_plane_tmap(&p.ld.tmW, wplanes, P, C, 9 * C, 9 * C, (int64_t)C * 9 * C, L::W_ROWS, what);
  if (rc != DKD_OK) return rc;
  p.ld.total_hrows = (int)(B * HW);
  p.ld.nterms = P == 2 ? 3 : 1;
  p.ep = ep;
  p.m_tiles = (p.ld.total_hrows + L::ROWS - 1) / L::ROWS;
  p.n_tiles = 1;
  return launch_tn<Cfg, L, E>(p, st, what, grid_out);
}
template <int MODE>
int run_conv(int hw, const __nv_bfloat16* in, const __nv_bfloat16* wplanes, const ConvEpiParams& ep, int64_t B, int C, int P, cudaStream_t st,
             const char* what, int* grid_out = nullptr) {
  return hw == 24 ? run_conv_grid<24, MODE>(in, wplanes, ep, B, C, P, st, what, grid_out)
                  : run_conv_grid<14, MODE>(in, wplanes, ep, B, C, P, st, what, grid_out);
}

// Items = (tap, ci half) x row splits over the clusters.  The split count is chosen so that the items fill whole waves of
// `slots` clusters: the former fixed 6 splits gave 324 items on 148 CTAs = 2.19 waves, i.e. a makespan of 3 waves for 2.19
// waves of work (27 % idle).
template <int HW>
int conv_wgrad_splits(int64_t B, int slots) {
  constexpr int rb = conv_wgrad_rows<HW>();
  return nt_best_splits(NtConvLoader<ConvWgradCfg<HW>, HW>::COMBOS_CLUSTER, slots, (int)((B * HW + rb - 1) / rb), 4, 16);
}

// dW[co][ci][tap] (PyTorch layout) = sum_m G[m, co] * X[m + shift(tap), ci], through dWt[split][tap][co][ci].  `part` null:
// the splits add into dWt with float atomics; else (deterministic mode) the split count depends on B alone and each split
// stores its own slot of `part`, which the transpose kernel folds in split order
template <int HW>
int run_conv_wgrad_grid(const __nv_bfloat16* G, const __nv_bfloat16* X, float* dWt, float* part, float* dW, int64_t B, int64_t M, int C,
                        int P, cudaStream_t st, const char* what) {
  using Cfg = ConvWgradCfg<HW>;
  using L = NtConvLoader<Cfg, HW>;
  GemmNtParamsT<Cfg, L> p;
  int rc = make_plane_tmap(&p.ld.tmG, G, P, M, C, C, M * C, Cfg::KROWS, what);
  if (rc != DKD_OK) return rc;
  rc = make_image_tmap(&p.ld.tmX, X, B, HW, C, P, what);
  if (rc != DKD_OK) return rc;
  p.ld.total_hrows = (int)(B * HW);
  p.ld.total_row_blocks = (p.ld.total_hrows + L::RB_ROWS - 1) / L::RB_ROWS;
  static const int resident = [] {
    auto kern = gemm_nt_kernel<Cfg, L>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
    return max_resident_clusters(kern, Cfg::CLUSTER, Cfg::THREADS, Cfg::SMEM);
  }();
  const int sp = conv_wgrad_splits<HW>(B, part ? kNumSMs / Cfg::CLUSTER : resident);
  nt_make_splits(p.ld.total_row_blocks, sp, &p.ld.splits, &p.ld.row_blocks_per_split);
  p.ep.ldd = C; p.ep.alpha = 1.f; p.ep.Dcol = nullptr;
  p.nterms = P == 2 ? 3 : 1;
  if (part) {
    p.ep.D = part; p.ep.store = 1; p.ep.split_stride = (int64_t)9 * C * C;   // C % 128 == 0: whole 128-byte slots
  } else {
    p.ep.D = dWt;
    cudaMemsetAsync(dWt, 0, (size_t)9 * C * C * sizeof(float), st);
  }
  // each item owns its slot in deterministic mode, so the grid (resident clusters) cannot change a bit
  int grid = min(resident, L::COMBOS_CLUSTER * p.ld.splits) * Cfg::CLUSTER;
  launch_gemm_nt<Cfg, L>(p, grid, st);
  rc = check_launch(what);
  if (rc != DKD_OK) return rc;
  return launch_conv_wgrad_transpose(part ? part : dWt, C, part ? p.ld.splits : 1, dW, st);
}
int run_conv_wgrad(int hw, const __nv_bfloat16* G, const __nv_bfloat16* X, float* dWt, float* part, float* dW, int64_t B, int64_t M, int C,
                   int P, cudaStream_t st, const char* what) {
  return hw == 24 ? run_conv_wgrad_grid<24>(G, X, dWt, part, dW, B, M, C, P, st, what)
                  : run_conv_wgrad_grid<14>(G, X, dWt, part, dW, B, M, C, P, st, what);
}

}  // namespace
}  // namespace dkd

extern "C" {

size_t dkd_masked_generation_workspace_bytes(int64_t B, int n_tok, int Ds, int Dt, int precision) {
  return dkd::carve(nullptr, B, n_tok, Ds, Dt, dkd::prec_planes(precision), dkd::prec_deterministic(precision)).bytes;
}

size_t dkd_masked_generation_hidden_offset(int64_t B, int n_tok, int Ds, int Dt, int precision) {
  dkd::Workspace w = dkd::carve(nullptr, B, n_tok, Ds, Dt, dkd::prec_planes(precision), dkd::prec_deterministic(precision));
  return (size_t)(reinterpret_cast<char*>(w.H) - static_cast<char*>(nullptr));
}

int dkd_masked_generation_fwdbwd(const void* s, const void* t, const float* mask, const float* W_align, const float* b_align,
                                 const float* mask_token, const float* conv1_w, const float* conv1_b, const float* conv2_w,
                                 const float* conv2_b, int64_t B, int Ts, int s_off, int Tt, int t_off, int Ds, int Dt, int dtype,
                                 int precision, float scale, void* g_s, float* g_W_align, float* g_b_align, float* g_mask_token,
                                 float* g_conv1_w, float* g_conv1_b, float* g_conv2_w, float* g_conv2_b, float* loss,
                                 void* workspace, size_t workspace_bytes, dkd_stream_t stream) {
  using namespace dkd;
  int rc = dkd_check_device();
  if (rc != DKD_OK) return rc;
  const char* fn = "dkd_masked_generation_fwdbwd";
  DKD_REQUIRE(dtype == DKD_F32 || dtype == DKD_BF16, DKD_E_DTYPE, "%s: dtype %d", fn, dtype);
  DKD_REQUIRE(prec_valid(precision), DKD_E_UNSUPPORTED, "%s: precision %d", fn, precision);
  const int n_tok = Ts - s_off, hw = grid_side(n_tok);
  DKD_REQUIRE(B > 0 && s_off >= 0 && t_off >= 0 && hw != 0 && Tt == t_off + n_tok, DKD_E_SHAPE,
              "%s: expects 196 (14x14 grid) or 576 (24x24 grid) patch tokens after the special tokens in both student and teacher, "
              "got %d and %d", fn, n_tok, Tt - t_off);
  DKD_REQUIRE(Ds == 192 && Dt == 384, DKD_E_SHAPE, "%s: built for widths 192 -> 384, got %d -> %d", fn, Ds, Dt);
  DKD_REQUIRE(s && t && mask && W_align && mask_token && conv1_w && conv1_b && conv2_w && conv2_b && loss && workspace, DKD_E_SHAPE,
              "%s: null pointer", fn);
  DKD_REQUIRE((((uintptr_t)workspace) & 1023) == 0, DKD_E_ALIGN, "%s: workspace must be 1024-byte aligned", fn);
  DKD_REQUIRE((((uintptr_t)g_s) & 31) == 0, DKD_E_ALIGN, "%s: g_s must be 32-byte aligned (256-bit stores)", fn);
  const int P = prec_planes(precision);
  const int64_t M = B * n_tok;
  DKD_REQUIRE(M < (1ll << 31) - 256, DKD_E_SHAPE, "%s: too many rows", fn);
  Workspace ws = carve(workspace, B, n_tok, Ds, Dt, P, prec_deterministic(precision));
  DKD_REQUIRE(workspace_bytes >= ws.bytes, DKD_E_WORKSPACE, "%s: workspace %zu < %zu", fn, workspace_bytes, ws.bytes);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const bool want_grads = g_s || g_W_align || g_b_align || g_mask_token || g_conv1_w || g_conv1_b || g_conv2_w || g_conv2_b;
  const int nterms = P == 2 ? 3 : 1;

  // ---- operand planes
  rc = launch_tokens_to_planes(s, dtype, B, Ts, s_off, n_tok, Ds, P, mask, ws.S, st);
  if (rc != DKD_OK) return rc;
  rc = launch_weight_to_planes(W_align, Dt, Ds, P, ws.Wa, want_grads ? ws.Wat : nullptr, st);
  if (rc != DKD_OK) return rc;
  rc = launch_conv_weight_to_planes(conv1_w, Dt, P, ws.W1c, ws.W1d, st);
  if (rc != DKD_OK) return rc;
  rc = launch_conv_weight_to_planes(conv2_w, Dt, P, ws.W2c, ws.W2d, st);
  if (rc != DKD_OK) return rc;

  ConvEpiParams ep{};
  ep.M = M; ep.N = Dt; ep.planes = P; ep.n_tok = n_tok; ep.Tt = Tt; ep.t_off = t_off; ep.t_is_bf16 = dtype == DKD_BF16;
  ep.mask = mask; ep.mask_token = mask_token; ep.t = t; ep.partials = ws.partials; ep.gscale = 2.f * scale;

  // ---- x_m = where(mask, mask_token, S' Wa^T + b)
  {
    using Cfg = AlignCfg;
    using L = PlaneLoader<Cfg>;
    using E = ConvEpi<Cfg, EPI_MASKFILL>;
    GemmParams<L, E> p;
    rc = make_plane_tmap(&p.ld.tmA, ws.S, P, M, Ds, Ds, M * Ds, Cfg::BM, "mgd S");
    if (rc != DKD_OK) return rc;
    rc = make_plane_tmap(&p.ld.tmB, ws.Wa, P, Dt, Ds, Ds, (int64_t)Dt * Ds, Cfg::BN, "mgd W_align");
    if (rc != DKD_OK) return rc;
    p.ld.k_blocks = Ds / 64; p.ld.nterms = nterms;
    p.ep = ep; p.ep.out = ws.X; p.ep.bias = b_align;
    p.m_tiles = (int)((M + Cfg::BM - 1) / Cfg::BM); p.n_tiles = Dt / Cfg::BN;
    rc = launch_tn<Cfg, L, E>(p, st, "mgd: align GEMM");
    if (rc != DKD_OK) return rc;
  }
  // ---- h = relu(conv1(x_m)), g = conv2(h), masked MSE
  {
    ConvEpiParams e1 = ep; e1.out = ws.H; e1.bias = conv1_b;
    rc = run_conv<EPI_RELU>(hw, ws.X, ws.W1c, e1, B, Dt, P, st, "mgd: conv1");
    if (rc != DKD_OK) return rc;
    ConvEpiParams e2 = ep; e2.out = ws.G; e2.bias = conv2_b;
    int grid = 0;
    rc = run_conv<EPI_MSE>(hw, ws.H, ws.W2c, e2, B, Dt, P, st, "mgd: conv2", &grid);
    if (rc != DKD_OK) return rc;
    rc = launch_fold_partials(ws.partials, grid, scale, loss, st);
    if (rc != DKD_OK) return rc;
  }
  if (!want_grads) return DKD_OK;

  // ---- conv2 backward
  if (g_conv2_w) {
    rc = run_conv_wgrad(hw, ws.G, ws.H, ws.dW2t, ws.wpart, g_conv2_w, B, M, Dt, P, st, "mgd: conv2 wgrad");
    if (rc != DKD_OK) return rc;
  }
  if (g_conv2_b) {
    rc = launch_colsum_planes(ws.G, M, Dt, P, nullptr, g_conv2_b, nullptr, st, ws.wpart);
    if (rc != DKD_OK) return rc;
  }
  {
    ConvEpiParams e = ep; e.out = ws.DH; e.act = ws.H;
    rc = run_conv<EPI_DRELU>(hw, ws.G, ws.W2d, e, B, Dt, P, st, "mgd: conv2 dgrad");
    if (rc != DKD_OK) return rc;
  }
  // ---- conv1 backward
  if (g_conv1_w) {
    rc = run_conv_wgrad(hw, ws.DH, ws.X, ws.dW1t, ws.wpart, g_conv1_w, B, M, Dt, P, st, "mgd: conv1 wgrad");
    if (rc != DKD_OK) return rc;
  }
  if (g_conv1_b) {
    rc = launch_colsum_planes(ws.DH, M, Dt, P, nullptr, g_conv1_b, nullptr, st, ws.wpart);
    if (rc != DKD_OK) return rc;
  }
  if (!(g_s || g_W_align || g_b_align || g_mask_token)) return DKD_OK;
  {
    ConvEpiParams e = ep; e.out = ws.G;  // dXm overwrites G (no longer needed)
    rc = run_conv<EPI_PLAIN>(hw, ws.DH, ws.W1d, e, B, Dt, P, st, "mgd: conv1 dgrad");
    if (rc != DKD_OK) return rc;
  }
  // ---- mask-token / alignment backward: masked rows feed mask_token, kept rows feed the Linear
  if (g_b_align || g_mask_token) {
    rc = launch_colsum_planes(ws.G, M, Dt, P, mask, g_b_align, g_mask_token, st, ws.wpart);
    if (rc != DKD_OK) return rc;
  }
  if (g_s) {
    using Cfg = DalignCfg;
    using L = PlaneLoader<Cfg>;
    using E = StoreRowsEpi<Cfg>;
    GemmParams<L, E> p;
    rc = make_plane_tmap(&p.ld.tmA, ws.G, P, M, Dt, Dt, M * Dt, Cfg::BM, "mgd dXm");
    if (rc != DKD_OK) return rc;
    rc = make_plane_tmap(&p.ld.tmB, ws.Wat, P, Ds, Dt, Dt, (int64_t)Dt * Ds, Cfg::BN, "mgd W_align^T");
    if (rc != DKD_OK) return rc;
    p.ld.k_blocks = Dt / 64; p.ld.nterms = nterms;
    p.ep.out = g_s; p.ep.drop_mask = mask; p.ep.bias = nullptr; p.ep.alpha = 1.f; p.ep.M = M; p.ep.N_total = Ds; p.ep.n_tok = n_tok; p.ep.T_out = Ts; p.ep.off = s_off;
    p.ep.out_is_bf16 = dtype == DKD_BF16;
    p.m_tiles = (int)((M + Cfg::BM - 1) / Cfg::BM); p.n_tiles = Ds / Cfg::BN;
    rc = launch_tn<Cfg, L, E>(p, st, "mgd: align dgrad");
    if (rc != DKD_OK) return rc;
  }
  if (g_W_align) {
    using Cfg = AlignWgradCfg;
    using L = NtPlainLoader<Cfg>;
    GemmNtParamsT<Cfg, L> p;
    rc = make_plane_tmap(&p.ld.tmA, ws.G, P, M, Dt, Dt, M * Dt, Cfg::KROWS, "mgd dXm^T");
    if (rc != DKD_OK) return rc;
    rc = make_plane_tmap(&p.ld.tmB, ws.S, P, M, Ds, Ds, M * Ds, Cfg::KROWS, "mgd S' (wgrad)");
    if (rc != DKD_OK) return rc;
    p.ld.tmOnes = p.ld.tmB;
    if (ws.wpart) {   // deterministic: slot per split, folded below
      p.ep.D = ws.wpart; p.ep.store = 1; p.ep.split_stride = nt_slot_floats((int64_t)Dt * Ds);
    } else {
      cudaMemsetAsync(g_W_align, 0, (size_t)Dt * Ds * sizeof(float), st);
      p.ep.D = g_W_align;
    }
    p.ep.Dcol = nullptr; p.ep.ldd = Ds; p.ep.alpha = 1.f;
    p.ld.ldd = Ds; p.ld.na_tiles = Dt / 128; p.ld.b_col0 = 0;
    p.ld.total_row_blocks = (int)((M + Cfg::KROWS - 1) / Cfg::KROWS);
    nt_make_splits(p.ld.total_row_blocks, kNumSMs / p.ld.na_tiles, &p.ld.splits, &p.ld.row_blocks_per_split);
    p.nterms = nterms;
    const int grid = min(kNumSMs, p.ld.na_tiles * p.ld.splits);
    auto kern = gemm_nt_kernel<Cfg, L>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
    kern<<<grid, Cfg::THREADS, Cfg::SMEM, st>>>(p);
    rc = check_launch("mgd: align wgrad");
    if (rc != DKD_OK) return rc;
    if (ws.wpart) {
      rc = launch_fold_splits(ws.wpart, p.ld.splits, p.ep.split_stride, (int64_t)Dt * Ds, g_W_align, 0, nullptr, 1.f, st);
      if (rc != DKD_OK) return rc;
    }
  }
  return DKD_OK;
}

}  // extern "C"
