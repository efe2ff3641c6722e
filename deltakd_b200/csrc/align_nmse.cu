// Normalised hidden-state matching (the feature term of DiffKD):
//     a = s[:, s_off:] W^T + b ;  a_hat = a / |a|,  t_hat = t[:, t_off:] / |t|   (L2 norm over the channel axis, per token)
//     loss += scale * sum (a_hat - t_hat)^2          and the gradients of s, W, b.
// Reference: diffkd branch, model/loss.py:112-116 (alignment heads), :139-140 (per-token normalisation) and :149
// (`F.mse_loss(s_feat, t_feat)`, whose 1/numel and the noise-aware weight w_t.mean() the caller folds into `scale`
// and into the autograd rescale).
//
//   1-2. operand planes (S, W) as in align_mse.cu
//   3.   gemm_tn with a 128 x 384 tile (the whole channel axis of a row lives in ONE accumulator row), epilogue
//        pass A: |a|^2, |t|^2 from TMEM + teacher row; pass B: d = a_hat - t_hat, loss partial and
//        g_a = 2 scale (d - (d . a_hat) a_hat) / |a|  written as bf16 planes (the teacher row is re-read from L2)
//   4-5. g_s = g_a W, g_W = g_a^T s, g_b = g_a^T 1 (align_ops.cuh)
#include "align_ops.cuh"

namespace dkd {
namespace {

using NmseCfg = GemmCfg<384, 2, 3, 1>;   // N = 384 (two 192-wide MMAs), 3-stage ring of 64 KB, one TMEM accumulator

struct NormMseParams {
  const void* t;          // teacher [B, Tt, N]
  const float* bias;      // [N] or null
  __nv_bfloat16* G;       // planes [P][M][N]
  double* partials;       // [gridDim.x]
  int64_t M;
  int N, n_tok, Tt, t_off, planes, t_is_bf16;
  float gscale;           // 2 * scale
};

struct NormMseEpi {
  using Params = NormMseParams;
  struct State { float acc; };
  static __device__ __forceinline__ void init(const Params&, State& st) { st.acc = 0.f; }

  static __device__ __forceinline__ void tile(const Params& p, State& st, int m0, int, int row_in_tile, uint32_t t_acc) {
    const int64_t m = (int64_t)m0 + row_in_tile;
    const bool live = m < p.M;
    const int64_t b = live ? m / p.n_tok : 0;
    const int64_t toff = (b * p.Tt + p.t_off + (live ? m - b * p.n_tok : 0)) * p.N;
    // pass A: squared norms of the aligned row and of the teacher row
    float saa = 0.f, stt = 0.f;
#pragma unroll 1
    for (int c0 = 0; c0 < NmseCfg::BN; c0 += 32) {
      float v[32], tv[32], bs[32];
      sm100::tmem_ld32(t_acc + c0, v);
      if (live) load_act32(p.t, toff + c0, p.t_is_bf16, tv);
      ldg_vec32(p.bias ? p.bias + c0 : nullptr, bs);
      sm100::tmem_ld_wait();
      if (live) {
#pragma unroll
        for (int j = 0; j < 32; ++j) { const float a = v[j] + bs[j]; saa = fmaf(a, a, saa); stt = fmaf(tv[j], tv[j], stt); }
      }
    }
    const float ia = rsqrtf(saa), it = rsqrtf(stt);
    // pass B (1): d . a_hat needs the whole row again; fold it from sums: d.a_hat = 1 - cos, cos = (a.t) ia it.
    // It is cheaper and more accurate to accumulate (a_hat - t_hat) directly: two sweeps over TMEM (no extra HBM).
    float dot = 0.f;   // sum (a_hat - t_hat) * a_hat
#pragma unroll 1
    for (int c0 = 0; c0 < NmseCfg::BN; c0 += 32) {
      float v[32], tv[32], bs[32];
      sm100::tmem_ld32(t_acc + c0, v);
      if (live) load_act32(p.t, toff + c0, p.t_is_bf16, tv);
      ldg_vec32(p.bias ? p.bias + c0 : nullptr, bs);
      sm100::tmem_ld_wait();
      if (live) {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float ah = (v[j] + bs[j]) * ia, d = ah - tv[j] * it;
          st.acc = fmaf(d, d, st.acc);
          dot = fmaf(d, ah, dot);
        }
      }
    }
    // pass B (2): g_a = gscale * (d - dot * a_hat) * ia
    const float gs = p.gscale * ia;
#pragma unroll 1
    for (int c0 = 0; c0 < NmseCfg::BN; c0 += 32) {
      float v[32], tv[32], bs[32];
      sm100::tmem_ld32(t_acc + c0, v);
      if (live) load_act32(p.t, toff + c0, p.t_is_bf16, tv);
      ldg_vec32(p.bias ? p.bias + c0 : nullptr, bs);
      sm100::tmem_ld_wait();
      if (!live) continue;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const float ah = (v[j] + bs[j]) * ia, d = ah - tv[j] * it;
        v[j] = gs * (d - dot * ah);
      }
      store_planes32(p.G + m * p.N + c0, p.M * p.N, p.planes, v);
    }
  }
  static __device__ __forceinline__ void finish(const Params& p, State& st, int tid) { epilogue_block_partial(st.acc, tid, p.partials); }
};

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct Workspace {
  __nv_bfloat16 *S, *Wp, *Wt, *G, *ones;
  double* partials;
  float* wpart;   // deterministic mode: per-split weight-gradient slots (align_wgrad), appended last
  size_t bytes;
};
Workspace carve(void* base, int64_t M, int Ds, int Dt, int P, bool det) {
  Workspace w;
  size_t off = 0;
  auto take = [&](size_t n) { size_t o = off; off = align_up(off + n, 1024); return reinterpret_cast<char*>(base) + o; };
  w.S = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * M * Ds * 2));
  w.G = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * M * Dt * 2));
  w.Wp = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * Dt * Ds * 2));
  w.Wt = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * Dt * Ds * 2));
  w.ones = reinterpret_cast<__nv_bfloat16*>(take((size_t)2 * 64 * 64 * 2));
  w.partials = reinterpret_cast<double*>(take((size_t)kNumSMs * sizeof(double)));
  w.wpart = det ? reinterpret_cast<float*>(take(align_wgrad_part_bytes(M, Ds, Dt, P))) : nullptr;
  w.bytes = off;
  return w;
}

}  // namespace
}  // namespace dkd

extern "C" {

size_t dkd_align_nmse_workspace_bytes(int64_t B, int n_tok, int Ds, int Dt, int precision) {
  return dkd::carve(nullptr, B * n_tok, Ds, Dt, dkd::prec_planes(precision), dkd::prec_deterministic(precision)).bytes;
}

int dkd_align_nmse_fwdbwd(const void* s, const void* t, const float* W, const float* bias, int64_t B, int Ts, int s_off, int Tt,
                          int t_off, int n_tok, int Ds, int Dt, int dtype, int precision, float scale, void* g_s, float* g_W,
                          float* g_b, float* loss, void* workspace, size_t workspace_bytes, dkd_stream_t stream) {
  using namespace dkd;
  int rc = dkd_check_device();
  if (rc != DKD_OK) return rc;
  const char* fn = "dkd_align_nmse_fwdbwd";
  DKD_REQUIRE(dtype == DKD_F32 || dtype == DKD_BF16, DKD_E_DTYPE, "%s: dtype %d", fn, dtype);
  DKD_REQUIRE(prec_valid(precision), DKD_E_UNSUPPORTED, "%s: precision %d", fn, precision);
  DKD_REQUIRE(B > 0 && n_tok > 0 && s_off >= 0 && t_off >= 0 && Ts >= s_off + n_tok && Tt >= t_off + n_tok, DKD_E_SHAPE,
              "%s: bad token geometry", fn);
  DKD_REQUIRE(Ds == 192 && Dt == 384, DKD_E_SHAPE, "%s: built for widths 192 -> 384, got %d -> %d", fn, Ds, Dt);
  DKD_REQUIRE(s && t && W && loss && workspace, DKD_E_SHAPE, "%s: null pointer", fn);
  DKD_REQUIRE((((uintptr_t)workspace) & 1023) == 0, DKD_E_ALIGN, "%s: workspace must be 1024-byte aligned", fn);
  DKD_REQUIRE((((uintptr_t)s | (uintptr_t)t | (uintptr_t)g_s) & 31) == 0, DKD_E_ALIGN, "%s: s, t and g_s must be 32-byte aligned", fn);
  const int P = prec_planes(precision);
  const int64_t M = B * n_tok;
  DKD_REQUIRE(M < (1ll << 31) - 256, DKD_E_SHAPE, "%s: too many rows", fn);
  Workspace ws = carve(workspace, M, Ds, Dt, P, prec_deterministic(precision));
  DKD_REQUIRE(workspace_bytes >= ws.bytes, DKD_E_WORKSPACE, "%s: workspace %zu < %zu", fn, workspace_bytes, ws.bytes);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const bool want_grads = g_s != nullptr || g_W != nullptr || g_b != nullptr;

  rc = launch_tokens_to_planes(s, dtype, B, Ts, s_off, n_tok, Ds, P, nullptr, ws.S, st);
  if (rc != DKD_OK) return rc;
  rc = launch_weight_to_planes(W, Dt, Ds, P, ws.Wp, want_grads ? ws.Wt : nullptr, st);
  if (rc != DKD_OK) return rc;
  {
    using Cfg = NmseCfg;
    using L = PlaneLoader<Cfg, 192>;
    GemmParams<L, NormMseEpi> p;
    rc = make_plane_tmap(&p.ld.tmA, ws.S, P, M, Ds, Ds, M * Ds, Cfg::BM, "align_nmse S");
    if (rc != DKD_OK) return rc;
    rc = make_plane_tmap(&p.ld.tmB, ws.Wp, P, Dt, Ds, Ds, (int64_t)Dt * Ds, 192, "align_nmse W");
    if (rc != DKD_OK) return rc;
    p.ld.k_blocks = Ds / 64; p.ld.nterms = P == 2 ? 3 : 1;
    p.ep.t = t; p.ep.bias = bias; p.ep.G = ws.G; p.ep.partials = ws.partials; p.ep.M = M; p.ep.N = Dt; p.ep.n_tok = n_tok;
    p.ep.Tt = Tt; p.ep.t_off = t_off; p.ep.planes = P; p.ep.t_is_bf16 = dtype == DKD_BF16; p.ep.gscale = 2.f * scale;
    p.m_tiles = (int)((M + Cfg::BM - 1) / Cfg::BM); p.n_tiles = 1;
    const int grid = min(kNumSMs, p.m_tiles);
    auto kern = gemm_tn_kernel<Cfg, L, NormMseEpi>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
    kern<<<grid, Cfg::THREADS, Cfg::SMEM, st>>>(p);
    rc = check_launch("dkd_align_nmse_fwdbwd: forward GEMM");
    if (rc != DKD_OK) return rc;
    rc = launch_fold_partials(ws.partials, grid, scale, loss, st);
    if (rc != DKD_OK) return rc;
  }
  if (!want_grads) return DKD_OK;
  if (g_s) {
    rc = align_dgrad(ws.G, ws.Wt, g_s, M, n_tok, Ts, s_off, Ds, Dt, P, dtype == DKD_BF16, 1.f, st, "dkd_align_nmse_fwdbwd: dgrad GEMM");
    if (rc != DKD_OK) return rc;
  }
  if (g_W || g_b) {
    DKD_REQUIRE(g_W != nullptr, DKD_E_UNSUPPORTED, "%s: g_b without g_W is not supported", fn);
    rc = align_wgrad(ws.G, ws.S, ws.ones, g_W, g_b, M, Ds, Dt, P, 1.f, st, "dkd_align_nmse_fwdbwd: wgrad GEMM", 0, ws.wpart);
    if (rc != DKD_OK) return rc;
  }
  return DKD_OK;
}

}  // extern "C"
