// Layer-wise hidden-state matching: loss += scale * || s[:,off:] W^T + b - t[:,off:] ||^2 with all gradients.
// Reference: curkd_loss early / mid (model/loss.py:376-393) and the ViTKD mimicking term (loss.py:277-289)
// — per layer `mse_loss(Linear(192->384)(student[:,1:]), teacher[:,2:], reduction='sum')` and its autograd
// backward (grad of the student feature, of the Linear weight and of its bias).
//
// Launch sequence per layer (all on `stream`, no host sync):
//   1. tokens_to_planes   s[B,Ts,Ds] (patch tokens only) -> bf16 planes S[P][M][Ds]      (P = 1 bf16 | 2 bf16x3)
//   2. weight_to_planes   W[Dt,Ds] -> Wp[P][Dt][Ds]   (step 3 reads it both K-major and MN-major: no transpose)
//   3. align_fused_fwd_dgrad (one persistent tcgen05 kernel, align_fused.cuh):
//        Y = S W^T ; d = Y + b - t ; loss partial ; G = 2*scale*d as bf16 planes G[P][M][Dt] (teacher read in place) ;
//        g_s[:,off:,:] = G W    (rows scattered into [B,Ts,Ds], CLS rows zeroed)
//   4. fold_partials      : loss += sum of the per-CTA partials, fixed order (deterministic)
//   5. gemm_nt (split-K, MN-major, 3-CTA clusters) : g_W += G^T S, g_b += G^T 1 (ones-column trick)
#include "align_fused.cuh"
#include "align_ops.cuh"

namespace dkd {
namespace {

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct Workspace {
  __nv_bfloat16 *S, *Wp, *G, *ones;
  double* partials;
  size_t bytes;
};
Workspace carve(void* base, int64_t M, int Ds, int Dt, int P) {
  Workspace w;
  size_t off = 0;
  auto take = [&](size_t n) { size_t o = off; off = align_up(off + n, 1024); return reinterpret_cast<char*>(base) + o; };
  w.S = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * M * Ds * 2));
  w.G = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * M * Dt * 2));
  w.Wp = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * Dt * Ds * 2));
  w.ones = reinterpret_cast<__nv_bfloat16*>(take((size_t)2 * 64 * 64 * 2));
  w.partials = reinterpret_cast<double*>(take((size_t)kNumSMs * sizeof(double)));
  w.bytes = off;
  return w;
}

}  // namespace
}  // namespace dkd

extern "C" {

size_t dkd_align_mse_workspace_bytes(int64_t B, int n_tok, int Ds, int Dt, int precision) {
  return dkd::carve(nullptr, B * n_tok, Ds, Dt, precision == DKD_PREC_BF16X3 ? 2 : 1).bytes;
}

int dkd_align_mse_fwdbwd(const void* s, const void* t, const float* W, const float* bias, int64_t B, int Ts, int s_off,
                         int Tt, int t_off, int n_tok, int Ds, int Dt, int dtype, int precision, float scale, void* g_s,
                         float* g_W, float* g_b, float* loss, void* workspace, size_t workspace_bytes, dkd_stream_t stream) {
  using namespace dkd;
  int rc = dkd_check_device();
  if (rc != DKD_OK) return rc;
  DKD_REQUIRE(dtype == DKD_F32 || dtype == DKD_BF16, DKD_E_DTYPE, "dkd_align_mse_fwdbwd: dtype %d", dtype);
  DKD_REQUIRE(precision == DKD_PREC_BF16 || precision == DKD_PREC_BF16X3, DKD_E_UNSUPPORTED, "dkd_align_mse_fwdbwd: precision %d", precision);
  DKD_REQUIRE(B > 0 && n_tok > 0 && s_off >= 0 && t_off >= 0 && Ts >= s_off + n_tok && Tt >= t_off + n_tok, DKD_E_SHAPE,
              "dkd_align_mse_fwdbwd: bad token geometry");
  DKD_REQUIRE(Ds == 192 && Dt == 384, DKD_E_SHAPE, "dkd_align_mse_fwdbwd: built for DeiT-Tiny -> DeiT-Small widths (192 -> 384), got %d -> %d", Ds, Dt);
  DKD_REQUIRE(s && t && W && loss && workspace, DKD_E_SHAPE, "dkd_align_mse_fwdbwd: null pointer");
  DKD_REQUIRE((((uintptr_t)workspace) & 1023) == 0, DKD_E_ALIGN, "dkd_align_mse_fwdbwd: workspace must be 1024-byte aligned");
  DKD_REQUIRE((((uintptr_t)s | (uintptr_t)t | (uintptr_t)g_s) & 31) == 0, DKD_E_ALIGN, "%s: s, t and g_s must be 32-byte aligned (256-bit accesses)", "dkd_align_mse_fwdbwd");
  const int P = precision == DKD_PREC_BF16X3 ? 2 : 1;
  const int64_t M = B * n_tok;
  DKD_REQUIRE(M < (1ll << 31) - 256, DKD_E_SHAPE, "dkd_align_mse_fwdbwd: too many rows");
  Workspace ws = carve(workspace, M, Ds, Dt, P);
  DKD_REQUIRE(workspace_bytes >= ws.bytes, DKD_E_WORKSPACE, "dkd_align_mse_fwdbwd: workspace %zu < %zu", workspace_bytes, ws.bytes);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);

  // 1-2. operand planes
  rc = launch_tokens_to_planes(s, dtype, B, Ts, s_off, n_tok, Ds, P, nullptr, ws.S, st);
  if (rc != DKD_OK) return rc;
  rc = launch_weight_to_planes(W, Dt, Ds, P, ws.Wp, nullptr, st);
  if (rc != DKD_OK) return rc;

  // 3. forward + residual + dgrad; the G planes it leaves feed step 5
  int grid = 0;
  const char* what = "dkd_align_mse_fwdbwd: fused forward + dgrad";
  rc = P == 2 ? align_fused_fwd_dgrad_t<2>(ws.S, ws.Wp, bias, t, dtype == DKD_BF16, Tt, t_off, n_tok, ws.G, ws.partials, 2.f * scale,
                                           g_s, Ts, s_off, dtype == DKD_BF16, 1.f, M, st, &grid, what)
              : align_fused_fwd_dgrad_t<1>(ws.S, ws.Wp, bias, t, dtype == DKD_BF16, Tt, t_off, n_tok, ws.G, ws.partials, 2.f * scale,
                                           g_s, Ts, s_off, dtype == DKD_BF16, 1.f, M, st, &grid, what);
  if (rc != DKD_OK) return rc;
  // 4. loss
  rc = launch_fold_partials(ws.partials, grid, scale, loss, st);
  if (rc != DKD_OK) return rc;
  // 5. g_W = G^T S, g_b = G^T 1
  if (g_W || g_b) {
    DKD_REQUIRE(g_W != nullptr, DKD_E_UNSUPPORTED, "dkd_align_mse_fwdbwd: g_b without g_W is not supported");
    rc = align_wgrad(ws.G, ws.S, ws.ones, g_W, g_b, M, Ds, Dt, P, 1.f, st, "dkd_align_mse_fwdbwd: wgrad GEMM");
    if (rc != DKD_OK) return rc;
  }
  return DKD_OK;
}

}  // extern "C"
