// The three tcgen05 GEMMs around a Linear(Ds -> Dt) alignment head, shared by the losses that need the aligned
// activations themselves (WassKD): forward rows, and the backward from a gradient-plane tensor G[P][M][Dt].
//   align_forward_rows : A[M, Dt] fp32 = S W^T + bias                 (gemm_tn, StoreRows epilogue)
//   align_dgrad        : g_s[:, off:, :] = alpha * G W                (gemm_tn, rows scattered, special tokens zeroed)
//   align_wgrad        : g_W = alpha * G^T S, g_b = alpha * G^T 1     (gemm_nt split-K in 3-CTA clusters, ones-column trick)
#pragma once
#include "epilogues.cuh"
#include "gemm_nt.cuh"
#include "planes.cuh"

namespace dkd {

using AlignCfg1 = GemmCfg<192, 1, 4, 2, 128, 1, 8>;   // one plane per stage (bf16 operands), 4-stage ring, 8 epilogue warps
using AlignCfg2 = GemmCfg<192, 1, 2, 2, 128, 2, 8>;   // both planes per stage (bf16x3), 2 stages of 80 KB, 8 epilogue warps
// wgrad: 3-CTA clusters (the three 128-wide teacher-channel tiles of one row split) with the S block multicast
using AlignWgradCfg1 = GemmNtCfg<3, true, 208, 0, 4, 64, false, 1, 3>;
// both planes per stage.  32 contraction rows per stage: 4 stages of 48 KB — with 64-row stages only two (96 KB each) fit and
// every stage exposed a full TMA round trip (the kernel ran at 2.1 us per 64 rows against 0.65 us of MMA time)
using AlignWgradCfg2 = GemmNtCfg<3, true, 208, 0, 4, 32, false, 2, 3>;

template <class Cfg>
inline int align_forward_rows_t(const __nv_bfloat16* S, const __nv_bfloat16* Wp, const float* bias, float* A, int64_t M, int Ds, int Dt,
                                int P, cudaStream_t st, const char* what) {
  using L = PlaneLoader<Cfg>;
  using E = StoreRowsEpi<Cfg>;
  GemmParams<L, E> p;
  int rc = make_plane_tmap(&p.ld.tmA, S, P, M, Ds, Ds, M * Ds, Cfg::BM, what);
  if (rc != DKD_OK) return rc;
  rc = make_plane_tmap(&p.ld.tmB, Wp, P, Dt, Ds, Ds, (int64_t)Dt * Ds, Cfg::BN, what);
  if (rc != DKD_OK) return rc;
  p.ld.k_blocks = Ds / 64; p.ld.nterms = P == 2 ? 3 : 1;
  p.ep.out = A; p.ep.drop_mask = nullptr; p.ep.bias = bias; p.ep.alpha = 1.f;
  p.ep.M = M; p.ep.N_total = Dt; p.ep.n_tok = (int)M; p.ep.T_out = (int)M; p.ep.off = 0; p.ep.out_is_bf16 = 0;
  p.m_tiles = (int)((M + Cfg::BM - 1) / Cfg::BM); p.n_tiles = Dt / Cfg::BN;
  const int grid = min(kNumSMs, p.m_tiles * p.n_tiles);
  auto kern = gemm_tn_kernel<Cfg, L, E>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
  kern<<<grid, Cfg::THREADS, Cfg::SMEM, st>>>(p);
  return check_launch(what);
}

template <class Cfg>
inline int align_dgrad_t(const __nv_bfloat16* G, const __nv_bfloat16* Wt, void* g_s, int64_t M, int n_tok, int Ts, int s_off, int Ds, int Dt,
                         int P, int out_is_bf16, float alpha, cudaStream_t st, const char* what, int g_lo_zero = 0) {
  using L = PlaneLoader<Cfg>;
  using E = StoreRowsEpi<Cfg>;
  GemmParams<L, E> p;
  int rc = make_plane_tmap(&p.ld.tmA, G, P, M, Dt, Dt, M * Dt, Cfg::BM, what);
  if (rc != DKD_OK) return rc;
  rc = make_plane_tmap(&p.ld.tmB, Wt, P, Ds, Dt, Dt, (int64_t)Dt * Ds, Cfg::BN, what);
  if (rc != DKD_OK) return rc;
  p.ld.k_blocks = Dt / 64; p.ld.nterms = P == 2 ? 3 : 1;
  p.a_lo_zero = p.ld.a_lo_zero = (Cfg::PLANES == 2 && g_lo_zero) ? 1 : 0;
  p.ep.out = g_s; p.ep.drop_mask = nullptr; p.ep.bias = nullptr; p.ep.alpha = alpha;
  p.ep.M = M; p.ep.N_total = Ds; p.ep.n_tok = n_tok; p.ep.T_out = Ts; p.ep.off = s_off; p.ep.out_is_bf16 = out_is_bf16;
  p.m_tiles = (int)((M + Cfg::BM - 1) / Cfg::BM); p.n_tiles = Ds / Cfg::BN;
  const int grid = min(kNumSMs, p.m_tiles * p.n_tiles);
  auto kern = gemm_tn_kernel<Cfg, L, E>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
  kern<<<grid, Cfg::THREADS, Cfg::SMEM, st>>>(p);
  return check_launch(what);
}

inline int align_forward_rows(const __nv_bfloat16* S, const __nv_bfloat16* Wp, const float* bias, float* A, int64_t M, int Ds, int Dt,
                              int P, cudaStream_t st, const char* what) {
  return P == 2 ? align_forward_rows_t<AlignCfg2>(S, Wp, bias, A, M, Ds, Dt, P, st, what)
                : align_forward_rows_t<AlignCfg1>(S, Wp, bias, A, M, Ds, Dt, P, st, what);
}
// g_lo_zero: the lo plane of G is identically zero and is neither read nor multiplied (WassKD's +-1 gradient plane)
inline int align_dgrad(const __nv_bfloat16* G, const __nv_bfloat16* Wt, void* g_s, int64_t M, int n_tok, int Ts, int s_off, int Ds, int Dt,
                       int P, int out_is_bf16, float alpha, cudaStream_t st, const char* what, int g_lo_zero = 0) {
  return P == 2 ? align_dgrad_t<AlignCfg2>(G, Wt, g_s, M, n_tok, Ts, s_off, Ds, Dt, P, out_is_bf16, alpha, st, what, g_lo_zero)
                : align_dgrad_t<AlignCfg1>(G, Wt, g_s, M, n_tok, Ts, s_off, Ds, Dt, P, out_is_bf16, alpha, st, what);
}

template <class Cfg>
inline int align_wgrad_t(const __nv_bfloat16* G, const __nv_bfloat16* S, __nv_bfloat16* ones, float* g_W, float* g_b, int64_t M, int Ds, int Dt,
                         int P, float alpha, cudaStream_t st, const char* what, int g_lo_zero = 0) {
  using L = NtPlainLoader<Cfg>;
  GemmNtParamsT<Cfg, L> p;
  int rc = make_plane_tmap(&p.ld.tmA, G, P, M, Dt, Dt, M * Dt, Cfg::KROWS, what);
  if (rc != DKD_OK) return rc;
  rc = make_plane_tmap(&p.ld.tmB, S, P, M, Ds, Ds, M * Ds, Cfg::KROWS, what);
  if (rc != DKD_OK) return rc;
  rc = make_plane_tmap(&p.ld.tmOnes, ones, 2, 64, 64, 64, 64 * 64, Cfg::KROWS, "ones tile");
  if (rc != DKD_OK) return rc;
  rc = launch_fill_ones_tile(ones, st);
  if (rc != DKD_OK) return rc;
  cudaMemsetAsync(g_W, 0, (size_t)Dt * Ds * sizeof(float), st);
  if (g_b) cudaMemsetAsync(g_b, 0, (size_t)Dt * sizeof(float), st);
  p.ep.D = g_W; p.ep.Dcol = g_b; p.ep.ldd = Ds; p.ep.alpha = alpha;
  p.ld.ldd = Ds; p.ld.na_tiles = Dt / 128; p.ld.b_col0 = 0;
  p.ld.total_row_blocks = (int)((M + Cfg::KROWS - 1) / Cfg::KROWS);
  p.nterms = P == 2 ? 3 : 1;
  p.a_lo_zero = (Cfg::PLANES == 2 && g_lo_zero) ? 1 : 0;
  static const int resident = [] {
    auto kern = gemm_nt_kernel<Cfg, L>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
    return max_resident_clusters(kern, Cfg::CLUSTER, Cfg::THREADS, Cfg::SMEM);
  }();
  nt_make_splits(p.ld.total_row_blocks, resident, &p.ld.splits, &p.ld.row_blocks_per_split);
  launch_gemm_nt<Cfg, L>(p, min(resident, p.ld.splits) * Cfg::CLUSTER, st);
  return check_launch(what);
}

inline int align_wgrad(const __nv_bfloat16* G, const __nv_bfloat16* S, __nv_bfloat16* ones, float* g_W, float* g_b, int64_t M, int Ds, int Dt,
                       int P, float alpha, cudaStream_t st, const char* what, int g_lo_zero = 0) {
  return P == 2 ? align_wgrad_t<AlignWgradCfg2>(G, S, ones, g_W, g_b, M, Ds, Dt, P, alpha, st, what, g_lo_zero)
                : align_wgrad_t<AlignWgradCfg1>(G, S, ones, g_W, g_b, M, Ds, Dt, P, alpha, st, what);
}

}  // namespace dkd
