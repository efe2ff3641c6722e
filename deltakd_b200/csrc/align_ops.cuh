// The three tcgen05 GEMMs around a Linear(Ds -> Dt) alignment head, shared by the losses that need the aligned
// activations themselves (WassKD): forward rows, and the backward from a gradient-plane tensor G[P][M][Dt].
//   align_forward_rows : A[M, Dt] fp32 = S W^T + bias                 (gemm_tn, StoreRows epilogue)
//   align_dgrad        : g_s[:, off:, :] = alpha * G W                (gemm_tn, rows scattered, special tokens zeroed)
//   align_wgrad        : g_W = alpha * G^T S, g_b = alpha * G^T 1     (gemm_nt split-K in 3-CTA clusters, ones-column trick;
//                        float atomics, or per-split slots and a fixed-order fold in deterministic mode)
// Dt = 384 or 768 (the fused CurKD kernel of align_fused.cuh covers the forward and dgrad of align_mse).
#pragma once
#include "epilogues.cuh"
#include "gemm_nt.cuh"
#include "planes.cuh"

namespace dkd {

using AlignCfg1 = GemmCfg<192, 1, 4, 2, 128, 1, 8>;   // one plane per stage (bf16 operands), 4-stage ring, 8 epilogue warps
using AlignCfg2 = GemmCfg<192, 1, 2, 2, 128, 2, 8>;   // both planes per stage (bf16x3), 2 stages of 80 KB, 8 epilogue warps
// wgrad: 3-CTA clusters (three 128-wide teacher-channel tiles of one row split) with the S block multicast; Dt = 768 has two
// such tile groups per row split
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

// Deterministic mode (`part` non-null): the split count depends on the shapes only (kNumSMs / CLUSTER clusters instead of
// the device's resident-cluster count), every work item stores its tile and its ones column with plain stores
// into slot part[split][nt_slot_floats(Dt * Ds + Dt)], and fold_splits_kernel adds the slots in split order in fp64 and applies alpha.
template <class Cfg, int GROUPS>
inline void align_wgrad_splits(int64_t M, int want, int* splits, int* per_split) {
  nt_make_splits((int)((M + Cfg::KROWS - 1) / Cfg::KROWS), want / GROUPS, splits, per_split);
}

template <class Cfg, int GROUPS>
inline size_t align_wgrad_part_bytes_t(int64_t M, int Ds, int Dt) {
  int splits, per;
  align_wgrad_splits<Cfg, GROUPS>(M, kNumSMs / Cfg::CLUSTER, &splits, &per);
  return (size_t)splits * nt_slot_floats((int64_t)Dt * Ds + Dt) * sizeof(float);
}

// bytes of the deterministic-mode partial slots of align_wgrad
inline size_t align_wgrad_part_bytes(int64_t M, int Ds, int Dt, int P) {
  if (Dt == 768)
    return P == 2 ? align_wgrad_part_bytes_t<AlignWgradCfg2, 2>(M, Ds, Dt) : align_wgrad_part_bytes_t<AlignWgradCfg1, 2>(M, Ds, Dt);
  return P == 2 ? align_wgrad_part_bytes_t<AlignWgradCfg2, 1>(M, Ds, Dt) : align_wgrad_part_bytes_t<AlignWgradCfg1, 1>(M, Ds, Dt);
}

template <class Cfg, int GROUPS>
inline int align_wgrad_t(const __nv_bfloat16* G, const __nv_bfloat16* S, __nv_bfloat16* ones, float* g_W, float* g_b, int64_t M, int Ds, int Dt,
                         int P, float alpha, cudaStream_t st, const char* what, int g_lo_zero, float* part) {
  using L = NtPlainLoader<Cfg, GROUPS>;
  GemmNtParamsT<Cfg, L> p;
  int rc = make_plane_tmap(&p.ld.tmA, G, P, M, Dt, Dt, M * Dt, Cfg::KROWS, what);
  if (rc != DKD_OK) return rc;
  rc = make_plane_tmap(&p.ld.tmB, S, P, M, Ds, Ds, M * Ds, Cfg::KROWS, what);
  if (rc != DKD_OK) return rc;
  rc = make_plane_tmap(&p.ld.tmOnes, ones, 2, 64, 64, 64, 64 * 64, Cfg::KROWS, "ones tile");
  if (rc != DKD_OK) return rc;
  rc = launch_fill_ones_tile(ones, st);
  if (rc != DKD_OK) return rc;
  const int64_t slot = nt_slot_floats((int64_t)Dt * Ds + Dt);
  if (part) {
    p.ep.D = part; p.ep.Dcol = g_b ? part + (int64_t)Dt * Ds : nullptr; p.ep.alpha = 1.f; p.ep.store = 1; p.ep.split_stride = slot;
  } else {
    cudaMemsetAsync(g_W, 0, (size_t)Dt * Ds * sizeof(float), st);
    if (g_b) cudaMemsetAsync(g_b, 0, (size_t)Dt * sizeof(float), st);
    p.ep.D = g_W; p.ep.Dcol = g_b; p.ep.alpha = alpha;
  }
  p.ep.ldd = Ds;
  p.ld.ldd = Ds; p.ld.na_tiles = Dt / 128; p.ld.b_col0 = 0;
  p.ld.total_row_blocks = (int)((M + Cfg::KROWS - 1) / Cfg::KROWS);
  p.nterms = P == 2 ? 3 : 1;
  p.a_lo_zero = (Cfg::PLANES == 2 && g_lo_zero) ? 1 : 0;
  static const int resident = [] {
    auto kern = gemm_nt_kernel<Cfg, L>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
    return max_resident_clusters(kern, Cfg::CLUSTER, Cfg::THREADS, Cfg::SMEM);
  }();
  // GROUPS work items (cluster tasks) per row split: about `resident` items in all, one wave of clusters.  The deterministic
  // split count is fixed by the shapes; its grid stays at the resident count, since each item owns its slot and which
  // cluster computes it cannot change a bit
  align_wgrad_splits<Cfg, GROUPS>(M, part ? kNumSMs / Cfg::CLUSTER : resident, &p.ld.splits, &p.ld.row_blocks_per_split);
  launch_gemm_nt<Cfg, L>(p, min(resident, GROUPS * p.ld.splits) * Cfg::CLUSTER, st);
  rc = check_launch(what);
  if (rc != DKD_OK || !part) return rc;
  return launch_fold_splits(part, p.ld.splits, slot, (int64_t)Dt * Ds, g_W, g_b ? Dt : 0, g_b, alpha, st);
}

// part: null = split-K reduction with float atomics into g_W / g_b; else deterministic mode, align_wgrad_part_bytes(...) bytes
inline int align_wgrad(const __nv_bfloat16* G, const __nv_bfloat16* S, __nv_bfloat16* ones, float* g_W, float* g_b, int64_t M, int Ds, int Dt,
                       int P, float alpha, cudaStream_t st, const char* what, int g_lo_zero = 0, float* part = nullptr) {
  if (Dt == 768)   // 6 teacher-channel tiles: two groups of 3
    return P == 2 ? align_wgrad_t<AlignWgradCfg2, 2>(G, S, ones, g_W, g_b, M, Ds, Dt, P, alpha, st, what, g_lo_zero, part)
                  : align_wgrad_t<AlignWgradCfg1, 2>(G, S, ones, g_W, g_b, M, Ds, Dt, P, alpha, st, what, 0, part);
  return P == 2 ? align_wgrad_t<AlignWgradCfg2, 1>(G, S, ones, g_W, g_b, M, Ds, Dt, P, alpha, st, what, g_lo_zero, part)
                : align_wgrad_t<AlignWgradCfg1, 1>(G, S, ones, g_W, g_b, M, Ds, Dt, P, alpha, st, what, 0, part);
}

}  // namespace dkd
