// bf16 "plane" operands of the tensor-core contractions.
// A value x is represented as hi = bf16(x) and, in the bf16x3 mode, lo = bf16(x - hi); products are
// formed as hi*hi + hi*lo + lo*hi in fp32 TMEM accumulators (relative error ~2^-16).
// Layout: [P planes][rows][cols] bf16, cols contiguous; plane 0 = hi, plane 1 = lo.
#pragma once
#include "common.cuh"

namespace dkd {

// patch tokens of src[B, T, D] (tokens off .. off+n_tok-1) -> dst[P][B*n_tok][D]
// rows whose drop_mask[m] != 0 are written as zeros (drop_mask may be null)
int launch_tokens_to_planes(const void* src, int dtype, int64_t B, int T, int off, int n_tok, int D, int P,
                            const float* drop_mask, __nv_bfloat16* dst, cudaStream_t st);
// conv weight [C][C][3][3] fp32 -> Wc[P][C][9C] (forward) and Wd[P][C][9C] (dgrad: taps flipped, channels swapped)
int launch_conv_weight_to_planes(const float* W, int C, int P, __nv_bfloat16* Wc, __nv_bfloat16* Wd, cudaStream_t st);
// dWt[splits][9][C][C] fp32 -> dW[C][C][3][3], the splits added in split order (fp64)
int launch_conv_wgrad_transpose(const float* dWt, int C, int splits, float* dW, cudaStream_t st);
// column sums of planes [P][M][N] split by an optional 0/1 row mask (outputs are overwritten).  `part` (deterministic
// mode, colsum_planes_part_bytes(N) bytes): per-CTA partial rows folded in a fixed order (fold_rows_kernel) instead of
// float atomics
int launch_colsum_planes(const __nv_bfloat16* X, int64_t M, int N, int P, const float* mask, float* out_keep, float* out_masked,
                         cudaStream_t st, float* part = nullptr);
size_t colsum_planes_part_bytes(int N);
// out0[0..n0) and out1[0..n1) = alpha * sum over s = 0..splits-1, in order, of part[s * stride + i] (fp64); null outputs skipped
int launch_fold_splits(const float* part, int splits, int64_t stride, int64_t n0, float* out0, int64_t n1, float* out1, float alpha,
                       cudaStream_t st);
// W[N, K] fp32 -> Wp[P][N][K] (optional) and Wt[P][K][N] (optional)
int launch_weight_to_planes(const float* W, int N, int K, int P, __nv_bfloat16* Wp, __nv_bfloat16* Wt, cudaStream_t st);
// ones[2][64][64]: plane 0 has column 0 = 1, everything else 0
int launch_fill_ones_tile(__nv_bfloat16* ones, cudaStream_t st);

// *loss += scale * sum(partials[0..n)), fixed order
int launch_fold_partials(const double* partials, int n, float scale, float* loss, cudaStream_t st);

}  // namespace dkd
