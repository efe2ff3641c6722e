// Conversion of fp32 / bf16 activations and fp32 weights into bf16 hi/lo plane tensors (planes.cuh).
// Pure streaming kernels: 16-byte vector loads and stores, grid sized to a multiple of the SM count.
#include "planes.cuh"

namespace dkd {
namespace {

template <typename T>
__global__ void tokens_to_planes_kernel(const T* __restrict__ src, int64_t B, int T_tok, int off, int n_tok, int D, int P,
                                        const float* __restrict__ drop_mask, __nv_bfloat16* __restrict__ dst) {
  const int vec_per_row = D / 8;
  const int64_t M = B * n_tok;
  const int64_t total = M * vec_per_row;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride) {
    const int64_t m = idx / vec_per_row;
    const int c = (int)(idx - m * vec_per_row) * 8;
    const int64_t b = m / n_tok;
    const int64_t srow = b * T_tok + off + (m - b * n_tok);
    float v[8];
    if (drop_mask != nullptr && __ldg(drop_mask + m) != 0.f) {  // masked token: its row is never used downstream
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = 0.f;
    } else if constexpr (sizeof(T) == 4) {
      Vec<float, 4>::load(reinterpret_cast<const float*>(src) + srow * D + c, *reinterpret_cast<float(*)[4]>(&v[0]));
      Vec<float, 4>::load(reinterpret_cast<const float*>(src) + srow * D + c + 4, *reinterpret_cast<float(*)[4]>(&v[4]));
    } else {
      Vec<__nv_bfloat16, 8>::load(reinterpret_cast<const __nv_bfloat16*>(src) + srow * D + c, v);
    }
    Vec<__nv_bfloat16, 8>::store(dst + m * D + c, v);
    if (P >= 2) {
      float lo[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) lo[j] = v[j] - __bfloat162float(__float2bfloat16_rn(v[j]));
      Vec<__nv_bfloat16, 8>::store(dst + M * D + m * D + c, lo);
      if (P >= 3) {  // third plane: all 24 mantissa bits (fp32-exact operands for 6-term products)
#pragma unroll
        for (int j = 0; j < 8; ++j) lo[j] = lo[j] - __bfloat162float(__float2bfloat16_rn(lo[j]));
        Vec<__nv_bfloat16, 8>::store(dst + 2 * M * D + m * D + c, lo);
      }
    }
  }
}

__global__ void weight_to_planes_kernel(const float* __restrict__ W, int N, int K, int P, __nv_bfloat16* __restrict__ Wp,
                                        __nv_bfloat16* __restrict__ Wt) {
  const int total = N * K;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int n = idx / K, k = idx - n * K;
    const float x = W[idx];
    const __nv_bfloat16 hi = __float2bfloat16_rn(x);
    const __nv_bfloat16 lo = __float2bfloat16_rn(x - __bfloat162float(hi));
    if (Wp) { Wp[idx] = hi; if (P == 2) Wp[total + idx] = lo; }
    if (Wt) { Wt[k * N + n] = hi; if (P == 2) Wt[total + k * N + n] = lo; }
  }
}

__global__ void fill_ones_tile_kernel(__nv_bfloat16* ones) {
  for (int idx = threadIdx.x; idx < 2 * 64 * 64; idx += blockDim.x)
    ones[idx] = __float2bfloat16_rn((idx < 64 * 64 && (idx & 63) == 0) ? 1.f : 0.f);
}

// conv weight W[co][ci][3][3] fp32 -> forward planes Wc[P][co][tap*C + ci] and dgrad planes Wd[P][ci][(8-tap)*C + co]
__global__ void conv_weight_to_planes_kernel(const float* __restrict__ W, int C, int P, __nv_bfloat16* __restrict__ Wc,
                                             __nv_bfloat16* __restrict__ Wd) {
  const int total = C * C * 9;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int tap = idx % 9, ci = (idx / 9) % C, co = idx / (9 * C);
    const float x = W[idx];
    const __nv_bfloat16 hi = __float2bfloat16_rn(x);
    const __nv_bfloat16 lo = __float2bfloat16_rn(x - __bfloat162float(hi));
    const int64_t fc = (int64_t)co * 9 * C + tap * C + ci;
    const int64_t fd = (int64_t)ci * 9 * C + (8 - tap) * C + co;
    Wc[fc] = hi; Wd[fd] = hi;
    if (P == 2) { Wc[total + fc] = lo; Wd[total + fd] = lo; }
  }
}

// dWt[split][tap][co][ci] fp32 -> dW[co][ci][tap] (PyTorch conv weight layout).  splits = 1: a gather in output order.
// splits > 1 (deterministic mode): the splits are added in split order in fp64, threads walking the source order so that
// the `splits` reads per element are coalesced and only its one store is strided.
__global__ void conv_wgrad_transpose_kernel(const float* __restrict__ dWt, int C, int splits, float* __restrict__ dW) {
  const int total = C * C * 9;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    if (splits == 1) {
      const int tap = idx % 9, ci = (idx / 9) % C, co = idx / (9 * C);
      dW[idx] = dWt[((int64_t)tap * C + co) * C + ci];
    } else {
      const int ci = idx % C, co = (idx / C) % C, tap = idx / (C * C);
      double a = dWt[idx];
#pragma unroll 4
      for (int s = 1; s < splits; ++s) a += (double)dWt[(int64_t)s * total + idx];
      dW[((int64_t)co * C + ci) * 9 + tap] = (float)a;
    }
  }
}

// out0[i] = alpha * sum_s part[s * stride + i] (i < n0), out1[i - n0] likewise (n0 <= i < n0 + n1): the per-split slots
// of a deterministic split-K product, added in slot order in fp64.  Null outputs are skipped.
__global__ void fold_splits_kernel(const float* __restrict__ part, int splits, int64_t stride, int64_t n0, float* __restrict__ out0,
                                   int64_t n1, float* __restrict__ out1, float alpha) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n0 + n1; i += (int64_t)gridDim.x * blockDim.x) {
    float* out = i < n0 ? (out0 ? out0 + i : nullptr) : (out1 ? out1 + (i - n0) : nullptr);
    if (out == nullptr) continue;
    double a = part[i];
#pragma unroll 4
    for (int s = 1; s < splits; ++s) a += (double)part[(int64_t)s * stride + i];
    *out = (float)(a * (double)alpha);
  }
}

// Column sums' fold: many partial rows (up to 592 per-CTA rows) over few columns (2N).  One CTA per 32 columns: warp w
// adds rows w, w + 32, w + 64, ... in increasing order (fp64), then warp 0 adds the 32 warp sums in warp order.  The
// order depends on `rows` only, so the result is deterministic, and each thread's chain is rows / 32 loads long instead
// of `rows` (fold_splits_kernel's one-thread-per-output form).
constexpr int kFoldRowsWarps = 32;
__global__ void __launch_bounds__(kFoldRowsWarps * 32) fold_rows_kernel(const float* __restrict__ part, int rows, int ncols, int64_t n0,
                                                                       float* __restrict__ out0, float* __restrict__ out1) {
  __shared__ double s_sum[kFoldRowsWarps][33];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int col = blockIdx.x * 32 + lane;
  double a = 0.0;
  if (col < ncols) {
#pragma unroll 4
    for (int r = warp; r < rows; r += kFoldRowsWarps) a += (double)part[(int64_t)r * ncols + col];
  }
  s_sum[warp][lane] = a;
  __syncthreads();
  if (warp == 0 && col < ncols) {
    double t = s_sum[0][lane];
    for (int w = 1; w < kFoldRowsWarps; ++w) t += s_sum[w][lane];
    float* out = col < n0 ? (out0 ? out0 + col : nullptr) : (out1 ? out1 + (col - n0) : nullptr);
    if (out) *out = (float)t;
  }
}

// column sums of plane tensors [P][M][N] (hi + lo), optionally split by a 0/1 row mask:
//   out_keep[c] += sum_{rows with mask==0 (or all rows if mask==null)} x[r,c];  out_masked[c] += sum_{mask!=0} x[r,c]
// One HBM pass: a thread owns 8 adjacent columns (16-byte loads of both planes), the CTA's row lanes stride over a
// contiguous block of rows with two rows in flight, lanes are combined in shared memory and each CTA issues one
// atomicAdd per column (592 CTAs x N atomics; the former one-row-per-CTA-iteration form took 85-95 us per call for
// 77-154 MB — 10 % of the bf16 MGD step).  With `part` (deterministic mode) the CTA stores its two sums as row
// part[cta][2][N] instead, and fold_rows_kernel adds the rows in a fixed order.
constexpr int kColsumThreads = 256;
__global__ void __launch_bounds__(kColsumThreads) colsum_planes_kernel(const __nv_bfloat16* __restrict__ X, int64_t M, int N, int P,
                                                                       const float* __restrict__ mask, int64_t rows_per_cta,
                                                                       float* __restrict__ out_keep, float* __restrict__ out_masked,
                                                                       float* __restrict__ part) {
  extern __shared__ float s_cs[];   // [2][RL][N]
  const int G = N >> 3, RL = kColsumThreads / G;
  const int cg = threadIdx.x % G, rl = threadIdx.x / G;
  float keep[8], msk[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) keep[j] = msk[j] = 0.f;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_cta;
  const int64_t r1 = r0 + rows_per_cta < M ? r0 + rows_per_cta : M;
  if (rl < RL) {
    auto row = [&](int64_t r, float (&v)[8]) {
      Vec<__nv_bfloat16, 8>::load(X + r * N + 8 * cg, v);
      if (P == 2) {
        float lo[8];
        Vec<__nv_bfloat16, 8>::load(X + M * N + r * N + 8 * cg, lo);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] += lo[j];
      }
    };
    auto add = [&](int64_t r, const float (&v)[8]) {
      if (mask != nullptr && __ldg(mask + r) != 0.f) {
#pragma unroll
        for (int j = 0; j < 8; ++j) msk[j] += v[j];
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) keep[j] += v[j];
      }
    };
    int64_t r = r0 + rl;
    for (; r + RL < r1; r += 2 * RL) {
      float u[8], w[8];
      row(r, u);
      row(r + RL, w);
      add(r, u);
      add(r + RL, w);
    }
    for (; r < r1; r += RL) {
      float u[8];
      row(r, u);
      add(r, u);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      s_cs[rl * N + 8 * cg + j] = keep[j];
      s_cs[(RL + rl) * N + 8 * cg + j] = msk[j];
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < 2 * N; k += kColsumThreads) {
    const int which = k / N, c = k - which * N;
    float* out = which ? out_masked : out_keep;
    if (out == nullptr) continue;
    float a = 0.f;
    for (int q = 0; q < RL; ++q) a += s_cs[(which * RL + q) * N + c];
    if (part) part[(int64_t)blockIdx.x * 2 * N + k] = a;
    else atomicAdd(out + c, a);
  }
}

// *loss += scale * sum(partials[0..n)): fixed thread -> partial assignment and fixed tree (bit-reproducible)
__global__ void __launch_bounds__(256) fold_partials_kernel(const double* __restrict__ partials, int n, float scale, float* __restrict__ loss) {
  __shared__ double s_w[8];
  double a = 0.0;
  for (int i = threadIdx.x; i < n; i += 256) a += partials[i];
  a = warp_sum(a);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += s_w[w];
    *loss += (float)(t * (double)scale);
  }
}

}  // namespace

int launch_fold_partials(const double* partials, int n, float scale, float* loss, cudaStream_t st) {
  fold_partials_kernel<<<1, 256, 0, st>>>(partials, n, scale, loss);
  return check_launch("fold_partials");
}

int launch_tokens_to_planes(const void* src, int dtype, int64_t B, int T, int off, int n_tok, int D, int P,
                            const float* drop_mask, __nv_bfloat16* dst, cudaStream_t st) {
  DKD_REQUIRE(D % 8 == 0, DKD_E_SHAPE, "tokens_to_planes: D %% 8 != 0");
  DKD_REQUIRE((((uintptr_t)src) & 15) == 0, DKD_E_ALIGN, "tokens_to_planes: source must be 16-byte aligned");
  const int64_t total = B * n_tok * (D / 8);
  int64_t blocks = (total + 255) / 256;
  if (blocks > (int64_t)kNumSMs * 8) blocks = (int64_t)kNumSMs * 8;
  if (dtype == DKD_F32)
    tokens_to_planes_kernel<float><<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const float*>(src), B, T, off, n_tok, D, P, drop_mask, dst);
  else
    tokens_to_planes_kernel<__nv_bfloat16><<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(src), B, T, off, n_tok, D, P, drop_mask, dst);
  return check_launch("tokens_to_planes");
}

int launch_weight_to_planes(const float* W, int N, int K, int P, __nv_bfloat16* Wp, __nv_bfloat16* Wt, cudaStream_t st) {
  const int total = N * K;
  int blocks = (total + 255) / 256;
  if (blocks > kNumSMs * 4) blocks = kNumSMs * 4;
  weight_to_planes_kernel<<<blocks, 256, 0, st>>>(W, N, K, P, Wp, Wt);
  return check_launch("weight_to_planes");
}

int launch_conv_weight_to_planes(const float* W, int C, int P, __nv_bfloat16* Wc, __nv_bfloat16* Wd, cudaStream_t st) {
  conv_weight_to_planes_kernel<<<kNumSMs * 4, 256, 0, st>>>(W, C, P, Wc, Wd);
  return check_launch("conv_weight_to_planes");
}

int launch_conv_wgrad_transpose(const float* dWt, int C, int splits, float* dW, cudaStream_t st) {
  conv_wgrad_transpose_kernel<<<kNumSMs * 4, 256, 0, st>>>(dWt, C, splits, dW);
  return check_launch("conv_wgrad_transpose");
}

int launch_fold_splits(const float* part, int splits, int64_t stride, int64_t n0, float* out0, int64_t n1, float* out1, float alpha,
                       cudaStream_t st) {
  int64_t blocks = (n0 + n1 + 255) / 256;
  if (blocks > (int64_t)kNumSMs * 8) blocks = (int64_t)kNumSMs * 8;
  fold_splits_kernel<<<(unsigned)blocks, 256, 0, st>>>(part, splits, stride, n0, out0, n1, out1, alpha);
  return check_launch("fold_splits");
}

size_t colsum_planes_part_bytes(int N) { return (size_t)kNumSMs * 4 * 2 * N * sizeof(float); }

int launch_colsum_planes(const __nv_bfloat16* X, int64_t M, int N, int P, const float* mask, float* out_keep, float* out_masked,
                         cudaStream_t st, float* part) {
  DKD_REQUIRE(N % 8 == 0 && N / 8 <= kColsumThreads, DKD_E_SHAPE, "colsum_planes: N");
  DKD_REQUIRE((((uintptr_t)X) & 15) == 0, DKD_E_ALIGN, "colsum_planes: 16-byte alignment");
  if (!part && out_keep) cudaMemsetAsync(out_keep, 0, (size_t)N * sizeof(float), st);
  if (!part && out_masked) cudaMemsetAsync(out_masked, 0, (size_t)N * sizeof(float), st);
  const int RL = kColsumThreads / (N / 8);
  int64_t blocks = (M + 2 * RL - 1) / (2 * RL);          // at least two rows per row lane
  if (blocks > (int64_t)kNumSMs * 4) blocks = (int64_t)kNumSMs * 4;
  if (blocks < 1) blocks = 1;
  const int64_t rows_per_cta = (M + blocks - 1) / blocks;
  blocks = (M + rows_per_cta - 1) / rows_per_cta;
  const size_t smem = (size_t)2 * RL * N * sizeof(float);
  colsum_planes_kernel<<<(unsigned)blocks, kColsumThreads, smem, st>>>(X, M, N, P, mask, rows_per_cta, out_keep, out_masked, part);
  int rc = check_launch("colsum_planes");
  if (rc != DKD_OK || !part) return rc;
  fold_rows_kernel<<<(2 * N + 31) / 32, kFoldRowsWarps * 32, 0, st>>>(part, (int)blocks, 2 * N, N, out_keep, out_masked);
  return check_launch("colsum_planes: fold");
}

int launch_fill_ones_tile(__nv_bfloat16* ones, cudaStream_t st) {
  fill_ones_tile_kernel<<<1, 256, 0, st>>>(ones);
  return check_launch("fill_ones_tile");
}

}  // namespace dkd
