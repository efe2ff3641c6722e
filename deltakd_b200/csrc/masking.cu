// Mask selection by rank-by-counting (bit-exact integer work) and the conditional gradient rescale.
// Reference: model/misc.py:14-30 (random_masking) and :72-81 / :118-128 / :150-160 (saliency_masking):
//   ids_shuffle = argsort(score); ids_restore = argsort(ids_shuffle); mask = gather(ones with the first
//   len_keep zeroed, ids_restore)   ==   rank_i = #{j : s_j < s_i or (s_j == s_i and j < i)},
//   mask_i = rank_i >= len_keep.
// One CTA per row; the row sits in shared memory; every thread counts for one token.
#include "common.cuh"

namespace dkd {
namespace {

__global__ void mask_rank_kernel(const float* __restrict__ score, int L, int len_keep, float* __restrict__ mask,
                                 int64_t* __restrict__ ids_restore, int64_t* __restrict__ ids_shuffle) {
  extern __shared__ float s_row[];
  const int64_t row = blockIdx.x;
  const float* src = score + row * L;
  for (int i = threadIdx.x; i < L; i += blockDim.x) s_row[i] = src[i];
  __syncthreads();
  for (int i = threadIdx.x; i < L; i += blockDim.x) {
    const float v = s_row[i];
    int rank = 0;
    if (v != v) {  // NaN sorts last (torch.sort semantics); among NaNs lower index first
      for (int j = 0; j < L; ++j) { const float u = s_row[j]; rank += (u == u) || (j < i); }
    } else {
      for (int j = 0; j < L; ++j) { const float u = s_row[j]; rank += (u < v) || (u == v && j < i); }
    }
    if (mask) mask[row * L + i] = rank >= len_keep ? 1.f : 0.f;
    if (ids_restore) ids_restore[row * L + i] = rank;
    if (ids_shuffle) ids_shuffle[row * L + rank] = i;
  }
}

template <typename T, int VEC>
__global__ void scale_if_not_one_kernel(T* __restrict__ x, int64_t n_vec, T* __restrict__ x2, int64_t n_vec2,
                                        const float* __restrict__ scale) {
  // launched with programmatic dependent launch: the predecessor (the op that wrote x / x2, or the one that wrote
  // *scale) may still be running until the wait returns
  grid_dep_wait();
  grid_dep_launch();
  const float s = *scale;
  if (s == 1.0f) return;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec + n_vec2; i += stride) {
    T* p = i < n_vec ? x + i * VEC : x2 + (i - n_vec) * VEC;
    float v[VEC];
    Vec<T, VEC>::load(p, v);
#pragma unroll
    for (int k = 0; k < VEC; ++k) v[k] *= s;
    Vec<T, VEC>::store(p, v);
  }
}

template <typename T>
int launch_scale(void* x, int64_t n, void* x2, int64_t n2, const float* scale, cudaStream_t st) {
  constexpr int MAXV = 16 / (int)sizeof(T);
  const bool vec_ok = (n % MAXV == 0) && ((((uintptr_t)x) & 15) == 0) && (n2 % MAXV == 0) && ((((uintptr_t)x2) & 15) == 0);
  const int64_t n_vec = vec_ok ? n / MAXV : n, n_vec2 = vec_ok ? n2 / MAXV : n2;
  int64_t blocks = (n_vec + n_vec2 + 255) / 256;
  if (blocks > (int64_t)kNumSMs * 16) blocks = (int64_t)kNumSMs * 16;
  if (blocks < 1) blocks = 1;
  T *a = reinterpret_cast<T*>(x), *b = reinterpret_cast<T*>(x2);
  if (vec_ok) launch_pdl(scale_if_not_one_kernel<T, MAXV>, dim3((unsigned)blocks), dim3(256), st, a, n_vec, b, n_vec2, scale);
  else launch_pdl(scale_if_not_one_kernel<T, 1>, dim3((unsigned)blocks), dim3(256), st, a, n_vec, b, n_vec2, scale);
  return check_launch("dkd_scale_if_not_one");
}

}  // namespace
}  // namespace dkd

extern "C" {

int dkd_mask_rank(const float* score, int64_t B, int64_t L, int64_t len_keep, float* mask,
                  int64_t* ids_restore, int64_t* ids_shuffle, dkd_stream_t stream) {
  using namespace dkd;
  int rc = dkd_check_device();
  if (rc != DKD_OK) return rc;
  DKD_REQUIRE(B >= 0 && L > 0 && L <= 1024 && B < (1ll << 31), DKD_E_SHAPE, "dkd_mask_rank: need 0 < L <= 1024 (B=%lld L=%lld)", (long long)B, (long long)L);
  DKD_REQUIRE(len_keep >= 0 && len_keep <= L, DKD_E_SHAPE, "dkd_mask_rank: len_keep %lld outside [0, L]", (long long)len_keep);
  if (B == 0) return DKD_OK;
  DKD_REQUIRE(score != nullptr, DKD_E_SHAPE, "dkd_mask_rank: null score");
  const int threads = L <= 256 ? (int)((L + 31) / 32 * 32) : 256;
  mask_rank_kernel<<<(unsigned)B, threads, (size_t)L * sizeof(float), reinterpret_cast<cudaStream_t>(stream)>>>(
      score, (int)L, (int)len_keep, mask, ids_restore, ids_shuffle);
  return check_launch("dkd_mask_rank");
}

int dkd_scale_if_not_one(void* x, int64_t n, void* x2, int64_t n2, int dtype, const float* scale, dkd_stream_t stream) {
  using namespace dkd;
  int rc = dkd_check_device();
  if (rc != DKD_OK) return rc;
  DKD_REQUIRE(n >= 0 && n2 >= 0 && scale != nullptr && (x != nullptr || n == 0) && (x2 != nullptr || n2 == 0), DKD_E_SHAPE,
              "dkd_scale_if_not_one: bad arguments");
  DKD_REQUIRE(dtype == DKD_F32 || dtype == DKD_BF16, DKD_E_DTYPE, "dkd_scale_if_not_one: dtype %d", dtype);
  if (n + n2 == 0) return DKD_OK;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  return dtype == DKD_F32 ? launch_scale<float>(x, n, x2, n2, scale, st) : launch_scale<__nv_bfloat16>(x, n, x2, n2, scale, st);
}

}  // extern "C"
