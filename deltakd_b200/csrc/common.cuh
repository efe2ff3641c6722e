// Shared device/host helpers for libdeltakd_sm100 (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/deltakd.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libdeltakd_sm100 is written for sm_100a (B200) only"
#endif

namespace dkd {

// ---- error plumbing (host) -------------------------------------------------
void set_error(const char* fmt, ...);
int check_launch(const char* what);  // cudaGetLastError -> DKD_E_LAUNCH

#define DKD_REQUIRE(cond, code, ...)  \
  do {                                \
    if (!(cond)) {                    \
      ::dkd::set_error(__VA_ARGS__);  \
      return (code);                  \
    }                                 \
  } while (0)

constexpr int kNumSMs = 148;  // B200

// ---- programmatic dependent launch ---------------------------------------------
// A kernel launched by launch_pdl may start while its predecessor on the stream is still running (its CTAs are resident
// and have called grid_dep_launch, or have exited), so launch latency and prologue overlap the predecessor's tail.  It
// must call grid_dep_wait before its first global-memory access: the wait returns once the predecessor grid has
// completed and its writes are visible.  Both are no-ops for a kernel launched without the attribute.
__device__ __forceinline__ void grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void grid_dep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = 0;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, args...);
}

// ---- element access ----------------------------------------------------------
template <typename T> struct Elt;
template <> struct Elt<float> {
  static __device__ __forceinline__ float ld(const float* p) { return *p; }
  static __device__ __forceinline__ void st(float* p, float v) { *p = v; }
};
template <> struct Elt<__nv_bfloat16> {
  static __device__ __forceinline__ float ld(const __nv_bfloat16* p) { return __bfloat162float(*p); }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
};

// VEC consecutive elements <-> fp32 registers with one 4/8/16-byte access.
template <typename T, int VEC> struct Vec {
  static_assert(VEC == 1 || VEC == 2 || VEC == 4 || VEC == 8, "VEC");
  static __device__ __forceinline__ void load(const T* p, float (&v)[VEC]) {
    constexpr int BYTES = VEC * (int)sizeof(T);
    if constexpr (BYTES == 16) {
      uint4 r = *reinterpret_cast<const uint4*>(p);
      unpack<4>(reinterpret_cast<const uint32_t*>(&r), v);
    } else if constexpr (BYTES == 8) {
      uint2 r = *reinterpret_cast<const uint2*>(p);
      unpack<2>(reinterpret_cast<const uint32_t*>(&r), v);
    } else if constexpr (BYTES == 4) {
      uint32_t r = *reinterpret_cast<const uint32_t*>(p);
      unpack<1>(&r, v);
    } else {
#pragma unroll
      for (int i = 0; i < VEC; ++i) v[i] = Elt<T>::ld(p + i);
    }
  }
  static __device__ __forceinline__ void store(T* p, const float (&v)[VEC]) {
    constexpr int BYTES = VEC * (int)sizeof(T);
    if constexpr (BYTES == 16) {
      uint4 r;
      pack<4>(v, reinterpret_cast<uint32_t*>(&r));
      *reinterpret_cast<uint4*>(p) = r;
    } else if constexpr (BYTES == 8) {
      uint2 r;
      pack<2>(v, reinterpret_cast<uint32_t*>(&r));
      *reinterpret_cast<uint2*>(p) = r;
    } else if constexpr (BYTES == 4) {
      uint32_t r;
      pack<1>(v, &r);
      *reinterpret_cast<uint32_t*>(p) = r;
    } else {
#pragma unroll
      for (int i = 0; i < VEC; ++i) Elt<T>::st(p + i, v[i]);
    }
  }

 private:
  template <int WORDS>
  static __device__ __forceinline__ void unpack(const uint32_t* w, float (&v)[VEC]) {
    if constexpr (sizeof(T) == 4) {
#pragma unroll
      for (int i = 0; i < WORDS; ++i) v[i] = __uint_as_float(w[i]);
    } else {
#pragma unroll
      for (int i = 0; i < WORDS; ++i) {  // bf16 -> fp32 is a 16-bit shift
        v[2 * i] = __uint_as_float(w[i] << 16);
        v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
      }
    }
  }
  template <int WORDS>
  static __device__ __forceinline__ void pack(const float (&v)[VEC], uint32_t* w) {
    if constexpr (sizeof(T) == 4) {
#pragma unroll
      for (int i = 0; i < WORDS; ++i) w[i] = __float_as_uint(v[i]);
    } else {
#pragma unroll
      for (int i = 0; i < WORDS; ++i) {
        __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
        w[i] = *reinterpret_cast<uint32_t*>(&h);
      }
    }
  }
};

// ---- 256-bit global accesses (sm_100: LDG/STG.E.256).  A thread that owns a contiguous run of a row moves it in
// 32-byte pieces: half the instructions and L1 wavefronts of 16-byte accesses, and every store fills a whole sector.
__device__ __forceinline__ void ldg256(const float* p, float (&v)[8]) {
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
               : "l"(p));
}
__device__ __forceinline__ void stg256(float* p, const float (&v)[8]) {
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]),
               "f"(v[5]), "f"(v[6]), "f"(v[7])
               : "memory");
}
// 16 bf16 <-> 16 fp32
__device__ __forceinline__ void ldg256(const __nv_bfloat16* p, float (&v)[16]) {
  uint32_t w[8];
  asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7])
               : "l"(p));
#pragma unroll
  for (int i = 0; i < 8; ++i) { v[2 * i] = __uint_as_float(w[i] << 16); v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u); }
}
__device__ __forceinline__ void stg256(__nv_bfloat16* p, const float (&v)[16]) {
  uint32_t w[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]); w[i] = *reinterpret_cast<uint32_t*>(&h); }
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]),
               "r"(w[5]), "r"(w[6]), "r"(w[7])
               : "memory");
}

// 32 consecutive fp32 of a small read-only vector (bias, mask token): every thread of the warp reads the same
// 128 bytes, so 8 broadcast 16-byte loads replace 32 scalar ones.  `p` may be null (-> zeros).
__device__ __forceinline__ void ldg_vec32(const float* p, float (&x)[32]) {
  if (p == nullptr) {
#pragma unroll
    for (int j = 0; j < 32; ++j) x[j] = 0.f;
    return;
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 w = __ldg(reinterpret_cast<const float4*>(p) + j);
    x[4 * j] = w.x; x[4 * j + 1] = w.y; x[4 * j + 2] = w.z; x[4 * j + 3] = w.w;
  }
}

// fp32 x[32] -> bf16 hi (and lo = x - hi) planes, 64 contiguous bytes each
__device__ __forceinline__ void store_planes32(__nv_bfloat16* hi_ptr, int64_t plane_stride, int planes, float (&x)[32]) {
  stg256(hi_ptr, *reinterpret_cast<float(*)[16]>(&x[0]));
  stg256(hi_ptr + 16, *reinterpret_cast<float(*)[16]>(&x[16]));
  if (planes == 2) {
    float lo[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) lo[j] = x[j] - __bfloat162float(__float2bfloat16_rn(x[j]));
    stg256(hi_ptr + plane_stride, *reinterpret_cast<float(*)[16]>(&lo[0]));
    stg256(hi_ptr + plane_stride + 16, *reinterpret_cast<float(*)[16]>(&lo[16]));
  }
}

// ---- packed fp32 pairs (sm_100: FFMA2 / FADD2 / FMUL2 — two IEEE fp32 operations per issued instruction) ----------
// For issue-bound elementwise kernels: the arithmetic is bit-identical to the scalar fmaf / + / *.
__device__ __forceinline__ unsigned long long f2_pack(float x, float y) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(x), "f"(y));
  return r;
}
__device__ __forceinline__ float2 f2_unpack(unsigned long long r) {
  float2 v;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(v.x), "=f"(v.y) : "l"(r));
  return v;
}
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
  unsigned long long r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(f2_pack(a.x, a.y)), "l"(f2_pack(b.x, b.y)), "l"(f2_pack(c.x, c.y)));
  return f2_unpack(r);
}
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
  unsigned long long r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2_pack(a.x, a.y)), "l"(f2_pack(b.x, b.y)));
  return f2_unpack(r);
}
__device__ __forceinline__ float2 sub2(float2 a, float2 b) {
  unsigned long long r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2_pack(a.x, a.y)), "l"(f2_pack(b.x, b.y)));
  return f2_unpack(r);
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
  unsigned long long r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2_pack(a.x, a.y)), "l"(f2_pack(b.x, b.y)));
  return f2_unpack(r);
}
__device__ __forceinline__ float2 splat2(float x) { return make_float2(x, x); }

// ---- reductions ----------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum of K values at once; result valid in every thread. `scratch` holds >= K*32 floats.
template <int K, int THREADS>
__device__ __forceinline__ void block_sum(float (&v)[K], float* scratch) {
  constexpr int WARPS = THREADS / 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k) v[k] = warp_sum(v[k]);
  if constexpr (THREADS == 32) return;   // a single warp owns the data: no shared memory, no barrier
  __syncthreads();  // protect scratch reuse
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < K; ++k) scratch[k * WARPS + warp] = v[k];
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < K; ++k) {
    float a = 0.f;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) a += scratch[k * WARPS + w];
    v[k] = a;
  }
}
template <int K, int THREADS>
__device__ __forceinline__ void block_max(float (&v)[K], float* scratch) {
  constexpr int WARPS = THREADS / 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k) v[k] = warp_max(v[k]);
  if constexpr (THREADS == 32) return;
  __syncthreads();
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < K; ++k) scratch[k * WARPS + warp] = v[k];
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < K; ++k) {
    float a = -INFINITY;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) a = fmaxf(a, scratch[k * WARPS + w]);
    v[k] = a;
  }
}

}  // namespace dkd
