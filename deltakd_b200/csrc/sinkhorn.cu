// WassKD 'sinkhorn' term: debiased Sinkhorn divergence between the 196 aligned student tokens and the 196 teacher
// tokens of every (sample, layer) pair.
// Reference: model/loss.py:200-225 — a Python loop of B x 3 calls of geomloss.SamplesLoss("sinkhorn", blur=0.05)
// (p = 2, scaling = 0.5, debias, uniform weights, tensorized backend), each with a host read-back of the diameter,
// and its autograd backward.  geomloss is an unlisted, absent third-party dependency: the algorithm follows
// upstream geomloss 0.2.x as restated in oracle/sinkhorn.py (PARITY UNPINNED, DESIGN.md §4).
//
// Per layer, all on `stream`, no host read-back (the eps schedule is built on the device):
//   1-3. a = S W^T + b (tcgen05, fp32 rows) as in wass_l1.cu
//   4.   x = a, y = t[:, t_off:] -> bf16 hi/mid/lo planes; row square norms; per pair: bounding-box diameter -> eps ladder
//   5.   cost matrices C_xy, C_xx, C_yy = 0.5(|u|^2 + |v|^2) - u.v : batched tcgen05 GEMMs (6 plane products = fp32-exact operands), one 128 x 208
//        TMEM tile per (pair, matrix, half), written with a 204-float row pitch (the shared-memory image)
//   6.   Sinkhorn loops, cost matrix resident in shared memory (one bulk copy), potentials in registers:
//        xy kernel — one CTA per pair, a thread per row (f_ba) and a thread per column (g_ab) of C_xy;
//        sym kernel — one CTA per (pair, xx | yy), a thread per row.  Softmins are base-2 log-sum-exps
//        (one pass per step: online maximum + MUFU ex2; the symmetric problems use two threads per row).  The last (extrapolation) step also emits the transport plans
//        P = softmax_j(h_b - C_xy/eps), Q = softmax_j(h_a - C_xx/eps) as bf16 hi/lo planes.
//   7.   g_a = scale/N (Q x - P y): batched tcgen05 GEMM (K-major plans x MN-major points), written as planes
//   8-9. g_s = g_a W, g_W = g_a^T s, g_b = g_a^T 1 (align_ops.cuh)
// Bound: MUFU ex2 throughput and the eps-step latency (on-chip); HBM traffic is hidden behind it.
#include "align_ops.cuh"

namespace dkd {
namespace {

constexpr int kTok = 196;                   // points per cloud (14 x 14 patch tokens)
constexpr int kD = 384;                     // teacher width
constexpr int kLD = 200;                    // pitch of a cost matrix in floats, global and shared: with four threads per row (LDS.128,
                                            // float4 chunks [0,12) [12,25) [25,37) [37,49)) the 2 rows x 4 parts of a quarter warp hit the 8
                                            // distinct 16-byte bank groups (50 = 2 mod 8; part offsets 0, 4, 1, 5), and with four threads
                                            // per column (LDS.32, rows = part mod 4) a warp hits 32 distinct banks (200 = 8 mod 32)
constexpr int kLDxy = kLD;
constexpr int kLDsym = kLD;
constexpr int kCostBytes = kTok * kLD * 4;  // 156 800 (one bulk copy)
constexpr int kLDP = 208;                   // plan row pitch in bf16 (416 B)
constexpr int kMaxEps = 64;
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ------------------------------------------------------------------ 4. norms, diameter, eps ladder (one kernel, one pass)
struct PrepParams {
  const float* A;     // [B*196, 384] aligned student
  const void* t;      // teacher [B, Tt, 384]
  float *nx, *ny;     // [B*196]
  float* eps;         // [B][kMaxEps]
  int* n_eps;         // [B]
  int Tt, t_off, t_is_bf16;
  float blur, scaling;
};

__device__ __forceinline__ float ld_t(const void* t, int64_t idx, int is_bf16) {
  return is_bf16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(t)[idx]) : reinterpret_cast<const float*>(t)[idx];
}

// One CTA per pair, ONE pass over the pair's 196 aligned-student rows and 196 teacher rows: a warp takes every 12th row,
// a lane 12 of its 384 coordinates (three float4) — square norms of the rows (lane-local sums in a fixed order, then a warp
// sum) and, per coordinate, the bounding box of x u y -> diameter -> eps list (geomloss epsilon_schedule).
__global__ void __launch_bounds__(kD) sinkhorn_prep_kernel(PrepParams p) {
  constexpr int kWarps = kD / 32;
  __shared__ float s_mn[kWarps][kD], s_mx[kWarps][kD];
  __shared__ double red[kWarps];
  const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float mn[12], mx[12];
#pragma unroll
  for (int j = 0; j < 12; ++j) { mn[j] = INFINITY; mx[j] = -INFINITY; }
  for (int i = warp; i < kTok; i += kWarps) {
    const int64_t row = (int64_t)b * kTok + i;
    const int64_t trow = ((int64_t)b * p.Tt + p.t_off + i) * kD;
    float sx = 0.f, sy = 0.f;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int c = lane * 4 + 128 * k;
      float a[4], y[4];
      Vec<float, 4>::load(p.A + row * kD + c, a);
      if (p.t_is_bf16) Vec<__nv_bfloat16, 4>::load(reinterpret_cast<const __nv_bfloat16*>(p.t) + trow + c, y);
      else Vec<float, 4>::load(reinterpret_cast<const float*>(p.t) + trow + c, y);
      sx += a[0] * a[0] + a[1] * a[1] + a[2] * a[2] + a[3] * a[3];
      sy += y[0] * y[0] + y[1] * y[1] + y[2] * y[2] + y[3] * y[3];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        mn[4 * k + q] = fminf(mn[4 * k + q], fminf(a[q], y[q]));
        mx[4 * k + q] = fmaxf(mx[4 * k + q], fmaxf(a[q], y[q]));
      }
    }
    sx = warp_sum(sx); sy = warp_sum(sy);
    if (lane == 0) { p.nx[row] = sx; p.ny[row] = sy; }
  }
#pragma unroll
  for (int k = 0; k < 3; ++k)
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      s_mn[warp][lane * 4 + 128 * k + q] = mn[4 * k + q];
      s_mx[warp][lane * 4 + 128 * k + q] = mx[4 * k + q];
    }
  __syncthreads();
  const int d = threadIdx.x;
  float lo = s_mn[0][d], hi = s_mx[0][d];
#pragma unroll
  for (int w = 1; w < kWarps; ++w) { lo = fminf(lo, s_mn[w][d]); hi = fmaxf(hi, s_mx[w][d]); }
  double r = (double)(hi - lo) * (double)(hi - lo);
  r = warp_sum(r);
  if ((d & 31) == 0) red[d >> 5] = r;
  __syncthreads();
  if (d == 0) {
    double s = 0.0;
    for (int w = 0; w < kWarps; ++w) s += red[w];
    const double diam = (double)(float)sqrt(s);   // torch: fp32 .norm().item()
    float* e = p.eps + (size_t)b * kMaxEps;
    const double start = 2.0 * log(diam), stop = 2.0 * log((double)p.blur), step = 2.0 * log((double)p.scaling);
    int n = (int)ceil((stop - start) / step);      // len(np.arange(start, stop, step))
    if (!(n > 0)) n = 0;
    if (n > kMaxEps - 2) n = kMaxEps - 2;
    e[0] = (float)(diam * diam);
    for (int k = 0; k < n; ++k) e[1 + k] = (float)exp(start + k * step);
    e[1 + n] = p.blur * p.blur;
    p.n_eps[b] = n + 2;
  }
}

// ------------------------------------------------------------------ 5. cost matrices (gemm_tn policies)
// tile index mt = (pair*3 + which)*2 + half ; which: 0 = C_xy (x rows, y cols), 1 = C_xx, 2 = C_yy
using CostCfg = GemmCfg<208, 1, 4, 2>;

struct CostLoaderParams {
  CUtensorMap tmXa, tmXb, tmYa, tmYb;   // 4-D {384, 196, B, planes}; a: box {64,128,1,1}, b: box {64,208,1,1}
  int nterms;
};
struct CostLoader {
  using Params = CostLoaderParams;
  static constexpr uint32_t TX_BYTES = CostCfg::STAGE_BYTES;
  static __device__ __forceinline__ int num_k_iters(const Params& p) { return (kD / 64) * p.nterms; }
  static __device__ __forceinline__ void prefetch(const Params& p) {
    sm100::tma_prefetch_desc(&p.tmXa); sm100::tma_prefetch_desc(&p.tmXb);
    sm100::tma_prefetch_desc(&p.tmYa); sm100::tma_prefetch_desc(&p.tmYb);
  }
  static __device__ __forceinline__ void issue(const Params& p, int kit, int mt, int, uint8_t* sA, uint8_t* sB, uint64_t* bar) {
    const int term = kit / (kD / 64), kb = kit - term * (kD / 64);
    int pa, pb;
    term_planes(term, p.nterms, pa, pb);
    const int half = mt & 1, which = (mt >> 1) % 3, pair = mt / 6;
    sm100::tma_load_4d(sA, which == 2 ? &p.tmYa : &p.tmXa, bar, kb * 64, half * 128, pair, pa);
    sm100::tma_load_4d(sB, which == 1 ? &p.tmXb : &p.tmYb, bar, kb * 64, 0, pair, pb);
  }
};

struct CostEpiParams {
  const float *nx, *ny;
  float* C;   // [pairs][3][196][kLD]
};
struct CostEpi {
  using Params = CostEpiParams;
  struct State {};
  static __device__ __forceinline__ void init(const Params&, State&) {}
  static __device__ __forceinline__ void tile(const Params& p, State&, int m0, int, int row_in_tile, uint32_t t_acc) {
    const int mt = m0 >> 7;
    const int half = mt & 1, which = (mt >> 1) % 3, pair = mt / 6;
    const int i = half * 128 + row_in_tile;
    const bool live = i < kTok;
    const float* na = (which == 2 ? p.ny : p.nx) + (size_t)pair * kTok;
    const float* nb = (which == 1 ? p.nx : p.ny) + (size_t)pair * kTok;
    const float ni = live ? __ldg(na + i) : 0.f;
    float* out = p.C + (size_t)(pair * 3 + which) * kTok * kLD + (size_t)(live ? i : 0) * (which == 0 ? kLDxy : kLDsym);
#pragma unroll 1
    for (int c0 = 0; c0 < 192; c0 += 32) {
      float v[32];
      sm100::tmem_ld32(t_acc + c0, v);
      sm100::tmem_ld_wait();
      if (!live) continue;
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        const float4 n4 = __ldg(reinterpret_cast<const float4*>(nb + c0 + j));
        *reinterpret_cast<float4*>(out + c0 + j) = make_float4(0.5f * (ni + n4.x) - v[j], 0.5f * (ni + n4.y) - v[j + 1],
                                                               0.5f * (ni + n4.z) - v[j + 2], 0.5f * (ni + n4.w) - v[j + 3]);
      }
    }
    float v[32];
    sm100::tmem_ld32(t_acc + 176, v);   // columns 176..207: the last four real ones are v[16..19]
    sm100::tmem_ld_wait();
    if (live) {
      const float4 n4 = __ldg(reinterpret_cast<const float4*>(nb + 192));
      *reinterpret_cast<float4*>(out + 192) = make_float4(0.5f * (ni + n4.x) - v[16], 0.5f * (ni + n4.y) - v[17],
                                                          0.5f * (ni + n4.z) - v[18], 0.5f * (ni + n4.w) - v[19]);
    }
  }
  static __device__ __forceinline__ void finish(const Params&, State&, int) {}
};

// ------------------------------------------------------------------ 6. Sinkhorn loops
struct SinkParams {
  const float* C;          // [pairs][3][196][kLD]
  const float* eps;        // [pairs][kMaxEps]
  const int* n_eps;        // [pairs]
  __nv_bfloat16* plans;    // [2: Q, -P][planes = 2][pairs][196][kLDP]
  double* partials;        // [pairs*3]
  int pairs, write_plans;
};

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// bulk copy of one cost matrix into shared memory (thread 0 issues, everybody waits)
__device__ __forceinline__ void load_cost(float* sC, const float* gC, uint64_t* bar) {
  using namespace sm100;
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
    mbar_expect_tx(bar, kCostBytes);
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(sC)),
                 "l"(gC), "r"(kCostBytes), "r"(smem_u32(bar))
                 : "memory");
  }
  __syncthreads();
  mbar_wait(bar, 0);
}

// One-pass ("online") base-2 log-sum-exp.  Values v_j = h[j] - C[.][j]*c2 are produced in chunks of NV; the running
// maximum m and the sum s = sum 2^(v - m) are rescaled when a chunk raises the maximum (one extra ex2 per chunk) —
// each cost entry is read from shared memory once per eps step instead of twice.
struct Lse { float m, s; };
template <int NV>
__device__ __forceinline__ void lse_push(Lse& a, const float (&v)[NV]) {
  static_assert(NV % 4 == 0, "chunks of whole float4");
  float c0 = v[0], c1 = v[1], c2 = v[2], c3 = v[3];
#pragma unroll
  for (int q = 4; q < NV; q += 4) { c0 = fmaxf(c0, v[q]); c1 = fmaxf(c1, v[q + 1]); c2 = fmaxf(c2, v[q + 2]); c3 = fmaxf(c3, v[q + 3]); }
  const float mn = fmaxf(a.m, fmaxf(fmaxf(c0, c1), fmaxf(c2, c3)));
  float s0 = a.s * ex2f(a.m - mn), s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
  for (int q = 0; q < NV; q += 4) {
    s0 += ex2f(v[q + 0] - mn); s1 += ex2f(v[q + 1] - mn);
    s2 += ex2f(v[q + 2] - mn); s3 += ex2f(v[q + 3] - mn);
  }
  a.m = mn; a.s = (s0 + s1) + (s2 + s3);
}
__device__ __forceinline__ Lse lse_merge(const Lse& a, const Lse& b) {
  const float m = fmaxf(a.m, b.m);
  return Lse{m, a.s * ex2f(a.m - m) + b.s * ex2f(b.m - m)};
}
// the four lanes 4i .. 4i+3 hold the parts of one row (or column): everybody gets the whole
__device__ __forceinline__ Lse lse_merge4(Lse a) {
#pragma unroll
  for (int o = 1; o <= 2; o <<= 1) {
    Lse b;
    b.m = __shfl_xor_sync(0xffffffffu, a.m, o);
    b.s = __shfl_xor_sync(0xffffffffu, a.s, o);
    a = lse_merge(a, b);
  }
  return a;
}
// float4 chunks [k0, k1) of one row: groups of four chunks, then single chunks
__device__ __forceinline__ Lse lse2_row_part(const float* __restrict__ crow, const float* __restrict__ h, float c2, int k0, int k1) {
  const float4* c4 = reinterpret_cast<const float4*>(crow);
  const float4* h4 = reinterpret_cast<const float4*>(h);
  Lse a{-INFINITY, 0.f};
  int kb = k0;
#pragma unroll 1
  for (; kb + 4 <= k1; kb += 4) {
    float v[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 c = c4[kb + q], hh = h4[kb + q];
      v[4 * q] = fmaf(-c.x, c2, hh.x); v[4 * q + 1] = fmaf(-c.y, c2, hh.y);
      v[4 * q + 2] = fmaf(-c.z, c2, hh.z); v[4 * q + 3] = fmaf(-c.w, c2, hh.w);
    }
    lse_push(a, v);
  }
#pragma unroll 1
  for (; kb < k1; ++kb) {
    const float4 c = c4[kb], hh = h4[kb];
    const float v[4] = {fmaf(-c.x, c2, hh.x), fmaf(-c.y, c2, hh.y), fmaf(-c.z, c2, hh.z), fmaf(-c.w, c2, hh.w)};
    lse_push(a, v);
  }
  return a;
}
// rows part, part + 4, part + 8, ... (49 of them) of column j of C_xy; hp = this part's slice of the part-major h vector
__device__ __forceinline__ Lse lse2_col_part(const float* __restrict__ ccol, const float* __restrict__ hp, float c2) {
  const float4* h4 = reinterpret_cast<const float4*>(hp);
  Lse a{-INFINITY, 0.f};
#pragma unroll 1
  for (int q0 = 0; q0 < 48; q0 += 16) {
    float v[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 hh = h4[(q0 >> 2) + q];
      const float* c = ccol + (size_t)(q0 + 4 * q) * 4 * kLDxy;
      v[4 * q] = fmaf(-c[0], c2, hh.x); v[4 * q + 1] = fmaf(-c[4 * kLDxy], c2, hh.y);
      v[4 * q + 2] = fmaf(-c[8 * kLDxy], c2, hh.z); v[4 * q + 3] = fmaf(-c[12 * kLDxy], c2, hh.w);
    }
    lse_push(a, v);
  }
  const float last = fmaf(-ccol[(size_t)48 * 4 * kLDxy], c2, hp[48]);
  return lse_merge(a, Lse{last, 1.f});
}

// plan row segment:  sign * 2^(h[j] - C[i][j]*c2 - m) / s  as bf16 hi / lo, float4 chunks [k0, k1), 8-byte stores
__device__ __forceinline__ void write_plan_part(const float* __restrict__ crow, const float* __restrict__ h, float c2, float m, float s,
                                                float sign, __nv_bfloat16* hi, __nv_bfloat16* lo, int k0, int k1) {
  const float4* c4 = reinterpret_cast<const float4*>(crow);
  const float4* h4 = reinterpret_cast<const float4*>(h);
  const float inv = sign / s;
#pragma unroll 4
  for (int k = k0; k < k1; ++k) {
    const float4 c = c4[k], hh = h4[k];
    float v[4], r[4];
    v[0] = inv * ex2f(fmaf(-c.x, c2, hh.x) - m); v[1] = inv * ex2f(fmaf(-c.y, c2, hh.y) - m);
    v[2] = inv * ex2f(fmaf(-c.z, c2, hh.z) - m); v[3] = inv * ex2f(fmaf(-c.w, c2, hh.w) - m);
#pragma unroll
    for (int q = 0; q < 4; ++q) r[q] = v[q] - __bfloat162float(__float2bfloat16_rn(v[q]));
    Vec<__nv_bfloat16, 4>::store(hi + 4 * k, v);
    Vec<__nv_bfloat16, 4>::store(lo + 4 * k, r);
  }
}

constexpr int kSinkThreads = 800;   // 25 warps: four threads per row — and, for C_xy, the same four per column
constexpr int kHP = 52;             // part-major h vector: [4][52] (49 used)
constexpr size_t kSinkSmem = (size_t)kCostBytes + (2 * kTok + 2 * 4 * kHP + kMaxEps) * sizeof(float) + 64;

// Step schedule (geomloss sinkhorn_loop): step -1 initialises the potentials at eps[0] from the log-weights alone,
// steps 0..n-1 average (symmetric update) at eps[k], step n is the final extrapolation at eps[n-1] (plain assignment).
//   XY  : one CTA per pair, cost C_xy; lanes 4i .. 4i+3 own row i (f_ba[i], a quarter of the row each) AND column i
//         (g_ab[i], rows = lane mod 4): every thread does the same work, 98 cost entries per eps step
//   !XY : one CTA per (pair, xx | yy); lanes 4i .. 4i+3 own row i (f_aa or g_bb)
// ncu of the previous layout (one thread per row / column, 14 warps, the 7th warp of each role nearly empty): XU pipe
// 54 % busy, top stalls MIO throttle (MUFU and LDS share the queue; the column threads issued 2 LDS per entry), wait,
// barrier (row warps waiting for the slower column warps) and long scoreboard (eps read from global memory each step).
template <bool XY>
__global__ void __launch_bounds__(kSinkThreads, 1) sinkhorn_kernel(SinkParams p) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  float* sC = reinterpret_cast<float*>(smem_raw);
  float* hR = sC + kTok * kLD;            // [2][196]     : h over columns j (from g_ab; xx, yy: from the potential itself), read by the row work
  float* hC = hR + 2 * kTok;              // [2][4][kHP]  : h over rows i (from f_ba), part-major: entry i at [i & 3][i >> 2]; read by the column work
  float* s_eps = hC + 2 * 4 * kHP;        // [kMaxEps]
  uint64_t* bar = reinterpret_cast<uint64_t*>(s_eps + kMaxEps);
  __shared__ double red[32];
  constexpr int LD = kLD;

  const int pair = XY ? blockIdx.x : blockIdx.x >> 1;
  const int which = XY ? 0 : 1 + (blockIdx.x & 1);
  const int n = p.n_eps[pair];
  if ((int)threadIdx.x < kMaxEps) s_eps[threadIdx.x] = p.eps[(size_t)pair * kMaxEps + threadIdx.x];
  if ((int)threadIdx.x < 2 * 4 * kHP) hC[threadIdx.x] = 0.f;
  load_cost(sC, p.C + (size_t)(pair * 3 + which) * kTok * kLD, bar);   // (contains the __syncthreads that publishes s_eps)

  const int idx = threadIdx.x >> 2, part = threadIdx.x & 3;   // row (and column) idx, quarter `part`
  const int k0 = part == 0 ? 0 : (part == 1 ? 12 : (part == 2 ? 25 : 37));
  const int k1 = part == 0 ? 12 : (part == 1 ? 25 : (part == 2 ? 37 : 49));
  const bool active = idx < kTok;
  const int row = active ? idx : 0;       // idle lanes of the last warp walk row 0 (results unused)
  const float logw = -__logf((float)kTok);
  float pot_f = 0.f, pot_g = 0.f;         // f_ba[idx] and (xy) g_ab[idx]; xx / yy: the one potential in pot_f
  Lse fin{0.f, 1.f};
  float c2_fin = 0.f;

  for (int step = -1; step <= n; ++step) {
    const float eps = s_eps[step < 0 ? 0 : (step < n ? step : n - 1)];
    const float inv_eps = 1.f / eps;
    const int buf = (step + 1) & 1;
    // the potentials become entries of the h vectors the other side reads (same side for the symmetric problems)
    if (active) {
      if (XY) {
        if (part == 0) hR[buf * kTok + idx] = (logw + (step < 0 ? 0.f : pot_g * inv_eps)) * kLog2e;
        if (part == 1) hC[(buf * 4 + (idx & 3)) * kHP + (idx >> 2)] = (logw + (step < 0 ? 0.f : pot_f * inv_eps)) * kLog2e;
      } else if (part == 0) {
        hR[buf * kTok + idx] = (logw + (step < 0 ? 0.f : pot_f * inv_eps)) * kLog2e;
      }
    }
    __syncthreads();
    const float c2 = kLog2e * inv_eps;
    const Lse a = lse_merge4(lse2_row_part(sC + row * LD, hR + buf * kTok, c2, k0, k1));
    fin = a; c2_fin = c2;
    const float upd_f = -eps * kLn2 * (a.m + __log2f(a.s));
    pot_f = (step < 0 || step == n) ? upd_f : 0.5f * (pot_f + upd_f);
    if (XY) {
      const Lse b = lse_merge4(lse2_col_part(sC + part * LD + row, hC + (buf * 4 + part) * kHP, c2));
      const float upd_g = -eps * kLn2 * (b.m + __log2f(b.s));
      pot_g = (step < 0 || step == n) ? upd_g : 0.5f * (pot_g + upd_g);
    }
  }

  // divergence partial: xy -> +(sum f_ba + sum g_ab)/N ; xx, yy -> -(sum f)/N
  double acc = (active && part == 0) ? (double)pot_f + (XY ? (double)pot_g : 0.0) : 0.0;
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
    p.partials[pair * 3 + which] = (XY ? s : -s) / (double)kTok;
  }
  // transport plans of the last step (rows only): -P from C_xy, Q from C_xx
  if (p.write_plans && active && which != 2) {
    const int mat = XY ? 1 : 0;
    const size_t plane = (size_t)p.pairs * kTok * kLDP;
    __nv_bfloat16* hi = p.plans + ((size_t)mat * 2 * p.pairs + pair) * kTok * kLDP + (size_t)idx * kLDP;
    write_plan_part(sC + idx * LD, hR + ((n + 1) & 1) * kTok, c2_fin, fin.m, fin.s, XY ? -1.f : 1.f, hi, hi + plane, k0, k1);
  }
}

// ------------------------------------------------------------------ 7. g_a = alpha (Q x - P y)  (gemm_nt, K-major A)
using GradCfg = GemmNtCfg<6, false, 256, 128, 3, 64, true>;

struct PlanLoaderParams {
  CUtensorMap tmPlan;    // 4-D {196 (pitch kLDP), 196, pairs, 4 = mat*2 + plane}, box {64,128,1,1}
  CUtensorMap tmX, tmY;  // 4-D {384, 196, pairs, 2}, box {64,64,1,1}
  int pairs;
};
struct PlanLoader {
  using Params = PlanLoaderParams;
  using Item = NtItem;
  static constexpr uint32_t TX_BYTES = GradCfg::STAGE_BYTES;
  static __device__ __forceinline__ int num_items(const Params& p) { return p.pairs * 2; }
  static __device__ __forceinline__ void prefetch(const Params& p) {
    sm100::tma_prefetch_desc(&p.tmPlan); sm100::tma_prefetch_desc(&p.tmX); sm100::tma_prefetch_desc(&p.tmY);
  }
  static __device__ __forceinline__ void decode(const Params&, int item, Item& it) {
    const int pair = item >> 1, half = item & 1;
    it.rb0 = 0; it.rb1 = 8;                 // 4 k-blocks of Q.x then 4 of (-P).y
    it.a_col0 = half * 128; it.b_col0 = 0;
    it.d_off = ((int64_t)pair * kTok + half * 128) * kD;
    it.dcol_off = -1; it.aux = pair;
    it.rows = half ? kTok - 128 : 128;
  }
  static __device__ __forceinline__ void issue(const Params& p, const Item& it, int term, int nterms, int rb, uint8_t* a, uint8_t* b, uint64_t* bar) {
    int pa, pb;
    term_planes(term, nterms, pa, pb);
    const int src = rb >> 2, kb = rb & 3;
    sm100::tma_load_4d(a, &p.tmPlan, bar, kb * 64, it.a_col0, it.aux, src * 2 + pa);
    const CUtensorMap* mb = src ? &p.tmY : &p.tmX;
#pragma unroll
    for (int i = 0; i < 6; ++i) sm100::tma_load_4d(b + (size_t)i * GradCfg::BOX_BYTES, mb, bar, i * 64, kb * 64, it.aux, pb);
  }
};

struct Workspace {
  __nv_bfloat16 *S, *Wp, *Wt, *ones, *Xp, *Yp, *plans, *G;
  float *A, *nx, *ny, *C, *eps;
  int* n_eps;
  double* partials;
  float* wpart;   // deterministic mode: per-split weight-gradient slots (align_wgrad), appended last
  size_t bytes;
};
Workspace carve(void* base, int64_t B, int Ds, int Dt, int P, bool det) {
  Workspace w;
  const int64_t M = B * kTok;
  size_t off = 0;
  auto take = [&](size_t n) { size_t o = off; off = align_up(off + n, 1024); return reinterpret_cast<char*>(base) + o; };
  w.S = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * M * Ds * 2));
  w.Wp = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * Dt * Ds * 2));
  w.Wt = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * Dt * Ds * 2));
  w.ones = reinterpret_cast<__nv_bfloat16*>(take((size_t)2 * 64 * 64 * 2));
  w.A = reinterpret_cast<float*>(take((size_t)M * Dt * 4));
  w.Xp = reinterpret_cast<__nv_bfloat16*>(take((size_t)3 * M * Dt * 2));
  w.Yp = reinterpret_cast<__nv_bfloat16*>(take((size_t)3 * M * Dt * 2));
  w.G = reinterpret_cast<__nv_bfloat16*>(take((size_t)2 * M * Dt * 2));
  w.nx = reinterpret_cast<float*>(take((size_t)M * 4));
  w.ny = reinterpret_cast<float*>(take((size_t)M * 4));
  w.C = reinterpret_cast<float*>(take((size_t)B * 3 * kCostBytes));
  w.plans = reinterpret_cast<__nv_bfloat16*>(take((size_t)4 * B * kTok * kLDP * 2));
  w.eps = reinterpret_cast<float*>(take((size_t)B * kMaxEps * 4));
  w.n_eps = reinterpret_cast<int*>(take((size_t)B * 4));
  w.partials = reinterpret_cast<double*>(take((size_t)B * 3 * sizeof(double)));
  w.wpart = det ? reinterpret_cast<float*>(take(align_wgrad_part_bytes(B * kTok, Ds, Dt, P))) : nullptr;
  w.bytes = off;
  return w;
}

int make_cloud_tmap(CUtensorMap* out, const void* base, int64_t B, int box_rows, const char* what) {
  const int64_t M = B * kTok;
  const uint64_t dims[4] = {(uint64_t)kD, (uint64_t)kTok, (uint64_t)B, 3};
  const uint64_t strides[3] = {(uint64_t)kD * 2, (uint64_t)kTok * kD * 2, (uint64_t)M * kD * 2};
  const uint32_t box[4] = {64, (uint32_t)box_rows, 1, 1};
  return make_tmap_bf16(out, base, 4, dims, strides, box, what);
}

}  // namespace
}  // namespace dkd

extern "C" {

size_t dkd_wass_sinkhorn_workspace_bytes(int64_t B, int n_tok, int Ds, int Dt, int precision) {
  (void)n_tok;
  return dkd::carve(nullptr, B, Ds, Dt, dkd::prec_planes(precision), dkd::prec_deterministic(precision)).bytes;
}

int dkd_wass_sinkhorn_fwdbwd(const void* s, const void* t, const float* W, const float* bias, int64_t B, int Ts, int s_off, int Tt,
                             int t_off, int n_tok, int Ds, int Dt, int dtype, int precision, float scale, void* g_s, float* g_W,
                             float* g_b, float* loss, void* workspace, size_t workspace_bytes, dkd_stream_t stream) {
  using namespace dkd;
  int rc = dkd_check_device();
  if (rc != DKD_OK) return rc;
  const char* fn = "dkd_wass_sinkhorn_fwdbwd";
  DKD_REQUIRE(dtype == DKD_F32 || dtype == DKD_BF16, DKD_E_DTYPE, "%s: dtype %d", fn, dtype);
  DKD_REQUIRE(prec_valid(precision), DKD_E_UNSUPPORTED, "%s: precision %d", fn, precision);
  DKD_REQUIRE(n_tok == kTok, DKD_E_SHAPE, "%s: built for %d patch tokens per sample, got %d", fn, kTok, n_tok);
  DKD_REQUIRE(B > 0 && s_off >= 0 && t_off >= 0 && Ts >= s_off + n_tok && Tt >= t_off + n_tok, DKD_E_SHAPE, "%s: bad token geometry", fn);
  DKD_REQUIRE(Ds == 192 && Dt == kD, DKD_E_SHAPE, "%s: built for widths 192 -> 384, got %d -> %d", fn, Ds, Dt);
  DKD_REQUIRE(s && t && W && loss && workspace, DKD_E_SHAPE, "%s: null pointer", fn);
  DKD_REQUIRE((((uintptr_t)workspace) & 1023) == 0, DKD_E_ALIGN, "%s: workspace must be 1024-byte aligned", fn);
  DKD_REQUIRE((((uintptr_t)s | (uintptr_t)t | (uintptr_t)g_s) & 31) == 0, DKD_E_ALIGN, "%s: s, t and g_s must be 32-byte aligned (256-bit accesses)", "dkd_wass_sinkhorn_fwdbwd");
  DKD_REQUIRE(B * 6 < (1ll << 24), DKD_E_SHAPE, "%s: too many samples", fn);
  const int P = prec_planes(precision);
  const int64_t M = B * kTok;
  Workspace ws = carve(workspace, B, Ds, Dt, P, prec_deterministic(precision));
  DKD_REQUIRE(workspace_bytes >= ws.bytes, DKD_E_WORKSPACE, "%s: workspace %zu < %zu", fn, workspace_bytes, ws.bytes);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const bool want_grads = g_s || g_W || g_b;
  const int pairs = (int)B;

  // 1-3. aligned student rows (fp32)
  rc = launch_tokens_to_planes(s, dtype, B, Ts, s_off, n_tok, Ds, P, nullptr, ws.S, st);
  if (rc != DKD_OK) return rc;
  rc = launch_weight_to_planes(W, Dt, Ds, P, ws.Wp, want_grads ? ws.Wt : nullptr, st);
  if (rc != DKD_OK) return rc;
  rc = align_forward_rows(ws.S, ws.Wp, bias, ws.A, M, Ds, Dt, P, st, "dkd_wass_sinkhorn_fwdbwd: align GEMM");
  if (rc != DKD_OK) return rc;

  // 4. point-cloud planes, norms, eps ladders
  rc = launch_tokens_to_planes(ws.A, DKD_F32, B, kTok, 0, kTok, Dt, 3, nullptr, ws.Xp, st);
  if (rc != DKD_OK) return rc;
  rc = launch_tokens_to_planes(t, dtype, B, Tt, t_off, kTok, Dt, 3, nullptr, ws.Yp, st);
  if (rc != DKD_OK) return rc;
  PrepParams pp;
  pp.A = ws.A; pp.t = t; pp.nx = ws.nx; pp.ny = ws.ny; pp.eps = ws.eps; pp.n_eps = ws.n_eps;
  pp.Tt = Tt; pp.t_off = t_off; pp.t_is_bf16 = dtype == DKD_BF16; pp.blur = 0.05f; pp.scaling = 0.5f;
  sinkhorn_prep_kernel<<<pairs, kD, 0, st>>>(pp);
  rc = check_launch("dkd_wass_sinkhorn_fwdbwd: norms, eps ladder");
  if (rc != DKD_OK) return rc;

  {  // 5. cost matrices
    using Cfg = CostCfg;
    GemmParams<CostLoader, CostEpi> p;
    rc = make_cloud_tmap(&p.ld.tmXa, ws.Xp, B, 128, "sinkhorn x (rows)");
    if (rc != DKD_OK) return rc;
    rc = make_cloud_tmap(&p.ld.tmXb, ws.Xp, B, 208, "sinkhorn x (cols)");
    if (rc != DKD_OK) return rc;
    rc = make_cloud_tmap(&p.ld.tmYa, ws.Yp, B, 128, "sinkhorn y (rows)");
    if (rc != DKD_OK) return rc;
    rc = make_cloud_tmap(&p.ld.tmYb, ws.Yp, B, 208, "sinkhorn y (cols)");
    if (rc != DKD_OK) return rc;
    p.ld.nterms = 6;   // fp32-exact operands: at eps = blur^2 the plans react to cost errors of ~1e-4 (bf16x3 gives ~1e-3)
    p.ep.nx = ws.nx; p.ep.ny = ws.ny; p.ep.C = ws.C;
    p.m_tiles = pairs * 6; p.n_tiles = 1;
    const int grid = min(kNumSMs, p.m_tiles);
    auto kern = gemm_tn_kernel<Cfg, CostLoader, CostEpi>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
    kern<<<grid, Cfg::THREADS, Cfg::SMEM, st>>>(p);
    rc = check_launch("dkd_wass_sinkhorn_fwdbwd: cost GEMM");
    if (rc != DKD_OK) return rc;
  }
  {  // 6. Sinkhorn loops
    SinkParams sp;
    sp.C = ws.C; sp.eps = ws.eps; sp.n_eps = ws.n_eps; sp.plans = ws.plans; sp.partials = ws.partials;
    sp.pairs = pairs; sp.write_plans = want_grads;
    cudaFuncSetAttribute(sinkhorn_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSinkSmem);
    cudaFuncSetAttribute(sinkhorn_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSinkSmem);
    sinkhorn_kernel<true><<<pairs, kSinkThreads, kSinkSmem, st>>>(sp);
    rc = check_launch("dkd_wass_sinkhorn_fwdbwd: sinkhorn xy");
    if (rc != DKD_OK) return rc;
    sinkhorn_kernel<false><<<pairs * 2, kSinkThreads, kSinkSmem, st>>>(sp);
    rc = check_launch("dkd_wass_sinkhorn_fwdbwd: sinkhorn xx/yy");
    if (rc != DKD_OK) return rc;
    rc = launch_fold_partials(ws.partials, pairs * 3, scale, loss, st);
    if (rc != DKD_OK) return rc;
  }
  if (!want_grads) return DKD_OK;

  {  // 7. g_a planes
    using Cfg = GradCfg;
    GemmNtParamsT<Cfg, PlanLoader> p;
    {
      const uint64_t dims[4] = {(uint64_t)kTok, (uint64_t)kTok, (uint64_t)B, 4};
      const uint64_t strides[3] = {(uint64_t)kLDP * 2, (uint64_t)kTok * kLDP * 2, (uint64_t)B * kTok * kLDP * 2};
      const uint32_t box[4] = {64, 128, 1, 1};
      rc = make_tmap_bf16(&p.ld.tmPlan, ws.plans, 4, dims, strides, box, "sinkhorn plans");
      if (rc != DKD_OK) return rc;
    }
    rc = make_cloud_tmap(&p.ld.tmX, ws.Xp, B, 64, "sinkhorn x (k rows)");
    if (rc != DKD_OK) return rc;
    rc = make_cloud_tmap(&p.ld.tmY, ws.Yp, B, 64, "sinkhorn y (k rows)");
    if (rc != DKD_OK) return rc;
    p.ld.pairs = pairs;
    p.nterms = 3;
    p.ep.D = nullptr; p.ep.Dcol = nullptr; p.ep.ldd = kD; p.ep.alpha = scale / (float)kTok;
    p.ep.Dplanes = ws.G; p.ep.plane_stride = M * kD; p.ep.n_planes = 2;
    const int grid = min(kNumSMs, pairs * 2);
    auto kern = gemm_nt_kernel<Cfg, PlanLoader>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
    kern<<<grid, Cfg::THREADS, Cfg::SMEM, st>>>(p);
    rc = check_launch("dkd_wass_sinkhorn_fwdbwd: plan GEMM");
    if (rc != DKD_OK) return rc;
  }
  // 8-9. through the alignment head (G planes are laid out [2][M][Dt]; a one-pass run reads the hi plane only)
  if (g_s) {
    rc = align_dgrad(ws.G, ws.Wt, g_s, M, n_tok, Ts, s_off, Ds, Dt, P, dtype == DKD_BF16, 1.f, st, "dkd_wass_sinkhorn_fwdbwd: dgrad GEMM");
    if (rc != DKD_OK) return rc;
  }
  if (g_W || g_b) {
    DKD_REQUIRE(g_W != nullptr, DKD_E_UNSUPPORTED, "%s: g_b without g_W is not supported", fn);
    rc = align_wgrad(ws.G, ws.S, ws.ones, g_W, g_b, M, Ds, Dt, P, 1.f, st, "dkd_wass_sinkhorn_fwdbwd: wgrad GEMM", 0, ws.wpart);
    if (rc != DKD_OK) return rc;
  }
  return DKD_OK;
}

}  // extern "C"
