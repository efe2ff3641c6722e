// WassKD 'l1' term: sorted-L1 (1-D Wasserstein) distance per (sample, channel) over the token axis.
// Reference: model/loss.py:187-199 —
//     a = align_wasskd[i](student[i][:, 1:]);  sort(a, dim=1), sort(teacher[i][:, 2:], dim=1);  mean|diff|
// and its autograd backward: g_a[b, pi(r), d] = sign(sorted_a[b,r,d] - sorted_t[b,r,d]) / numel, with pi the
// student sort permutation.
//
//   1-2. operand planes (S, W) as in align_mse.cu
//   3.   a = S W^T + b  (gemm_tn, fp32 rows to scratch)
//   4.   sort kernel: one CTA per (sample, 32-channel group); the [n_tok x 32] student and teacher tiles are
//        staged (transposed) in shared memory from coalesced 128-byte rows; 4 adjacent lanes sort one column with
//        a 256-wide keys-only bitonic network held in registers (64 keys per lane: 33 of the 36 stages are
//        in-register FMNMX pairs, 3 use warp shuffles); the permutation is recovered by a binary search of each
//        student value in its sorted column (duplicates ordered by token index); |diff| is block-reduced and
//        sign(diff) goes back through shared memory so the +-1 gradient plane is written with full rows.
//   5-6. g_s = c * G W, g_W = c * G^T S, g_b = c * G^T 1  (tcgen05; c = scale folded into the epilogues)
// The sort is on-chip (shared memory + registers): HBM traffic is the a/t tile reads and the +-1 plane write.
#include "align_ops.cuh"

namespace dkd {
namespace {

constexpr int kSortThreads = 128;   // 4 warps x 4 columns x 8 lanes
constexpr int kCh = 16;             // channels (columns) per CTA
constexpr int kMaxTok = 256;        // bitonic width
constexpr int kPerLane = 32;        // keys per lane: a column is held by 8 adjacent lanes
constexpr int kQuad = kMaxTok / kPerLane;   // 8 lanes per column
constexpr int kSearchIlp = 4;

// Keys-only bitonic sort of 256 floats held by 8 adjacent lanes (sorted position e = sub*32 + r, sub = lane & 7).
// Strides below 32 are in-register compare-exchanges (two FMNMX, 30 stages); strides 32/64/128 (6 stages) cross
// lanes by shuffle.  Descending sub-sequences (phases k = 32, 64, 128 on the lanes whose position has bit k set) are run
// as ascending ones on negated keys, so every compare-exchange has a compile-time direction.  Ascending on exit;
// ties need no order (equal keys are interchangeable in the sorted sequence).
__device__ __forceinline__ void bitonic256_oct(float (&key)[kPerLane], int sub) {
#pragma unroll
  for (int k = 2; k <= 256; k <<= 1) {
    // sign flips as multiplications by +-1 (exact): FMUL runs on the FMA pipe — the kernel is bound by the ALU pipe
    // (FMNMX, selects and compares issue at half rate there; ncu: 70 % ALU-pipe active at 52 % issue utilisation)
    const float sgn = (k >= kPerLane && k < 256 && ((sub * kPerLane) & k) != 0) ? -1.f : 1.f;
    if (k >= kPerLane && k < 256) {
#pragma unroll
      for (int r = 0; r < kPerLane; ++r) key[r] *= sgn;
    }
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (j >= kPerLane) {
        const int lx = j / kPerLane;                        // partner lane = lane ^ lx
        const bool keep_min = (sub & lx) == 0;              // lower position of the pair keeps the minimum
#pragma unroll
        for (int r = 0; r < kPerLane; ++r) {
          const float o = __shfl_xor_sync(0xffffffffu, key[r], lx);
          key[r] = keep_min ? fminf(key[r], o) : fmaxf(key[r], o);
        }
      } else {
#pragma unroll
        for (int r = 0; r < kPerLane; ++r) {
          if ((r & j) == 0) {
            const int pr = r | j;
            const bool up = k >= kPerLane || (r & k) == 0;     // compile-time
            const float a = key[r], b = key[pr];
            key[r] = up ? fminf(a, b) : fmaxf(a, b);
            key[pr] = up ? fmaxf(a, b) : fminf(a, b);
          }
        }
      }
    }
    if (k >= kPerLane && k < 256) {
#pragma unroll
      for (int r = 0; r < kPerLane; ++r) key[r] *= sgn;
    }
  }
}

struct SortParams {
  const float* a;        // [M, N] fp32 aligned student (scratch)
  const void* t;         // teacher [B, Tt, N]
  __nv_bfloat16* G;      // [M][N] sign(diff) in {-1, 0, +1} (exact in bf16: the GEMMs that consume it skip the lo plane)
  double* partials;      // [gridDim]
  int64_t M;
  int N, n_tok, Tt, t_off, planes, t_is_bf16, write_grad, pitch;
};

// One CTA per (sample, 16-channel group).  Shared memory holds three transposed tiles [16 columns][pitch]:
//   sa  : student values (later: the +-1 gradient, in place)      st : teacher values -> sorted teacher (in place)
//   ssa : sorted student
// A warp owns 4 columns (8 lanes each).  Both sequences are sorted keys-only; the permutation is never carried:
// the rank of a student value is its lower bound in the sorted student column (duplicates are ordered by token
// index, as the oracle's stable sort does), and d|.|/da = sign(a - sorted_t[rank]).
__global__ void __launch_bounds__(kSortThreads) wass_sort_kernel(SortParams p) {
  extern __shared__ __align__(16) float smem_f[];
  const int pitch = p.pitch;     // 264
  float* sa = smem_f;
  float* st = sa + kCh * pitch;
  float* ssa = st + kCh * pitch;
  __shared__ float red[kSortThreads / 32];
  const int groups = p.N / kCh;
  const int b = blockIdx.x / groups, c0 = (blockIdx.x % groups) * kCh;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n_tok = p.n_tok;

  // tile loads: a thread owns one 16-byte chunk (4 channels) of every 32nd token; all loads are issued before the
  // first transposing store (the fill is otherwise a chain of DRAM round trips)
  {
    constexpr int kSlots = kMaxTok / (kSortThreads / 4);   // 8 token slots per thread
    const int ch = (threadIdx.x & 3) * 4, tok0 = threadIdx.x >> 2;
    float4 va[kSlots], vt[kSlots];
#pragma unroll
    for (int k = 0; k < kSlots; ++k) {
      const int tok = tok0 + k * (kSortThreads / 4);
      if (tok < n_tok) {
        va[k] = __ldg(reinterpret_cast<const float4*>(p.a + ((int64_t)b * n_tok + tok) * p.N + c0 + ch));
        const int64_t toff = ((int64_t)b * p.Tt + p.t_off + tok) * p.N + c0 + ch;
        if (p.t_is_bf16) {
          float v[4];
          Vec<__nv_bfloat16, 4>::load(reinterpret_cast<const __nv_bfloat16*>(p.t) + toff, v);
          vt[k] = make_float4(v[0], v[1], v[2], v[3]);
        } else {
          vt[k] = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.t) + toff));
        }
      }
    }
    float* da = sa + ch * pitch + tok0;
    float* dt = st + ch * pitch + tok0;
#pragma unroll
    for (int k = 0; k < kSlots; ++k) {
      const int o = k * (kSortThreads / 4);
      if (tok0 + o < n_tok) {
        da[o] = va[k].x; da[pitch + o] = va[k].y; da[2 * pitch + o] = va[k].z; da[3 * pitch + o] = va[k].w;
        dt[o] = vt[k].x; dt[pitch + o] = vt[k].y; dt[2 * pitch + o] = vt[k].z; dt[3 * pitch + o] = vt[k].w;
      }
    }
  }
  __syncthreads();

  const int sub = lane & (kQuad - 1);
  const int col = warp * 4 + (lane >> 3);
  float* ca = sa + col * pitch;
  float* ct = st + col * pitch;
  float* cs = ssa + col * pitch;
  float key[kPerLane];
  float local = 0.f;

  // pass 0: teacher column, pass 1: student column — gather (token q*8 + sub: conflict-free), sort, store sorted
#pragma unroll 1
  for (int pass = 0; pass < 2; ++pass) {
    const float* src = pass ? ca : ct;
    float* dst = pass ? cs : ct;
#pragma unroll
    for (int q = 0; q < kPerLane; ++q) { const int tok = q * kQuad + sub; key[q] = tok < n_tok ? src[tok] : INFINITY; }
    __syncwarp();
    bitonic256_oct(key, sub);
#pragma unroll
    for (int r = 0; r < kPerLane; r += 4)
      if (sub * kPerLane + r < pitch) *reinterpret_cast<float4*>(dst + sub * kPerLane + r) = make_float4(key[r], key[r + 1], key[r + 2], key[r + 3]);
  }
#pragma unroll
  for (int r = 0; r < kPerLane; r += 4) {   // key[] still holds the sorted student column
    const int e = sub * kPerLane + r;
    if (e < n_tok) {                          // n_tok % 4 == 0 is not required: +inf - +inf never enters (guards below)
      const float4 tv = *reinterpret_cast<const float4*>(ct + e);
      if (e + 0 < n_tok) local += fabsf(key[r + 0] - tv.x);
      if (e + 1 < n_tok) local += fabsf(key[r + 1] - tv.y);
      if (e + 2 < n_tok) local += fabsf(key[r + 2] - tv.z);
      if (e + 3 < n_tok) local += fabsf(key[r + 3] - tv.w);
    }
  }
  __syncwarp();

  if (p.write_grad) {
    // sign of (student value - its teacher partner), two bit masks per lane (token q*8 + sub -> bit q);
    // 4 independent searches in flight (each is a chain of 8 dependent shared-memory loads; 8 in flight measured slower)
    unsigned pos = 0u, neg = 0u;
#pragma unroll 1
    for (int q0 = 0; q0 * kQuad + sub < n_tok; q0 += kSearchIlp) {
      float v[kSearchIlp];
      int r[kSearchIlp];
#pragma unroll
      for (int u = 0; u < kSearchIlp; ++u) {
        const int tok = (q0 + u) * kQuad + sub;
        v[u] = tok < n_tok ? ca[tok] : INFINITY;
        r[u] = 0;
      }
#pragma unroll
      for (int step = 128; step > 0; step >>= 1) {
#pragma unroll
        for (int u = 0; u < kSearchIlp; ++u) r[u] += cs[r[u] + step - 1] < v[u] ? step : 0;
      }
#pragma unroll
      for (int u = 0; u < kSearchIlp; ++u) {
        const int tok = (q0 + u) * kQuad + sub;
        if (tok < n_tok) {
          int rk = r[u];
          if (cs[rk + 1] == v[u])                          // duplicates: earlier tokens first
            for (int j = 0; j < tok; ++j) rk += (ca[j] == v[u]) ? 1 : 0;
          const float d = v[u] - ct[rk];
          pos |= (unsigned)(d > 0.f) << (q0 + u);
          neg |= (unsigned)(d < 0.f) << (q0 + u);
        }
      }
    }
    __syncwarp();   // every lane of the column is done reading the student values
#pragma unroll 4
    for (int q = 0; q < kPerLane; ++q)
      if (q * kQuad + sub < n_tok) ca[q * kQuad + sub] = ((pos >> q) & 1u) ? 1.f : (((neg >> q) & 1u) ? -1.f : 0.f);
  }

  local = warp_sum(local);
  if (lane == 0) red[warp] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < kSortThreads / 32; ++w) s += (double)red[w];
    p.partials[blockIdx.x] = s;
  }
  if (!p.write_grad) return;
  // +-1 gradient plane: a thread converts 4 channels of a token (8-byte stores, 32-byte rows per CTA)
  {
    const int ch = (threadIdx.x & 3) * 4;
    for (int tok = threadIdx.x >> 2; tok < n_tok; tok += kSortThreads / 4) {
      float v[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) v[q] = sa[(ch + q) * pitch + tok];
      const int64_t off = ((int64_t)b * n_tok + tok) * p.N + c0 + ch;
      Vec<__nv_bfloat16, 4>::store(p.G + off, v);
      if (p.planes == 2) {
        const float z[4] = {0.f, 0.f, 0.f, 0.f};
        Vec<__nv_bfloat16, 4>::store(p.G + p.M * p.N + off, z);
      }
    }
  }
}

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct Workspace {
  __nv_bfloat16 *S, *Wp, *Wt, *G, *ones;
  float* A;
  double* partials;
  float* wpart;   // deterministic mode: per-split weight-gradient slots (align_wgrad), appended last
  size_t bytes;
};
Workspace carve(void* base, int64_t B, int64_t M, int Ds, int Dt, int P, bool det) {
  Workspace w;
  size_t off = 0;
  auto take = [&](size_t n) { size_t o = off; off = align_up(off + n, 1024); return reinterpret_cast<char*>(base) + o; };
  w.S = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * M * Ds * 2));
  w.G = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * M * Dt * 2));
  w.A = reinterpret_cast<float*>(take((size_t)M * Dt * 4));
  w.Wp = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * Dt * Ds * 2));
  w.Wt = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * Dt * Ds * 2));
  w.ones = reinterpret_cast<__nv_bfloat16*>(take((size_t)2 * 64 * 64 * 2));
  w.partials = reinterpret_cast<double*>(take((size_t)B * (Dt / kCh) * sizeof(double)));
  w.wpart = det ? reinterpret_cast<float*>(take(align_wgrad_part_bytes(M, Ds, Dt, P))) : nullptr;
  w.bytes = off;
  return w;
}

}  // namespace
}  // namespace dkd

extern "C" {

size_t dkd_wass_l1_workspace_bytes(int64_t B, int n_tok, int Ds, int Dt, int precision) {
  return dkd::carve(nullptr, B, B * n_tok, Ds, Dt, dkd::prec_planes(precision), dkd::prec_deterministic(precision)).bytes;
}

int dkd_wass_l1_fwdbwd(const void* s, const void* t, const float* W, const float* bias, int64_t B, int Ts, int s_off, int Tt,
                       int t_off, int n_tok, int Ds, int Dt, int dtype, int precision, float scale, void* g_s, float* g_W,
                       float* g_b, float* loss, void* workspace, size_t workspace_bytes, dkd_stream_t stream) {
  using namespace dkd;
  int rc = dkd_check_device();
  if (rc != DKD_OK) return rc;
  const char* fn = "dkd_wass_l1_fwdbwd";
  DKD_REQUIRE(dtype == DKD_F32 || dtype == DKD_BF16, DKD_E_DTYPE, "%s: dtype %d", fn, dtype);
  DKD_REQUIRE(prec_valid(precision), DKD_E_UNSUPPORTED, "%s: precision %d", fn, precision);
  DKD_REQUIRE(B > 0 && n_tok > 0 && n_tok <= kMaxTok && s_off >= 0 && t_off >= 0 && Ts >= s_off + n_tok && Tt >= t_off + n_tok,
              DKD_E_SHAPE, "%s: bad token geometry (n_tok <= %d)", fn, kMaxTok);
  DKD_REQUIRE(Ds == 192 && (Dt == 384 || Dt == 768), DKD_E_SHAPE,
              "%s: built for widths 192 -> 384 (DeiT-Tiny -> DeiT-Small) and 192 -> 768 (DeiT-Tiny -> DeiT-Base), got %d -> %d", fn, Ds, Dt);
  DKD_REQUIRE(s && t && W && loss && workspace, DKD_E_SHAPE, "%s: null pointer", fn);
  DKD_REQUIRE((((uintptr_t)workspace) & 1023) == 0, DKD_E_ALIGN, "%s: workspace must be 1024-byte aligned", fn);
  DKD_REQUIRE((((uintptr_t)s | (uintptr_t)t | (uintptr_t)g_s) & 31) == 0, DKD_E_ALIGN, "%s: s, t and g_s must be 32-byte aligned (256-bit accesses)", "dkd_wass_l1_fwdbwd");
  const int P = prec_planes(precision);
  const int64_t M = B * n_tok;
  DKD_REQUIRE(M < (1ll << 31) - 256 && B * (Dt / kCh) < (1ll << 31), DKD_E_SHAPE, "%s: too many rows", fn);
  Workspace ws = carve(workspace, B, M, Ds, Dt, P, prec_deterministic(precision));
  DKD_REQUIRE(workspace_bytes >= ws.bytes, DKD_E_WORKSPACE, "%s: workspace %zu < %zu", fn, workspace_bytes, ws.bytes);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const bool want_grads = g_s || g_W || g_b;

  rc = launch_tokens_to_planes(s, dtype, B, Ts, s_off, n_tok, Ds, P, nullptr, ws.S, st);
  if (rc != DKD_OK) return rc;
  rc = launch_weight_to_planes(W, Dt, Ds, P, ws.Wp, want_grads ? ws.Wt : nullptr, st);
  if (rc != DKD_OK) return rc;

  rc = align_forward_rows(ws.S, ws.Wp, bias, ws.A, M, Ds, Dt, P, st, "dkd_wass_l1_fwdbwd: align GEMM");   // a = S W^T + b
  if (rc != DKD_OK) return rc;
  const int sort_grid = (int)(B * (Dt / kCh));
  {
    SortParams sp;
    sp.a = ws.A; sp.t = t; sp.G = ws.G; sp.partials = ws.partials; sp.M = M; sp.N = Dt; sp.n_tok = n_tok; sp.Tt = Tt;
    sp.t_off = t_off; sp.planes = 1; sp.t_is_bf16 = dtype == DKD_BF16; sp.write_grad = want_grads;   // +-1 is exact in bf16: no lo plane
    sp.pitch = kMaxTok + 8;   // all 256 sorted slots (+inf padded) are stored; 264 = 8 mod 32: a warp's 4 columns gather from 32 banks
    const size_t sort_smem = (size_t)3 * kCh * sp.pitch * sizeof(float);
    cudaFuncSetAttribute(wass_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sort_smem);
    wass_sort_kernel<<<sort_grid, kSortThreads, sort_smem, st>>>(sp);
    rc = check_launch("dkd_wass_l1_fwdbwd: sort");
    if (rc != DKD_OK) return rc;
    rc = launch_fold_partials(ws.partials, sort_grid, scale, loss, st);
    if (rc != DKD_OK) return rc;
  }
  if (!want_grads) return DKD_OK;

  if (g_s) {  // g_s = scale * G W
    rc = align_dgrad(ws.G, ws.Wt, g_s, M, n_tok, Ts, s_off, Ds, Dt, P, dtype == DKD_BF16, scale, st, "dkd_wass_l1_fwdbwd: dgrad GEMM", 1);
    if (rc != DKD_OK) return rc;
  }
  if (g_W || g_b) {
    DKD_REQUIRE(g_W != nullptr, DKD_E_UNSUPPORTED, "%s: g_b without g_W is not supported", fn);
    rc = align_wgrad(ws.G, ws.S, ws.ones, g_W, g_b, M, Ds, Dt, P, scale, st, "dkd_wass_l1_fwdbwd: wgrad GEMM", 1, ws.wpart);
    if (rc != DKD_OK) return rc;
  }
  return DKD_OK;
}

}  // extern "C"
