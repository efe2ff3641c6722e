// LRKD: low-rank projection matching.
// Reference: lrkd branch (model/loss.py:80-103) + lrkd_loss (:314-330): per layer pair (student 0,1,-1 / teacher 0,1,11)
//     T = teacher[:, 2:].reshape(M, Dt) ;  U, S, _ = svd(T) ;  A = U[:, :k] diag(S[:k])       ( = T V_k )
//     s' = Linear(Ds -> k)(student[:, 1:]).reshape(M, k) ;  loss += coef * mean((A - s')^2)
// and its autograd backward (to the student feature and the Linear).
//
// The tall SVD is replaced by the eigen-decomposition of the Dt x Dt Gram matrix (A = T V_k needs only V_k):
//   1. teacher -> bf16 planes (hi, mid, lo = all 24 mantissa bits) + exact fp64 column sums of squares
//   2. Gram  G = T^T T  on tcgen05 (gemm_nt, split over rows, 6 plane products = fp32-exact operands); each split
//      stores its fp32 partial tile, a second kernel adds the partials in fp64 in a fixed order (deterministic),
//      symmetrises and puts the exact diagonal in
//   3. eigenvectors of G: one-sided (Hestenes) Jacobi in fp64, all layers in ONE launch.  Default: cluster-resident —
//      one 16-CTA thread-block cluster per matrix, the columns live in shared memory / registers and move between CTAs
//      through distributed shared memory, one hardware cluster barrier per group round (section 3b); stops when the
//      `rank` leading columns are orthogonal to every other column.  Fallback (no 16-CTA cluster schedulable):
//      cooperative launch, 12 or 24 CTAs per matrix exchanging column groups through global memory (section 3)
//   4. select: column norms = eigenvalues, rank them (descending, ties by index), V_k = top-k normalised columns;
//      builds the fused operand [W' | -V_k] (bf16 hi/lo planes) and the transposed head for the backward
//   5. d = [s | T] [W' | -V_k]^T + b' = s' - A  in ONE tcgen05 GEMM (K = Ds + Dt), epilogue: loss partial and
//      g_s' = 2 coef/(M k) d as planes ;  6. g_s = g_s' W' ;  7. g_W' = g_s'^T s, g_b' = g_s'^T 1
// Column signs of singular vectors are arbitrary (LAPACK's differ between fp32 and fp64, SURVEY §7): V_k and S_k
// can be returned so that callers / tests align signs; here each v is normalised to a positive largest component.
#include <cooperative_groups.h>

#include "epilogues.cuh"
#include "gemm_nt.cuh"
#include "planes.cuh"

namespace dkd {
namespace {

constexpr int kN = 384;              // Dt: order of the Gram matrix
// Columns per group G: a CTA holds 2G columns and runs one warp per column pair (G warps).  G = 8 (24 CTAs per matrix)
// is the default — with fewer pairs per SM the fp64 pipe of each SM is less contended and a round is ~20 % shorter
// than with G = 16 (G = 4 measured slower again: 95 grid barriers per sweep); G = 16 (12 CTAs per matrix) is used when
// 24 * n_layers CTAs would not be co-resident.
template <int G> struct JacobiCfg {
  static constexpr int CTAS = kN / G / 2;
  static constexpr int THREADS = 32 * G;
  static constexpr size_t SMEM = (size_t)2 * G * kN * sizeof(double);
};
constexpr int kMaxSweeps = 14;
constexpr int kMaxSweepsCluster = 30;   // decaying spectra (real features) need ~20 until the leading columns stop moving
constexpr double kJacobiTol = 1e-10;   // pairs with |cos| below this are not rotated
// Jacobi converges quadratically: a sweep that SAW no |cos| above 1e-6 leaves the columns orthogonal to ~1e-12, so it
// is the last one (no separate verification sweep).
constexpr double kJacobiStop = 1e-6;
constexpr int kMaxLayers = 8;

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---------------------------------------------------------------- 1. teacher planes + exact column sums of squares
template <typename T>
__global__ void __launch_bounds__(192) teacher_planes_kernel(const T* __restrict__ src, int64_t B, int T_tok, int off, int n_tok,
                                                             int P, __nv_bfloat16* __restrict__ dst, double* __restrict__ sumsq_part) {
  // 48 threads cover one 384-wide row (8 channels each); 4 rows per block iteration; a thread keeps its channel group
  const int cg = (threadIdx.x % 48) * 8, rl = threadIdx.x / 48;
  const int64_t M = B * n_tok;
  double acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.0;
  for (int64_t m = (int64_t)blockIdx.x * 4 + rl; m < M; m += (int64_t)gridDim.x * 4) {
    const int64_t b = m / n_tok;
    const int64_t srow = b * T_tok + off + (m - b * n_tok);
    float v[8];
    if constexpr (sizeof(T) == 4) {
      Vec<float, 4>::load(reinterpret_cast<const float*>(src) + srow * kN + cg, *reinterpret_cast<float(*)[4]>(&v[0]));
      Vec<float, 4>::load(reinterpret_cast<const float*>(src) + srow * kN + cg + 4, *reinterpret_cast<float(*)[4]>(&v[4]));
    } else {
      Vec<__nv_bfloat16, 8>::load(reinterpret_cast<const __nv_bfloat16*>(src) + srow * kN + cg, v);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = fma((double)v[j], (double)v[j], acc[j]);
    float r[8];
    Vec<__nv_bfloat16, 8>::store(dst + m * kN + cg, v);
    if (P >= 2) {
#pragma unroll
      for (int j = 0; j < 8; ++j) r[j] = v[j] - __bfloat162float(__float2bfloat16_rn(v[j]));
      Vec<__nv_bfloat16, 8>::store(dst + M * kN + m * kN + cg, r);
    }
    if (P >= 3) {
#pragma unroll
      for (int j = 0; j < 8; ++j) r[j] = r[j] - __bfloat162float(__float2bfloat16_rn(r[j]));
      Vec<__nv_bfloat16, 8>::store(dst + 2 * M * kN + m * kN + cg, r);
    }
  }
  __shared__ double red[4][kN];
#pragma unroll
  for (int j = 0; j < 8; ++j) red[rl][cg + j] = acc[j];
  __syncthreads();
  for (int c = threadIdx.x; c < kN; c += 192)
    sumsq_part[(size_t)blockIdx.x * kN + c] = (red[0][c] + red[1][c]) + (red[2][c] + red[3][c]);
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---------------------------------------------------------------- 2. Gram: per-split partial tiles -> fp64, symmetric
using GramCfg = GemmNtCfg<6, false, 256, 128, 3, 64>;   // 128 x 384 fp32 tile in TMEM, 64 rows per stage

struct NtGramLoader : NtPlainLoader<GramCfg> {
  static __device__ __forceinline__ void decode(const Params& p, int item, Item& it) {
    const int tile = item % p.na_tiles, split = item / p.na_tiles;
    it.rb0 = split * p.row_blocks_per_split;
    it.rb1 = min(it.rb0 + p.row_blocks_per_split, p.total_row_blocks);
    it.a_col0 = tile * 128;
    it.b_col0 = 0;
    it.d_off = ((int64_t)split * kN + tile * 128) * kN;   // partial[split][tile*128 ..][0 .. 384)
    it.dcol_off = -1;
    it.aux = 0;
  }
};

__global__ void gram_reduce_kernel(const float* __restrict__ part, int splits, double* __restrict__ gsum) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= kN * kN) return;
  double a = 0.0;
  for (int s = 0; s < splits; ++s) a += (double)part[(size_t)s * kN * kN + idx];
  gsum[idx] = a;
}

// off-diagonal: 0.5 (g_ij + g_ji); diagonal: the exact fp64 column sums of squares, folded over the partial blocks by
// one warp per column in a fixed order (a thread-per-column loop over 296 partials was a 26 us chain of L2 round trips)
__global__ void __launch_bounds__(256) gram_symmetrize_kernel(const double* __restrict__ gsum, const double* __restrict__ sumsq_part,
                                                              int nparts, double* __restrict__ W) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < kN * kN) {
    const int i = idx / kN, j = idx - i * kN;
    if (i != j) W[idx] = 0.5 * (gsum[idx] + gsum[j * kN + i]);
  }
  const int warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp_global < kN) {
    double v = 0.0;
    for (int s = lane; s < nparts; s += 32) v += sumsq_part[(size_t)s * kN + warp_global];
    v = warp_sum_d(v);
    if (lane == 0) W[(size_t)warp_global * kN + warp_global] = v;
  }
}

// ---------------------------------------------------------------- 3. batched one-sided Jacobi (cooperative launch)
struct JacobiParams {
  double* W;                       // [L][n][n], column j contiguous at j*n (symmetric start)
  unsigned* bar;                   // [L] barrier counters, zeroed before launch
  unsigned long long* offmax;      // [L][2] max |cos| of the sweep (bits of a non-negative double), zeroed
  int* sweeps_out;                 // [L]
  int k;                           // cluster-resident version: number of leading eigenpairs the caller needs (1..n)
};

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ void layer_barrier(unsigned* ctr, unsigned target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(ctr, 1u);
    const long long t0 = clock64();
    while (ld_acquire_u32(ctr) < target) {
      if (clock64() - t0 > 4000000000ll) {
        printf("dkd: LRKD Jacobi barrier timed out (block %d,%d)\n", blockIdx.x, blockIdx.y);
        __trap();
      }
    }
    __threadfence();
  }
  __syncthreads();
}

// Two-level (block) one-sided Jacobi.  The 384 columns form 24 groups of 16; in an outer round every CTA owns a pair
// of groups (round-robin tournament over the groups: 23 outer rounds per sweep), copies its 32 columns (96 KB of fp64)
// into shared memory, rotates the 16 x 16 cross pairs there (16 inner rounds, 16 warps = 16 disjoint column pairs per
// inner round, __syncthreads between rounds; the pairs inside a group are done once per sweep, in outer round 0) and
// writes them back.  One grid barrier per OUTER round: 23 per sweep instead of the 383 of a flat ordering — the
// solver is bound by the latency of its sequential rounds, not by arithmetic.
template <int G>
__global__ void __launch_bounds__(32 * G) jacobi_kernel(JacobiParams p) {
  constexpr int n = kN, PER = n / 32;          // 12 elements per lane
  constexpr int NG = n / G;                    // column groups
  constexpr int kJacobiThreads = 32 * G;
  constexpr int LC = 2 * G;                    // 32 columns per CTA
  extern __shared__ double scol[];             // [LC][n]
  const int layer = blockIdx.y;
  double* W = p.W + (size_t)layer * n * n;
  unsigned* bar = p.bar + layer;
  unsigned long long* offmax = p.offmax + 2 * layer;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;   // 16 warps
  // columns whose norm is below 1e-13 * trace(G) belong to the null space (rank-deficient teacher): never rotated
  __shared__ double s_tiny;
  __shared__ double s_off[kJacobiThreads / 32];
  if (warp == 0) {
    double tr = 0.0;
    for (int i = lane; i < n; i += 32) tr += W[(size_t)i * n + i];
    tr = warp_sum_d(tr);
    if (lane == 0) s_tiny = (1e-13 * tr) * (1e-13 * tr);
  }
  __syncthreads();
  const double tiny = s_tiny;
  unsigned epoch = 0;
  int sweep = 0;
  for (; sweep < kMaxSweeps; ++sweep) {
    double local_off = 0.0;
    for (int r = 0; r < NG - 1; ++r) {
      // round-robin tournament over groups: position 0 is fixed, the others rotate; this CTA takes (pos c, pos NG-1-c)
      const int pi = blockIdx.x, pj = NG - 1 - blockIdx.x;
      const int gp = pi == 0 ? 0 : 1 + (pi - 1 + r) % (NG - 1);
      const int gq = 1 + (pj - 1 + r) % (NG - 1);
      for (int idx = threadIdx.x; idx < LC * n; idx += kJacobiThreads) {
        const int c = idx / n, i = idx - c * n;
        const int gc = (c < G ? gp * G : gq * G - G) + c;
        scol[idx] = __ldcg(W + (size_t)gc * n + i);
      }
      __syncthreads();
      // inner rounds: in outer round 0 first the pairs INSIDE each of the two groups (15 rounds, 8 pairs per group),
      // then — every outer round — the 16 x 16 cross pairs (16 rounds of 16 disjoint pairs).  Per sweep every column
      // pair is rotated exactly once: 23 * 16 + 15 = 383 sequential rounds, as in a flat ordering, but 360 of the
      // 383 synchronisations are __syncthreads instead of grid barriers.
      const int n_inner = (r == 0 ? G - 1 : 0) + G;
      for (int ir = 0; ir < n_inner; ++ir) {
        int cp, cq;
        if (r == 0 && ir < G - 1) {            // within-group tournament: first half of the warps group P, second half group Q
          const int base = (warp / (G / 2)) * G, w8 = warp % (G / 2);
          const int qi = w8, qj = G - 1 - w8;
          cp = base + (qi == 0 ? 0 : 1 + (qi - 1 + ir) % (G - 1));
          cq = base + 1 + (qj - 1 + ir) % (G - 1);
        } else {
          const int k = ir - (r == 0 ? G - 1 : 0);
          cp = warp;
          cq = G + ((warp + k) & (G - 1));
        }
        double* a = scol + cp * n;
        double* b = scol + cq * n;
        double x[PER], y[PER];
        double aa = 0.0, bb = 0.0, ab = 0.0;
#pragma unroll
        for (int k = 0; k < PER; ++k) { x[k] = a[lane + 32 * k]; y[k] = b[lane + 32 * k]; }
#pragma unroll
        for (int k = 0; k < PER; ++k) { aa = fma(x[k], x[k], aa); bb = fma(y[k], y[k], bb); ab = fma(x[k], y[k], ab); }
        aa = warp_sum_d(aa); bb = warp_sum_d(bb); ab = warp_sum_d(ab);
        const double prod = aa * bb;
        const double cosv = (prod > 0.0 && (aa > tiny || bb > tiny)) ? fabs(ab) * rsqrt(prod) : 0.0;
        local_off = fmax(local_off, cosv);
        if (cosv > kJacobiTol) {
          // t = sign(zeta) / (|zeta| + sqrt(1 + zeta^2)), zeta = (bb - aa) / (2 ab), written with one division:
          // t = sign(d h) |h| / (|d| + sqrt(d^2 + h^2)), d = bb - aa, h = 2 ab ;  c = 1/sqrt(1 + t^2), s = c t
          const double d = bb - aa, h = 2.0 * ab;
          const double t = ((d >= 0.0) == (h >= 0.0) ? fabs(h) : -fabs(h)) / (fabs(d) + sqrt(fma(d, d, h * h)));
          const double c = rsqrt(fma(t, t, 1.0)), sn = c * t;
#pragma unroll
          for (int k = 0; k < PER; ++k) {
            a[lane + 32 * k] = c * x[k] - sn * y[k];
            b[lane + 32 * k] = sn * x[k] + c * y[k];
          }
        }
        __syncthreads();
      }
      for (int idx = threadIdx.x; idx < LC * n; idx += kJacobiThreads) {
        const int c = idx / n, i = idx - c * n;
        const int gc = (c < G ? gp * G : gq * G - G) + c;
        W[(size_t)gc * n + i] = scol[idx];
      }
      if (r == NG - 2) {   // end of the sweep: publish this CTA's largest |cos|
        if (lane == 0) s_off[warp] = local_off;
        __syncthreads();
        if (threadIdx.x == 0) {
          double m = 0.0;
          for (int w = 0; w < kJacobiThreads / 32; ++w) m = fmax(m, s_off[w]);
          atomicMax(offmax + (sweep & 1), (unsigned long long)__double_as_longlong(m));
        }
      }
      ++epoch;
      layer_barrier(bar, epoch * gridDim.x);
      if (r == 0 && blockIdx.x == 0 && threadIdx.x == 0) offmax[(sweep + 1) & 1] = 0ull;  // buffer of the next sweep
    }
    const double off = __longlong_as_double((long long)__ldcg(offmax + (sweep & 1)));
    if (off <= kJacobiStop) { ++sweep; break; }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && p.sweeps_out) p.sweeps_out[layer] = sweep;
}

// ---------------------------------------------------------------- 3b. cluster-resident Jacobi (the default)
// One 16-CTA thread-block cluster per matrix; the matrix never leaves the SMs during the solve.  Every CTA holds two
// groups of 12 columns ("slot 0", "slot 1", 36 KB each).  A group round rotates the 12 x 12 cross pairs of the two
// resident groups; then every warp stores its columns straight into the shared memory of the CTA that needs them next
// (st.shared::cluster into the other half of a double buffer), so the exchange costs no extra pass and ONE hardware
// cluster barrier per group round replaces the global-memory round trip + software grid barrier of the cooperative
// version (11 us per group round there).
// Inside a group round the work is laid out for what bounds it — the latency of the dependent chain of a pair rotation
// (dot product -> 5-level double butterfly, 176 cycles -> rotation parameters -> update), the fp64 pipes (16 lanes per SM
// sub-partition: a warp-wide DFMA issues every 2 cycles; measured 64 lanes/clk/SM) and the 128 B/clk shared-memory
// port (measured with clock64: a first version that kept every column in shared memory and gave one pair to each of 12
// warps spent 1 150 of its 2 370 cycles per pair round moving 2 x 73 KB through that port and 610 in a branchy,
// IEEE-division parameter chain): 4 warps, one per sub-partition; a warp keeps THREE slot-0 columns in registers for
// the whole group round and takes three slot-1 columns per macro round (4 macro rounds; the slot-1 triples walk around
// the warps), rotating the 3 x 3 cross pairs in three steps of three independent pairs whose chains interleave in the
// one instruction stream — 9 pair rotations per 3 columns loaded + 3 stored.  1 380 cycles per step of 3 pairs per warp
// (0.73 us per sequential pair round; the cooperative version needs 1.4 us).
// Ordering over the cluster (content-agnostic: it only says where the CONTENT of a slot goes, so sweeps chain without
// returning the columns home): recursive halving.  Phase R = 16, 8, 4, 2, 1 works in sub-rings of R consecutive CTAs
// for R rounds: slot 0 stays, slot 1 moves to the next CTA of the sub-ring, so every slot-0 group of the sub-ring meets
// every slot-1 group (only ONE group per CTA crosses the cluster network per round).  The last round of a phase sends
// all slot-0 groups of a sub-ring to its lower half and all slot-1 groups to its upper half: the next phase pairs them
// up among themselves.  16 + 8 + 4 + 2 + 1 = 31 group rounds = C(32, 2) / 16 group pairs; the pairs INSIDE a group are
// done in the last group round of the sweep (a tournament over the 4 column triples of a group, 12 steps).
// Arithmetic per pair is cut to what the fp64 pipe must do: squared norms travel with the columns (element [384] of a
// column, updated from the rotation, recomputed once per sweep), so one dot product per pair instead of three; the
// rotation parameters are formed in fp32 (MUFU) from scale-free quantities and (c, s) is then made orthonormal in
// fp64 by one Newton step (c^2 + s^2 = 1 to ~1e-21) — a 1e-7 error of the ANGLE only leaves a residual 1e-7 |cos| for
// the next sweep, it does not perturb the result.
constexpr int kCS = 16;                       // CTAs per matrix
constexpr int kCG = kN / (2 * kCS);           // 12 columns per group
constexpr int kCC = 3;                        // columns of each slot per warp
constexpr int kCW = kCG / kCC;                // 4 warps per CTA (one per SM sub-partition: the fp64 pipes are per sub-partition)
constexpr int kCStride = kN + 8;              // doubles per column buffer; [kN] holds the squared norm
constexpr size_t kClusterSmem = (size_t)2 * 2 * kCG * kCStride * sizeof(double);   // [parity][slot][col][stride] = 150 528 B
constexpr int kPER = kN / 32;                 // 12 elements of a column per lane

__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t cta) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(cta));
  return r;
}
__device__ __forceinline__ void st_cluster_f64(uint32_t addr, double v) {
  asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory");
}

__device__ __forceinline__ void col_load(const double* c, int lane, double (&x)[kPER], double& nrm) {
#pragma unroll
  for (int k = 0; k < kPER; ++k) x[k] = c[lane + 32 * k];
  nrm = c[kN];
}
__device__ __forceinline__ void col_store(double* c, int lane, const double (&x)[kPER], double nrm) {
#pragma unroll
  for (int k = 0; k < kPER; ++k) c[lane + 32 * k] = x[k];
  if (lane == 0) c[kN] = nrm;
}
__device__ __forceinline__ void col_store_cluster(uint32_t addr, int lane, const double (&x)[kPER], double nrm) {
#pragma unroll
  for (int k = 0; k < kPER; ++k) st_cluster_f64(addr + 8u * (lane + 32 * k), x[k]);
  if (lane == 0) st_cluster_f64(addr + 8u * kN, nrm);
}
__device__ __forceinline__ double col_norm2(const double (&x)[kPER]) {
  double s0 = 0.0, s1 = 0.0;
#pragma unroll
  for (int k = 0; k < kPER; k += 2) { s0 = fma(x[k], x[k], s0); s1 = fma(x[k + 1], x[k + 1], s1); }
  return warp_sum_d(s0 + s1);
}

__device__ __forceinline__ float rsqrt_approx(float x) { float y; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float sqrt_approx(float x) { float y; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// Rotation of one pair from its squared norms and dot product (all warp-uniform): (c, s) — (1, 0) when the pair is not
// rotated — and the new squared norms.  Straight-line code (selects, single-MUFU approximations): this chain sits between
// the dot product and the column update of every pair, and the chains of a step's pairs must interleave in one warp.
// The fp64 part is kept short because warp-uniform scalars still cost a full warp instruction on the fp64 pipe.
struct JacobiRot { double c, sn; };
__device__ __forceinline__ JacobiRot jacobi_rotation(double& aa, double& bb, double ab, float thr2, float& seen) {
  constexpr float tiny = 1e-26f;   // (1e-13 * trace)^2 in scaled units: null-space columns are never rotated
  const float aaf = (float)aa, bbf = (float)bb, abf = (float)ab, big = fmaxf(aaf, bbf);
  const bool live = fminf(aaf, bbf) > 1e-36f && big > tiny;
  const float rn = live ? rsqrt_approx(aaf) * rsqrt_approx(bbf) : 0.f;   // 1 / (|a| |b|): d and h below are scale-free
  const float cosv = fabsf(abf) * rn;
  const bool rot = cosv > (float)kJacobiTol;
  // t = sign(d h) |h| / (|d| + sqrt(d^2 + h^2)), d = bb - aa, h = 2 ab ;  c = 1/sqrt(1 + t^2), s = c t
  const float df = (float)(bb - aa) * rn, hf = 2.f * abf * rn;      // |h| = 2 cos >= 2e-10, |d| <= 2e18: no under/overflow
  const float den = fabsf(df) + sqrt_approx(fmaf(df, df, hf * hf));
  const float tf = rot ? (df >= 0.f ? hf : -hf) * rcp_approx(den) : 0.f;
  // What the pair still does to a wanted column: the smaller of |cos| and |tan| of the rotation.  A leading column and a
  // small unconverged one keep |cos| = O(1) for many sweeps (the small column is dominated by what leaks into it from
  // the leading directions) while the rotation they get, ~ cos |b| / |a|, is already negligible.
  seen = big >= thr2 ? fmaxf(seen, fminf(cosv, fabsf(tf))) : seen;
  const double td = (double)tf, q = fma(td, td, 1.0);
  const double c0 = (double)rsqrt_approx(fmaf(tf, tf, 1.f));
  const double e = fma(-q, c0 * c0, 1.0);                   // c0 = (1 + delta) / sqrt(q): e = -2 delta - delta^2
  JacobiRot r;
  r.c = c0 * fma(e, fma(e, 0.375, 0.5), 1.0);               // (1 - e)^(-1/2) to second order: c^2 (1 + t^2) = 1 + O(e^3); t = 0 -> exactly 1
  r.sn = r.c * td;
  // |a'|^2 = aa - t ab, |b'|^2 = bb + t ab at the exact Jacobi angle, and the derivative of |a'|^2 with respect to the
  // angle there is -2 a'.b' = 0: the 1e-7 relative error of t enters the carried norms only in second order
  const double tab = td * ab;
  aa -= tab; bb += tab;
  return r;
}

// One step: NP independent pairs (col[Sel::a(i)], col[Sel::b(i)]) of the warp's register-resident columns, their chains
// (dot product -> butterfly -> rotation parameters -> update) interleaved by the unrolled loops.
template <int NP, class Sel, int NC>
__device__ __forceinline__ void jacobi_step(double (&col)[NC][kPER], double (&nrm)[NC], float thr2, float& seen) {
  double ab[NP];
#pragma unroll
  for (int i = 0; i < NP; ++i) {
    double p0 = 0.0, p1 = 0.0;
#pragma unroll
    for (int k = 0; k < kPER; k += 2) {
      p0 = fma(col[Sel::a(i)][k], col[Sel::b(i)][k], p0);
      p1 = fma(col[Sel::a(i)][k + 1], col[Sel::b(i)][k + 1], p1);
    }
    ab[i] = p0 + p1;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int i = 0; i < NP; ++i) ab[i] += __shfl_xor_sync(0xffffffffu, ab[i], o);
  }
  JacobiRot r[NP];
#pragma unroll
  for (int i = 0; i < NP; ++i) r[i] = jacobi_rotation(nrm[Sel::a(i)], nrm[Sel::b(i)], ab[i], thr2, seen);
#pragma unroll
  for (int i = 0; i < NP; ++i) {
#pragma unroll
    for (int k = 0; k < kPER; ++k) {
      const double xv = col[Sel::a(i)][k], yv = col[Sel::b(i)][k];
      col[Sel::a(i)][k] = fma(r[i].c, xv, -r[i].sn * yv);
      col[Sel::b(i)][k] = fma(r[i].sn, xv, r[i].c * yv);
    }
  }
}
// columns 0..C-1 = first set, C..2C-1 = second set.  Cross<S>: pair i = (i, C + (i + S) mod C); Inner3<R>: round R of the
// tournament inside each set of 3 (one pair per set).
template <int S> struct SelCross {
  static constexpr __device__ int a(int i) { return i; }
  static constexpr __device__ int b(int i) { return kCC + (i + S) % kCC; }
};
template <int R> struct SelInner3 {   // R = 0: (0,1), 1: (0,2), 2: (1,2)
  static constexpr __device__ int a(int i) { return (i ? kCC : 0) + (R == 2 ? 1 : 0); }
  static constexpr __device__ int b(int i) { return (i ? kCC : 0) + (R == 0 ? 1 : 2); }
};
static_assert(kCC == 3, "the step selectors are written for 3 columns of each set per warp");

__global__ void __launch_bounds__(32 * kCW, 1) jacobi_cluster_kernel(JacobiParams p) {
  constexpr int n = kN, G = kCG, C = kCC;
  constexpr int T = 2 * kCS - 1;               // group rounds per sweep
  extern __shared__ __align__(16) double sbuf[];   // [2][2][G][kCStride]
  __shared__ double s_scale;
  __shared__ float s_warp_off[kCW];
  __shared__ float s_cta_off[2][kCS];          // [sweep parity][cta]: written by every CTA of the cluster
  __shared__ double s_norms[kN];               // squared norms of all columns at the start of a sweep (written by every CTA)
  __shared__ double s_thr2;
  const int rank = (int)sm100::cluster_ctarank();
  const int layer = blockIdx.x / kCS;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double* W = p.W + (size_t)layer * n * n;
  auto col_ptr = [&](int par, int slot, int c) { return sbuf + ((size_t)(par * 2 + slot) * G + c) * kCStride; };

  if (warp == 0) {
    double tr = 0.0;
    for (int i = lane; i < n; i += 32) tr += W[(size_t)i * n + i];
    tr = warp_sum_d(tr);
    if (lane == 0) s_scale = (tr > 0.0 && tr < 1e300) ? scalbn(1.0, -ilogb(tr)) : 1.0;   // trace * scale in [1, 2)
  }
  __syncthreads();
  const double scale = s_scale;
  for (int c = warp; c < 2 * G; c += kCW) {    // this CTA's 24 columns: global column rank * 24 + c -> (slot c / 12, column c % 12)
    const double* src = W + (size_t)(rank * 2 * G + c) * n;
    double x[kPER];
#pragma unroll
    for (int k = 0; k < kPER; ++k) x[k] = __ldcg(src + lane + 32 * k) * scale;
    col_store(col_ptr(0, c / G, c % G), lane, x, col_norm2(x));
  }
  sm100::cluster_sync();   // every CTA of the cluster is running (its shared memory may be written) and has loaded its columns

  int par = 0, sweep = 0;
  for (; sweep < kMaxSweepsCluster; ++sweep) {
    // Convergence is judged on the pairs that involve a WANTED column — one of the k largest (by the norms at the start
    // of the sweep, 2 % margin).  A wanted column that is orthogonal to every other column is an eigenvector of G^2,
    // hence of G; the columns of small eigenvalues converge last (for a decaying spectrum of condition 1e8 three times
    // later than the leading ones, and the numerically-zero columns of a rank-deficient matrix never do) and nobody
    // reads them.  All pairs are still rotated.
    if (p.k < n) {
      if (threadIdx.x < 2 * G) {
        const double v = col_ptr(par, threadIdx.x / G, threadIdx.x % G)[n];
        const uint32_t local = sm100::smem_u32(&s_norms[rank * 2 * G + threadIdx.x]);
#pragma unroll
        for (int c = 0; c < kCS; ++c) st_cluster_f64(mapa_shared(local, (uint32_t)c), v);
      }
      sm100::cluster_sync();
      for (int j = threadIdx.x; j < n; j += 32 * kCW) {
        const double v = s_norms[j];
        int cnt = 0;
        for (int i = 0; i < n; ++i) { const double u = s_norms[i]; cnt += (u > v) || (u == v && i < j); }
        if (cnt == p.k - 1) s_thr2 = 0.98 * v;
      }
    } else if (threadIdx.x == 0) {
      s_thr2 = 0.0;
    }
    __syncthreads();
    const float thr2 = (float)s_thr2;
    float seen = 0.f;                          // what this warp saw on the wanted pairs (see jacobi_rotation)
    for (int t = 0; t < T; ++t) {
      // phase (ring size R) and round r inside it: t = 0..15 -> R = 16, 16..23 -> 8, 24..27 -> 4, 28..29 -> 2, 30 -> 1
      int R = kCS, r = t;
      while (r >= R) { r -= R; R >>= 1; }
      const int i = rank & (R - 1), base = rank - i;
      int dcta0 = rank, dslot0 = 0, dcta1 = rank, dslot1 = 1;
      if (R > 1) {
        if (r < R - 1) {
          dcta1 = base + ((i + 1) & (R - 1));
        } else if (i < R / 2) {
          dcta1 = rank + R / 2; dslot1 = 0;
        } else {
          dcta0 = rank - R / 2; dslot0 = 1;
        }
      }
      double col[2 * C][kPER], nrm[2 * C];
      if (t == T - 1) {
        // pairs inside each group, once per sweep: warps 0, 1 take slot 0, warps 2, 3 slot 1; tournament over the 4
        // column triples {3s, 3s+1, 3s+2} of the group (3 rounds of 2 meetings); a meeting rotates the 3 x 3 cross pairs,
        // the first round also the pairs inside each of the two triples.  The carried squared norms are recomputed.
        const int slot = warp >> 1, v = warp & 1, vj = 3 - v;
        for (int rr = 0; rr < 3; ++rr) {
          const int sa = v == 0 ? 0 : 1 + (v - 1 + rr) % 3, sb = 1 + (vj - 1 + rr) % 3;
#pragma unroll
          for (int c = 0; c < C; ++c) {
            col_load(col_ptr(par, slot, C * sa + c), lane, col[c], nrm[c]);
            col_load(col_ptr(par, slot, C * sb + c), lane, col[C + c], nrm[C + c]);
          }
#pragma unroll
          for (int c = 0; c < 2 * C; ++c) nrm[c] = col_norm2(col[c]);
          if (rr == 0) {
            jacobi_step<2, SelInner3<0>>(col, nrm, thr2, seen);
            jacobi_step<2, SelInner3<1>>(col, nrm, thr2, seen);
            jacobi_step<2, SelInner3<2>>(col, nrm, thr2, seen);
          }
          jacobi_step<C, SelCross<0>>(col, nrm, thr2, seen);
          jacobi_step<C, SelCross<1>>(col, nrm, thr2, seen);
          jacobi_step<C, SelCross<2>>(col, nrm, thr2, seen);
#pragma unroll
          for (int c = 0; c < C; ++c) {
            col_store(col_ptr(par, slot, C * sa + c), lane, col[c], nrm[c]);
            col_store(col_ptr(par, slot, C * sb + c), lane, col[C + c], nrm[C + c]);
          }
          __syncthreads();
        }
      }
      // cross pairs of the two groups: slot-0 columns 3w .. 3w+2 stay in this warp's registers, the slot-1 column
      // triples walk around the warps
#pragma unroll
      for (int c = 0; c < C; ++c) col_load(col_ptr(par, 0, C * warp + c), lane, col[c], nrm[c]);
      for (int m = 0; m < kCW; ++m) {
        const int j = (warp + m) & (kCW - 1);
#pragma unroll
        for (int c = 0; c < C; ++c) col_load(col_ptr(par, 1, C * j + c), lane, col[C + c], nrm[C + c]);
        jacobi_step<C, SelCross<0>>(col, nrm, thr2, seen);
        jacobi_step<C, SelCross<1>>(col, nrm, thr2, seen);
        jacobi_step<C, SelCross<2>>(col, nrm, thr2, seen);
        if (m < kCW - 1) {
#pragma unroll
          for (int c = 0; c < C; ++c) col_store(col_ptr(par, 1, C * j + c), lane, col[C + c], nrm[C + c]);
          __syncthreads();
        } else {
          // end of the group round: the columns go to the buffers of the NEXT group round, in the CTA that holds them then
          const uint32_t d1 = mapa_shared(sm100::smem_u32(col_ptr(par ^ 1, dslot1, C * j)), (uint32_t)dcta1);
          const uint32_t d0 = mapa_shared(sm100::smem_u32(col_ptr(par ^ 1, dslot0, C * warp)), (uint32_t)dcta0);
#pragma unroll
          for (int c = 0; c < C; ++c) {
            col_store_cluster(d1 + 8u * kCStride * c, lane, col[C + c], nrm[C + c]);
            col_store_cluster(d0 + 8u * kCStride * c, lane, col[c], nrm[c]);
          }
        }
      }
      if (t == T - 1) {                        // end of the sweep: every CTA learns what every CTA saw
        if (lane == 0) s_warp_off[warp] = seen;
        __syncthreads();
        if (threadIdx.x < kCS) {
          float m = 0.f;
#pragma unroll
          for (int w = 0; w < kCW; ++w) m = fmaxf(m, s_warp_off[w]);
          const uint32_t dst = mapa_shared(sm100::smem_u32(&s_cta_off[sweep & 1][rank]), (uint32_t)threadIdx.x);
          asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(dst), "f"(m) : "memory");
        }
      }
      sm100::cluster_sync();
      par ^= 1;
    }
    float off = 0.f;
#pragma unroll
    for (int c = 0; c < kCS; ++c) off = fmaxf(off, s_cta_off[sweep & 1][c]);
    if (off <= (float)kJacobiStop) { ++sweep; break; }
  }
  // back to global memory, unscaled (power of two: exact); the column ORDER is a permutation of the input order
  const double inv = 1.0 / scale;
  for (int c = warp; c < 2 * G; c += kCW) {
    const double* src = col_ptr(par, c / G, c % G);
    double* dst = W + (size_t)(rank * 2 * G + c) * n;
#pragma unroll
    for (int k = 0; k < kPER; ++k) dst[lane + 32 * k] = src[lane + 32 * k] * inv;
  }
  if (rank == 0 && threadIdx.x == 0 && p.sweeps_out) p.sweeps_out[layer] = sweep;
}

// host: can a 16-CTA cluster of this kernel be scheduled on this device?  (non-portable cluster size; cached)
bool jacobi_cluster_available() {
  static const bool ok = [] {
    if (cudaFuncSetAttribute(jacobi_cluster_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess ||
        cudaFuncSetAttribute(jacobi_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kClusterSmem) != cudaSuccess) {
      cudaGetLastError();
      return false;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(kCS);
    cfg.blockDim = dim3(32 * kCW);
    cfg.dynamicSmemBytes = kClusterSmem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = kCS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int ncl = 0;
    if (cudaOccupancyMaxActiveClusters(&ncl, jacobi_cluster_kernel, &cfg) != cudaSuccess) { cudaGetLastError(); return false; }
    return ncl >= 1;
  }();
  return ok;
}

cudaError_t launch_jacobi_cluster(const JacobiParams& jp, int n_layers, cudaStream_t st) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(kCS * n_layers));
  cfg.blockDim = dim3(32 * kCW);
  cfg.dynamicSmemBytes = kClusterSmem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = kCS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, jacobi_cluster_kernel, jp);
}

// host: eigensolver launch.  algo 0 = default (cluster-resident when a 16-CTA cluster can be scheduled, else cooperative),
// 1 = cluster-resident, 2 = cooperative.  bar / offmax (cooperative version only) must be zeroed on the stream before.
int run_jacobi(double* Wm, int n_layers, int k, unsigned* bar, unsigned long long* offmax, int* sweeps_out, int algo, const char* fn,
               cudaStream_t st) {
  JacobiParams jp;
  jp.W = Wm; jp.bar = bar; jp.offmax = offmax; jp.sweeps_out = sweeps_out; jp.k = k;
  void* kargs[] = {&jp};
  cudaError_t e;
  if (algo == 1 && !jacobi_cluster_available()) {
    set_error("%s: a %d-CTA cluster of the Jacobi eigensolver cannot be scheduled on this device", fn, kCS);
    return DKD_E_LAUNCH;
  }
  if (algo == 1 || (algo == 0 && jacobi_cluster_available())) {
    e = launch_jacobi_cluster(jp, n_layers, st);
  } else if (JacobiCfg<8>::CTAS * n_layers <= kNumSMs) {
    cudaFuncSetAttribute(jacobi_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)JacobiCfg<8>::SMEM);
    e = cudaLaunchCooperativeKernel((const void*)jacobi_kernel<8>, dim3(JacobiCfg<8>::CTAS, n_layers), dim3(JacobiCfg<8>::THREADS), kargs,
                                    JacobiCfg<8>::SMEM, st);
  } else {
    cudaFuncSetAttribute(jacobi_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)JacobiCfg<16>::SMEM);
    e = cudaLaunchCooperativeKernel((const void*)jacobi_kernel<16>, dim3(JacobiCfg<16>::CTAS, n_layers), dim3(JacobiCfg<16>::THREADS),
                                    kargs, JacobiCfg<16>::SMEM, st);
  }
  if (e != cudaSuccess) {
    set_error("%s: launch of the Jacobi eigensolver failed: %s", fn, cudaGetErrorString(e));
    cudaGetLastError();
    return DKD_E_LAUNCH;
  }
  return check_launch("dkd_lrkd: Jacobi eigensolver");
}

// ---------------------------------------------------------------- 4. select top-k, build fused operands
struct SelectParams {
  const double* W;                 // [L][n][n] after Jacobi: column j = lambda_j v_j
  const float* head_w[kMaxLayers];  // W' [k, Ds]
  const float* head_b[kMaxLayers];  // b' [k] or null
  float* Vk_out[kMaxLayers];        // [k, n] or null
  float* S_out[kMaxLayers];         // [k] or null
  __nv_bfloat16* Wcat;             // [L][P][BN][Ds + n]   K-major operand [W' | -V_k], rows >= k zero
  __nv_bfloat16* Wt;               // [L][P][Ds][BN]       W'^T (dgrad operand), cols >= k zero
  float* bias_pad;                 // [L][BN]
  double* lam;                     // [L][n] column norms (scratch between the two select kernels)
  int* order;                      // [L][n] order[r] = column with rank r
  float* sgn;                      // [L][n]
  int k, BN, Ds, P;
};

// 4a. column norms (= eigenvalues) and the sign convention: one warp per column (coalesced 256-byte reads), 8 columns per
// CTA so that the columns' global-memory round trips overlap; the largest-magnitude component is found with its index
// so that ties resolve to the first row, as a sequential scan would.  Then one CTA per layer ranks the norms.
__global__ void __launch_bounds__(256) eig_norm_kernel(SelectParams p) {
  constexpr int n = kN;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int layer = blockIdx.x / (n / 8), j = (blockIdx.x % (n / 8)) * 8 + warp;
  const double* col = p.W + (size_t)layer * n * n + (size_t)j * n;
  // (the magnitude is tracked in its own variable: with `fabs(v) > fabs(big)` nvcc 12.9 drops the fabs of `big` in the
  // second unrolled comparison — DSETP.GT |v1|, v0 in the SASS — and a negative first element loses)
  double a = 0.0, big = 0.0, mag = 0.0;
  int bi = n;
#pragma unroll
  for (int k = 0; k < n / 32; ++k) {
    const double v = col[lane + 32 * k], av = fabs(v);
    a = fma(v, v, a);
    if (av > mag) { mag = av; big = v; bi = lane + 32 * k; }
  }
  a = warp_sum_d(a);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double om = __shfl_xor_sync(0xffffffffu, mag, o);
    const double ob = __shfl_xor_sync(0xffffffffu, big, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (om > mag || (om == mag && oi < bi)) { mag = om; big = ob; bi = oi; }
  }
  if (lane == 0) {
    p.lam[layer * n + j] = sqrt(a);
    p.sgn[layer * n + j] = big < 0.0 ? -1.f : 1.f;   // sign convention: largest-magnitude component positive
  }
}
__global__ void __launch_bounds__(kN) eig_rank_kernel(SelectParams p) {
  constexpr int n = kN;
  __shared__ double lam[n];
  const int layer = blockIdx.x, j = threadIdx.x;
  lam[j] = p.lam[layer * n + j];
  __syncthreads();
  const double v = lam[j];
  int rank = 0;
  for (int i = 0; i < n; ++i) rank += (lam[i] > v) || (lam[i] == v && i < j);
  p.order[layer * n + rank] = j;
}

// 4b. one CTA per (output row r, layer): row r of [W' | -V_k] and column r of W'^T as bf16 planes
__global__ void __launch_bounds__(kN) select_kernel(SelectParams p) {
  constexpr int n = kN;
  const int r = blockIdx.x, layer = blockIdx.y, j = threadIdx.x;
  const double* W = p.W + (size_t)layer * n * n;
  const int K = p.Ds + n;
  __nv_bfloat16* wc = p.Wcat + (size_t)layer * p.P * p.BN * K;
  __nv_bfloat16* wt = p.Wt + (size_t)layer * p.P * p.Ds * p.BN;
  const float* hw = p.head_w[layer];
  const float* hb = p.head_b[layer];
  float* vk = p.Vk_out[layer];
  float* so = p.S_out[layer];
  auto put = [&](__nv_bfloat16* base, size_t plane_stride, size_t off, float x) {
    const __nv_bfloat16 hi = __float2bfloat16_rn(x);
    base[off] = hi;
    if (p.P == 2) base[plane_stride + off] = __float2bfloat16_rn(x - __bfloat162float(hi));
  };
  const bool real = r < p.k;
  float v = 0.f;                       // V part: thread j = channel
  if (real) {
    const int col = p.order[layer * n + r];
    const double l = p.lam[layer * n + col];
    v = l > 0.0 ? (float)(W[(size_t)col * n + j] / l) * p.sgn[layer * n + col] : 0.f;
    if (vk) vk[(size_t)r * n + j] = v;
    if (so && j == 0) so[r] = (float)sqrt(l);
  }
  put(wc, (size_t)p.BN * K, (size_t)r * K + p.Ds + j, -v);
  if (j < p.Ds) {
    const float w = real ? hw[(size_t)r * p.Ds + j] : 0.f;
    put(wc, (size_t)p.BN * K, (size_t)r * K + j, w);
    put(wt, (size_t)p.Ds * p.BN, (size_t)j * p.BN + r, w);
  }
  if (j == 0) p.bias_pad[(size_t)layer * p.BN + r] = (real && hb) ? hb[r] : 0.f;
}

// ---------------------------------------------------------------- 5. residual GEMM over the concatenated K = Ds + Dt
struct ConcatLoaderParams {
  CUtensorMap tmS, tmT, tmW;
  int s_blocks;   // Ds / 64
  int k_blocks;   // (Ds + Dt) / 64
  int nterms;
};
template <class Cfg>
struct ConcatLoader {
  using Params = ConcatLoaderParams;
  static constexpr uint32_t TX_BYTES = Cfg::STAGE_BYTES;
  static __device__ __forceinline__ int num_k_iters(const Params& p) { return p.k_blocks * p.nterms; }
  static __device__ __forceinline__ void prefetch(const Params& p) {
    sm100::tma_prefetch_desc(&p.tmS);
    sm100::tma_prefetch_desc(&p.tmT);
    sm100::tma_prefetch_desc(&p.tmW);
  }
  static __device__ __forceinline__ void issue(const Params& p, int kit, int mt, int nt, uint8_t* sA, uint8_t* sB, uint64_t* bar) {
    const int term = kit / p.k_blocks, kb = kit - term * p.k_blocks;
    int pa, pb;
    term_planes(term, p.nterms, pa, pb);
    if (kb < p.s_blocks) sm100::tma_load_3d(sA, &p.tmS, bar, kb * 64, mt * Cfg::BM, pa);
    else sm100::tma_load_3d(sA, &p.tmT, bar, (kb - p.s_blocks) * 64, mt * Cfg::BM, pa);
    sm100::tma_load_3d(sB, &p.tmW, bar, kb * 64, nt * Cfg::BN, pb);
  }
};

using DgradCfg = GemmCfg<192, 1, 4, 2>;
using WgradCfg = GemmNtCfg<3, true, 208, 0, 4>;

struct Workspace {
  __nv_bfloat16 *Tp[kMaxLayers], *Sp, *Gp, *Wcat, *Wt, *ones;
  float *part, *bias_pad;
  double *gsum, *W, *sumsq, *partials;
  unsigned* bar;
  unsigned long long* offmax;
  size_t bytes;
};
constexpr int kSumsqBlocks = 296;

Workspace carve(void* base, int L, int64_t M, int Ds, int BN, int PT, int P) {
  Workspace w;
  size_t off = 0;
  auto take = [&](size_t n) { size_t o = off; off = align_up(off + n, 1024); return reinterpret_cast<char*>(base) + o; };
  for (int l = 0; l < kMaxLayers; ++l) w.Tp[l] = l < L ? reinterpret_cast<__nv_bfloat16*>(take((size_t)PT * M * kN * 2)) : nullptr;
  w.Sp = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * M * Ds * 2));
  w.Gp = reinterpret_cast<__nv_bfloat16*>(take((size_t)P * M * BN * 2));
  w.Wcat = reinterpret_cast<__nv_bfloat16*>(take((size_t)L * P * BN * (Ds + kN) * 2));
  w.Wt = reinterpret_cast<__nv_bfloat16*>(take((size_t)L * P * Ds * BN * 2));
  w.ones = reinterpret_cast<__nv_bfloat16*>(take((size_t)2 * 64 * 64 * 2));
  w.part = reinterpret_cast<float*>(take((size_t)kNumSMs * kN * kN * 4 / 3 + (size_t)kN * kN * 4));
  w.bias_pad = reinterpret_cast<float*>(take((size_t)L * BN * 4));
  w.gsum = reinterpret_cast<double*>(take((size_t)kN * kN * 8));
  w.W = reinterpret_cast<double*>(take((size_t)L * kN * kN * 8));
  w.sumsq = reinterpret_cast<double*>(take((size_t)kSumsqBlocks * kN * 8));
  w.partials = reinterpret_cast<double*>(take((size_t)kNumSMs * 8));
  w.bar = reinterpret_cast<unsigned*>(take((size_t)kMaxLayers * 4));
  w.offmax = reinterpret_cast<unsigned long long*>(take((size_t)kMaxLayers * 2 * 8));
  w.bytes = off;
  return w;
}

int bn_for_rank(int rank) { return rank <= 64 ? 64 : 128; }

template <int BN>
int run_residual(const Workspace& ws, int layer, int64_t M, int Ds, int P, float gscale, cudaStream_t st, int* grid_out) {
  using Cfg = GemmCfg<BN, 1, 4, 2>;
  using L = ConcatLoader<Cfg>;
  using E = ResidualMseEpi<Cfg>;
  GemmParams<L, E> p;
  const int K = Ds + kN;
  int rc = make_plane_tmap(&p.ld.tmS, ws.Sp, P, M, Ds, Ds, M * Ds, Cfg::BM, "lrkd S");
  if (rc != DKD_OK) return rc;
  rc = make_plane_tmap(&p.ld.tmT, ws.Tp[layer], P, M, kN, kN, M * kN, Cfg::BM, "lrkd T");
  if (rc != DKD_OK) return rc;
  rc = make_plane_tmap(&p.ld.tmW, ws.Wcat + (size_t)layer * P * BN * K, P, BN, K, K, (int64_t)BN * K, Cfg::BN, "lrkd [W'|-V]");
  if (rc != DKD_OK) return rc;
  p.ld.s_blocks = Ds / 64; p.ld.k_blocks = K / 64; p.ld.nterms = P == 2 ? 3 : 1;
  p.ep.t = nullptr; p.ep.bias = ws.bias_pad + (size_t)layer * BN; p.ep.G = ws.Gp; p.ep.partials = ws.partials;
  p.ep.M = M; p.ep.N = BN; p.ep.n_tok = 1; p.ep.Tt = 1; p.ep.t_off = 0; p.ep.planes = P; p.ep.gscale = gscale; p.ep.t_is_bf16 = 0;
  p.m_tiles = (int)((M + Cfg::BM - 1) / Cfg::BM);
  p.n_tiles = 1;
  const int grid = min(kNumSMs, p.m_tiles);
  auto kern = gemm_tn_kernel<Cfg, L, E>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
  kern<<<grid, Cfg::THREADS, Cfg::SMEM, st>>>(p);
  *grid_out = grid;
  return check_launch("dkd_lrkd_fwdbwd: residual GEMM");
}

}  // namespace
}  // namespace dkd

extern "C" {

size_t dkd_lrkd_workspace_bytes(int n_layers, int64_t B, int n_tok, int Ds, int Dt, int rank, int dtype, int precision) {
  using namespace dkd;
  if (n_layers < 1 || n_layers > kMaxLayers || Dt != kN) return 0;
  const int P = precision == DKD_PREC_BF16X3 ? 2 : 1;
  const int PT = dtype == DKD_F32 ? 3 : P;
  return carve(nullptr, n_layers, B * n_tok, Ds, bn_for_rank(rank), PT, P).bytes;
}

size_t dkd_lrkd_eigensolve_workspace_bytes(void) { return 1024; }

int dkd_lrkd_eigensolve(double* Wm, int n_layers, int k, int* sweeps_out, int algo, void* workspace, size_t workspace_bytes,
                        dkd_stream_t stream) {
  using namespace dkd;
  const char* fn = "dkd_lrkd_eigensolve";
  DKD_REQUIRE(Wm != nullptr && workspace != nullptr, DKD_E_SHAPE, "%s: null pointer", fn);
  DKD_REQUIRE(n_layers >= 1 && n_layers <= kMaxLayers, DKD_E_SHAPE, "%s: n_layers must be 1..%d", fn, kMaxLayers);
  DKD_REQUIRE(k >= 1 && k <= kN, DKD_E_SHAPE, "%s: k must be 1..%d", fn, kN);
  DKD_REQUIRE(algo >= 0 && algo <= 2, DKD_E_UNSUPPORTED, "%s: algo must be 0 (default), 1 (cluster) or 2 (cooperative)", fn);
  DKD_REQUIRE(workspace_bytes >= 1024, DKD_E_WORKSPACE, "%s: workspace %zu < 1024", fn, workspace_bytes);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  cudaMemsetAsync(workspace, 0, 1024, st);
  unsigned* bar = reinterpret_cast<unsigned*>(workspace);
  unsigned long long* offmax = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(workspace) + 512);
  return run_jacobi(Wm, n_layers, k, bar, offmax, sweeps_out, algo, fn, st);
}

int dkd_lrkd_fwdbwd(int n_layers, const void* const* s, const void* const* t, const float* const* W, const float* const* bias,
                    const float* coef, int64_t B, int Ts, int s_off, int Tt, int t_off, int n_tok, int Ds, int Dt, int rank,
                    int dtype, int precision, void* const* g_s, float* const* g_W, float* const* g_b, float* loss,
                    float* const* Vk_out, float* const* S_out, int* sweeps_out, void* workspace, size_t workspace_bytes,
                    dkd_stream_t stream) {
  using namespace dkd;
  int rc = dkd_check_device();
  if (rc != DKD_OK) return rc;
  const char* fn = "dkd_lrkd_fwdbwd";
  DKD_REQUIRE(dtype == DKD_F32 || dtype == DKD_BF16, DKD_E_DTYPE, "%s: dtype %d", fn, dtype);
  DKD_REQUIRE(precision == DKD_PREC_BF16 || precision == DKD_PREC_BF16X3, DKD_E_UNSUPPORTED, "%s: precision %d", fn, precision);
  DKD_REQUIRE(n_layers >= 1 && n_layers <= kMaxLayers, DKD_E_SHAPE, "%s: 1..%d layers", fn, kMaxLayers);
  DKD_REQUIRE(B > 0 && n_tok > 0 && s_off >= 0 && t_off >= 0 && Ts >= s_off + n_tok && Tt >= t_off + n_tok, DKD_E_SHAPE,
              "%s: bad token geometry", fn);
  DKD_REQUIRE(Ds == 192 && Dt == kN, DKD_E_SHAPE, "%s: built for widths 192 -> 384, got %d -> %d", fn, Ds, Dt);
  DKD_REQUIRE(rank >= 1 && rank <= 128, DKD_E_SHAPE, "%s: rank %d outside [1, 128]", fn, rank);
  DKD_REQUIRE(s && t && W && coef && loss && workspace, DKD_E_SHAPE, "%s: null pointer", fn);
  for (int l = 0; l < n_layers; ++l) {
    DKD_REQUIRE(s[l] && t[l] && W[l], DKD_E_SHAPE, "%s: null pointer in layer %d", fn, l);
    DKD_REQUIRE(g_s == nullptr || (((uintptr_t)g_s[l]) & 31) == 0, DKD_E_ALIGN, "%s: g_s[%d] must be 32-byte aligned", fn, l);
  }
  DKD_REQUIRE((((uintptr_t)workspace) & 1023) == 0, DKD_E_ALIGN, "%s: workspace must be 1024-byte aligned", fn);
  const int P = precision == DKD_PREC_BF16X3 ? 2 : 1;
  const int PT = dtype == DKD_F32 ? 3 : P;
  const int BN = bn_for_rank(rank);
  const int64_t M = B * n_tok;
  DKD_REQUIRE(M < (1ll << 31) - 256, DKD_E_SHAPE, "%s: too many rows", fn);
  DKD_REQUIRE(M >= rank, DKD_E_SHAPE, "%s: rank %d exceeds the %lld teacher rows", fn, rank, (long long)M);
  Workspace ws = carve(workspace, n_layers, M, Ds, BN, PT, P);
  DKD_REQUIRE(workspace_bytes >= ws.bytes, DKD_E_WORKSPACE, "%s: workspace %zu < %zu", fn, workspace_bytes, ws.bytes);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  bool want_grads = false;
  for (int l = 0; l < n_layers; ++l)
    want_grads = want_grads || (g_s && g_s[l]) || (g_W && g_W[l]) || (g_b && g_b[l]);

  cudaMemsetAsync(ws.bar, 0, (size_t)kMaxLayers * 4, st);
  cudaMemsetAsync(ws.offmax, 0, (size_t)kMaxLayers * 2 * 8, st);

  // ---- 1-2. per layer: teacher planes, Gram partials, fp64 reduction
  for (int l = 0; l < n_layers; ++l) {
    if (dtype == DKD_F32)
      teacher_planes_kernel<float><<<kSumsqBlocks, 192, 0, st>>>(reinterpret_cast<const float*>(t[l]), B, Tt, t_off, n_tok, PT, ws.Tp[l], ws.sumsq);
    else
      teacher_planes_kernel<__nv_bfloat16><<<kSumsqBlocks, 192, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(t[l]), B, Tt, t_off, n_tok, PT, ws.Tp[l], ws.sumsq);
    rc = check_launch("dkd_lrkd_fwdbwd: teacher planes");
    if (rc != DKD_OK) return rc;
    using Cfg = GramCfg;
    using L = NtGramLoader;
    GemmNtParamsT<Cfg, L> p;
    rc = make_plane_tmap(&p.ld.tmA, ws.Tp[l], PT, M, kN, kN, M * kN, Cfg::KROWS, "lrkd Gram A");
    if (rc != DKD_OK) return rc;
    p.ld.tmB = p.ld.tmA;
    p.ld.tmOnes = p.ld.tmA;
    p.ld.na_tiles = kN / 128;
    p.ld.total_row_blocks = (int)((M + Cfg::KROWS - 1) / Cfg::KROWS);
    nt_make_splits(p.ld.total_row_blocks, kNumSMs / p.ld.na_tiles, &p.ld.splits, &p.ld.row_blocks_per_split);
    p.ld.b_col0 = 0; p.ld.ldd = kN;
    p.ep.D = ws.part; p.ep.Dcol = nullptr; p.ep.ldd = kN; p.ep.alpha = 1.f; p.ep.store = 1; p.ep.rows_valid = 128;
    p.nterms = dtype == DKD_F32 ? 6 : 1;
    const int grid = min(kNumSMs, p.ld.na_tiles * p.ld.splits);
    auto kern = gemm_nt_kernel<Cfg, L>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
    kern<<<grid, Cfg::THREADS, Cfg::SMEM, st>>>(p);
    rc = check_launch("dkd_lrkd_fwdbwd: Gram GEMM");
    if (rc != DKD_OK) return rc;
    gram_reduce_kernel<<<(kN * kN + 255) / 256, 256, 0, st>>>(ws.part, p.ld.splits, ws.gsum);
    rc = check_launch("dkd_lrkd_fwdbwd: Gram reduce");
    if (rc != DKD_OK) return rc;
    gram_symmetrize_kernel<<<(kN * kN + 255) / 256, 256, 0, st>>>(ws.gsum, ws.sumsq, kSumsqBlocks, ws.W + (size_t)l * kN * kN);
    rc = check_launch("dkd_lrkd_fwdbwd: Gram symmetrize");
    if (rc != DKD_OK) return rc;
  }

  // ---- 3. eigenvectors: all layers in one launch
  rc = run_jacobi(ws.W, n_layers, rank, ws.bar, ws.offmax, sweeps_out, 0, fn, st);
  if (rc != DKD_OK) return rc;

  // ---- 4. top-k selection and fused operands
  {
    SelectParams sp{};
    sp.W = ws.W;
    for (int l = 0; l < n_layers; ++l) {
      sp.head_w[l] = W[l];
      sp.head_b[l] = bias ? bias[l] : nullptr;
      sp.Vk_out[l] = Vk_out ? Vk_out[l] : nullptr;
      sp.S_out[l] = S_out ? S_out[l] : nullptr;
    }
    sp.Wcat = ws.Wcat; sp.Wt = ws.Wt; sp.bias_pad = ws.bias_pad; sp.k = rank; sp.BN = BN; sp.Ds = Ds; sp.P = P;
    // scratch: the Gram sum buffer is free once every layer's matrix has been built
    sp.lam = ws.gsum;
    sp.order = reinterpret_cast<int*>(ws.gsum + (size_t)kMaxLayers * kN);
    sp.sgn = reinterpret_cast<float*>(sp.order + (size_t)kMaxLayers * kN);
    eig_norm_kernel<<<n_layers * (kN / 8), 256, 0, st>>>(sp);
    rc = check_launch("dkd_lrkd_fwdbwd: eigenvalues");
    if (rc != DKD_OK) return rc;
    eig_rank_kernel<<<n_layers, kN, 0, st>>>(sp);
    rc = check_launch("dkd_lrkd_fwdbwd: eigenvalue ranking");
    if (rc != DKD_OK) return rc;
    select_kernel<<<dim3(BN, n_layers), kN, 0, st>>>(sp);
    rc = check_launch("dkd_lrkd_fwdbwd: select");
    if (rc != DKD_OK) return rc;
  }

  // ---- 5-7. per layer: residual GEMM (+ loss), dgrad, wgrad
  for (int l = 0; l < n_layers; ++l) {
    rc = launch_tokens_to_planes(s[l], dtype, B, Ts, s_off, n_tok, Ds, P, nullptr, ws.Sp, st);
    if (rc != DKD_OK) return rc;
    const float c = coef[l] / ((float)M * (float)rank);
    int grid = 0;
    rc = BN == 64 ? run_residual<64>(ws, l, M, Ds, P, 2.f * c, st, &grid) : run_residual<128>(ws, l, M, Ds, P, 2.f * c, st, &grid);
    if (rc != DKD_OK) return rc;
    rc = launch_fold_partials(ws.partials, grid, c, loss, st);
    if (rc != DKD_OK) return rc;
    if (!want_grads) continue;
    void* gs = g_s ? g_s[l] : nullptr;
    float* gW = g_W ? g_W[l] : nullptr;
    float* gb = g_b ? g_b[l] : nullptr;
    if (gs) {
      using Cfg = DgradCfg;
      using L = PlaneLoader<Cfg>;
      using E = StoreRowsEpi<Cfg>;
      GemmParams<L, E> p;
      rc = make_plane_tmap(&p.ld.tmA, ws.Gp, P, M, BN, BN, M * BN, Cfg::BM, "lrkd G");
      if (rc != DKD_OK) return rc;
      rc = make_plane_tmap(&p.ld.tmB, ws.Wt + (size_t)l * P * Ds * BN, P, Ds, BN, BN, (int64_t)Ds * BN, Cfg::BN, "lrkd W'^T");
      if (rc != DKD_OK) return rc;
      p.ld.k_blocks = BN / 64; p.ld.nterms = P == 2 ? 3 : 1;
      p.ep.out = gs; p.ep.drop_mask = nullptr; p.ep.bias = nullptr; p.ep.alpha = 1.f; p.ep.M = M; p.ep.N_total = Ds; p.ep.n_tok = n_tok;
      p.ep.T_out = Ts; p.ep.off = s_off; p.ep.out_is_bf16 = dtype == DKD_BF16;
      p.m_tiles = (int)((M + Cfg::BM - 1) / Cfg::BM); p.n_tiles = Ds / Cfg::BN;
      const int g2 = min(kNumSMs, p.m_tiles * p.n_tiles);
      auto kern = gemm_tn_kernel<Cfg, L, E>;
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
      kern<<<g2, Cfg::THREADS, Cfg::SMEM, st>>>(p);
      rc = check_launch("dkd_lrkd_fwdbwd: dgrad GEMM");
      if (rc != DKD_OK) return rc;
    }
    if (gW || gb) {
      using Cfg = WgradCfg;
      using L = NtPlainLoader<Cfg>;
      DKD_REQUIRE(gW != nullptr, DKD_E_UNSUPPORTED, "%s: g_b without g_W is not supported", fn);
      GemmNtParamsT<Cfg, L> p;
      rc = make_plane_tmap(&p.ld.tmA, ws.Gp, P, M, BN, BN, M * BN, Cfg::KROWS, "lrkd G^T");
      if (rc != DKD_OK) return rc;
      rc = make_plane_tmap(&p.ld.tmB, ws.Sp, P, M, Ds, Ds, M * Ds, Cfg::KROWS, "lrkd S (wgrad)");
      if (rc != DKD_OK) return rc;
      rc = make_plane_tmap(&p.ld.tmOnes, ws.ones, 2, 64, 64, 64, 64 * 64, Cfg::KROWS, "ones tile");
      if (rc != DKD_OK) return rc;
      rc = launch_fill_ones_tile(ws.ones, st);
      if (rc != DKD_OK) return rc;
      cudaMemsetAsync(gW, 0, (size_t)rank * Ds * sizeof(float), st);
      if (gb) cudaMemsetAsync(gb, 0, (size_t)rank * sizeof(float), st);
      p.ep.D = gW; p.ep.Dcol = gb; p.ep.ldd = Ds; p.ep.alpha = 1.f; p.ep.store = 0; p.ep.rows_valid = rank;
      p.ld.ldd = Ds; p.ld.na_tiles = 1; p.ld.b_col0 = 0;
      p.ld.total_row_blocks = (int)((M + Cfg::KROWS - 1) / Cfg::KROWS);
      nt_make_splits(p.ld.total_row_blocks, kNumSMs, &p.ld.splits, &p.ld.row_blocks_per_split);
      p.nterms = P == 2 ? 3 : 1;
      const int g3 = min(kNumSMs, p.ld.splits);
      auto kern = gemm_nt_kernel<Cfg, L>;
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
      kern<<<g3, Cfg::THREADS, Cfg::SMEM, st>>>(p);
      rc = check_launch("dkd_lrkd_fwdbwd: wgrad GEMM");
      if (rc != DKD_OK) return rc;
    }
  }
  return DKD_OK;
}

}  // extern "C"
