// Fused base-CE + soft/hard KD on logits, forward + backward in one sweep.
// Reference arithmetic: model/loss.py:35 (timm SoftTargetCrossEntropy / LabelSmoothingCrossEntropy,
// loss.py:244-249), :57-64 (soft KD, note the /numel), :66-67 (hard KD), :241 (mix).
//
// One CTA per batch row.  The row of each operand is read from HBM exactly once (held in registers
// when C <= THREADS*VEC*NV, otherwise re-read through L1/L2), max / log-sum-exp are block-reduced,
// both gradient rows are written in the same launch, and a one-CTA launch behind it folds the per-row
// partials in a fixed order (deterministic) into {total, base, kd}.
// HBM-bound: algorithmic bytes = (reads + grad writes) * B * C * sizeof(elt); no tensor-core work.
#include "common.cuh"

// Phase stamps (point, value the stamp must wait for) of the one-CTA-per-row kernel and of the fold.
// tools/probes/logit_phase_probe.cu defines both before including this file; the library compiles them to nothing.
#ifndef DKD_LOGIT_STAMP
#define DKD_LOGIT_STAMP(point, dep) ((void)0)
#endif
#ifndef DKD_LOGIT_FOLD_STAMP
#define DKD_LOGIT_FOLD_STAMP(point, dep) ((void)0)
#endif

namespace dkd {
namespace {

constexpr int kThreads = 128;

// e^x through MUFU.EX2 (2 instructions instead of expf's ~20).  Arguments here are <= 0 (maximum subtracted) and O(10):
// the relative error (~2^-22 plus the rounding of x*log2(e)) is ~1e-6, far inside the 1e-5 / 1e-4 parity gates —
// and with ~100 instructions per logit the exact expf made the kernel issue-bound instead of HBM-bound.
__device__ __forceinline__ float fexp(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x * 1.4426950408889634f));
  return y;
}
// e^(x*k - m) with k*log2(e) and m*log2(e) pre-multiplied by the caller: one FFMA + MUFU
__device__ __forceinline__ float fexp2(float x, float k2, float m2) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(fmaf(x, k2, -m2)));
  return y;
}

// both lanes of a pair: 2^(x)
__device__ __forceinline__ float2 ex2_2(float2 x) {
  float2 y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y.x) : "f"(x.x));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y.y) : "f"(x.y));
  return y;
}

struct LogitKdParams {
  const void* z;      // outputs
  const void* zk;     // outputs_kd
  const void* zt;     // teacher logits
  const void* y;      // soft labels or int64 ids
  void* gz;
  void* gzk;
  float* loss_out;    // [3]
  float* row_base;    // [B]
  float* row_kd;      // [B]
  unsigned int* ticket;
  int64_t B, C;
  int label_kind, kd_kind;
  float smoothing, alpha, tau;
  const float* mix_lam;   // int labels only: if set, row r's target is lam * smooth_onehot(y[r]) + (1 - lam) * smooth_onehot(y[B-1-r])
};

// NV > 0: row cached in registers (C <= kThreads*VEC*NV).  NV == 0: streaming (re-read) path.
// One batch row: block-reduced maxima / sums, both gradient rows written, per-row loss partials stored.
// z / zk / zt / y point at the row's operands — in global memory (one CTA per row) or in a shared-memory stage
// filled by bulk copies (streaming kernel below); the arithmetic is the same code.
// LK / KK: label_kind / kd_kind as compile-time constants (kRuntimeMode = read them from the parameters).  The common
// modes are instantiated so that the per-element mode tests vanish from the unrolled inner loops.
constexpr int kRuntimeMode = -2;
constexpr float kL2e = 1.4426950408889634f;
// gz_row / gzk_row: where this row's gradients go (global rows, or the ring stage of the streaming kernel; null = not
// wanted).  PACK2: fp32-pair arithmetic in passes 2 and 3.  publish(base_row, kd_row) runs in every thread once the row's
// loss terms are known, after pass 3 has issued the gradient stores.
template <typename T, int VEC, int NV, int THREADS = kThreads, int LK = kRuntimeMode, int KK = kRuntimeMode,
          bool PACK2 = (THREADS == kThreads), typename Publish>
__device__ __forceinline__ void logit_row(const LogitKdParams& p, int64_t row, const T* z, const T* zk, const T* zt, const T* y,
                                          T* gz_row, T* gzk_row, float* scratch, int* s_arg, float* s_argv, float& base_out,
                                          float& kd_out, Publish&& publish) {
  const int64_t C = p.C;
  const int label_kind = LK == kRuntimeMode ? p.label_kind : LK;
  const int kd_kind = KK == kRuntimeMode ? p.kd_kind : KK;
  const int tid = THREADS == 32 ? (int)(threadIdx.x & 31) : (int)threadIdx.x;   // THREADS == 32: one warp per row
  const int64_t label = label_kind == 1 ? reinterpret_cast<const int64_t*>(p.y)[row] : -1;
  // Mixup / CutMix targets generated on the fly (timm mixup_target, tools/train.py:288-295 + engine.py:16-18): the
  // [B, C] soft-label tensor is never materialised — 5 instead of 6 row streams.  label2 = -1 when not mixing.
  const bool mixing = label_kind == 1 && p.mix_lam != nullptr;
  const int64_t label2 = mixing ? reinterpret_cast<const int64_t*>(p.y)[p.B - 1 - row] : -1;
  const float lam = mixing ? __ldg(p.mix_lam) : 1.f;
  const float invT = kd_kind == 1 ? 1.f / p.tau : 1.f;

  constexpr int NVR = NV > 0 ? NV : 1;
  float rz[NVR][VEC], rk[NVR][VEC], rt[NVR][VEC], ry[NVR][VEC];
  const int nchunk = (int)((C + (int64_t)THREADS * VEC - 1) / ((int64_t)THREADS * VEC));

  auto col_of = [&](int it) -> int64_t { return ((int64_t)it * THREADS + tid) * VEC; };
  // Loads are unconditional and branch-free: columns past the row end are clamped to column 0 (the passes test
  // col < C themselves), and operands a mode does not use alias one it does (their values are never read; the
  // duplicate loads hit L1).  Kernel-uniform branches on the mode split the loads into basic blocks, each exposing
  // its own DRAM round trip (ncu: six equal long-scoreboard stalls per row); this way they issue back to back.
  const T* any = label_kind >= 0 ? z : zk;
  const T* lz = label_kind >= 0 ? z : any;
  const T* lzk = kd_kind ? zk : any;
  const T* lzt = kd_kind ? zt : any;
  const T* ly = label_kind == 0 ? y : any;
  auto load4 = [&](int it, float (&a)[VEC], float (&b)[VEC], float (&c)[VEC], float (&d)[VEC]) {
    const int64_t col0 = col_of(it);
    const int64_t col = col0 < C ? col0 : 0;  // C % VEC == 0 by construction
    Vec<T, VEC>::load(lz + col, a);
    Vec<T, VEC>::load(lzk + col, b);
    Vec<T, VEC>::load(lzt + col, c);
    Vec<T, VEC>::load(ly + col, d);
    if (label_kind < 0) {
#pragma unroll
      for (int v = 0; v < VEC; ++v) a[v] = 0.f;
    }
  };

  // ---- pass 1: maxima (and teacher argmax for hard KD) -------------------------------------
  // maxima of the RAW logits; zk / zt are scaled by invT after the reduction (invT > 0 and rounding is monotone, so
  // max_i fl(x_i * invT) == fl(max_i x_i * invT) exactly) — two multiplies per logit fewer
  float mx[3] = {-INFINITY, -INFINITY, -INFINITY};  // z, zk, zt
  float best = -INFINITY;
  int64_t best_i = INT64_MAX;
  auto pass1 = [&](int it, float (&a)[VEC], float (&b)[VEC], float (&c)[VEC]) {
    const int64_t col = col_of(it);
    if (col < C) {
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        mx[0] = fmaxf(mx[0], a[v]);
        if (kd_kind) {
          mx[1] = fmaxf(mx[1], b[v]);
          mx[2] = fmaxf(mx[2], c[v]);
          if (kd_kind == 2 && c[v] > best) { best = c[v]; best_i = col + v; }  // first max within thread
        }
      }
    }
  };
  if constexpr (NV > 0) {
    // all of the row's loads are issued before the first value is used: one DRAM round trip per row, not one per chunk
#pragma unroll
    for (int it = 0; it < NV; ++it)
      if (it < nchunk) load4(it, rz[it], rk[it], rt[it], ry[it]);
#pragma unroll
    for (int it = 0; it < NV; ++it)
      if (it < nchunk) pass1(it, rz[it], rk[it], rt[it]);
  } else {
    for (int it = 0; it < nchunk; ++it) {
      load4(it, rz[0], rk[0], rt[0], ry[0]);
      pass1(it, rz[0], rk[0], rt[0]);
    }
  }
  DKD_LOGIT_STAMP(1, mx[0]);   // loads landed
  block_max<3, THREADS>(mx, scratch);
  DKD_LOGIT_STAMP(2, mx[0]);
  mx[1] *= invT;
  mx[2] *= invT;
  int64_t tgt = label;  // index whose one-hot enters the KD gradient (hard) -- label handled separately
  int64_t hard_idx = -1;
  if (kd_kind == 2) {
    // argmax with first-index tie-break: warp shuffle, then across warps
    float bv = best;
    long long bi = (long long)best_i;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    if constexpr (THREADS > 32) {
      __syncthreads();
      if ((threadIdx.x & 31) == 0) { s_argv[threadIdx.x >> 5] = bv; s_arg[threadIdx.x >> 5] = (int)bi; }
      __syncthreads();
      bv = s_argv[0]; bi = s_arg[0];
#pragma unroll
      for (int w = 1; w < THREADS / 32; ++w) {
        if (s_argv[w] > bv || (s_argv[w] == bv && s_arg[w] < bi)) { bv = s_argv[w]; bi = s_arg[w]; }
      }
    }
    hard_idx = bi;
  }
  (void)tgt;

  // ---- pass 2: sums --------------------------------------------------------------------------
  // s[0]=sum exp(z-m0)  s[1]=sum exp(a-m1)  s[2]=sum exp(b-m2)  s[3]=sum exp(b-m2)*(b-a)   (a = zk/T, b = zt/T;
  //                                              s[3] is accumulated on the raw logits and scaled by 1/T once)
  // t[0]=sum y          t[1]=sum y*z (soft labels) | sum z (int labels)   t[2]=z[label]  t[3]=zk[hard_idx]
  // In the register-resident case the exponentials replace the logits in rz / rk / rt (pass 3 needs only them,
  // the soft labels and the column index), so every exp is evaluated once.
  float st8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float (&s)[4] = *reinterpret_cast<float(*)[4]>(&st8[0]);
  float (&t)[4] = *reinterpret_cast<float(*)[4]>(&st8[4]);
  // Register-resident rows with an even vector width run pass 2 and pass 3 on fp32 PAIRS (FFMA2 / FADD2 / FMUL2): 22 %
  // fewer instructions per row.  Measured A/B on one B200: the latency-chain case (B = 256, 4-warp CTAs) gains
  // 5.87 -> 5.71 us; the large-batch 2-warp variant is bound by bytes in flight, not by issue, and loses 3 %
  // (56.2 -> 58.0 us at B = 16 384) — so only the small-batch shape uses the packed forms.
  constexpr bool PACKED = NV > 0 && VEC % 2 == 0 && PACK2;
  float2 S2[4], T2[2];   // pair accumulators of s[0..3], t[0..1]
#pragma unroll
  for (int k = 0; k < 4; ++k) S2[k] = make_float2(0.f, 0.f);
  T2[0] = T2[1] = make_float2(0.f, 0.f);
  auto pass2 = [&](int it, float (&a)[VEC], float (&b)[VEC], float (&c)[VEC], float (&d)[VEC]) {
    const int64_t col = col_of(it);
    if (col < C) {
      if constexpr (PACKED) {
        const float2 kz = splat2(kL2e), nm0 = splat2(-mx[0] * kL2e);
        const float2 kt = splat2(invT * kL2e), nm1 = splat2(-mx[1] * kL2e), nm2 = splat2(-mx[2] * kL2e);
#pragma unroll
        for (int v = 0; v < VEC; v += 2) {
          const float2 A = make_float2(a[v], a[v + 1]);
          const float2 ea = ex2_2(fma2(A, kz, nm0));
          S2[0] = add2(S2[0], ea);
          if (label_kind == 0) {
            const float2 D = make_float2(d[v], d[v + 1]);
            T2[0] = add2(T2[0], D);
            T2[1] = fma2(D, A, T2[1]);
          } else {
            T2[1] = add2(T2[1], A);
            if (col + v == label) t[2] = a[v];
            if (col + v + 1 == label) t[2] = a[v + 1];
            if (col + v == label2) t[0] = a[v];
            if (col + v + 1 == label2) t[0] = a[v + 1];
          }
          a[v] = ea.x; a[v + 1] = ea.y;
          if (kd_kind == 1) {
            const float2 Bv = make_float2(b[v], b[v + 1]), Cv = make_float2(c[v], c[v + 1]);
            const float2 eb = ex2_2(fma2(Cv, kt, nm2)), es = ex2_2(fma2(Bv, kt, nm1));
            S2[1] = add2(S2[1], es);
            S2[2] = add2(S2[2], eb);
            S2[3] = fma2(eb, sub2(Cv, Bv), S2[3]);
            b[v] = es.x; b[v + 1] = es.y;
            c[v] = eb.x; c[v + 1] = eb.y;
          } else if (kd_kind == 2) {
            const float2 Bv = make_float2(b[v], b[v + 1]);
            const float2 es = ex2_2(fma2(Bv, kz, nm1));
            S2[1] = add2(S2[1], es);
            if (col + v == hard_idx) t[3] = b[v];
            if (col + v + 1 == hard_idx) t[3] = b[v + 1];
            b[v] = es.x; b[v + 1] = es.y;
          }
        }
        return;
      }
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        const float ea = fexp2(a[v], kL2e, mx[0] * kL2e);
        s[0] += ea;
        if (label_kind == 0) { t[0] += d[v]; t[1] += d[v] * a[v]; }
        else { t[1] += a[v]; if (col + v == label) t[2] = a[v]; if (col + v == label2) t[0] = a[v]; }
        if (NV > 0) a[v] = ea;
        if (kd_kind == 1) {
          const float eb = fexp2(c[v], invT * kL2e, mx[2] * kL2e), es = fexp2(b[v], invT * kL2e, mx[1] * kL2e);
          s[1] += es;
          s[2] += eb;
          s[3] = fmaf(eb, c[v] - b[v], s[3]);
          if (NV > 0) { b[v] = es; c[v] = eb; }
        } else if (kd_kind == 2) {
          const float es = fexp2(b[v], kL2e, mx[1] * kL2e);
          s[1] += es;
          if (col + v == hard_idx) t[3] = b[v];
          if (NV > 0) b[v] = es;
        }
      }
    }
  };
  if constexpr (NV > 0) {
#pragma unroll
    for (int it = 0; it < NV; ++it) if (it < nchunk) pass2(it, rz[it], rk[it], rt[it], ry[it]);
  } else {
    for (int it = 0; it < nchunk; ++it) {
      load4(it, rz[0], rk[0], rt[0], ry[0]);
      pass2(it, rz[0], rk[0], rt[0], ry[0]);
    }
  }
  if constexpr (PACKED) {
#pragma unroll
    for (int k = 0; k < 4; ++k) s[k] = S2[k].x + S2[k].y;
    if (label_kind == 0) t[0] = T2[0].x + T2[0].y;   // (int labels: t[0] carries z[label2] of the mixed target)
    t[1] = T2[1].x + T2[1].y;
  }
  block_sum<8, THREADS>(st8, scratch);
  DKD_LOGIT_STAMP(3, s[0]);
  s[3] *= invT;

  // s[] >= 1 (the maximum contributes e^0): lg2.approx (absolute error 2^-22) and approximate reciprocals are exact
  // enough by two orders of magnitude, and the IEEE logf / division sequences were ~10 % of the kernel's instructions
  const float Bf = (float)p.B, Cf = (float)C;
  const float lse0 = mx[0] + __logf(s[0]);
  float base_row, kd_row = 0.f;
  if (label_kind < 0) base_row = 0.f;
  else if (label_kind == 0) base_row = lse0 * t[0] - t[1];
  else base_row = (1.f - p.smoothing) * (lse0 - (lam * t[2] + (1.f - lam) * t[0])) + p.smoothing * (lse0 - t[1] / Cf);

  // ---- pass 3: gradients -----------------------------------------------------------------------
  const float wb = (kd_kind == 0 ? 1.f : 1.f - p.alpha) / Bf;           // d total / d base_row
  const float wk = kd_kind == 1 ? p.alpha * p.tau / (Bf * Cf) : p.alpha / Bf;
  const float inv_s0 = __frcp_rn(s[0]), inv_s1 = kd_kind ? __frcp_rn(s[1]) : 0.f, inv_s2 = kd_kind == 1 ? __frcp_rn(s[2]) : 0.f;
  // the per-row factors are folded so that a gradient element costs one multiply and one FMA:
  //   g0 = e0 * k0 - y * wb  (soft labels) | e0 * k0 - (onehot * (1-eps) + eps/C) * wb  (int labels)
  //   g1 = es * k1 - et * k2 (soft KD)     | es * k1 - onehot * wk                      (hard KD)
  const float k0 = (label_kind == 0 ? inv_s0 * t[0] : inv_s0) * wb;
  const float k1 = inv_s1 * wk, k2 = inv_s2 * wk;
  const float sm_wb = p.smoothing / Cf * wb, hot_wb = (1.f - p.smoothing) * wb * lam, hot2_wb = (1.f - p.smoothing) * wb * (1.f - lam);
  T* gz = label_kind >= 0 ? gz_row : nullptr;
  T* gzk = kd_kind ? gzk_row : nullptr;
  auto pass3 = [&](int it, float (&a)[VEC], float (&b)[VEC], float (&c)[VEC], float (&d)[VEC]) {
    const int64_t col = col_of(it);
    if (col < C) {
      float g0[VEC], g1[VEC];
      if constexpr (PACKED) {
        const float2 K0 = splat2(k0), K1 = splat2(k1), NK2 = splat2(-k2), NWB = splat2(-wb), NSM = splat2(-sm_wb);
#pragma unroll
        for (int v = 0; v < VEC; v += 2) {
          const float2 e0 = make_float2(a[v], a[v + 1]);
          float2 r0;
          if (label_kind == 0) r0 = fma2(e0, K0, mul2(make_float2(d[v], d[v + 1]), NWB));
          else {
            r0 = fma2(e0, K0, NSM);
            if (col + v == label) r0.x -= hot_wb;
            if (col + v + 1 == label) r0.y -= hot_wb;
            if (col + v == label2) r0.x -= hot2_wb;
            if (col + v + 1 == label2) r0.y -= hot2_wb;
          }
          g0[v] = r0.x; g0[v + 1] = r0.y;
          if (kd_kind == 1) {
            const float2 r1 = fma2(make_float2(b[v], b[v + 1]), K1, mul2(make_float2(c[v], c[v + 1]), NK2));
            g1[v] = r1.x; g1[v + 1] = r1.y;
          } else if (kd_kind == 2) {
            float2 r1 = mul2(make_float2(b[v], b[v + 1]), K1);
            if (col + v == hard_idx) r1.x -= wk;
            if (col + v + 1 == hard_idx) r1.y -= wk;
            g1[v] = r1.x; g1[v + 1] = r1.y;
          }
        }
      } else {
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        const float e0 = NV > 0 ? a[v] : fexp(a[v] - mx[0]);
        if (label_kind == 0) g0[v] = fmaf(e0, k0, -(d[v] * wb));
        else g0[v] = fmaf(e0, k0, -sm_wb) - (col + v == label ? hot_wb : 0.f) - (col + v == label2 ? hot2_wb : 0.f);
        if (kd_kind == 1) {
          const float es = NV > 0 ? b[v] : fexp(b[v] * invT - mx[1]);
          const float et = NV > 0 ? c[v] : fexp(c[v] * invT - mx[2]);
          g1[v] = fmaf(es, k1, -(et * k2));
        } else if (kd_kind == 2) {
          const float es = NV > 0 ? b[v] : fexp(b[v] - mx[1]);
          g1[v] = fmaf(es, k1, col + v == hard_idx ? -wk : 0.f);
        }
      }
      }
      if (gz) Vec<T, VEC>::store(gz + col, g0);
      if (gzk) Vec<T, VEC>::store(gzk + col, g1);
    }
  };
  if (gz || gzk) {
    if constexpr (NV > 0) {
#pragma unroll
      for (int it = 0; it < NV; ++it) if (it < nchunk) pass3(it, rz[it], rk[it], rt[it], ry[it]);
    } else {
      for (int it = 0; it < nchunk; ++it) {
        load4(it, rz[0], rk[0], rt[0], ry[0]);
        pass3(it, rz[0], rk[0], rt[0], ry[0]);
      }
    }
  }
  DKD_LOGIT_STAMP(4, 0.f);   // gradient stores issued

  // The KD term is formed after the gradient stores are issued: its latency overlaps their drain instead of delaying them.
  if (kd_kind == 1) {
    // sum_c p_t (log p_t - log p_s) = s3/s2 - lse2 + lse1, regrouped so that no term of size max/T enters the sum: with
    // M1, M2 the shifts pass 2 subtracted in its exponents (log2 units, the same rounded values),
    //   = s3/s2 + (M1 - M2) ln 2 + ln(s1/s2).
    // Each term is O(|zt - zk| / T) and the row's KL is their small difference when the student is near the teacher.
    // As lse1 - lse2, two O(max/T) values each rounded (and each off by the rounding of its own shift), the error was up
    // to ~300 times the fp32 reference's at trained-logit scales.  __fmul_rn: the shifts are not contracted into FMAs.
    const float M1 = __fmul_rn(mx[1], kL2e), M2 = __fmul_rn(mx[2], kL2e);
    kd_row = fmaf(s[3], inv_s2, (M1 - M2) * 0.6931471805599453f) + log1pf((s[1] - s[2]) * inv_s2);
  } else if (kd_kind == 2) {
    kd_row = mx[1] + __logf(s[1]) - t[3];
  }
  publish(base_row, kd_row);

  base_out = base_row;   // valid in every thread (block-wide sums); the caller stores or accumulates them
  kd_out = kd_row;
}

// One CTA folds the per-row partials in a fixed order (bit-reproducible) into {total, base, kd}.
// `n_part`: number of partial sums in row_base / row_kd (one per row, or one per warp of the ring kernel).
// Thread t adds rows t, t + THREADS, t + 2 * THREADS, ... in that order, then a fixed tree combines the threads.  The
// loads of 8 rows per thread are all issued before the first add, so up to 8 * THREADS partials cost one L2 round trip.
template <int THREADS = kThreads>
__device__ __forceinline__ void logit_fold(const LogitKdParams& p, float* scratch, int64_t n_part) {
  const float Bf = (float)p.B, Cf = (float)p.C;
  float acc[2] = {0.f, 0.f};
  auto batch = [&](int64_t r0) {
    float b[8], k[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      // a row past the end adds +0.f: acc is never -0.f (it starts at +0.f), so this gives the bits of skipping the add
      const int64_t r = r0 + (int64_t)u * THREADS;
      b[u] = r < n_part ? __ldcg(p.row_base + r) : 0.f;
      k[u] = r < n_part ? __ldcg(p.row_kd + r) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) { acc[0] += b[u]; acc[1] += k[u]; }
  };
  batch(threadIdx.x);
  for (int64_t r0 = threadIdx.x + 8 * THREADS; r0 < n_part; r0 += 8 * THREADS) batch(r0);
  DKD_LOGIT_FOLD_STAMP(6, acc[0]);
  block_sum<2, THREADS>(acc, scratch);
  if (threadIdx.x == 0) {
    const float base = acc[0] / Bf;  // 0 when label_kind < 0 (KD term only: total = alpha * kd)
    float kd = 0.f, total = base;
    if (p.kd_kind == 1) { kd = acc[1] * p.tau * p.tau / (Bf * Cf); total = base * (1.f - p.alpha) + kd * p.alpha; }
    else if (p.kd_kind == 2) { kd = acc[1] / Bf; total = base * (1.f - p.alpha) + kd * p.alpha; }
    p.loss_out[0] = total;
    p.loss_out[1] = base;
    p.loss_out[2] = kd;
    DKD_LOGIT_FOLD_STAMP(7, 0.f);
  }
}

// Ticket and fold for a kernel whose partials are final only at its end (the ring kernel's per-warp sums): one add per
// CTA on a word of the workspace, and the CTA that draws gridDim.x - 1 folds and resets the word for the next call.
template <int THREADS>
__device__ __forceinline__ void logit_finalize(const LogitKdParams& p, float* scratch, bool* s_last, int64_t n_part) {
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned int done = atomicAdd(p.ticket, 1u);
    *s_last = (done == gridDim.x - 1);
  }
  __syncthreads();
  if (!*s_last) return;
  __threadfence();
  logit_fold<THREADS>(p, scratch, n_part);
  if (threadIdx.x == 0) *p.ticket = 0u;
}

// fold by the first warp only (block size not known at compile time)
__device__ __forceinline__ void logit_finalize_any(const LogitKdParams& p, float* scratch, bool* s_last, int64_t n_part) {
  const float Bf = (float)p.B, Cf = (float)p.C;
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned int done = atomicAdd(p.ticket, 1u);
    *s_last = (done == gridDim.x - 1);
  }
  __syncthreads();
  if (!*s_last || threadIdx.x >= 32) return;
  __threadfence();
  float a0 = 0.f, a1 = 0.f;
  for (int64_t r = threadIdx.x; r < n_part; r += 32) { a0 += __ldcg(p.row_base + r); a1 += __ldcg(p.row_kd + r); }
  a0 = warp_sum(a0); a1 = warp_sum(a1);
  if (threadIdx.x == 0) {
    const float base = a0 / Bf;
    float kd = 0.f, total = base;
    if (p.kd_kind == 1) { kd = a1 * p.tau * p.tau / (Bf * Cf); total = base * (1.f - p.alpha) + kd * p.alpha; }
    else if (p.kd_kind == 2) { kd = a1 / Bf; total = base * (1.f - p.alpha) + kd * p.alpha; }
    p.loss_out[0] = total; p.loss_out[1] = base; p.loss_out[2] = kd;
    *p.ticket = 0u;
  }
}

// The row kernel's partials are folded by a one-CTA launch right behind it (launch_pdl): its CTA is resident while the
// rows run, and its dependency wait returns once every row CTA has exited and its partials are visible.  That grid
// boundary is the whole inter-CTA protocol — no row CTA waits for another, and none pays a fence or an atomic.
// Behind the 128-thread row kernel (B < 1024, or rows too long for the 2-warp one): kThreads threads, logit_fold's
// thread -> row assignment and reduction tree.
__global__ void __launch_bounds__(kThreads) logit_fold_small_kernel(LogitKdParams p) {
  __shared__ float scratch[2 * (kThreads / 32)];
  grid_dep_wait();
  DKD_LOGIT_FOLD_STAMP(9, 0.f);
  grid_dep_launch();
  logit_fold<kThreads>(p, scratch, p.B);
}

// Large batches: a 1024-thread CTA with 8 independent loads in flight per thread (a 128-thread fold of 16 384 rows is
// ~130 dependent L2 round trips — it was most of the runtime of the fused form at B = 16 384).
// Fixed thread -> row assignment and fixed reduction tree: bit-reproducible.
constexpr int kFoldThreads = 1024;
__global__ void __launch_bounds__(kFoldThreads) logit_fold_kernel(LogitKdParams p) {
  __shared__ float scratch[2 * (kFoldThreads / 32)];
  grid_dep_wait();
  grid_dep_launch();
  float a0[8], a1[8];
#pragma unroll
  for (int u = 0; u < 8; ++u) a0[u] = a1[u] = 0.f;
  for (int64_t r0 = threadIdx.x; r0 < p.B; r0 += 8 * kFoldThreads) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int64_t r = r0 + (int64_t)u * kFoldThreads;
      if (r < p.B) { a0[u] += __ldcg(p.row_base + r); a1[u] += __ldcg(p.row_kd + r); }
    }
  }
  float acc[2] = {((a0[0] + a0[1]) + (a0[2] + a0[3])) + ((a0[4] + a0[5]) + (a0[6] + a0[7])),
                  ((a1[0] + a1[1]) + (a1[2] + a1[3])) + ((a1[4] + a1[5]) + (a1[6] + a1[7]))};
  block_sum<2, kFoldThreads>(acc, scratch);
  if (threadIdx.x == 0) {
    const float Bf = (float)p.B, Cf = (float)p.C;
    const float base = acc[0] / Bf;
    float kd = 0.f, total = base;
    if (p.kd_kind == 1) { kd = acc[1] * p.tau * p.tau / (Bf * Cf); total = base * (1.f - p.alpha) + kd * p.alpha; }
    else if (p.kd_kind == 2) { kd = acc[1] / Bf; total = base * (1.f - p.alpha) + kd * p.alpha; }
    p.loss_out[0] = total;
    p.loss_out[1] = base;
    p.loss_out[2] = kd;
  }
}

// Asks L2 for `bytes` bytes at `src` without loading anything into the SM: one bulk prefetch when the range is 16-byte
// aligned at both ends, otherwise one prefetch per 128-byte line spread over the CTA.  A hint only — it orders nothing
// and returns no data.
template <int THREADS>
__device__ __forceinline__ void prefetch_l2(const void* src, int64_t bytes) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(src);
  if (((a | (uintptr_t)bytes) & 15) == 0) {
    const uint32_t n = (uint32_t)min(bytes, (int64_t)0xfffffff0);   // the size operand is 32-bit: a hint may stop short
    if (threadIdx.x == 0) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(n) : "memory");
  } else {
    for (uintptr_t l = (a & ~(uintptr_t)127) + (uintptr_t)threadIdx.x * 128; l < a + (uintptr_t)bytes; l += THREADS * 128)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(l));
  }
}

// Thread 0 stores its row's partials after its gradient stores are issued; logit_fold_small_kernel or logit_fold_kernel
// folds them in the next launch, whose dependency wait returns only once every row CTA has finished.  Launched with programmatic dependent launch (launch_pdl).
template <typename T, int VEC, int NV, int THREADS = kThreads, int LK = kRuntimeMode, int KK = kRuntimeMode>
__global__ void __launch_bounds__(THREADS) logit_kd_kernel(LogitKdParams p) {
  __shared__ float scratch[8 * (kThreads / 32)];
  __shared__ int s_arg[kThreads / 32];
  __shared__ float s_argv[kThreads / 32];
  DKD_LOGIT_STAMP(0, 0.f);
  const int label_kind = LK == kRuntimeMode ? p.label_kind : LK;
  const int kd_kind = KK == kRuntimeMode ? p.kd_kind : KK;
  const int64_t row = blockIdx.x, C = p.C;
  const T* z = label_kind >= 0 ? reinterpret_cast<const T*>(p.z) + row * C : nullptr;
  const T* zk = kd_kind ? reinterpret_cast<const T*>(p.zk) + row * C : nullptr;
  const T* zt = kd_kind ? reinterpret_cast<const T*>(p.zt) + row * C : nullptr;
  const T* y = label_kind == 0 ? reinterpret_cast<const T*>(p.y) + row * C : nullptr;
  T* gz = p.gz ? reinterpret_cast<T*>(p.gz) + row * C : nullptr;
  T* gzk = p.gzk ? reinterpret_cast<T*>(p.gzk) + row * C : nullptr;
  // The predecessor may still be running until the wait returns: the op that wrote the logits, or the previous call on
  // this workspace (partials) and on gradient memory reused from it.  Before the wait, the CTA only asks L2 for its
  // operand rows, so that the loads after it find them there instead of in DRAM.  L2 is the GPU's point of coherence:
  // stores of the predecessor that land after a prefetch update the prefetched lines, so no stale copy can be read.
  const T* rows[4] = {z, zk, zt, y};
#pragma unroll
  for (int i = 0; i < 4; ++i)
    if (rows[i]) prefetch_l2<THREADS>(rows[i], C * (int64_t)sizeof(T));
  grid_dep_wait();
  DKD_LOGIT_STAMP(8, 0.f);
  grid_dep_launch();
  float base_row, kd_row;
  logit_row<T, VEC, NV, THREADS, LK, KK>(p, row, z, zk, zt, y, gz, gzk, scratch, s_arg, s_argv, base_row, kd_row,
                                         [&](float base, float kd) {
                                           if (threadIdx.x == 0) {
                                             p.row_base[row] = base;
                                             p.row_kd[row] = kd;
                                           }
                                         });
}

// ---------------------------------------------------------------------------------------------------------------
// Large batches: persistent CTAs, ONE WARP PER ROW, rows streamed through a per-warp ring of shared-memory stages by
// bulk copies (cp.async.bulk + mbarrier complete_tx) — no thread ever waits on a global load:
//   lane 0   issues the 2-4 operand rows of row k+2 into the stage row k-1 has left,
//   the warp waits on row k's mbarrier, reads the stage once into registers (the three passes of logit_row run on
//            registers, warp shuffles only: no block barrier anywhere), writes both gradient rows back INTO the stage
//            (over z and zk) and lane 0 sends them to HBM with bulk stores.
// The one-CTA-per-row form keeps a row's loads in flight only for the first third of the CTA's life (two block
// reductions sit between its load and store phases): 56 % of the HBM copy rate at B = 16 384; here every warp always
// has 1-2 rows (8-16 KB) of bulk loads in flight and the stores drain asynchronously.
constexpr int kRingStages = 3;
constexpr int kRingMaxWarps = 8;
constexpr int kRingSmemBudget = 224 * 1024;

__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   (uint32_t)__cvta_generic_to_shared(dst)),
               "l"(src), "r"(bytes), "r"((uint32_t)__cvta_generic_to_shared(bar))
               : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* dst, const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"((uint32_t)__cvta_generic_to_shared(src)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void ring_bar_init(uint64_t* bar) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)) : "memory");
}
__device__ __forceinline__ void ring_bar_expect(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void ring_bar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(bar);
  uint32_t ok = 0;
  const long long t0 = clock64();
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(a), "r"(parity)
        : "memory");
    if (ok) return;
    if (clock64() - t0 > 4000000000ll) {   // a protocol bug traps instead of hanging the GPU
      printf("dkd: logit ring wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
      __trap();
    }
  }
}

template <typename T, int VEC, int NV, int LK, int KK>
__global__ void __launch_bounds__(32 * kRingMaxWarps, 1) logit_ring_kernel(LogitKdParams p, int row_stride /* bytes, multiple of 128 */) {
  extern __shared__ __align__(128) uint8_t ring_smem[];
  constexpr int NOPS = (LK >= 0 ? 1 : 0) + (LK == 0 ? 1 : 0) + (KK ? 2 : 0);
  // stage layout: [z][zk][zt][y] (only the operands the mode reads); gradients overwrite z and zk
  constexpr int O_Z = 0, O_ZK = (LK >= 0 ? 1 : 0), O_ZT = O_ZK + 1, O_Y = O_ZK + (KK ? 2 : 0);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  const int64_t C = p.C;
  const uint32_t row_bytes = (uint32_t)(C * sizeof(T));
  const int stage_bytes = NOPS * row_stride;
  uint8_t* wbase = ring_smem + (size_t)warp * kRingStages * stage_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(ring_smem + (size_t)nw * kRingStages * stage_bytes) + warp * kRingStages;
  const int64_t gw = (int64_t)blockIdx.x * nw + warp, GW = (int64_t)gridDim.x * nw;
  const int64_t nrows = gw < p.B ? (p.B - gw + GW - 1) / GW : 0;
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < kRingStages; ++s) ring_bar_init(&bars[s]);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  const T* gZ = reinterpret_cast<const T*>(p.z);
  const T* gZK = reinterpret_cast<const T*>(p.zk);
  const T* gZT = reinterpret_cast<const T*>(p.zt);
  const T* gY = reinterpret_cast<const T*>(p.y);
  auto issue = [&](int64_t k) {   // lane 0 only
    const int s = (int)(k % kRingStages);
    const int64_t off = (gw + k * GW) * C;
    uint8_t* st = wbase + (size_t)s * stage_bytes;
    ring_bar_expect(&bars[s], NOPS * row_bytes);
    if (LK >= 0) bulk_g2s(st + O_Z * row_stride, gZ + off, row_bytes, &bars[s]);
    if (KK) {
      bulk_g2s(st + O_ZK * row_stride, gZK + off, row_bytes, &bars[s]);
      bulk_g2s(st + O_ZT * row_stride, gZT + off, row_bytes, &bars[s]);
    }
    if (LK == 0) bulk_g2s(st + O_Y * row_stride, gY + off, row_bytes, &bars[s]);
  };
  if (lane == 0) {
    for (int64_t k = 0; k < kRingStages - 1 && k < nrows; ++k) issue(k);
  }
  float acc_base = 0.f, acc_kd = 0.f;
  for (int64_t k = 0; k < nrows; ++k) {
    const int s = (int)(k % kRingStages);
    const uint32_t parity = (uint32_t)((k / kRingStages) & 1);
    uint8_t* st = wbase + (size_t)s * stage_bytes;
    const int64_t row = gw + k * GW;
    ring_bar_wait(&bars[s], parity);
    T* sz = reinterpret_cast<T*>(st + O_Z * row_stride);
    T* szk = reinterpret_cast<T*>(st + O_ZK * row_stride);
    const T* szt = reinterpret_cast<const T*>(st + O_ZT * row_stride);
    const T* sy = reinterpret_cast<const T*>(st + O_Y * row_stride);
    float base_row, kd_row;
    logit_row<T, VEC, NV, 32, LK, KK, true>(p, row, LK >= 0 ? sz : nullptr, KK ? szk : nullptr, KK ? szt : nullptr, LK == 0 ? sy : nullptr,
                                            (p.gz && LK >= 0) ? sz : nullptr, (p.gzk && KK) ? szk : nullptr, nullptr, nullptr, nullptr,
                                            base_row, kd_row, [](float, float) {});
    acc_base += base_row;   // this warp's rows, in row order: fixed for a given (B, grid)
    acc_kd += kd_row;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the gradient rows (generic-proxy writes) -> visible to the bulk stores
    __syncwarp();
    if (lane == 0) {
      const int64_t off = row * C;
      if (p.gz && LK >= 0) bulk_s2g(reinterpret_cast<T*>(p.gz) + off, sz, row_bytes);
      if (p.gzk && KK) bulk_s2g(reinterpret_cast<T*>(p.gzk) + off, szk, row_bytes);
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      // the stage of row k-1 is free once ITS stores have read shared memory (all but the newest group)
      asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
      if (k + kRingStages - 1 < nrows) issue(k + kRingStages - 1);
    }
    __syncwarp();
  }
  if (lane == 0) {
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // stores complete before the CTA's shared memory goes away
    if (gw < p.B) {              // one partial per warp that owns rows (the workspace holds B entries)
      p.row_base[gw] = acc_base;
      p.row_kd[gw] = acc_kd;
    }
  }
  const int64_t n_part = GW < p.B ? GW : p.B;
  // last CTA folds the GW per-warp partials in a fixed order: no second launch
  __shared__ float scratch[2 * kRingMaxWarps];
  __shared__ bool s_last;
  __syncthreads();
  if (blockDim.x == 32 * kRingMaxWarps) logit_finalize<32 * kRingMaxWarps>(p, scratch, &s_last, n_part);
  else logit_finalize_any(p, scratch, &s_last, n_part);
}

// one block size; NV by row length; the six usual (label_kind, kd_kind) modes are compiled in
template <typename T, int VEC, int THREADS, int LK, int KK>
void launch_nv(const LogitKdParams& p, int64_t nchunk, dim3 grid, cudaStream_t stream) {
  if (nchunk <= 1) launch_pdl(logit_kd_kernel<T, VEC, 1, THREADS, LK, KK>, grid, dim3(THREADS), stream, p);
  else if (nchunk <= 2) launch_pdl(logit_kd_kernel<T, VEC, 2, THREADS, LK, KK>, grid, dim3(THREADS), stream, p);
  else launch_pdl(logit_kd_kernel<T, VEC, 4, THREADS, LK, KK>, grid, dim3(THREADS), stream, p);
}
template <typename T, int VEC, int THREADS>
void launch_mode(const LogitKdParams& p, int64_t nchunk, dim3 grid, cudaStream_t stream) {
  if constexpr (VEC * sizeof(T) == 16) {   // specialise the vectorised kernels only
    const int lk = p.label_kind, kk = p.kd_kind;
    if (lk == 0 && kk == 1) return launch_nv<T, VEC, THREADS, 0, 1>(p, nchunk, grid, stream);
    if (lk == 1 && kk == 1) return launch_nv<T, VEC, THREADS, 1, 1>(p, nchunk, grid, stream);
    if (lk == 0 && kk == 2) return launch_nv<T, VEC, THREADS, 0, 2>(p, nchunk, grid, stream);
    if (lk == 1 && kk == 2) return launch_nv<T, VEC, THREADS, 1, 2>(p, nchunk, grid, stream);
    if (lk == 0 && kk == 0) return launch_nv<T, VEC, THREADS, 0, 0>(p, nchunk, grid, stream);
    if (lk == 1 && kk == 0) return launch_nv<T, VEC, THREADS, 1, 0>(p, nchunk, grid, stream);
  }
  launch_nv<T, VEC, THREADS, kRuntimeMode, kRuntimeMode>(p, nchunk, grid, stream);
}

// streaming launch for one compiled (label_kind, kd_kind) mode; false when the mode / shape is not covered
template <typename T, int VEC, int NV, int LK, int KK>
int launch_ring_mode(const LogitKdParams& p, cudaStream_t stream) {
  constexpr int NOPS = (LK >= 0 ? 1 : 0) + (LK == 0 ? 1 : 0) + (KK ? 2 : 0);
  const int row_stride = (int)((p.C * (int64_t)sizeof(T) + 127) / 128 * 128);
  int warps = kRingSmemBudget / (kRingStages * NOPS * row_stride);
  if (warps > kRingMaxWarps) warps = kRingMaxWarps;
  if (warps < 2) return 1;   // rows too long for the ring: caller falls back
  const size_t smem = (size_t)warps * kRingStages * NOPS * row_stride + (size_t)warps * kRingStages * sizeof(uint64_t);
  int64_t grid = (p.B + warps - 1) / warps;
  if (grid > kNumSMs) grid = kNumSMs;
  auto kern = logit_ring_kernel<T, VEC, NV, LK, KK>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  kern<<<(unsigned)grid, 32 * warps, smem, stream>>>(p, row_stride);
  return 0;
}
template <typename T, int VEC, int NV>
int launch_ring(const LogitKdParams& p, cudaStream_t stream) {
  const int lk = p.label_kind, kk = p.kd_kind;
  if (lk == 0 && kk == 1) return launch_ring_mode<T, VEC, NV, 0, 1>(p, stream);
  if (lk == 1 && kk == 1) return launch_ring_mode<T, VEC, NV, 1, 1>(p, stream);
  if (lk == 0 && kk == 2) return launch_ring_mode<T, VEC, NV, 0, 2>(p, stream);
  if (lk == 1 && kk == 2) return launch_ring_mode<T, VEC, NV, 1, 2>(p, stream);
  if (lk == 0 && kk == 0) return launch_ring_mode<T, VEC, NV, 0, 0>(p, stream);
  if (lk == 1 && kk == 0) return launch_ring_mode<T, VEC, NV, 1, 0>(p, stream);
  return 1;
}

template <typename T, int VEC>
int launch_logit_kd(const LogitKdParams& p, cudaStream_t stream) {
  const int64_t per_chunk = (int64_t)kThreads * VEC;
  const int64_t nchunk = (p.C + per_chunk - 1) / per_chunk;
  dim3 grid((unsigned)p.B), block(kThreads);
  const int64_t nchunk64 = (p.C + 64 * VEC - 1) / (64 * VEC);
  if constexpr (VEC * sizeof(T) == 16) {   // large batch, 16-byte aligned rows of 1-4 KB: persistent bulk-copy ring
    constexpr int NV = 32 / VEC;           // 32 elements per lane and operand: C <= 1024
    if (p.B >= 1024 && p.C * (int64_t)sizeof(T) >= 1024 && p.C <= 32 * VEC * NV) {
      if (launch_ring<T, VEC, NV>(p, stream) == 0) return check_launch("dkd_logit_kd_fwdbwd: ring");
    }
  }
  if (p.B >= 1024 && nchunk64 <= 4) {   // large batch: 2-warp CTAs (4-warp measured 3 % slower), 1024-thread fold
    launch_mode<T, VEC, 64>(p, nchunk64, grid, stream);
    int rc = check_launch("dkd_logit_kd_fwdbwd");
    if (rc != DKD_OK) return rc;
    launch_pdl(logit_fold_kernel, dim3(1), dim3(kFoldThreads), stream, p);
    return check_launch("dkd_logit_kd_fwdbwd: fold");
  }
  if (nchunk <= 4) launch_mode<T, VEC, kThreads>(p, nchunk, grid, stream);
  else launch_pdl(logit_kd_kernel<T, VEC, 0>, grid, block, stream, p);
  int rc = check_launch("dkd_logit_kd_fwdbwd");
  if (rc != DKD_OK) return rc;
  launch_pdl(logit_fold_small_kernel, dim3(1), dim3(kThreads), stream, p);
  return check_launch("dkd_logit_kd_fwdbwd: fold");
}

template <typename T>
int dispatch_vec(const LogitKdParams& p, cudaStream_t stream) {
  constexpr int MAXV = 16 / (int)sizeof(T);
  auto aligned = [&](int vec) {
    const uintptr_t m = (uintptr_t)vec * sizeof(T) - 1;
    auto ok = [&](const void* q) { return q == nullptr || (((uintptr_t)q) & m) == 0; };
    return p.C % vec == 0 && ok(p.z) && ok(p.zk) && ok(p.zt) && (p.label_kind == 1 || ok(p.y)) && ok(p.gz) && ok(p.gzk);
  };
  if (aligned(MAXV)) return launch_logit_kd<T, MAXV>(p, stream);
  if (aligned(MAXV / 2)) return launch_logit_kd<T, MAXV / 2>(p, stream);
  return launch_logit_kd<T, 1>(p, stream);
}

}  // namespace
}  // namespace dkd

extern "C" {

size_t dkd_logit_kd_workspace_bytes(int64_t B) {
  return (size_t)(B > 0 ? B : 0) * 2 * sizeof(float) + 256;
}

int dkd_logit_kd_fwdbwd(const void* outputs, const void* outputs_kd, const void* teacher_logits,
                        const void* labels, int label_kind, int kd_kind, int64_t B, int64_t C, int dtype,
                        float smoothing, float alpha, float tau, const float* mix_lam, void* g_outputs, void* g_outputs_kd,
                        float* loss_out, void* workspace, size_t workspace_bytes, dkd_stream_t stream) {
  using namespace dkd;
  int rc = dkd_check_device();
  if (rc != DKD_OK) return rc;
  DKD_REQUIRE(B > 0 && C > 0 && B < (1ll << 31), DKD_E_SHAPE, "dkd_logit_kd_fwdbwd: bad shape B=%lld C=%lld", (long long)B, (long long)C);
  DKD_REQUIRE(dtype == DKD_F32 || dtype == DKD_BF16, DKD_E_DTYPE, "dkd_logit_kd_fwdbwd: dtype %d", dtype);
  DKD_REQUIRE(label_kind >= -1 && label_kind <= 1, DKD_E_UNSUPPORTED, "dkd_logit_kd_fwdbwd: label_kind %d", label_kind);
  DKD_REQUIRE(kd_kind >= 0 && kd_kind <= 2, DKD_E_UNSUPPORTED, "dkd_logit_kd_fwdbwd: kd_kind %d", kd_kind);
  DKD_REQUIRE(loss_out && workspace && (label_kind < 0 || (outputs && labels)), DKD_E_SHAPE, "dkd_logit_kd_fwdbwd: null pointer");
  DKD_REQUIRE(label_kind >= 0 || kd_kind != 0, DKD_E_UNSUPPORTED, "dkd_logit_kd_fwdbwd: nothing to compute (no base term and no KD term)");
  DKD_REQUIRE(kd_kind == 0 || (outputs_kd && teacher_logits), DKD_E_SHAPE, "dkd_logit_kd_fwdbwd: KD needs outputs_kd and teacher_logits");
  DKD_REQUIRE(kd_kind != 1 || tau > 0.f, DKD_E_SHAPE, "dkd_logit_kd_fwdbwd: tau must be > 0");
  DKD_REQUIRE(workspace_bytes >= dkd_logit_kd_workspace_bytes(B), DKD_E_WORKSPACE, "dkd_logit_kd_fwdbwd: workspace too small");
  DKD_REQUIRE((((uintptr_t)workspace) & 15) == 0, DKD_E_ALIGN, "dkd_logit_kd_fwdbwd: workspace must be 16-byte aligned");
  LogitKdParams p;
  p.z = outputs; p.zk = outputs_kd; p.zt = teacher_logits; p.y = labels;
  p.gz = g_outputs; p.gzk = g_outputs_kd; p.loss_out = loss_out;
  p.ticket = reinterpret_cast<unsigned int*>(workspace);
  p.row_base = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + 256);
  p.row_kd = p.row_base + B;
  p.B = B; p.C = C; p.label_kind = label_kind; p.kd_kind = kd_kind;
  p.smoothing = smoothing; p.alpha = alpha; p.tau = tau;
  DKD_REQUIRE(mix_lam == nullptr || label_kind == 1, DKD_E_UNSUPPORTED, "dkd_logit_kd_fwdbwd: mix_lam needs int64 labels (label_kind 1)");
  p.mix_lam = mix_lam;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  return dtype == DKD_F32 ? dispatch_vec<float>(p, st) : dispatch_vec<__nv_bfloat16>(p, st);
}

}  // extern "C"
