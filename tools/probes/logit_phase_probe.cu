// Phase probe (not part of the library) of the fused logit KD kernel at the headline shape (soft KD + soft-label base CE,
// B = 256, C = 1000, bf16).  It compiles deltakd_b200/csrc/logit_kd.cu with DKD_LOGIT_STAMP defined: thread 0 of every CTA
// records clock64 (SM cycles, comparable within a CTA) and %globaltimer (ns, comparable across CTAs) at
//   0 kernel entry, 8 dependency resolved (after griddepcontrol.wait, where the kernel has one), 1 loads landed,
//   2 block max done, 3 block sums done, 4 gradient stores issued, 5 ticket returned (builds whose last row CTA folds),
//   9 fold kernel's dependency resolved (builds that fold in a launch of their own), 6 fold loads summed, 7 loss stored.
// The workload is a CUDA graph of K calls on one stream and one workspace, inputs rotated through 97 sets (189 MiB > 126 MiB
// of L2; K >= 97 so that a replay reads them all and the rows come from DRAM, as in bench.py); each replay leaves the
// stamps of its last call, and R replays give R samples per CTA.  Times are reported from
// the first row CTA's start (entry, or dependency resolved) as the median row CTA and as the last row CTA (the one whose
// final stamp is latest: the folding CTA where a row CTA folds).  A fold kernel stamps a slot of its own; its points are
// reported in both columns, its cycles counted from its dependency resolving.
//
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 --expt-relaxed-constexpr -I deltakd_b200/csrc \
//        -o build/logit_phase_probe tools/probes/logit_phase_probe.cu deltakd_b200/csrc/abi.cu
//   build/logit_phase_probe [K=100] [R=200]
// (-I another directory holding a stamped logit_kd.cu probes that version instead.)
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include <cuda_bf16.h>
#include <cuda_runtime.h>

constexpr int kPoints = 10;
constexpr int kMaxRows = 1024;
constexpr int kFoldSlot = kMaxRows;
struct Stamp {
  long long clk;
  unsigned long long ns;
};
__device__ Stamp g_stamp[kMaxRows + 1][kPoints];

__device__ __forceinline__ void probe_stamp(unsigned slot, int point, float dep) {
  asm volatile("" ::"f"(dep));   // the stamp is taken after `dep` is available
  if (threadIdx.x == 0 && slot <= kMaxRows) {
    unsigned long long ns;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
    g_stamp[slot][point] = {clock64(), ns};
  }
}
#define DKD_LOGIT_STAMP(point, dep) probe_stamp(blockIdx.x < kMaxRows ? blockIdx.x : ~0u, point, dep)
#define DKD_LOGIT_FOLD_STAMP(point, dep) probe_stamp(kFoldSlot, point, dep)
#include "logit_kd.cu"

#define CK(x)                                                                          \
  do {                                                                                 \
    cudaError_t e_ = (x);                                                              \
    if (e_ != cudaSuccess) {                                                           \
      fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); \
      exit(1);                                                                         \
    }                                                                                  \
  } while (0)

__global__ void fill_kernel(__nv_bfloat16* x, int64_t n, uint32_t seed, float lo, float hi) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    uint32_t h = (uint32_t)i * 2654435761u ^ seed;
    h ^= h >> 15; h *= 2246822519u; h ^= h >> 13; h *= 3266489917u; h ^= h >> 16;
    x[i] = __float2bfloat16(lo + (hi - lo) * (h >> 8) * (1.f / 16777216.f));
  }
}

// %globaltimer resolution: distinct successive readings of one thread
__global__ void timer_kernel(unsigned long long* d, int n) {
  unsigned long long prev, t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(prev));
  int k = 0;
  for (int i = 0; i < 1 << 22 && k < n; ++i) {
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    if (t != prev) { d[k++] = t - prev; prev = t; }
  }
}

static double median(std::vector<double> v) {
  if (v.empty()) return 0.0 / 0.0;
  std::sort(v.begin(), v.end());
  return v[v.size() / 2];
}

int main(int argc, char** argv) {
  const int K = argc > 1 ? atoi(argv[1]) : 100, R = argc > 2 ? atoi(argv[2]) : 200;
  const int64_t B = 256, Cn = 1000, set_elems = 4 * B * Cn, nsets = 97;
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, 0));

  unsigned long long* dt;
  const int nt = 256;
  CK(cudaMalloc(&dt, nt * sizeof(unsigned long long)));
  timer_kernel<<<1, 1>>>(dt, nt);
  std::vector<unsigned long long> ht(nt);
  CK(cudaMemcpy(ht.data(), dt, nt * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  std::vector<double> tdel(ht.begin() + 1, ht.end());
  std::sort(tdel.begin(), tdel.end());

  __nv_bfloat16 *in, *g0, *g1;
  float* loss;
  void* ws;
  CK(cudaMalloc(&in, nsets * set_elems * sizeof(__nv_bfloat16)));
  CK(cudaMalloc(&g0, B * Cn * sizeof(__nv_bfloat16)));
  CK(cudaMalloc(&g1, B * Cn * sizeof(__nv_bfloat16)));
  CK(cudaMalloc(&loss, 3 * sizeof(float)));
  const size_t ws_bytes = dkd_logit_kd_workspace_bytes(B);
  CK(cudaMalloc(&ws, ws_bytes));
  CK(cudaMemset(ws, 0, ws_bytes));
  for (int64_t s = 0; s < nsets; ++s) {
    __nv_bfloat16* base = in + s * set_elems;
    fill_kernel<<<296, 256>>>(base, 3 * B * Cn, 1234u + 17u * (uint32_t)s, -4.f, 4.f);                 // z, zk, zt
    fill_kernel<<<296, 256>>>(base + 3 * B * Cn, B * Cn, 99u + 17u * (uint32_t)s, 0.f, 2.f / Cn);     // soft labels
  }
  CK(cudaDeviceSynchronize());

  cudaStream_t st;
  CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  int call = 0;
  auto one = [&]() {
    const __nv_bfloat16* s = in + (int64_t)(call++ % nsets) * set_elems;
    const int rc = dkd_logit_kd_fwdbwd(s, s + B * Cn, s + 2 * B * Cn, s + 3 * B * Cn, 0, 1, B, Cn, DKD_BF16, 0.f, 0.1f, 3.f,
                                       nullptr, g0, g1, loss, ws, ws_bytes, (dkd_stream_t)st);
    if (rc) { fprintf(stderr, "dkd_logit_kd_fwdbwd: %s\n", dkd_last_error()); exit(1); }
  };
  for (int i = 0; i < 3; ++i) one();
  CK(cudaStreamSynchronize(st));
  cudaGraph_t graph;
  cudaGraphExec_t exec;
  CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
  for (int i = 0; i < K; ++i) one();
  CK(cudaStreamEndCapture(st, &graph));
  CK(cudaGraphInstantiate(&exec, graph, 0));
  CK(cudaGraphLaunch(exec, st));
  CK(cudaStreamSynchronize(st));

  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  std::vector<double> call_us;
  // per point: samples of (median CTA) and (last CTA), ns from the first CTA's start; per phase: cycles
  std::vector<std::vector<double>> med_ns(kPoints), last_ns(kPoints), med_cyc(kPoints), last_cyc(kPoints);
  std::vector<double> mhz;
  std::vector<Stamp> h((kMaxRows + 1) * kPoints);
  for (int r = 0; r < R; ++r) {
    CK(cudaEventRecord(e0, st));
    CK(cudaGraphLaunch(exec, st));
    CK(cudaEventRecord(e1, st));
    CK(cudaStreamSynchronize(st));
    float ms;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    call_us.push_back(ms * 1e3 / K);
    CK(cudaMemcpyFromSymbol(h.data(), g_stamp, h.size() * sizeof(Stamp)));
    auto at = [&](int cta, int pt) -> const Stamp& { return h[cta * kPoints + pt]; };
    auto start = [&](int cta) { return at(cta, 8).ns ? at(cta, 8) : at(cta, 0); };
    unsigned long long t0 = ~0ull;
    for (int c = 0; c < B; ++c) t0 = std::min(t0, start(c).ns);
    auto final_pt = [&](int cta) {   // the CTA's latest stamp of this call
      int f = -1;
      for (int pt = 0; pt < kPoints; ++pt)
        if (at(cta, pt).ns >= t0 && (f < 0 || at(cta, pt).ns > at(cta, f).ns)) f = pt;
      return f;
    };
    int last = -1;
    for (int c = 0; c < B; ++c)
      if (final_pt(c) >= 0 && (last < 0 || at(c, final_pt(c)).ns > at(last, final_pt(last)).ns)) last = c;
    const bool fold_slot = at(kFoldSlot, 7).ns >= t0;
    if (last < 0 || !(fold_slot || at(last, 7).ns >= t0)) { fprintf(stderr, "no CTA stored the loss in replay %d\n", r); return 1; }
    for (int pt = 0; pt < kPoints; ++pt) {
      std::vector<double> ns, cyc;
      for (int c = 0; c < B; ++c) {
        if (at(c, pt).ns < t0) continue;   // not stamped in this call (fold points in other CTAs, point 8 without PDL)
        ns.push_back((double)(at(c, pt).ns - t0));
        cyc.push_back((double)(at(c, pt).clk - start(c).clk));
      }
      if (!ns.empty()) { med_ns[pt].push_back(median(ns)); med_cyc[pt].push_back(median(cyc)); }
      if (at(last, pt).ns >= t0) {
        last_ns[pt].push_back((double)(at(last, pt).ns - t0));
        last_cyc[pt].push_back((double)(at(last, pt).clk - start(last).clk));
      }
      if (fold_slot && at(kFoldSlot, pt).ns >= t0) {
        const double fns = (double)(at(kFoldSlot, pt).ns - t0), fcyc = (double)(at(kFoldSlot, pt).clk - at(kFoldSlot, 9).clk);
        med_ns[pt].push_back(fns); last_ns[pt].push_back(fns);
        med_cyc[pt].push_back(fcyc); last_cyc[pt].push_back(fcyc);
      }
    }
    const int f = final_pt(last);
    const double dns = (double)(at(last, f).ns - at(last, 0).ns), dclk = (double)(at(last, f).clk - at(last, 0).clk);
    if (dns > 0) mhz.push_back(dclk / dns * 1e3);
  }
  const char* names[kPoints] = {"entry", "loads landed", "block max", "block sums", "grad stores issued", "ticket returned",
                                "fold loads summed", "loss stored", "dependency resolved", "fold dependency resolved"};
  const int order[kPoints] = {0, 8, 1, 2, 3, 4, 5, 9, 6, 7};
  printf("{\"device\": \"%s\", \"K\": %d, \"replays\": %d, \"call_us_median\": %.3f, \"globaltimer_step_ns\": "
         "{\"min\": %.0f, \"median\": %.0f}, \"sm_mhz_from_stamps\": %.0f, \"points\": [\n",
         prop.name, K, R, median(call_us), tdel.front(), median(tdel), median(mhz));
  bool first = true;
  for (int i = 0; i < kPoints; ++i) {
    const int pt = order[i];
    if (med_ns[pt].empty() && last_ns[pt].empty()) continue;
    printf("%s  {\"point\": %d, \"name\": \"%s\", \"median_cta_ns\": %.0f, \"last_cta_ns\": %.0f, \"median_cta_cycles\": %.0f, "
           "\"last_cta_cycles\": %.0f}",
           first ? "" : ",\n", pt, names[pt], median(med_ns[pt]), median(last_ns[pt]), median(med_cyc[pt]), median(last_cyc[pt]));
    first = false;
  }
  printf("\n]}\n");
  return 0;
}
