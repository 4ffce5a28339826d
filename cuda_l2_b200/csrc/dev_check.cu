// dev_check — standalone bring-up / tuning tool for libb200_hgemm.so (developer tool, not product).
//
//   dev_check check <acc_bits> <cfg|-1> <M> <N> <K> [gm splits]   exactness vs an independent GPU checker
//                                                     (splits: 1 none, >1 workspace, -2/-4/-8 cluster, 100/101 stream-K)
//   dev_check time  <acc_bits> <cfg|-1> <M> <N> <K> [iters gm splits]  CUDA-event timing (+ cuBLAS for scale)
//   dev_check sustain <acc_bits> <cfg|-1> <M> <N> <K> [seconds gm splits]   burst vs power-capped throughput, ours and cuBLAS
//   dev_check sweep <acc_bits> <M> <N> <K> [iters]           time every config and group_m variant
//   dev_check wall  <acc_bits> <M> <N> <K> [seconds [tune_warm tune_bench]]  the harness's protocol (one baseline/ours pair at a time,
//                                                     fresh operands per iteration, zero-filled output) vs 6 library baselines
//   dev_check wallgrid <acc_bits> <part> <nparts> [seconds tune_warm tune_bench limit]   `wall` over a share of the grid
//   dev_check_trace trace <acc_bits> <cfg|-1> <M> <N> <K> [gm splits cold]   per-CTA phase timestamps of one launch (trace build only)
//   dev_check grid  <acc_bits> [part nparts budget_ms min_gflop max_gflop [wall]]  time every config on the whole shape grid (CSV);
//                                                     "wall": rank by the harness metric instead of CUDA-event time
//
// Inputs are small integers, so every product and partial sum is exact in fp16 and fp32: any
// mismatch is a kernel bug, never rounding. C is surrounded by guard bands to catch stray writes.
#include <cublas_v2.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <array>
#include <cstring>
#include <functional>
#include <string>
#include <vector>

#include "../../include/b200_baselines.h"
#include "../../include/b200_hgemm.h"
#include <chrono>
#include <random>
#include <thread>

#define CK(x)                                                                              \
  do {                                                                                     \
    cudaError_t e_ = (x);                                                                  \
    if (e_ != cudaSuccess) {                                                               \
      printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__);      \
      exit(2);                                                                             \
    }                                                                                      \
  } while (0)

__global__ void fill_ternary(__half* p, size_t n, uint32_t seed) {
  size_t i = blockIdx.x * size_t(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  uint32_t x = uint32_t(i) * 2654435761u ^ seed;
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  p[i] = __float2half(float(int(x % 3u) - 1));
}
__global__ void fill_normalish(__half* p, size_t n, uint32_t seed) {
  size_t i = blockIdx.x * size_t(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  uint32_t x = uint32_t(i) * 2654435761u ^ seed;
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  p[i] = __float2half((float(x & 0xffff) / 65536.f - 0.5f) * 2.f);
}
// N(0,1) like the harness's torch.randn(...).half() operands (Box-Muller on a counter hash; benchmarking_utils.py:36-37)
__global__ void fill_randn(__half* p, size_t n, uint32_t seed) {
  size_t i = blockIdx.x * size_t(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  uint32_t x = uint32_t(i) * 2654435761u ^ seed, y = uint32_t(i >> 32) * 0x9E3779B9u + uint32_t(i) * 0x85ebca6bu + ~seed;
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  y ^= y >> 16; y *= 0x7feb352du; y ^= y >> 15; y *= 0x846ca68bu; y ^= y >> 16;
  const float u1 = (float(x >> 8) + 1.0f) * (1.0f / 16777217.0f), u2 = float(y >> 8) * (1.0f / 16777216.0f);
  p[i] = __float2half(sqrtf(-2.0f * __logf(u1)) * __cosf(6.28318530718f * u2));
}
// row-major [R,C] -> row-major [C,R] (tools/utils.py:110-115 as_col_major on the device, for the harness protocol)
__global__ void transpose_rc(const __half* __restrict__ in, __half* __restrict__ out, int R, int C) {
  __shared__ __half tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += 8) {
    const int r = r0 + j, c = c0 + threadIdx.x;
    if (r < R && c < C) tile[j][threadIdx.x] = in[size_t(r) * C + c];
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += 8) {
    const int c = c0 + j, r = r0 + threadIdx.x;
    if (r < R && c < C) out[size_t(c) * R + r] = tile[threadIdx.x][j];
  }
}
__global__ void fill_u16(uint16_t* p, size_t n, uint16_t v) {
  size_t i = blockIdx.x * size_t(blockDim.x) + threadIdx.x;
  if (i < n) p[i] = v;
}
// independent checker: one thread per C element, fp32 accumulation, RN to fp16
__global__ void naive_tn(const __half* A, const __half* Bt, __half* C, int M, int N, int K) {
  int n = blockIdx.x * blockDim.x + threadIdx.x;
  int m = blockIdx.y * blockDim.y + threadIdx.y;
  if (m >= M || n >= N) return;
  float acc = 0.f;
  for (int k = 0; k < K; ++k) acc += __half2float(A[size_t(m) * K + k]) * __half2float(Bt[size_t(n) * K + k]);
  C[size_t(m) * N + n] = __float2half_rn(acc);
}
__global__ void compare(const uint16_t* a, const uint16_t* b, size_t n, unsigned long long* nbad, unsigned long long* first) {
  size_t i = blockIdx.x * size_t(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  uint16_t x = a[i], y = b[i];
  if (x == y) return;
  if ((x & 0x7fff) == 0 && (y & 0x7fff) == 0) return;   // +0 vs -0
  atomicAdd(nbad, 1ull);
  atomicMin(first, (unsigned long long)i);
}
__global__ void check_guard(const uint16_t* p, size_t n, uint16_t v, unsigned long long* nbad) {
  size_t i = blockIdx.x * size_t(blockDim.x) + threadIdx.x;
  if (i < n && p[i] != v) atomicAdd(nbad, 1ull);
}

static inline dim3 g1(size_t n) { return dim3(unsigned((n + 255) / 256)); }

struct Problem {
  int M, N, K;
  __half *A, *Bt, *Cbuf, *C, *Cref;
  static constexpr size_t kGuard = 16384;
  void alloc(int m, int n, int k) {
    M = m; N = n; K = k;
    CK(cudaMalloc(&A, size_t(M) * K * 2));
    CK(cudaMalloc(&Bt, size_t(N) * K * 2));
    CK(cudaMalloc(&Cbuf, (size_t(M) * N + 2 * kGuard) * 2));
    CK(cudaMalloc(&Cref, size_t(M) * N * 2));
    C = Cbuf + kGuard;
    fill_ternary<<<g1(size_t(M) * K), 256>>>(A, size_t(M) * K, 0x1234567u);
    fill_ternary<<<g1(size_t(N) * K), 256>>>(Bt, size_t(N) * K, 0x89abcdeu);
    CK(cudaDeviceSynchronize());
  }
  void reset_c() {
    fill_u16<<<g1(size_t(M) * N + 2 * kGuard), 256>>>((uint16_t*)Cbuf, size_t(M) * N + 2 * kGuard, 0x7bffu);
  }
  void release() { cudaFree(A); cudaFree(Bt); cudaFree(Cbuf); cudaFree(Cref); }
};

static cublasHandle_t g_blas;
static void cublas_tn(const Problem& p, __half* out) {
  // row-major C = A * Bt^T  <=>  column-major C^T[N,M] = Bt(op T)[N,K] * A^T[K,M]
  const float alpha = 1.f, beta = 0.f;
  cublasStatus_t s = cublasGemmEx(g_blas, CUBLAS_OP_T, CUBLAS_OP_N, p.N, p.M, p.K, &alpha, p.Bt, CUDA_R_16F, p.K,
                                  p.A, CUDA_R_16F, p.K, &beta, out, CUDA_R_16F, p.N, CUBLAS_COMPUTE_32F,
                                  CUBLAS_GEMM_DEFAULT_TENSOR_OP);
  if (s != CUBLAS_STATUS_SUCCESS) { printf("cublas error %d\n", int(s)); exit(3); }
}

static int run_ours(int acc, int cfg, const Problem& p, int group_m = 0, int splits = 1) {
  if (cfg < 0)
    return acc == 32 ? b200_hgemm_f32acc(p.A, nullptr, p.Bt, p.C, p.M, p.N, p.K, nullptr)
                     : b200_hgemm_f16acc(p.A, nullptr, p.Bt, p.C, p.M, p.N, p.K, nullptr);
  return b200_hgemm_run_config(acc, cfg, p.A, p.Bt, p.C, p.M, p.N, p.K, group_m, 0, splits, nullptr);
}

static int do_check(int acc, int cfg, int M, int N, int K, int gm = 0, int splits = 1) {
  Problem p; p.alloc(M, N, K);
  const bool use_naive = double(M) * N * K <= 2.2e10;
  if (use_naive) {
    dim3 b(32, 8), g((N + 31) / 32, (M + 7) / 8);
    naive_tn<<<g, b>>>(p.A, p.Bt, p.Cref, M, N, K);
  } else {
    cublas_tn(p, p.Cref);
  }
  CK(cudaDeviceSynchronize());
  p.reset_c();
  CK(cudaDeviceSynchronize());
  int st = run_ours(acc, cfg, p, gm, splits);
  if (splits != 1 && st == 0) st = run_ours(acc, cfg, p, gm, splits);   // twice: the counters / flags must reset themselves
  cudaError_t e = cudaDeviceSynchronize();
  int sel = cfg < 0 ? b200_hgemm_select_config(acc, M, N, K) : cfg;
  if (st != 0 || e != cudaSuccess) {
    printf("CHECK acc=%d cfg=%d(%d) %dx%dx%d  LAUNCH-FAIL status=%d (%s) sync=%s\n", acc, cfg, sel, M, N, K, st,
           b200_hgemm_strerror(st), cudaGetErrorString(e));
    return 1;
  }
  unsigned long long *d, h[3] = {0, ~0ull, 0};
  CK(cudaMalloc(&d, 24));
  CK(cudaMemcpy(d, h, 24, cudaMemcpyHostToDevice));
  compare<<<g1(size_t(M) * N), 256>>>((uint16_t*)p.C, (uint16_t*)p.Cref, size_t(M) * N, d, d + 1);
  check_guard<<<g1(Problem::kGuard), 256>>>((uint16_t*)p.Cbuf, Problem::kGuard, 0x7bffu, d + 2);
  check_guard<<<g1(Problem::kGuard), 256>>>((uint16_t*)(p.C + size_t(M) * N), Problem::kGuard, 0x7bffu, d + 2);
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(h, d, 24, cudaMemcpyDeviceToHost));
  const bool ok = h[0] == 0 && h[2] == 0;
  printf("CHECK acc=%d cfg=%d(%d) gm=%d splits=%d %dx%dx%d  %s mismatches=%llu first=(%lld,%lld) guard_bad=%llu checker=%s\n", acc, cfg,
         sel, gm, splits, M, N, K, ok ? "PASS" : "FAIL", h[0], h[0] ? (long long)(h[1] / N) : -1LL,
         h[0] ? (long long)(h[1] % N) : -1LL, h[2], use_naive ? "naive" : "cublas");
  if (!ok && h[0]) {
    // dump a small corner of both matrices around the first mismatch to make layout bugs readable
    size_t r0 = h[1] / N, c0 = (h[1] % N) & ~size_t(7);
    std::vector<__half> a(8), b(8);
    for (size_t r = r0; r < r0 + 4 && r < size_t(M); ++r) {
      CK(cudaMemcpy(a.data(), p.C + r * N + c0, 16, cudaMemcpyDeviceToHost));
      CK(cudaMemcpy(b.data(), p.Cref + r * N + c0, 16, cudaMemcpyDeviceToHost));
      printf("   row %zu col %zu..: got", r, c0);
      for (int i = 0; i < 8; ++i) printf(" %g", __half2float(a[i]));
      printf(" | want");
      for (int i = 0; i < 8; ++i) printf(" %g", __half2float(b[i]));
      printf("\n");
    }
  }
  cudaFree(d);
  p.release();
  fflush(stdout);
  return ok ? 0 : 1;
}

template <class F>
static float time_ms(F&& f, int iters, int warm = 5) {
  cudaEvent_t a, b;
  CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
  for (int i = 0; i < warm; ++i) f();
  CK(cudaDeviceSynchronize());
  CK(cudaEventRecord(a));
  for (int i = 0; i < iters; ++i) f();
  CK(cudaEventRecord(b));
  CK(cudaEventSynchronize(b));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, a, b));
  cudaEventDestroy(a); cudaEventDestroy(b);
  return ms / iters;
}

// One launch at a time, device time between two events, median over `iters` — what a caller that
// synchronises after every call (the harness) can at best observe as kernel time.
template <class F>
static float time_isolated_ms(F&& f, int iters, int warm = 2) {
  cudaEvent_t a, b;
  CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
  std::vector<float> t;
  for (int i = 0; i < warm + iters; ++i) {
    CK(cudaEventRecord(a));
    f();
    CK(cudaEventRecord(b));
    CK(cudaEventSynchronize(b));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, a, b));
    if (i >= warm) t.push_back(ms);
  }
  cudaEventDestroy(a); cudaEventDestroy(b);
  std::sort(t.begin(), t.end());
  return t[t.size() / 2];
}

static void alloc_random(Problem& p, int M, int N, int K) {
  p.alloc(M, N, K);
  fill_normalish<<<g1(size_t(M) * K), 256>>>(p.A, size_t(M) * K, 0x1234567u);
  fill_normalish<<<g1(size_t(N) * K), 256>>>(p.Bt, size_t(N) * K, 0x89abcdeu);
  CK(cudaDeviceSynchronize());
}

static int do_time(int acc, int cfg, int M, int N, int K, int iters, int gm = 0, int splits = 1) {
  Problem p; alloc_random(p, M, N, K);
  const double flops = 2.0 * M * N * K;
  int st = run_ours(acc, cfg, p, gm, splits);
  cudaError_t e = cudaDeviceSynchronize();
  if (st != 0 || e != cudaSuccess) { printf("TIME launch fail %d %s\n", st, cudaGetErrorString(e)); return 1; }
  float ours = time_ms([&] { run_ours(acc, cfg, p, gm, splits); }, iters);
  float blas = time_ms([&] { cublas_tn(p, p.Cref); }, iters);
  int sel = cfg < 0 ? b200_hgemm_select_config(acc, M, N, K) : cfg;
  // the same two, one launch at a time (event pair around each launch, median): what a caller that synchronises after
  // every call can see, with the kernel's ramp-up and tail no longer hidden behind its neighbours
  const float ours_iso = time_isolated_ms([&] { run_ours(acc, cfg, p, gm, splits); }, std::max(iters, 9));
  const float blas_iso = time_isolated_ms([&] { cublas_tn(p, p.Cref); }, std::max(iters, 9));
  printf("TIME-ISOLATED acc=%d cfg=%d(%d) gm=%d splits=%d %dx%dx%d  ours %.2f us | cublas %.2f us | ratio %.3f\n", acc, cfg, sel, gm,
         splits, M, N, K, ours_iso * 1e3, blas_iso * 1e3, blas_iso / ours_iso);
  printf("TIME acc=%d cfg=%d(%d) gm=%d splits=%d %dx%dx%d  ours %.2f us %.1f TFLOP/s | cublas(fp32acc) %.2f us %.1f TFLOP/s | ratio %.3f\n",
         acc, cfg, sel, gm, splits, M, N, K, ours * 1e3, flops / ours * 1e-9, blas * 1e3, flops / blas * 1e-9, blas / ours);
  p.release();
  fflush(stdout);
  return 0;
}

// sustain: back-to-back launches of one kernel for `seconds`, throughput per ~50 ms window. The first windows run at
// burst clocks, the last ones at whatever the power cap leaves: the gap between a kernel's two figures is its power
// appetite, and the harness (seven efficient kernels in rotation, seconds per shape) lives in the second state.
// Run nvidia-smi -lms alongside (tools/gpu/*.sh) to see clocks and watts for each phase.
static int do_sustain(int acc, int cfg, int M, int N, int K, double seconds, int gm, int splits) {
  Problem p; alloc_random(p, M, N, K);
  const double flops = 2.0 * M * N * K;
  if (run_ours(acc, cfg, p, gm, splits) || cudaDeviceSynchronize() != cudaSuccess) { printf("SUSTAIN launch fail\n"); return 1; }
  struct Fn { const char* name; std::function<void()> f; };
  std::vector<Fn> fns = {{"ours", [&] { run_ours(acc, cfg, p, gm, splits); }}, {"cublas", [&] { cublas_tn(p, p.Cref); }}};
  cudaEvent_t a, b; CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
  for (auto& fn : fns) {
    // idle first, so that every kernel starts from the same cool state
    CK(cudaDeviceSynchronize());
    std::this_thread::sleep_for(std::chrono::milliseconds(1500));
    float one = time_ms(fn.f, 3, 1);
    const int per_window = std::max(1, int(50.0 / std::max(one, 1e-3f)));
    std::vector<double> tf;
    const auto t_end = std::chrono::steady_clock::now() + std::chrono::duration<double>(seconds);
    while (std::chrono::steady_clock::now() < t_end) {
      CK(cudaEventRecord(a));
      for (int i = 0; i < per_window; ++i) fn.f();
      CK(cudaEventRecord(b));
      CK(cudaEventSynchronize(b));
      float ms; CK(cudaEventElapsedTime(&ms, a, b));
      tf.push_back(flops * per_window / ms * 1e-9);
    }
    const size_t n = tf.size(), tail = std::max<size_t>(1, n / 4);
    double first = tf[0], last = 0;
    for (size_t i = n - tail; i < n; ++i) last += tf[i] / tail;
    printf("SUSTAIN acc=%d %s cfg=%d gm=%d splits=%d %dx%dx%d  windows=%zu x %d launches  first %.1f TFLOP/s  last-quarter %.1f TFLOP/s  (%.3f)\n",
           acc, fn.name, cfg, gm, splits, M, N, K, n, per_window, first, last, last / first);
    fflush(stdout);
  }
  cudaEventDestroy(a); cudaEventDestroy(b);
  p.release();
  return 0;
}

static int do_sweep(int acc, int M, int N, int K, int iters) {
  Problem p; alloc_random(p, M, N, K);
  const double flops = 2.0 * M * N * K;
  float blas = time_ms([&] { cublas_tn(p, p.Cref); }, iters);
  printf("SWEEP acc=%d %dx%dx%d cublas %.2f us %.1f TFLOP/s\n", acc, M, N, K, blas * 1e3, flops / blas * 1e-9);
  const int ncfg = b200_hgemm_num_configs();
  const int gms[] = {1, 2, 4, 8, 16, 32};
  for (int c = 0; c < ncfg; ++c) {
    int bn, st_, cg, cm, cn; b200_hgemm_config_info(c, &bn, &st_, &cg); b200_hgemm_config_cluster(c, &cm, &cn);
    const int mr = b200_hgemm_config_m_rep(c);
    if ((M + 127) / 128 < cg * cm * mr || (N + bn - 1) / bn < cn) continue;
    for (int gm : gms) {
      const int nm = (M + 128 * cg * cm * mr - 1) / (128 * cg * cm * mr);
      if (gm > 1 && gm / 2 >= nm) continue;   // wider than the problem: same schedule as the previous one
      int st = run_ours(acc, c, p, gm);
      cudaError_t e = cudaDeviceSynchronize();
      if (st != 0 || e != cudaSuccess) { printf("  cfg %d gm %d FAIL %d %s\n", c, gm, st, cudaGetErrorString(e)); return 1; }
      float t = time_ms([&] { run_ours(acc, c, p, gm); }, iters, 3);
      printf("  cfg=%d (BN=%d st=%d cg=%d cl=%dx%d) gm=%-2d  %.2f us  %.1f TFLOP/s  vs cublas %.3f\n", c, bn, st_, cg, cm, cn, gm,
             t * 1e3, flops / t * 1e-9, blas / t);
    }
  }
  p.release();
  fflush(stdout);
  return 0;
}

// grid: time every configuration on every shape of the harness grid (+ the extra LLM shape); one CSV line per
// shape:  M,N,K,cublas_us,best_cfg,best_gm,best_us,<cfg>:<gm>:<us>...   Used by tools/tune_b200.py.
// wall_metric: time each launch the way the harness does (host clock around one call bracketed by device
// synchronisation, reference benchmarking_utils.py:23-31) and rank candidates by their mean TFLOP/s over the rounds —
// the quantity the sweep is scored on — instead of the median CUDA-event time of the isolated launch.
static int do_grid(int acc, int part, int nparts, double budget_ms, double min_gflop = 0.0, double max_gflop = 1e30,
                   bool wall_metric = false) {
  const int G[10] = {64, 128, 256, 512, 1024, 2048, 4096, 8192, 12288, 16384};
  std::vector<std::array<int, 3>> shapes;
  for (int a : G) for (int b : G) for (int c : G) shapes.push_back({a, b, c});
  shapes.push_back({2048, 11008, 4096});
  const int ncfg = b200_hgemm_num_configs();
  // one allocation, sized for the largest problem, reused by every shape
  const size_t maxe = size_t(16384) * 16384;
  Problem p;
  CK(cudaMalloc(&p.A, maxe * 2)); CK(cudaMalloc(&p.Bt, maxe * 2));
  CK(cudaMalloc(&p.Cbuf, maxe * 2)); CK(cudaMalloc(&p.Cref, maxe * 2));
  p.C = p.Cbuf;
  fill_normalish<<<g1(maxe), 256>>>(p.A, maxe, 0x1234567u);
  fill_normalish<<<g1(maxe), 256>>>(p.Bt, maxe, 0x89abcdeu);
  CK(cudaDeviceSynchronize());
  for (size_t si = 0; si < shapes.size(); ++si) {
    if (int(si % nparts) != part) continue;
    p.M = shapes[si][0]; p.N = shapes[si][1]; p.K = shapes[si][2];
    const double flops = 2.0 * p.M * p.N * p.K;
    if (flops * 1e-9 < min_gflop || flops * 1e-9 > max_gflop) continue;
    const double est_ms = flops / 1.0e15 * 1e3 + 0.004;
    const int iters = std::max(3, std::min(40, int(budget_ms / est_ms)));
    float blas = 0.f;
    std::string line;
    int best_c = -1, best_g = 0, best_s = 1; float best_t = 1e30f;
    struct Cand { int c, gm, sp; std::vector<float> t; };
    std::vector<Cand> all;
    // B200_TUNE_CFGS="3,26,27": only these configurations are candidates (a focused pass over one size class);
    // B200_TUNE_KEEP_ALL=1: the wall-metric mode ranks every candidate instead of a shortlist
    static const std::vector<int> only_cfgs = [] {
      std::vector<int> v;
      if (const char* e = getenv("B200_TUNE_CFGS")) { for (const char* q = e; *q;) { v.push_back(atoi(q)); while (*q && *q != ',') ++q; if (*q) ++q; } }
      return v;
    }();
    static const bool keep_all = getenv("B200_TUNE_KEEP_ALL") != nullptr;
    for (int c = 0; c < ncfg; ++c) {
      if (!only_cfgs.empty() && std::find(only_cfgs.begin(), only_cfgs.end(), c) == only_cfgs.end()) continue;
      int bn, st_, cg, cm, cn; b200_hgemm_config_info(c, &bn, &st_, &cg); b200_hgemm_config_cluster(c, &cm, &cn);
      const int mr = b200_hgemm_config_m_rep(c);
      if ((p.M + 127) / 128 < cg * cm * mr || (p.N + bn - 1) / bn < cn) continue;   // part of the tile would only see padding
      if (mr > 1 && p.K < 2048) continue;   // no accumulator ring: the epilogue is exposed, only a long K amortises it
      // pair + multicast: exact, but slower than plain pairs in every event-time run; the wall-metric mode keeps them,
      // because they move the fewest bytes per FLOP (what cuBLAS's 2x2_2cta kernels do) and that is what counts at the power cap
      if (cg == 2 && cm * cn > 1 && !wall_metric) continue;
      const bool plain = (cm * cn == 1) && bn >= 64 && mr == 1;
      const int nm = (p.M + 128 * cg * cm * mr - 1) / (128 * cg * cm * mr);
      const int nn = (p.N + bn * cn - 1) / (bn * cn);
      std::vector<std::pair<int, int>> cands = {{0, 1}};   // (group_m, splits)
      if (nm * nn > 148 / (cg * cm * cn) && nm > 1 && nn > 1) {
        cands = {{1, 1}, {4, 1}, {8, 1}, {16, 1}};
        if (nm >= 32) cands.push_back({32, 1});
      }
      const int nkb = (p.K + 63) / 64;
      if (plain && cg == 1 && nm * nn * 2 <= 148 && nkb >= 4)
        for (int sp : {2, 3, 4, 6, 8, 12, 16, 24, 32})
          if (sp <= 148 / (nm * nn) && sp <= nkb) cands.push_back({0, sp});
      if (plain && cg == 1 && nkb >= 8 && nm * nn <= 148)
        for (int cs : {2, 4, 8})
          if (nm * nn * cs <= 296 && nkb >= 2 * cs) cands.push_back({0, -cs});   // cluster (DSMEM) split-K
      // stream-K (splits code 100: the partial last wave, 101: that plus one full wave) where the tile count leaves
      // more than 5 % of the last wave empty
      // (round 2: in the harness's synchronised-call metric stream-K won 41 of the 51 tensor-bound shapes it was tuned
      //  into, also where the last wave is nearly full, so it is a candidate wherever the tile count is not a wave multiple)
      const int workers = 148 / cg;
      if (plain && (nm * nn) % workers != 0 && nkb >= 8) {
        const std::vector<int> sk_gms = (nm * nn > workers && nm > 1 && nn > 1) ? std::vector<int>{4, 16} : std::vector<int>{0};
        for (int g : sk_gms) {
          cands.push_back({g, 100});
          if (nm * nn > workers) cands.push_back({g, 101});
        }
      }
      for (const auto& cand_ : cands) {
        const int gm = cand_.first, sp = cand_.second;
        if (gm > 1 && gm / 2 >= nm) continue;
        if (run_ours(acc, c, p, gm, sp) != 0 || cudaDeviceSynchronize() != cudaSuccess) { printf("GRIDFAIL %d %d %d cfg %d gm %d sp %d\n", p.M, p.N, p.K, c, gm, sp); return 1; }
        all.push_back({c, gm, sp, {}});
      }
    }
    // Interleave: every round times each candidate (and cuBLAS) once, one isolated launch each, so that all of
    // them see the same clock / thermal state — what the harness's alternating calls see.
    std::vector<float> blas_t;
    cudaEvent_t ea, eb; CK(cudaEventCreate(&ea)); CK(cudaEventCreate(&eb));
    auto once_event = [&](auto&& f) {
      float ms;
      CK(cudaEventRecord(ea)); f(); CK(cudaEventRecord(eb)); CK(cudaEventSynchronize(eb));
      CK(cudaEventElapsedTime(&ms, ea, eb));
      return ms;
    };
    auto once_wall = [&](auto&& f) {
      CK(cudaDeviceSynchronize());
      const auto t0 = std::chrono::steady_clock::now();
      f();
      CK(cudaDeviceSynchronize());
      return std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    };
    auto median = [](std::vector<float> v) { std::sort(v.begin(), v.end()); return v[v.size() / 2]; };
    if (wall_metric) {
      // Two phases. A rotation through ~40 candidates, most of them far from the best, leaves the chip below its power
      // cap, and the ranking of the good ones in that state is not their ranking in the harness, whose rotation holds
      // only efficient kernels (ours + six cuBLAS flavours) and sits at the cap: in round 1 the event-time tuner
      // preferred 128x256 single-CTA tiles on many large shapes where the 256x256 CTA-pair tile is 2-5 % better in
      // the harness. So: a quick event-time pass shortlists, the shortlist is ranked in a harness-like rotation.
      // An isolated launch between two events never measures less than ≈13 us on this system (round 1: twelve very
      // different candidates of 256x2048x2048 all read 14.2-14.5 us), so short kernels are shortlisted on bursts of
      // back-to-back launches, whose per-launch time does expose the kernel's own duration.
      const int quick = std::max(2, iters / 4);
      const int burst = est_ms < 0.03 ? 8 : 1;
      for (int r = 0; r < quick + 1; ++r)
        for (auto& cd : all) {
          const float t = once_event([&] { for (int b = 0; b < burst; ++b) run_ours(acc, cd.c, p, cd.gm, cd.sp); }) / burst;
          if (r) cd.t.push_back(t);
        }
      std::sort(all.begin(), all.end(), [&](const Cand& x, const Cand& y) { return median(x.t) < median(y.t); });
      std::vector<Cand> keep;
      auto have_cfg = [&](int c) { for (auto& k : keep) if (k.c == c) return true; return false; };
      int plain_kept = 0;
      for (auto& cd : all) {
        int bn, st_, cg, cm, cn; b200_hgemm_config_info(cd.c, &bn, &st_, &cg); b200_hgemm_config_cluster(cd.c, &cm, &cn);
        const bool mcast = cm * cn > 1;
        // the six fastest, plus the fastest schedule of every CTA-pair configuration within 8 % of the best, plus — always —
        // the three fastest candidates WITHOUT a multicast cluster: how well a multicast cluster performs depends on the
        // GPC layout of the individual GPU (round 2: configurations 18/19 ranked first on the tuning box and lost 8-10 %
        // on the sweep's box), so the table must always have a portable alternative to compare against
        const bool want_plain = !mcast && plain_kept < 3;
        if (keep_all || keep.size() < 6 || (cg == 2 && !have_cfg(cd.c) && median(cd.t) <= 1.08f * median(all[0].t)) || want_plain) {
          keep.push_back(cd);
          if (!mcast) ++plain_kept;
        }
      }
      all.swap(keep);
      for (auto& cd : all) cd.t.clear();
      int rounds = est_ms < 0.03 ? 3 * iters : iters;   // host-clock samples of a 15 us call scatter by ~1 us: average more of them
      // and long kernels need the rotation to last: the power cap settles over tens of milliseconds (aim at >= 0.3 s)
      rounds = std::max(rounds, std::min(40, int(300.0 / (13.0 * est_ms))));
      rounds = std::max(rounds, 6);   // millisecond kernels at the power cap scatter by several per cent: never fewer than six samples
      for (int r = 0; r < rounds + 1; ++r) {
        // three library calls per round keep the mix (and the power state) close to the harness's rotation
        for (int rep = 0; rep < 3; ++rep) { const float tb = once_wall([&] { cublas_tn(p, p.Cref); }); if (r) blas_t.push_back(tb); }
        for (auto& cd : all) { const float t = once_wall([&] { run_ours(acc, cd.c, p, cd.gm, cd.sp); }); if (r) cd.t.push_back(t); }
      }
    } else {
      for (int r = 0; r < iters + 1; ++r) {
        const float tb = once_event([&] { cublas_tn(p, p.Cref); });
        if (r) blas_t.push_back(tb);
        for (auto& cd : all) { const float t = once_event([&] { run_ours(acc, cd.c, p, cd.gm, cd.sp); }); if (r) cd.t.push_back(t); }
      }
    }
    cudaEventDestroy(ea); cudaEventDestroy(eb);
    // event metric: median time; wall metric: the time whose rate is the mean rate (the harness averages TFLOP/s)
    auto med = [&](std::vector<float>& v) {
      if (wall_metric) { double r = 0; for (float t : v) r += 1.0 / t; return float(v.size() / r); }
      std::sort(v.begin(), v.end());
      return v[v.size() / 2];
    };
    blas = med(blas_t);
    for (auto& cd : all) {
      const float t = med(cd.t);
      char buf[64]; snprintf(buf, sizeof buf, ",%d:%d:%d:%.2f", cd.c, cd.gm, cd.sp, t * 1e3); line += buf;
      if (t < best_t) { best_t = t; best_c = cd.c; best_g = cd.gm; best_s = cd.sp; }
    }
    printf("GRID,%d,%d,%d,%d,%.2f,%d,%d,%d,%.2f%s\n", acc, p.M, p.N, p.K, blas * 1e3, best_c, best_g, best_s, best_t * 1e3, line.c_str());
    fflush(stdout);
  }
  return 0;
}


#ifdef B200_HGEMM_TRACE
// trace (dev_check_trace only, linked against libb200_hgemm_trace.so): where one launch spends its time, from
// per-CTA timestamps written by the instrumented kernel (slots documented next to kTraceSlots in hgemm_sm100.cuh).
extern "C" int b200_hgemm_trace_slots(void);
extern "C" int b200_hgemm_trace_arm(int max_ctas);
extern "C" int b200_hgemm_trace_read(unsigned long long* out, int ctas);

// cold != 0: before the traced launch, other work (a cuBLAS GEMM on other operands, 512 MB of memset) evicts this
// kernel's instructions, descriptors and operands from the caches and the TLBs — the state every call of the
// harness's rotation starts from, as opposed to the back-to-back state of `dev_check time`.
static int do_trace(int acc, int cfg, int M, int N, int K, int gm, int splits, int cold) {
  Problem p; alloc_random(p, M, N, K);
  for (int i = 0; i < 3; ++i) if (run_ours(acc, cfg, p, gm, splits)) { printf("TRACE launch failed\n"); return 1; }
  CK(cudaDeviceSynchronize());
  if (cold) {
    Problem other; alloc_random(other, 2048, 2048, 2048);
    void* scratch; const size_t bytes = size_t(512) << 20;
    CK(cudaMalloc(&scratch, bytes));
    for (int i = 0; i < 2; ++i) { cublas_tn(other, other.Cref); CK(cudaMemsetAsync(scratch, i, bytes)); }
    CK(cudaDeviceSynchronize());
    cudaFree(scratch);
    other.release();
  }
  const int kMaxCtas = 320, S = b200_hgemm_trace_slots();
  if (b200_hgemm_trace_arm(kMaxCtas)) { printf("TRACE arm failed\n"); return 1; }
  if (run_ours(acc, cfg, p, gm, splits)) { printf("TRACE launch failed\n"); return 1; }
  std::vector<unsigned long long> buf(size_t(kMaxCtas) * S * 2);
  if (b200_hgemm_trace_read(buf.data(), kMaxCtas)) { printf("TRACE read failed\n"); return 1; }
  b200_hgemm_trace_arm(0);
  auto gt = [&](int cta, int slot) { return double(buf[(size_t(cta) * S + slot) * 2]); };          // ns
  auto ck = [&](int cta, int slot) { return double(buf[(size_t(cta) * S + slot) * 2 + 1]); };      // SM cycles
  int ctas = 0;
  double t0 = 1e300, t_end = 0;
  for (int c = 0; c < kMaxCtas; ++c) if (gt(c, 0) > 0) { ctas = c + 1; t0 = std::min(t0, gt(c, 0)); t_end = std::max(t_end, gt(c, 8)); }
  if (!ctas) { printf("TRACE: no CTA wrote a timestamp\n"); return 1; }
  struct Row { const char* name; std::vector<double> v; };
  std::vector<Row> rows = {{"entry after first CTA [us]", {}}, {"setup (entry -> barrier) [us]", {}},
                           {"entry -> first TMA issued [us]", {}}, {"entry -> first stage landed [us]", {}},
                           {"main loop: first stage landed -> last accumulator complete [us]", {}},
                           {"MMA issue: cycles per k-block", {}}, {"MMA issue: ns per k-block", {}},
                           {"producer finished before last accumulator by [us]", {}},
                           {"tail: last accumulator complete -> epilogue drained [us]", {}},
                           {"teardown: epilogue drained -> after last barrier [us]", {}},
                           {"CTA lifetime [us]", {}}, {"k-blocks issued", {}}, {"units", {}}};
  for (int c = 0; c < ctas; ++c) {
    if (gt(c, 0) == 0) continue;
    rows[0].v.push_back((gt(c, 0) - t0) * 1e-3);
    rows[1].v.push_back((gt(c, 1) - gt(c, 0)) * 1e-3);
    if (gt(c, 2) > 0) rows[2].v.push_back((gt(c, 2) - gt(c, 0)) * 1e-3);
    if (gt(c, 4) > 0) {   // leader CTAs only (the MMA issuer)
      rows[3].v.push_back((gt(c, 4) - gt(c, 0)) * 1e-3);
      if (gt(c, 10) > 0) rows[4].v.push_back((gt(c, 10) - gt(c, 4)) * 1e-3);
      const double kb = gt(c, 9);
      if (kb > 0) { rows[5].v.push_back((ck(c, 5) - ck(c, 4)) / kb); rows[6].v.push_back((gt(c, 5) - gt(c, 4)) / kb); }
      rows[11].v.push_back(kb); rows[12].v.push_back(gt(c, 11));
    }
    if (gt(c, 3) > 0 && gt(c, 10) > 0) rows[7].v.push_back((gt(c, 10) - gt(c, 3)) * 1e-3);
    if (gt(c, 7) > 0 && gt(c, 10) > 0) rows[8].v.push_back((gt(c, 7) - gt(c, 10)) * 1e-3);
    if (gt(c, 7) > 0) rows[9].v.push_back((gt(c, 8) - gt(c, 7)) * 1e-3);
    rows[10].v.push_back((gt(c, 8) - gt(c, 0)) * 1e-3);
  }
  int sel = cfg < 0 ? b200_hgemm_select_config(acc, M, N, K) : cfg;
  printf("TRACE acc=%d cfg=%d(%d) gm=%d splits=%d %s %dx%dx%d  ctas=%d  first entry -> last exit %.2f us\n", acc, cfg, sel, gm, splits,
         cold ? "COLD" : "warm", M, N, K, ctas, (t_end - t0) * 1e-3);
  for (auto& r : rows) {
    if (r.v.empty()) continue;
    std::sort(r.v.begin(), r.v.end());
    printf("  %-72s min %10.2f  median %10.2f  max %10.2f  (n=%zu)\n", r.name, r.v.front(), r.v[r.v.size() / 2], r.v.back(), r.v.size());
  }
  p.release();
  return 0;
}
#endif

// wall: the harness's measurement PROTOCOL in C++ (reference benchmarking_offline.py:119-161, benchmarking_utils.py:12-69;
// eval_one_file.sh:71-135), one (baseline, ours) pair at a time as the reference runs one pair per process:
//   per pair     warm-up loop in the fixed order [baseline, ours], then the timed loop with the order shuffled per iteration;
//   per iteration  fresh N(0,1) A [M,K] and B [K,N]; every function gets ITS OWN copies (a clone of A, a clone of B, the
//                K-major transpose of B) and its own output filled with noise; device sync;
//   per call     the output is zero-filled, device sync, host clock, ONE call, device sync, host clock;
//   metric       mean over iterations of 2MNK / t per function; speed-up of a pair = ours / baseline FROM THAT PAIR;
//                "-max" = the harder layout = the smaller speed-up (summarize_result.py:43-53).
// cuBLASLt auto-tuning first runs the reference's search (50 warm-up + 100 timed rounds over every candidate the heuristic
// returns) unless other round counts are given. `seconds` is the timed loop of each auto-tuning pair; the four pairs
// that only fill the other CSV columns get 40 % of it. The pairs run in shuffled order.
struct WallBuffers {   // sized once for the largest problem of a run
  __half *A0, *B0;                 // this iteration's operands
  __half *A[2], *Brow[2], *Bt[2], *C[2];   // [0] baseline's copies, [1] ours
  void alloc(size_t maxe) {
    CK(cudaMalloc(&A0, maxe * 2)); CK(cudaMalloc(&B0, maxe * 2));
    for (int f = 0; f < 2; ++f) {
      CK(cudaMalloc(&A[f], maxe * 2)); CK(cudaMalloc(&Brow[f], maxe * 2)); CK(cudaMalloc(&Bt[f], maxe * 2)); CK(cudaMalloc(&C[f], maxe * 2));
    }
  }
  void release() {
    cudaFree(A0); cudaFree(B0);
    for (int f = 0; f < 2; ++f) { cudaFree(A[f]); cudaFree(Brow[f]); cudaFree(Bt[f]); cudaFree(C[f]); }
  }
};

static int wall_one(int acc, int M, int N, int K, WallBuffers& w, double seconds, int tune_warm, int tune_bench) {
  int cand[2] = {0, 0}; float best_ms[2] = {0, 0};
  if (tune_warm < 0) {
    // adaptive: the reference's 50 + 100 rounds where they are cheap, fewer for long kernels so that the search of one
    // layout stays near `-tune_warm` x 10 ms (8 candidates is what the heuristic returns on this library), never below 10 + 20
    const double est = std::max(std::max(2.0 * M * N * K / 1.2e15, 2.0 * (double(M) * K + double(N) * K + double(M) * N) / 5e12), 5e-6) + 8e-6;
    const double budget = -tune_warm * 0.01;
    const int rounds = std::max(30, std::min(150, int(budget / (8.0 * est))));
    tune_warm = rounds / 3; tune_bench = rounds - tune_warm;
  }
  for (int lay = 0; lay < 2; ++lay) {
    int st = b200_bl_lt_autotune_find(acc, lay, M, N, K, tune_warm, tune_bench);
    if (st) { printf("WALLFAIL,%d,%d,%d,%d,autotune find status %d\n", acc, M, N, K, st); return 1; }
    b200_bl_lt_autotune_info(acc, lay, &cand[lay], &best_ms[lay]);
  }
  // baseline f(copies index 0); ours always works on copies index 1
  struct Fn { const char* name; bool primary; std::function<int()> f; };
  std::vector<Fn> base = {
      {"cublas_tn", false, [&] { return b200_bl_cublas(acc, 1, w.A[0], w.Bt[0], w.C[0], M, N, K); }},
      {"cublas_nn", false, [&] { return b200_bl_cublas(acc, 0, w.A[0], w.Brow[0], w.C[0], M, N, K); }},
      {"lt_heur_tn", false, [&] { return b200_bl_lt_heuristic(acc, 1, w.A[0], w.Bt[0], w.C[0], M, N, K); }},
      {"lt_heur_nn", false, [&] { return b200_bl_lt_heuristic(acc, 0, w.A[0], w.Brow[0], w.C[0], M, N, K); }},
      {"lt_auto_tn", true, [&] { return b200_bl_lt_autotune(acc, 1, w.A[0], w.Bt[0], w.C[0], M, N, K); }},
      {"lt_auto_nn", true, [&] { return b200_bl_lt_autotune(acc, 0, w.A[0], w.Brow[0], w.C[0], M, N, K); }},
  };
  auto ours = [&] {
    return acc == 32 ? b200_hgemm_f32acc(w.A[1], w.Brow[1], w.Bt[1], w.C[1], M, N, K, nullptr)
                     : b200_hgemm_f16acc(w.A[1], w.Brow[1], w.Bt[1], w.C[1], M, N, K, nullptr);
  };
  const size_t ea = size_t(M) * K, eb = size_t(K) * N, ec = size_t(M) * N;
  const double flops = 2.0 * M * N * K;
  static uint32_t draw = 1;
  auto new_operands = [&] {   // run_all_perf_funcs_once, benchmarking_utils.py:35-58
    fill_randn<<<g1(ea), 256>>>(w.A0, ea, 0x1234567u + 7919u * draw);
    fill_randn<<<g1(eb), 256>>>(w.B0, eb, 0x89abcdeu + 104729u * draw);
    ++draw;
    for (int f = 0; f < 2; ++f) {
      CK(cudaMemcpyAsync(w.A[f], w.A0, ea * 2, cudaMemcpyDeviceToDevice));
      CK(cudaMemcpyAsync(w.Brow[f], w.B0, eb * 2, cudaMemcpyDeviceToDevice));
      transpose_rc<<<dim3((N + 31) / 32, (K + 31) / 32), dim3(32, 8)>>>(w.Brow[f], w.Bt[f], K, N);
      fill_randn<<<g1(ec), 256>>>(w.C[f], ec, 0x5555u + 31u * draw + f);
    }
    CK(cudaDeviceSynchronize());
  };
  auto now = [] { return std::chrono::steady_clock::now(); };
  auto timed = [&](int which, const std::function<int()>& f, double* ms, double* call_ms) {   // run_benchmark, :12-33
    CK(cudaMemsetAsync(w.C[which], 0, ec * 2));
    CK(cudaDeviceSynchronize());
    const auto t0 = now();
    const int st = f();
    const auto t_ret = now();
    CK(cudaDeviceSynchronize());
    *ms = std::chrono::duration<double, std::milli>(now() - t0).count();
    *call_ms = std::chrono::duration<double, std::milli>(t_ret - t0).count();
    return st;
  };
  std::vector<int> order(base.size());
  for (size_t i = 0; i < order.size(); ++i) order[i] = int(i);
  std::mt19937 rng(12345u + uint32_t(M) * 31u + uint32_t(N) * 17u + uint32_t(K));
  std::shuffle(order.begin(), order.end(), rng);
  std::vector<double> base_tf(base.size(), 0.0), ours_tf(base.size(), 0.0), base_ms(base.size(), 0.0), ours_ms(base.size(), 0.0);
  std::vector<int> iters(base.size(), 0);
  double ours_call_ms = 0.0, base_call_ms = 0.0; int calls = 0;
  for (int bi : order) {
    const double bench_s = base[bi].primary ? seconds : 0.4 * seconds, warm_s = 0.25 * bench_s;
    new_operands();
    if (base[bi].f() || ours()) { printf("WALLFAIL,%d,%d,%d,%d,first call failed: %s\n", acc, M, N, K, base[bi].name); return 1; }
    CK(cudaDeviceSynchronize());
    const auto t_begin = now();
    int warm_iters = 0;
    while (warm_iters < 1 || std::chrono::duration<double>(now() - t_begin).count() < warm_s) {
      new_operands();
      double ms, cm;
      timed(0, base[bi].f, &ms, &cm); timed(1, ours, &ms, &cm);
      ++warm_iters;
    }
    const auto t_bench = now();
    while (iters[bi] < 3 || std::chrono::duration<double>(now() - t_bench).count() < bench_s) {
      new_operands();
      const bool ours_first = rng() & 1u;   // random.shuffle of the two-element list
      double ms_b = 0, ms_o = 0, cm_b = 0, cm_o = 0;
      if (ours_first) { timed(1, ours, &ms_o, &cm_o); timed(0, base[bi].f, &ms_b, &cm_b); }
      else { timed(0, base[bi].f, &ms_b, &cm_b); timed(1, ours, &ms_o, &cm_o); }
      base_tf[bi] += flops / ms_b * 1e-9; ours_tf[bi] += flops / ms_o * 1e-9;
      base_ms[bi] += ms_b; ours_ms[bi] += ms_o;
      ours_call_ms += cm_o; base_call_ms += cm_b; ++calls;
      ++iters[bi];
    }
  }
  int cfg, gm, sp; b200_hgemm_select(acc, M, N, K, &cfg, &gm, &sp);
  double ours_mean = 0.0, ours_ms_mean = 0.0; int samples = 0;
  for (size_t i = 0; i < base.size(); ++i) { ours_mean += ours_tf[i] / iters[i]; ours_ms_mean += ours_ms[i] / iters[i]; samples += iters[i]; }
  ours_mean /= base.size(); ours_ms_mean /= base.size();
  printf("WALL,%d,%d,%d,%d,samples=%d,cfg=%d,gm=%d,splits=%d,lt_candidates=%d/%d,tune_rounds=%d+%d,protocol=pairs,ours=%.6g", acc, M, N, K,
         samples, cfg, gm, sp, cand[1], cand[0], tune_warm, tune_bench, ours_mean);
  double sp_auto[2] = {0, 0};
  for (size_t i = 0; i < base.size(); ++i) {
    const double b = base_tf[i] / iters[i], o = ours_tf[i] / iters[i];
    printf(",%s=%.6g,%s_speedup=%.4f,%s_n=%d", base[i].name, b, base[i].name, o / b, base[i].name, iters[i]);
    if (i == 4) sp_auto[0] = o / b;
    if (i == 5) sp_auto[1] = o / b;
  }
  printf(",speedup_vs_lt_auto_max=%.4f,ours_us=%.2f,lt_auto_tn_us=%.2f,ours_call_us=%.2f,baseline_call_us=%.2f\n", std::min(sp_auto[0], sp_auto[1]),
         ours_ms_mean * 1e3, base_ms[4] / iters[4] * 1e3, ours_call_ms / calls * 1e3, base_call_ms / calls * 1e3);
  fflush(stdout);
  return 0;
}

static int do_wall(int acc, int M, int N, int K, double seconds, int tune_warm, int tune_bench) {
  WallBuffers w;
  w.alloc(std::max(std::max(size_t(M) * K, size_t(K) * N), size_t(M) * N));
  if (b200_bl_init(acc)) { printf("baseline init failed\n"); return 1; }
  int rc = wall_one(acc, M, N, K, w, seconds, tune_warm, tune_bench);
  w.release();
  return rc;
}

// wallgrid: `wall` over this process's share of the 1001-shape grid (shapes sorted by cost, dealt round-robin
// to `nparts` processes — one per GPU), all in one process so that CUDA/cuBLAS start-up is paid once.
// B200_WALLGRID_SHAPES=<file of "M N K" lines> replaces the grid (stratified samples, reruns of single shapes).
static int do_wallgrid(int acc, int part, int nparts, double seconds, int tune_warm, int tune_bench, int limit) {
  const int G[10] = {64, 128, 256, 512, 1024, 2048, 4096, 8192, 12288, 16384};
  std::vector<std::array<int, 3>> shapes;
  if (const char* path = getenv("B200_WALLGRID_SHAPES")) {
    FILE* f = fopen(path, "r");
    if (!f) { printf("cannot open %s\n", path); return 1; }
    int a, b, c;
    while (fscanf(f, "%d %d %d", &a, &b, &c) == 3) shapes.push_back({a, b, c});
    fclose(f);
  } else {
    for (int a : G) for (int b : G) for (int c : G) shapes.push_back({a, b, c});
    shapes.push_back({2048, 11008, 4096});
  }
  auto cost = [](const std::array<int, 3>& s) { return double(s[0]) * s[1] * s[2] + 3e9 * (double(s[0]) * s[1] + double(s[1]) * s[2] + double(s[0]) * s[2]) / 1e6; };
  std::stable_sort(shapes.begin(), shapes.end(), [&](const auto& x, const auto& y) { return cost(x) > cost(y); });
  size_t maxe = 0;
  for (const auto& sh : shapes)
    maxe = std::max(maxe, std::max(std::max(size_t(sh[0]) * sh[2], size_t(sh[2]) * sh[1]), size_t(sh[0]) * sh[1]));
  WallBuffers w;
  w.alloc(maxe);
  if (b200_bl_init(acc)) { printf("baseline init failed\n"); return 1; }
  int done = 0, failed = 0;
  const auto t0 = std::chrono::steady_clock::now();
  for (size_t si = 0; si < shapes.size(); ++si) {
    if (int(si % nparts) != part) continue;
    if (limit > 0 && done >= limit) break;
    failed += wall_one(acc, shapes[si][0], shapes[si][1], shapes[si][2], w, seconds, tune_warm, tune_bench);
    ++done;
  }
  printf("WALLGRID done=%d failed=%d seconds=%.1f\n", done, failed, std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
  w.release();
  return failed ? 1 : 0;
}

int main(int argc, char** argv) {
  if (argc < 2) { printf("usage: see source header\n"); return 64; }
  CK(cudaSetDevice(0));
  cublasCreate(&g_blas);
  std::string mode = argv[1];
  if (mode == "check" && argc >= 7)
    return do_check(atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), atoi(argv[5]), atoi(argv[6]), argc > 7 ? atoi(argv[7]) : 0,
                    argc > 8 ? atoi(argv[8]) : 1);
  if (mode == "time" && argc >= 7)
    return do_time(atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), atoi(argv[5]), atoi(argv[6]), argc > 7 ? atoi(argv[7]) : 20,
                   argc > 8 ? atoi(argv[8]) : 0, argc > 9 ? atoi(argv[9]) : 1);
  if (mode == "sustain" && argc >= 7)
    return do_sustain(atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), atoi(argv[5]), atoi(argv[6]), argc > 7 ? atof(argv[7]) : 3.0,
                      argc > 8 ? atoi(argv[8]) : 0, argc > 9 ? atoi(argv[9]) : 1);
  if (mode == "sweep" && argc >= 6)
    return do_sweep(atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), atoi(argv[5]), argc > 6 ? atoi(argv[6]) : 20);
#ifdef B200_HGEMM_TRACE
  if (mode == "trace" && argc >= 7)
    return do_trace(atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), atoi(argv[5]), atoi(argv[6]), argc > 7 ? atoi(argv[7]) : 0,
                    argc > 8 ? atoi(argv[8]) : 1, argc > 9 ? atoi(argv[9]) : 0);
#endif
  if (mode == "wall" && argc >= 6)
    return do_wall(atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), atoi(argv[5]), argc > 6 ? atof(argv[6]) : 1.0,
                   argc > 7 ? atoi(argv[7]) : 0, argc > 8 ? atoi(argv[8]) : 0);
  if (mode == "wallgrid" && argc >= 5)
    return do_wallgrid(atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), argc > 5 ? atof(argv[5]) : 0.3, argc > 6 ? atoi(argv[6]) : 5,
                       argc > 7 ? atoi(argv[7]) : 15, argc > 8 ? atoi(argv[8]) : 0);
  if (mode == "grid" && argc >= 3)
    return do_grid(atoi(argv[2]), argc > 3 ? atoi(argv[3]) : 0, argc > 4 ? atoi(argv[4]) : 1, argc > 5 ? atof(argv[5]) : 3.0, argc > 6 ? atof(argv[6]) : 0.0, argc > 7 ? atof(argv[7]) : 1e30,
                   argc > 8 && std::string(argv[8]) == "wall");
  printf("bad arguments\n");
  return 64;
}
