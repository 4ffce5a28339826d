// libb200_hgemm.so — C-ABI entry points declared in include/b200_hgemm.h.
// Holds every kernel configuration and the per-shape dispatcher. No torch, no CUTLASS, no cuBLAS.
#include "../../include/b200_hgemm.h"

#include <atomic>
#include <cstdlib>
#include <map>
#include <memory>
#include <mutex>

#include "hgemm_configs.cuh"
#include "hgemm_dispatch.cuh"

namespace {

std::atomic<unsigned long long> g_launches{0};
constexpr int kBf16Acc32 = 0xB32;   // internal selector of run(): bf16 operands, fp32 accumulation

template <bool kAccF32, bool kBf16 = false>
int run_config(int id, const void* A, const void* Bt, void* C, int M, int N, int K, int group_m, int max_ctas,
               int splits, cudaStream_t s) {
  using namespace b200;
  int st;
  switch (id) {
#define B200_CASE(ID, BN, STAGES, CG, CM, CN, MR)                                                      \
  case ID:                                                                                         \
    st = host::launch<Config<BN, STAGES, CG, kAccF32, CM, CN, MR, kBf16>>(A, Bt, C, M, N, K, s, group_m, max_ctas, splits); \
    break;
    B200_HGEMM_CONFIGS(B200_CASE)
#undef B200_CASE
    default:
      return host::kBadConfig;
  }
  if (st == host::kOk) g_launches.fetch_add(1, std::memory_order_relaxed);
  return st;
}

template <class Cfg>
int schedule_units(int M, int N, int K, int splits, int num_sms, int worker, int* units, int max_units,
                   int* num_workers, int* sk_tiles, int* contributors) {
  using namespace b200;
  const host::Plan p = host::make_plan<Cfg>(M, N, K, num_sms / Cfg::CLUSTER_CTAS, splits);
  if (num_workers) *num_workers = p.workers;
  if (sk_tiles) *sk_tiles = p.sk_tiles;
  if (worker < 0 || worker >= p.workers) return host::kBadShape;
  WorkIter it(worker, p.workers, p.num_tiles, p.nkb, p.splits, p.sk_tiles);
  WorkUnit u;
  int n = 0;
  while (it.next(u)) {
    if (n < max_units && units) {
      units[3 * n] = u.tile; units[3 * n + 1] = u.kb0; units[3 * n + 2] = u.kb1;
      if (contributors)
        contributors[n] = (p.sk_tiles && u.kb0 == 0 && u.kb1 < p.nkb)
                              ? streamk_contributors(worker, p.workers, p.sk_tiles * p.nkb, u.tile, p.nkb) : 0;
    }
    ++n;
  }
  return n;
}

int run(int acc_bits, int id, const void* A, const void* Bt, void* C, int M, int N, int K, int group_m,
        int max_ctas, int splits, void* stream) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (acc_bits == 32) return run_config<true>(id, A, Bt, C, M, N, K, group_m, max_ctas, splits, s);
  if (acc_bits == 16) return run_config<false>(id, A, Bt, C, M, N, K, group_m, max_ctas, splits, s);
  if (acc_bits == kBf16Acc32) return run_config<true, true>(id, A, Bt, C, M, N, K, group_m, max_ctas, splits, s);
  return b200::host::kBadConfig;
}

constexpr int kHostBlocks = 8;   // at most this many row blocks in the pipelined host entry
struct HostCtx {
  std::mutex mu;
  void* dbuf = nullptr; size_t dcap = 0;
  cudaStream_t in = nullptr, run = nullptr, out = nullptr;
  cudaEvent_t b_in = nullptr, a_in[kHostBlocks] = {}, done[kHostBlocks] = {};
};
std::mutex g_host_mu;
std::map<int, std::unique_ptr<HostCtx>> g_host_ctx;
HostCtx& host_ctx(int dev) {
  std::lock_guard<std::mutex> lock(g_host_mu);
  auto& slot = g_host_ctx[dev];
  if (!slot) slot.reset(new HostCtx());
  return *slot;
}

}  // namespace

extern "C" {

int b200_hgemm_num_configs(void) { return b200::kNumConfigs; }

int b200_hgemm_config_info(int config_id, int* bn, int* stages, int* cta_group) {
  switch (config_id) {
#define B200_CASE(ID, BN, STAGES, CG, CM, CN, MR)  \
  case ID:                             \
    if (bn) *bn = BN;                  \
    if (stages) *stages = STAGES;      \
    if (cta_group) *cta_group = CG;    \
    return 0;
    B200_HGEMM_CONFIGS(B200_CASE)
#undef B200_CASE
    default:
      return b200::host::kBadConfig;
  }
}

int b200_hgemm_config_cluster(int config_id, int* cluster_m, int* cluster_n) {
  switch (config_id) {
#define B200_CASE(ID, BN, STAGES, CG, CM, CN, MR) \
  case ID:                                    \
    if (cluster_m) *cluster_m = CM;           \
    if (cluster_n) *cluster_n = CN;           \
    return 0;
    B200_HGEMM_CONFIGS(B200_CASE)
#undef B200_CASE
    default:
      return b200::host::kBadConfig;
  }
}

int b200_hgemm_schedule_units(int config_id, int M, int N, int K, int splits, int num_sms, int worker, int* units,
                              int max_units, int* num_workers, int* sk_tiles, int* contributors) {
  if (M <= 0 || N <= 0 || K <= 0 || num_sms <= 0) return b200::host::kBadShape;
  switch (config_id) {
#define B200_CASE(ID, BN, STAGES, CG, CM, CN, MR)                                                                   \
  case ID:                                                                                                          \
    return schedule_units<b200::Config<BN, STAGES, CG, true, CM, CN, MR>>(M, N, K, splits, num_sms, worker, units, \
                                                                          max_units, num_workers, sk_tiles, contributors);
    B200_HGEMM_CONFIGS(B200_CASE)
#undef B200_CASE
    default:
      return b200::host::kBadConfig;
  }
}

int b200_hgemm_config_m_rep(int config_id) {
  switch (config_id) {
#define B200_CASE(ID, BN, STAGES, CG, CM, CN, MR) \
  case ID:                                        \
    return MR;
    B200_HGEMM_CONFIGS(B200_CASE)
#undef B200_CASE
    default:
      return b200::host::kBadConfig;
  }
}

int b200_hgemm_select_config(int acc_bits, int M, int N, int K) {
  if (acc_bits != 32 && acc_bits != 16) return b200::host::kBadConfig;
  if (M <= 0 || N <= 0 || K <= 0) return b200::host::kBadShape;
  return b200::dispatch::select(acc_bits, M, N, K).config_id;
}

int b200_hgemm_select(int acc_bits, int M, int N, int K, int* config_id, int* group_m, int* splits) {
  if (acc_bits != 32 && acc_bits != 16) return b200::host::kBadConfig;
  if (M <= 0 || N <= 0 || K <= 0) return b200::host::kBadShape;
  const b200::dispatch::Choice ch = b200::dispatch::select(acc_bits, M, N, K);
  if (config_id) *config_id = ch.config_id;
  if (group_m) *group_m = ch.group_m;
  if (splits) *splits = ch.splits;
  return 0;
}

int b200_hgemm_run_config(int acc_bits, int config_id, const void* A, const void* B_kmajor, void* C, int M,
                          int N, int K, int group_m, int max_ctas, int splits, void* stream) {
  return run(acc_bits, config_id, A, B_kmajor, C, M, N, K, group_m, max_ctas, splits, stream);
}

int b200_hgemm_f32acc(const void* A, const void* /*B_rowmajor*/, const void* B_kmajor, void* C, int M, int N,
                      int K, void* stream) {
  int st = b200::host::validate(A, B_kmajor, C, M, N, K);
  if (st) return st;
  const b200::dispatch::Choice ch = b200::dispatch::select(32, M, N, K);
  return run(32, ch.config_id, A, B_kmajor, C, M, N, K, ch.group_m, 0, ch.splits, stream);
}

int b200_hgemm_f16acc(const void* A, const void* /*B_rowmajor*/, const void* B_kmajor, void* C, int M, int N,
                      int K, void* stream) {
  int st = b200::host::validate(A, B_kmajor, C, M, N, K);
  if (st) return st;
  const b200::dispatch::Choice ch = b200::dispatch::select(16, M, N, K);
  return run(16, ch.config_id, A, B_kmajor, C, M, N, K, ch.group_m, 0, ch.splits, stream);
}

int b200_bgemm_f32acc(const void* A, const void* /*B_rowmajor*/, const void* B_kmajor, void* C, int M, int N,
                      int K, void* stream) {
  int st = b200::host::validate(A, B_kmajor, C, M, N, K);
  if (st) return st;
  // same data movement and the same MMA rate as the fp16 / fp32-accumulate kernel: its tuned table applies
  const b200::dispatch::Choice ch = b200::dispatch::select(32, M, N, K);
  return run(kBf16Acc32, ch.config_id, A, B_kmajor, C, M, N, K, ch.group_m, 0, ch.splits, stream);
}

int b200_bgemm_run_config(int config_id, const void* A, const void* B_kmajor, void* C, int M, int N, int K,
                          int group_m, int max_ctas, int splits, void* stream) {
  return run(kBf16Acc32, config_id, A, B_kmajor, C, M, N, K, group_m, max_ctas, splits, stream);
}

int b200_hgemm_host(int acc_bits, const void* hA, const void* hB_kmajor, void* hC, int M, int N, int K) {
  if (!hA || !hB_kmajor || !hC) return b200::host::kNullPointer;
  if (M <= 0 || N <= 0 || K <= 0) return b200::host::kBadShape;
  if (acc_bits != 32 && acc_bits != 16) return b200::host::kBadConfig;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return int(e);
  // Per-device context (device scratch that grows monotonically, three private streams and their events), created on
  // first use, shared by all host threads and freed by b200_hgemm_release(). The call is synchronous, so callers on
  // one device take turns (ctx.mu); callers on different devices do not meet.
  HostCtx& ctx = host_ctx(dev);
  std::lock_guard<std::mutex> turn(ctx.mu);
  const size_t a_bytes = size_t(M) * K * 2, b_bytes = size_t(N) * K * 2, c_bytes = size_t(M) * N * 2;
  auto up = [](size_t x) { return (x + 255) & ~size_t(255); };
  const size_t need = up(a_bytes) + up(b_bytes) + up(c_bytes);
  if (need > ctx.dcap) {
    if (ctx.dbuf) cudaFree(ctx.dbuf);
    ctx.dbuf = nullptr; ctx.dcap = 0;
    if ((e = cudaMalloc(&ctx.dbuf, need)) != cudaSuccess) return int(e);
    ctx.dcap = need;
  }
  char* dA = static_cast<char*>(ctx.dbuf);
  char* dB = dA + up(a_bytes);
  char* dC = dB + up(b_bytes);
  auto gemm = [&](const void* a, void* c, int m, cudaStream_t s) {
    return acc_bits == 32 ? b200_hgemm_f32acc(a, nullptr, dB, c, m, N, K, s) : b200_hgemm_f16acc(a, nullptr, dB, c, m, N, K, s);
  };

  // Large problems are PCIe time: B goes first, then A in row blocks; the GEMM of block i runs while block i+1 is on
  // its way in and block i-1 on its way out (PCIe is full duplex), on three private streams joined before returning.
  // Row blocks are independent GEMMs (C_i = A_i * B), so the result does not depend on the blocking.
  // Blocks of >= 512 rows (a GEMM of fewer rows under-fills the device), at most kHostBlocks of them: the tail that
  // nothing overlaps — the last block's GEMM and copy out — shrinks with the block size.
  const int blocks = std::min(kHostBlocks, M / 512);
  const bool pipelined = blocks >= 2 && (a_bytes + c_bytes) >= (size_t(8) << 20);
  if (!pipelined) {
    if ((e = cudaMemcpyAsync(dA, hA, a_bytes, cudaMemcpyHostToDevice, 0)) != cudaSuccess) return int(e);
    if ((e = cudaMemcpyAsync(dB, hB_kmajor, b_bytes, cudaMemcpyHostToDevice, 0)) != cudaSuccess) return int(e);
    int st = gemm(dA, dC, M, nullptr);
    if (st) return st;
    if ((e = cudaMemcpyAsync(hC, dC, c_bytes, cudaMemcpyDeviceToHost, 0)) != cudaSuccess) return int(e);
    e = cudaStreamSynchronize(0);
    return e == cudaSuccess ? 0 : int(e);
  }

  if (!ctx.in) {
    if ((e = cudaStreamCreateWithFlags(&ctx.in, cudaStreamNonBlocking)) != cudaSuccess) return int(e);
    if ((e = cudaStreamCreateWithFlags(&ctx.run, cudaStreamNonBlocking)) != cudaSuccess) return int(e);
    if ((e = cudaStreamCreateWithFlags(&ctx.out, cudaStreamNonBlocking)) != cudaSuccess) return int(e);
    if ((e = cudaEventCreateWithFlags(&ctx.b_in, cudaEventDisableTiming)) != cudaSuccess) return int(e);
    for (int i = 0; i < kHostBlocks; ++i) {
      if ((e = cudaEventCreateWithFlags(&ctx.a_in[i], cudaEventDisableTiming)) != cudaSuccess) return int(e);
      if ((e = cudaEventCreateWithFlags(&ctx.done[i], cudaEventDisableTiming)) != cudaSuccess) return int(e);
    }
  }
  // work queued by the caller on the legacy default stream (non-blocking streams do not wait for it on their own)
  if ((e = cudaStreamSynchronize(0)) != cudaSuccess) return int(e);
  const int rows_per = ((M + blocks - 1) / blocks + 127) / 128 * 128;   // whole 128-row tiles per block
  if ((e = cudaMemcpyAsync(dB, hB_kmajor, b_bytes, cudaMemcpyHostToDevice, ctx.in)) != cudaSuccess) return int(e);
  if ((e = cudaEventRecord(ctx.b_in, ctx.in)) != cudaSuccess) return int(e);
  if ((e = cudaStreamWaitEvent(ctx.run, ctx.b_in, 0)) != cudaSuccess) return int(e);
  for (int i = 0; i < blocks; ++i) {
    const int r0 = i * rows_per, rows = std::min(rows_per, M - r0);
    if (rows <= 0) break;
    const size_t a_off = size_t(r0) * K * 2, c_off = size_t(r0) * N * 2;
    if ((e = cudaMemcpyAsync(dA + a_off, static_cast<const char*>(hA) + a_off, size_t(rows) * K * 2, cudaMemcpyHostToDevice, ctx.in)) != cudaSuccess) return int(e);
    if ((e = cudaEventRecord(ctx.a_in[i], ctx.in)) != cudaSuccess) return int(e);
    if ((e = cudaStreamWaitEvent(ctx.run, ctx.a_in[i], 0)) != cudaSuccess) return int(e);
    int st = gemm(dA + a_off, dC + c_off, rows, ctx.run);
    if (st) { cudaDeviceSynchronize(); return st; }
    if ((e = cudaEventRecord(ctx.done[i], ctx.run)) != cudaSuccess) return int(e);
    if ((e = cudaStreamWaitEvent(ctx.out, ctx.done[i], 0)) != cudaSuccess) return int(e);
    if ((e = cudaMemcpyAsync(static_cast<char*>(hC) + c_off, dC + c_off, size_t(rows) * N * 2, cudaMemcpyDeviceToHost, ctx.out)) != cudaSuccess) return int(e);
  }
  if ((e = cudaStreamSynchronize(ctx.out)) != cudaSuccess) return int(e);   // the last copy out is behind everything else
  if ((e = cudaStreamSynchronize(ctx.run)) != cudaSuccess) return int(e);
  e = cudaStreamSynchronize(ctx.in);
  return e == cudaSuccess ? 0 : int(e);
}

int b200_hgemm_prewarm(void* stream) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return int(e);
  b200::host::SplitKScratch* sk = nullptr;
  return b200::host::splitk_scratch(dev, static_cast<cudaStream_t>(stream), &sk);
}

int b200_hgemm_release(void) {
  b200::host::release_scratch();
  int cur = 0;
  cudaGetDevice(&cur);
  std::lock_guard<std::mutex> lock(g_host_mu);
  for (auto& kv : g_host_ctx) {
    HostCtx& c = *kv.second;
    std::lock_guard<std::mutex> turn(c.mu);
    cudaSetDevice(kv.first);
    cudaDeviceSynchronize();
    if (c.dbuf) cudaFree(c.dbuf);
    c.dbuf = nullptr; c.dcap = 0;
    if (c.in) {
      cudaStreamDestroy(c.in); cudaStreamDestroy(c.run); cudaStreamDestroy(c.out);
      cudaEventDestroy(c.b_in);
      for (int i = 0; i < kHostBlocks; ++i) { cudaEventDestroy(c.a_in[i]); cudaEventDestroy(c.done[i]); }
      c.in = c.run = c.out = nullptr;
    }
  }
  cudaSetDevice(cur);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? 0 : int(e);
}

#ifdef B200_HGEMM_TRACE
// Developer-only entry points of libb200_hgemm_trace.so (see kTraceSlots in hgemm_sm100.cuh); not part of the C ABI.
static unsigned long long* g_trace_dev = nullptr;
static int g_trace_ctas = 0;
int b200_hgemm_trace_slots(void) { return b200::kTraceSlots; }
int b200_hgemm_trace_arm(int max_ctas) {   // zero the buffer and point the kernels at it (max_ctas <= 0: disarm)
  unsigned long long* none = nullptr;
  if (max_ctas <= 0) return int(cudaMemcpyToSymbol(b200::g_trace_buf, &none, sizeof(none)));
  const size_t bytes = size_t(max_ctas) * b200::kTraceSlots * 2 * sizeof(unsigned long long);
  if (max_ctas > g_trace_ctas) {
    if (g_trace_dev) cudaFree(g_trace_dev);
    g_trace_dev = nullptr; g_trace_ctas = 0;
    cudaError_t e = cudaMalloc(&g_trace_dev, bytes);
    if (e != cudaSuccess) return int(e);
    g_trace_ctas = max_ctas;
  }
  cudaError_t e = cudaMemset(g_trace_dev, 0, bytes);
  if (e != cudaSuccess) return int(e);
  return int(cudaMemcpyToSymbol(b200::g_trace_buf, &g_trace_dev, sizeof(g_trace_dev)));
}
int b200_hgemm_trace_read(unsigned long long* out, int ctas) {
  if (!g_trace_dev || ctas > g_trace_ctas) return b200::host::kBadShape;
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return int(e);
  return int(cudaMemcpy(out, g_trace_dev, size_t(ctas) * b200::kTraceSlots * 2 * sizeof(unsigned long long),
                        cudaMemcpyDeviceToHost));
}
#endif

unsigned long long b200_hgemm_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

const char* b200_hgemm_strerror(int status) { return b200::host::status_string(status); }

}  // extern "C"
