// Host side of the B200 HGEMM: tensor-map construction (cached), one-time kernel attribute setup,
// and the cluster launch. Shared by the C-ABI library (b200_hgemm_capi.cu) and by the per-shape
// translation units under kernels/b200_*/ that the reference-style JIT harness compiles.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <algorithm>
#include <deque>
#include <mutex>

#include "hgemm_sm100.cuh"

namespace b200 {
namespace host {

enum Status : int {
  kOk = 0,
  kBadShape = -1,        // M, N or K <= 0
  kBadAlignment = -2,    // pointers must be 16-byte aligned, K % 8 == 0 and N % 8 == 0 (TMA strides)
  kNoDriver = -3,        // cuTensorMapEncodeTiled could not be resolved
  kEncodeFailed = -4,
  kNullPointer = -5,
  kBadConfig = -6,
  kNotBlackwell = -7,
  kNoScratch = -8,       // internal: no split-K scratch for this (device, stream) and none can be allocated now (stream capture)
  // > 0: a cudaError_t from the launch
};

inline const char* status_string(int s) {
  switch (s) {
    case kOk: return "ok";
    case kBadShape: return "M, N and K must be positive";
    case kBadAlignment: return "operands must be 16-byte aligned with K % 8 == 0 and N % 8 == 0";
    case kNoDriver: return "cuTensorMapEncodeTiled unavailable (driver too old?)";
    case kEncodeFailed: return "cuTensorMapEncodeTiled failed";
    case kNullPointer: return "null operand pointer";
    case kBadConfig: return "unknown kernel configuration id";
    case kNotBlackwell: return "device is not compute capability 10.x (sm_100a build)";
    case kNoScratch: return "split-K scratch unavailable (allocate it outside stream capture with b200_hgemm_prewarm)";
    default: return s > 0 ? cudaGetErrorString(static_cast<cudaError_t>(s)) : "unknown error";
  }
}

using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                   CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                   CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

// Row-major fp16 matrix [rows, cols] (cols contiguous) -> 2-D tiled map, 128B swizzle,
// box = {box_cols (64 or 32) columns, box_rows}. Out-of-bounds elements read as zero / are not written.
inline int encode_2d(CUtensorMap* map, const void* ptr, int rows, int cols, int box_rows, int box_cols = kBlockK,
                     bool bf16 = false) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return kNoDriver;
  cuuint64_t dims[2] = {cuuint64_t(cols), cuuint64_t(rows)};
  cuuint64_t strides[1] = {cuuint64_t(cols) * 2};
  cuuint32_t box[2] = {cuuint32_t(box_cols), cuuint32_t(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  // the swizzle span equals the box's inner extent: 64 fp16 = 128 B, 32 fp16 = 64 B
  const CUtensorMapSwizzle swz = box_cols == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  CUresult r = fn(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? kOk : kEncodeFailed;
}

// Small direct-mapped cache of encoded maps: benchmark loops re-present the same few pointers
// (the caching allocator recycles them), and an encode costs about a microsecond of host time.
struct MapKey {
  const void* ptr; int rows, cols, box_rows, box_cols; bool bf16;
  bool operator==(const MapKey& o) const {
    return ptr == o.ptr && rows == o.rows && cols == o.cols && box_rows == o.box_rows && box_cols == o.box_cols && bf16 == o.bf16;
  }
};
struct MapCache {
  static constexpr int kSlots = 64;
  MapKey keys[kSlots];
  CUtensorMap maps[kSlots];
  bool valid[kSlots];
  MapCache() { std::memset(valid, 0, sizeof(valid)); }
  // Copies the map out: two operands of one call may share a slot, so a pointer into the cache would alias.
  int get(const void* ptr, int rows, int cols, int box_rows, CUtensorMap* out, int box_cols = kBlockK, bool bf16 = false) {
    MapKey k{ptr, rows, cols, box_rows, box_cols, bf16};
    uint64_t h = (reinterpret_cast<uint64_t>(ptr) >> 8) * 0x9E3779B97F4A7C15ull;
    h ^= uint64_t(uint32_t(rows)) * 0xC2B2AE3D27D4EB4Full + uint64_t(uint32_t(cols)) * 0x165667B19E3779F9ull +
         uint64_t(box_rows) * 131u + uint64_t(box_cols);
    int slot = int((h >> 32) % kSlots);
    if (!(valid[slot] && keys[slot] == k)) {
      int st = encode_2d(&maps[slot], ptr, rows, cols, box_rows, box_cols, bf16);
      if (st != kOk) { valid[slot] = false; return st; }
      keys[slot] = k;
      valid[slot] = true;
    }
    std::memcpy(out, &maps[slot], sizeof(CUtensorMap));
    return kOk;
  }
};
inline MapCache& map_cache() {
  static thread_local MapCache c;
  return c;
}

struct DeviceInfo { int dev; int num_sms; int cc_major; };
inline const DeviceInfo& device_info() {
  // per-device, resolved once (the harness pins one device per process)
  static thread_local int cached_dev = -1;
  static thread_local DeviceInfo info{-1, 0, 0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev != cached_dev) {
    cudaDeviceGetAttribute(&info.num_sms, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&info.cc_major, cudaDevAttrComputeCapabilityMajor, dev);
    info.dev = dev;
    cached_dev = dev;
  }
  return info;
}

inline int validate(const void* A, const void* Bt, const void* C, int M, int N, int K) {
  if (!A || !Bt || !C) return kNullPointer;
  if (M <= 0 || N <= 0 || K <= 0) return kBadShape;
  if ((K % 8) || (N % 8)) return kBadAlignment;
  if ((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(Bt) | reinterpret_cast<uintptr_t>(C)) & 15)
    return kBadAlignment;
  return kOk;
}

// Split-K / stream-K scratch: fp32 partial tiles + arrival counters, one per (device, stream), allocated on first use
// (or ahead of time by b200_hgemm_prewarm — required before a CUDA-graph capture, where cudaMalloc is illegal) and kept
// until b200_hgemm_release(). Process-wide and mutex-protected: any host thread that launches on a (device, stream)
// finds the same scratch, and the pool grows with the number of streams instead of silently running out. Counters are
// zero between launches (the kernel resets them), so consecutive launches on a stream need no host-side clearing.
// Launches that share a scratch must be ordered by their stream — which they are, being on the same stream.
struct SplitKScratch {
  int dev = -1; cudaStream_t stream = nullptr; float* ws = nullptr; unsigned* ctr = nullptr;
};
constexpr size_t kSplitKWsBytes = size_t(kMaxStreamKSlots) * kBlockM * 256 * sizeof(float);   // 160 units of 128x256 fp32
// split-K arrive/done counters, then one stream-K flag per (CTA slot, epilogue warp)
constexpr size_t kSplitKCtrBytes = (2 * kMaxSplitTiles + kMaxStreamKSlots * kStreamKFlagsPerSlot) * sizeof(unsigned);
struct ScratchPool {
  std::mutex mu;
  std::deque<SplitKScratch> entries;   // deque: growing never moves an entry another thread holds a pointer to
};
inline ScratchPool& scratch_pool() {
  static ScratchPool pool;
  return pool;
}
inline int splitk_scratch(int dev, cudaStream_t stream, SplitKScratch** out) {
  ScratchPool& pool = scratch_pool();
  std::lock_guard<std::mutex> lock(pool.mu);
  for (auto& e : pool.entries)
    if (e.ws && e.dev == dev && e.stream == stream) { *out = &e; return kOk; }
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(stream, &cap) != cudaSuccess) { cudaGetLastError(); return kNoScratch; }
  if (cap != cudaStreamCaptureStatusNone) return kNoScratch;   // cudaMalloc would invalidate the capture
  SplitKScratch e;
  cudaError_t err = cudaMalloc(&e.ws, kSplitKWsBytes);
  if (err != cudaSuccess) return int(err);
  err = cudaMalloc(&e.ctr, kSplitKCtrBytes);
  if (err != cudaSuccess) { cudaFree(e.ws); return int(err); }
  err = cudaMemsetAsync(e.ctr, 0, kSplitKCtrBytes, stream);
  if (err != cudaSuccess) { cudaFree(e.ws); cudaFree(e.ctr); return int(err); }
  e.dev = dev; e.stream = stream;
  SplitKScratch* slot = nullptr;
  for (auto& old : pool.entries) if (!old.ws) { slot = &old; break; }   // reuse a released entry
  if (slot) *slot = e; else { pool.entries.push_back(e); slot = &pool.entries.back(); }
  *out = slot;
  return kOk;
}
// Frees every scratch allocation of this process (all devices). The caller guarantees that no launch of this
// library is in flight or issued concurrently.
inline void release_scratch() {
  ScratchPool& pool = scratch_pool();
  std::lock_guard<std::mutex> lock(pool.mu);
  int cur = 0;
  cudaGetDevice(&cur);
  for (auto& e : pool.entries) {
    if (!e.ws) continue;
    cudaSetDevice(e.dev);
    cudaDeviceSynchronize();
    cudaFree(e.ws); cudaFree(e.ctr);
    e = SplitKScratch{};
  }
  cudaSetDevice(cur);
}

// Largest usable split factor for this problem/config: units must fit the SMs (one CTA per unit), every
// split must own at least one k-block, and the partial tiles must fit the workspace.
template <class Cfg>
int clamp_splits(int splits, int M, int N, int K, int num_sms) {
  if (splits <= 1 || Cfg::CTA_GROUP != 1) return 1;
  const int tiles = ((M + kBlockM - 1) / kBlockM) * ((N + Cfg::BN - 1) / Cfg::BN);   // CTA_GROUP == 1: callers exclude M_REP > 1
  const int nkb = (K + kBlockK - 1) / kBlockK;
  if (tiles > kMaxSplitTiles) return 1;
  splits = std::min(splits, std::min(num_sms / tiles, std::min(nkb, 32)));   // <= 32: the slices of all partials must fit the pipeline smem
  while (splits > 1 && (splits - 1) * ((nkb + splits - 1) / splits) >= nkb) --splits;   // no empty split
  while (splits > 1 && size_t(tiles) * splits * kBlockM * Cfg::BN * sizeof(float) > kSplitKWsBytes) --splits;
  return std::max(splits, 1);
}

// `splits` values with a special meaning (besides > 1: workspace split-K, -2/-4/-8: cluster split-K)
constexpr int kStreamKTail = 100;           // stream-K over the tiles of the partial last wave
constexpr int kStreamKTailPlusWave = 101;   // ... plus one full wave, so that every worker's slice is longer than a tile
constexpr int kMinStreamKSlice = 4;         // k-blocks; shorter slices are all pipeline fill and fix-up

// What a launch will run: how many workers (CTAs, CTA pairs or clusters), which K-decomposition.
struct Plan {
  int num_tiles, nkb;
  int workers;          // grid = workers * (CTAs per worker)
  int splits;           // > 1: split-K, one worker per (tile, split)
  int cluster_reduce;   // != 0: the splits of a tile form a cluster of this many CTAs and reduce through DSMEM
  int sk_tiles;         // > 0: stream-K over the first sk_tiles tiles
};

// `workers_avail`: workers the device can hold at once (SMs / CTAs per worker, after max_ctas and cluster occupancy).
template <class Cfg>
Plan make_plan(int M, int N, int K, int workers_avail, int splits) {
  Plan p{};
  const int num_m_blocks = (M + Cfg::TILE_M * Cfg::CLUSTER_M - 1) / (Cfg::TILE_M * Cfg::CLUSTER_M);
  const int num_n_blocks = (N + Cfg::BN * Cfg::CLUSTER_N - 1) / (Cfg::BN * Cfg::CLUSTER_N);
  p.num_tiles = num_m_blocks * num_n_blocks;
  p.nkb = (K + kBlockK - 1) / kBlockK;
  p.workers = std::max(workers_avail, 1);
  const bool plain = Cfg::STREAM_K;   // no multicast cluster, BN >= 64, 128 rows per CTA: the K-decompositions are wired for these
  int sk_mode = 0;
  if (splits == kStreamKTail || splits == kStreamKTailPlusWave) { sk_mode = splits; splits = 1; }
  if (!plain) splits = 1;
  if (splits < -1) {
    int cs = -splits;
    if (Cfg::CTA_GROUP == 1 && (cs == 2 || cs == 4 || cs == 8)) {
      // every CTA of the cluster must own at least one k-block: halve the cluster until no k-range is empty
      while (cs > 1 && (cs - 1) * ((p.nkb + cs - 1) / cs) >= p.nkb) cs /= 2;
      if (cs > 1) p.cluster_reduce = cs;
    }
    splits = 1;
  }
  p.splits = clamp_splits<Cfg>(splits, M, N, K, p.workers);
  if (p.cluster_reduce) {
    p.workers = p.num_tiles * p.cluster_reduce;   // one cluster per tile, one CTA per k-range
    p.splits = p.cluster_reduce;
  } else if (p.splits > 1) {
    p.workers = p.num_tiles * p.splits;           // exactly one CTA per (tile, split) unit
  } else {
    if (sk_mode && plain && p.num_tiles % p.workers != 0 && p.workers * Cfg::CTA_GROUP <= kMaxStreamKSlots) {
      int sk = p.num_tiles % p.workers;
      if (sk_mode == kStreamKTailPlusWave && p.num_tiles > p.workers) sk += p.workers;
      if (sk * p.nkb / p.workers >= kMinStreamKSlice) p.sk_tiles = sk;
    }
    if (!p.sk_tiles && p.workers > p.num_tiles) p.workers = p.num_tiles;
  }
  return p;
}

inline bool cache_hints_enabled() {
  static const bool on = [] { const char* e = std::getenv("B200_HGEMM_NO_CACHE_HINTS"); return !(e && e[0] == '1'); }();
  return on;
}

// How many clusters of this configuration the device holds at once (asked once per device).
template <class Cfg>
int max_resident_clusters(const DeviceInfo& di) {
  static thread_local int max_clusters = 0, max_clusters_dev = -1;
  if (max_clusters_dev != di.dev) {
    cudaLaunchConfig_t probe{};
    probe.gridDim = dim3(unsigned(di.num_sms / Cfg::CLUSTER_CTAS * Cfg::CLUSTER_CTAS), 1, 1);
    probe.blockDim = dim3(Cfg::NUM_THREADS, 1, 1);
    probe.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cudaLaunchAttribute pa[1];
    pa[0].id = cudaLaunchAttributeClusterDimension;
    pa[0].val.clusterDim.x = Cfg::CLUSTER_CTAS; pa[0].val.clusterDim.y = 1; pa[0].val.clusterDim.z = 1;
    probe.attrs = pa; probe.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, hgemm_tn_kernel<Cfg>, &probe) != cudaSuccess || n < 1) {
      cudaGetLastError();
      n = std::max(1, di.num_sms / Cfg::CLUSTER_CTAS * 7 / 8);
    }
    max_clusters = n; max_clusters_dev = di.dev;
  }
  return max_clusters;
}

// B200_HGEMM_NO_PDL=1 launches without programmatic stream serialisation (developer A/B).
inline bool pdl_enabled() {
  static const bool on = [] { const char* e = std::getenv("B200_HGEMM_NO_PDL"); return !(e && e[0] == '1'); }();
  return on;
}

// One (configuration, K-mode) instance of the kernel: opt into its dynamic shared memory once, then launch.
// Function attributes are per device AND per copy of the kernel: when two shared objects instantiate this template
// (libb200_hgemm.so and a JIT-built hgemm_lib.so in one process), a function-local static may be merged across
// them (STB_GNU_UNIQUE) while each object still launches its own kernel copy. Key on both.
struct LaunchArgs {
  CUtensorMap ma, mb, mc;
  int M, N, K, group_m;
  Plan plan;
  float* ws; unsigned* ctr; __half* c;
  uint64_t hint_a, hint_b;
  cudaStream_t stream;
};

template <class Cfg, int KMODE>
int launch_mode(const DeviceInfo& di, const LaunchArgs& a) {
  static thread_local int attr_dev = -1;
  static thread_local const void* attr_fn = nullptr;
  const void* this_fn = reinterpret_cast<const void*>(&hgemm_tn_kernel<Cfg, KMODE>);
  if (attr_dev != di.dev || attr_fn != this_fn) {
    cudaError_t e = cudaFuncSetAttribute(hgemm_tn_kernel<Cfg, KMODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         Cfg::SMEM_BYTES);
    if (e != cudaSuccess) return int(e);
    attr_dev = di.dev;
    attr_fn = this_fn;
  }
  constexpr bool kSplit = (KMODE == kWorkspaceSplitK || KMODE == kClusterSplitK);
  const int cluster = (KMODE == kClusterSplitK) ? a.plan.cluster_reduce : Cfg::CLUSTER_CTAS;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(unsigned(a.plan.workers * (kSplit ? 1 : Cfg::CLUSTER_CTAS)), 1, 1);   // split-K: one CTA per (tile, split)
  cfg.blockDim = dim3(Cfg::NUM_THREADS, 1, 1);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = a.stream;
  cudaLaunchAttribute attr[3];
  unsigned na = 0;
  if (cluster > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = unsigned(cluster);
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  // Workspace split-K and stream-K CTAs wait for sibling CTAs of the same grid (arrival counters / flags in global
  // memory), so the whole grid must be resident at once. A cooperative launch makes that the driver's guarantee: the
  // grid starts only when all of it fits (other kernels holding SMs delay it instead of starving half of it into
  // the watchdog), and a grid that can never fit is refused with cudaErrorCooperativeLaunchTooLarge, which launch()
  // turns into the undivided schedule. (Cluster split-K needs nothing: a cluster is co-scheduled by the hardware.)
  constexpr bool coop = (KMODE == kWorkspaceSplitK || KMODE == kStreamK);
  if (coop) {
    attr[na].id = cudaLaunchAttributeCooperative;
    attr[na].val.cooperative = 1;
    ++na;
  }
  // programmatic dependent launch: this kernel's prologue may overlap the tail of the stream's previous kernel; the
  // kernel itself waits (griddepcontrol.wait) before its first global-memory access. Back-to-back GEMMs lose the
  // 2-3 us of launch + set-up between them; a caller that synchronises after every call sees no difference.
  // Not for a cooperative launch: the pair was measured to change nothing (DESIGN.md §6).
  if (!coop && pdl_enabled()) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  const cudaError_t e = cudaLaunchKernelEx(&cfg, hgemm_tn_kernel<Cfg, KMODE>, a.ma, a.mb, a.mc, a.M, a.N, a.K,
                                           a.group_m, a.plan.splits, a.plan.sk_tiles, a.ws, a.ctr, a.c, a.hint_a, a.hint_b);
  return e == cudaSuccess ? kOk : int(e);
}

// group_m <= 0 selects the default rasterisation width. max_ctas <= 0 means "all SMs". `splits`: 1 none, > 1 workspace
// split-K, -2/-4/-8 cluster split-K, kStreamKTail / kStreamKTailPlusWave stream-K — each clamped to what the problem and
// the configuration allow. MODES: bit mask of the K-modes this call site may need (a per-shape translation unit
// names its one mode and so compiles two kernels instead of four; the plain mode is always available as fallback).
template <class Cfg, unsigned MODES = 0xFu>
int launch(const void* A, const void* Bt, void* C, int M, int N, int K, cudaStream_t stream,
           int group_m = 0, int max_ctas = 0, int splits = 1) {
  int st = validate(A, Bt, C, M, N, K);
  if (st != kOk) return st;
  const DeviceInfo& di = device_info();
  if (di.cc_major != 10) return kNotBlackwell;

  LaunchArgs a{};
  MapCache& cache = map_cache();
  if ((st = cache.get(A, M, K, Cfg::A_BOX_ROWS, &a.ma, kBlockK, Cfg::BF16)) != kOk) return st;
  if ((st = cache.get(Bt, N, K, Cfg::B_BOX_ROWS, &a.mb, kBlockK, Cfg::BF16)) != kOk) return st;
  if ((st = cache.get(C, M, N, 32, &a.mc, Cfg::EPI_N, Cfg::BF16)) != kOk) return st;

  constexpr bool kCanSplit = Cfg::SPLIT_K && (MODES & ((1u << kWorkspaceSplitK) | (1u << kClusterSplitK)));
  constexpr bool kCanStream = Cfg::STREAM_K && (MODES & (1u << kStreamK));
  const bool wants_stream_k = (splits == kStreamKTail || splits == kStreamKTailPlusWave);
  if ((wants_stream_k && !kCanStream) || (!wants_stream_k && splits != 1 && !kCanSplit)) splits = 1;
  if (splits > 1 && !(MODES & (1u << kWorkspaceSplitK))) splits = 1;
  if (splits < -1 && !(MODES & (1u << kClusterSplitK))) splits = 1;

  int workers = (max_ctas > 0 ? max_ctas : di.num_sms) / Cfg::CLUSTER_CTAS;
  // Clusters must fit inside a GPC, so fewer than SMs / cluster size may be resident at once. Larger clusters are
  // always sized to what fits; CTA pairs only when stream-K is requested, whose owners wait for contributors
  // that must therefore be running (for the plain schedule a pair that starts late is merely late).
  if (Cfg::CLUSTER_CTAS > 2 || (Cfg::CLUSTER_CTAS == 2 && wants_stream_k && splits != 1)) {
    workers = std::min(workers, max_resident_clusters<Cfg>(di));
  }
  a.plan = make_plan<Cfg>(M, N, K, workers, splits);
  if ((a.plan.splits > 1 && !a.plan.cluster_reduce) || a.plan.sk_tiles) {
    SplitKScratch* sk = nullptr;
    if (splitk_scratch(di.dev, stream, &sk) == kOk) {
      a.ws = sk->ws; a.ctr = sk->ctr;
    } else {
      cudaGetLastError();
      a.plan = make_plan<Cfg>(M, N, K, workers, 1);   // no scratch (allocation failed, or first use inside a stream capture): run undivided
    }
  }
  a.M = M; a.N = N; a.K = K;
  a.group_m = group_m > 0 ? group_m : (Cfg::CTA_GROUP == 2 ? 8 : 16);
  a.c = static_cast<__half*>(C);
  a.stream = stream;
  // L2 eviction priorities: when one operand is streamed (about) once while the other is re-read by every tile row
  // or column and is small enough to live in L2, keep the small one and let the streamed one go first.
  a.hint_a = ptx::kL2EvictNormal; a.hint_b = ptx::kL2EvictNormal;
  if (cache_hints_enabled()) {
    const size_t a_bytes = size_t(M) * K * 2, b_bytes = size_t(N) * K * 2;
    const int n_tiles = (N + Cfg::BN - 1) / Cfg::BN, m_tiles = (M + Cfg::TILE_M - 1) / Cfg::TILE_M;
    constexpr size_t kL2Keep = size_t(48) << 20, kStream = size_t(96) << 20;
    if (a_bytes >= kStream && b_bytes <= kL2Keep && n_tiles <= 4) { a.hint_a = ptx::kL2EvictFirst; a.hint_b = ptx::kL2EvictLast; }
    else if (b_bytes >= kStream && a_bytes <= kL2Keep && m_tiles <= 4) { a.hint_b = ptx::kL2EvictFirst; a.hint_a = ptx::kL2EvictLast; }
  }
  // a co-resident mode the device cannot hold (refused before anything ran) falls back to the undivided schedule
  auto undivided = [&](int err) {
    if (err != int(cudaErrorCooperativeLaunchTooLarge) && err != int(cudaErrorLaunchOutOfResources)) return err;
    cudaGetLastError();
    a.plan = make_plan<Cfg>(M, N, K, workers, 1);
    return launch_mode<Cfg, kPlain>(di, a);
  };
  if constexpr (kCanStream) {
    if (a.plan.sk_tiles > 0) return undivided(launch_mode<Cfg, kStreamK>(di, a));
  }
  if constexpr (Cfg::SPLIT_K && (MODES & (1u << kClusterSplitK))) {
    if (a.plan.cluster_reduce) return launch_mode<Cfg, kClusterSplitK>(di, a);
  }
  if constexpr (Cfg::SPLIT_K && (MODES & (1u << kWorkspaceSplitK))) {
    if (a.plan.splits > 1) return undivided(launch_mode<Cfg, kWorkspaceSplitK>(di, a));
  }
  return launch_mode<Cfg, kPlain>(di, a);
}

}  // namespace host
}  // namespace b200
