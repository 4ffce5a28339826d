// B200 (sm_100a) HGEMM:  C[M,N] (fp16) = A[M,K] (fp16, K-contiguous) * Bt[N,K]^T (fp16, K-contiguous)
// with fp32 (F32F16F16F32) or fp16 (F16F16F16F16) accumulation in tensor memory.
//
// Replaces, for --device_type b200, the per-shape kernels the reference ships for older GPUs
// (reference: kernels/a100_F32F16F16F32/4096_4096_4096.cu:22-177 mainloop+epilogue, :179-279 launcher;
//  kernels/h100_F32F16F16F32/4096_4096_4096.cu:21-80 for the TMA/wgmma flavour). Same contract:
// TN operands (A row-major, B supplied K-major as `b_col_major`, tools/utils.py:110-115), C row-major
// fully overwritten, one round-to-nearest fp32->fp16 conversion at the end.
//
// Design (nothing below is translated from the reference; it is written for Blackwell):
//   * persistent CTAs (one per SM, or one CTA pair per 2 SMs), static tile schedule with grouped
//     rasterisation for L2 reuse;
//   * warp-specialised: warp 0 = TMA producer, warp 1 = tcgen05.mma issuer (warp-uniform loops, one elected lane issues),
//     warp 2 = TMEM allocator, warps 4..11 = epilogue (TMEM -> regs -> swizzled smem -> TMA store), two warps
//     per TMEM lane quadrant, each taking half of a tile's column chunks;
//   * operands land in 128B-swizzled smem via cp.async.bulk.tensor (OOB rows/cols zero-filled, so no
//     harness padding is ever needed), consumed in place by tcgen05.mma through smem descriptors;
//   * kStages-deep full/empty mbarrier ring between TMA and MMA, and a 2-deep TMEM accumulator ring
//     between MMA and epilogue so the epilogue of tile i overlaps the main loop of tile i+1;
//   * CTA_GROUP == 2: cta_group::2 MMA (256 x BN per CTA pair), each CTA loads its 128 rows of A and
//     half of the B tile, the leader CTA issues the MMAs and multicasts the commit to both CTAs;
//   * CLUSTER_M x CLUSTER_N > 1: thread-block clusters of single-CTA groups on adjacent tiles. The CTAs of a
//     cluster row need the same A tile, those of a cluster column the same B tile: each CTA loads only a
//     1/CLUSTER_N slice of A and a 1/CLUSTER_M slice of B and TMA-multicasts it to the CTAs that need it, so the
//     L2->SM traffic per CTA drops while every CTA still holds full tiles for its MMAs. A stage is released by
//     a tcgen05.commit multicast to every CTA of the consumer's cluster row and column;
//   * split-K for problems with few output tiles and long K, two flavours, both deterministic: partial tiles
//     through an fp32 global workspace with a distributed reduction (up to 32 splits), or the splits of a tile
//     form a cluster and reduce through distributed shared memory (2/4/8 splits, no workspace);
//   * stream-K for tile counts that leave the last wave partly empty: the first tiles of the schedule are cut along
//     K into one equal slice per worker (hgemm_schedule.cuh), the partial sums of a tile meet in its owner's
//     epilogue through the same workspace, in fixed k order.
#pragma once
#include <cuda.h>          // CUtensorMap (type only; the encoder is fetched at run time)
#include <cuda_runtime.h>
#include <cstdint>

#include "hgemm_schedule.cuh"
#include "ptx_sm100.cuh"


namespace b200 {

constexpr int kBlockK = 64;          // 64 fp16 = 128 B = one swizzle row
constexpr int kUmmaK = 16;           // K per tcgen05.mma.kind::f16
constexpr int kBlockM = 128;         // rows per CTA (all 128 TMEM lanes)
constexpr int kNumThreads = 384;     // 12 warps: 0 TMA, 1 MMA, 2 TMEM alloc, 3 idle, 4-11 epilogue (two per TMEM lane quadrant);
                                     // 8 warps (256 threads) for tiles of one 64-column chunk, whose second epilogue set would idle
constexpr int kEpiWarp0 = 4;
constexpr int kAccStages = 2;        // TMEM accumulator ring depth
// How a launch divides K. The kernel is compiled once per (configuration, mode), so that the plain schedule — nearly
// every launch — carries none of the three other epilogues: a quarter of the instructions, and registers to spare.
enum KMode : int { kPlain = 0, kWorkspaceSplitK = 1, kClusterSplitK = 2, kStreamK = 3 };

// Developer instrumentation (only in builds with -DB200_HGEMM_TRACE, i.e. libb200_hgemm_trace.so; the product build
// contains none of it): per-CTA timestamps of the kernel's phases, read back by `dev_check_trace trace`.
//   slot 0 entry | 1 setup done | 2 first TMA issued | 3 last TMA issued | 4 first stage landed (MMA warp)
//   5 last MMA commit issued | 6 first accumulator complete (epilogue) | 7 epilogue drained | 8 after the teardown
//   barrier | 9 k-blocks issued (a count) | 10 last accumulator complete (epilogue) | 11 units run (a count)
constexpr int kTraceSlots = 12;      // each slot: {%globaltimer ns, clock64}
#ifdef B200_HGEMM_TRACE
__device__ unsigned long long* g_trace_buf = nullptr;   // [gridDim.x][kTraceSlots][2], zeroed by the host before the launch
__device__ __forceinline__ void trace_mark(int slot) {
  if (g_trace_buf) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    unsigned long long* e = g_trace_buf + (size_t(blockIdx.x) * kTraceSlots + slot) * 2;
    e[0] = t;
    e[1] = (unsigned long long)clock64();
  }
}
__device__ __forceinline__ void trace_value(int slot, unsigned long long v) {
  if (g_trace_buf) g_trace_buf[(size_t(blockIdx.x) * kTraceSlots + slot) * 2] = v;
}
#define B200_TRACE(slot) ::b200::trace_mark(slot)
#define B200_TRACE_VALUE(slot, v) ::b200::trace_value(slot, v)
#define B200_TRACE_ONLY(...) __VA_ARGS__
#else
#define B200_TRACE(slot) ((void)0)
#define B200_TRACE_VALUE(slot, v) ((void)0)
#define B200_TRACE_ONLY(...)
#endif

template <int BN_, int STAGES_, int CTA_GROUP_, bool ACC_F32_, int CLUSTER_M_ = 1, int CLUSTER_N_ = 1, int M_REP_ = 1, bool BF16_ = false>
struct Config {
  static constexpr int BN = BN_;               // tile N (= UMMA N)
  static constexpr int STAGES = STAGES_;
  static constexpr int CTA_GROUP = CTA_GROUP_; // 1: 128xBN per CTA; 2: 256xBN per CTA pair
  static constexpr bool ACC_F32 = ACC_F32_;
  // bf16 operands and bf16 output instead of fp16 (README.md:73 "denser configurations" territory): same pipeline, two
  // instruction-descriptor fields and the epilogue's convert differ. tcgen05 kind::f16 accumulates bf16 products in fp32 only.
  static constexpr bool BF16 = BF16_;
  static_assert(!BF16_ || ACC_F32_, "bf16 operands accumulate in fp32");
  // Multicast cluster: CLUSTER_M x CLUSTER_N groups (single CTAs or CTA pairs) work on a block of adjacent tiles;
  // the groups of a cluster row share their A tile, those of a cluster column their B tile. Each CTA loads a
  // 1/CLUSTER_N slice of its A rows and a 1/CLUSTER_M slice of its B rows and TMA-multicasts it to the CTAs
  // (same position inside their pair) of the groups that need it. Cluster rank = (cm + CLUSTER_M * cn) * CTA_GROUP + r.
  static constexpr int CLUSTER_M = CLUSTER_M_;
  static constexpr int CLUSTER_N = CLUSTER_N_;
  static constexpr int MCAST_CTAS = CLUSTER_M * CLUSTER_N;
  static constexpr int CLUSTER_CTAS = CTA_GROUP * MCAST_CTAS;
  // M_REP = 2: every CTA owns 256 rows — two 128-row MMAs per k-step that share the B tile in shared memory and fill
  // two accumulators — so a CTA pair covers 512 x BN and each B byte fetched from L2 feeds twice the MMA work (the
  // shape of cuBLAS's largest kernel, nvjet_hsh_256x256_64x4_2x1_2cta). With BN = 256 the two accumulators fill all
  // 512 TMEM columns: no accumulator ring, the epilogue of a tile is not overlapped with the next main loop, which
  // only a long K amortises. No split-K / stream-K in this mode.
  static constexpr int M_REP = M_REP_;
  static constexpr int CTA_M = kBlockM * M_REP;             // rows per CTA
  static constexpr int TILE_M = CTA_M * CTA_GROUP;
  static constexpr int LOAD_N = BN / CTA_GROUP;             // B rows each CTA holds per stage
  static constexpr int A_BOX_ROWS = CTA_M / CLUSTER_N;      // A rows each CTA loads per stage
  static constexpr int B_BOX_ROWS = LOAD_N / CLUSTER_M;     // B rows each CTA loads per stage
  static constexpr int A_STAGE_BYTES = CTA_M * kBlockK * 2;
  static constexpr int B_STAGE_BYTES = LOAD_N * kBlockK * 2;
  static constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
  static constexpr int EPI_N = BN < 64 ? BN : 64;            // columns per epilogue step / TMA store box
  static constexpr int EPI_CHUNKS = BN / EPI_N;
  // two epilogue warps per TMEM lane quadrant share a tile's column chunks when there are at least two of them
  static constexpr int EPI_GROUPS = EPI_CHUNKS >= 2 ? 2 : 1;
  static constexpr int EPI_CHUNKS_PER_GROUP = (EPI_CHUNKS + EPI_GROUPS - 1) / EPI_GROUPS;
  static constexpr int NUM_THREADS = EPI_GROUPS == 2 ? kNumThreads : kNumThreads - 128;   // no warps that would only wait
  // which K-decompositions this configuration's kernel can be instantiated with
  static constexpr bool SPLIT_K = CTA_GROUP_ * CLUSTER_M_ * CLUSTER_N_ == 1 && BN_ >= 64 && M_REP_ == 1;
  static constexpr bool STREAM_K = CLUSTER_M_ * CLUSTER_N_ == 1 && BN_ >= 64 && M_REP_ == 1;
  static constexpr int EPI_BUF_BYTES = 32 * EPI_N * 2;       // one warp, one chunk: 32 rows x EPI_N fp16
  static constexpr int EPI_BYTES = 8 * 32 * 64 * 2;          // 8 warps x one staging buffer (sized for EPI_N = 64)
  static constexpr int BAR_BYTES = 512;
  // stream-K, owner unit that ends a worker's schedule: the partial tiles are fetched by bulk copies into the (then
  // idle) pipeline shared memory, one region per epilogue warp holding a ring of chunk images
  static constexpr int FIX_REGION_BYTES = ((STAGES * STAGE_BYTES) / 8) & ~1023;
  static constexpr int FIX_BARS = 8 * 3;
  static constexpr int SMEM_BYTES = 1024 /*align slack*/ + STAGES * STAGE_BYTES + EPI_BYTES + BAR_BYTES;
  static constexpr int ACC_COLS = M_REP * BN;                // TMEM columns of one accumulator stage
  static constexpr int ACC_STAGES = (kAccStages * ACC_COLS <= 512) ? kAccStages : 1;   // ring depth that fits TMEM
  static constexpr int TMEM_COLS_USED = ACC_STAGES * ACC_COLS;
  static constexpr int TMEM_COLS = TMEM_COLS_USED <= 32 ? 32 : TMEM_COLS_USED <= 64 ? 64
                                 : TMEM_COLS_USED <= 128 ? 128 : TMEM_COLS_USED <= 256 ? 256 : 512;
  static_assert(BN == 32 || BN % 64 == 0, "tile N is 32 or a multiple of 64");
  static_assert(BN >= 32 && BN <= 256 && (BN % 16) == 0, "UMMA N constraints");
  static_assert(CLUSTER_CTAS <= 8, "portable cluster size");
  static_assert(A_BOX_ROWS % 8 == 0 && B_BOX_ROWS % 8 == 0, "slices must cover whole 8-row swizzle atoms");
  static_assert(M_REP == 1 || M_REP == 2, "one or two 128-row blocks per CTA");
  static_assert(A_BOX_ROWS <= 256 && B_BOX_ROWS <= 256, "TMA box dimension limit");
  static_assert(TMEM_COLS_USED <= 512, "accumulator ring exceeds TMEM");
  static_assert(SMEM_BYTES <= 232448, "exceeds 227 KB of shared memory");
  static_assert(A_STAGE_BYTES % 1024 == 0 && B_STAGE_BYTES % 1024 == 0, "swizzle-128B tiles need 1 KB alignment");
  static_assert(8 * (2 * STAGES + 2 * kAccStages + 1) + 8 + 8 * FIX_BARS <= BAR_BYTES, "barrier block too small");   // ACC_STAGES <= kAccStages
};

// 32-bit tcgen05 instruction descriptor for kind::f16, fp16 A/B, both K-major.
// [4,6) D fmt (0=f16,1=f32) | [7,10) A fmt (0=f16) | [10,13) B fmt | [15] A major | [16] B major
// | [17,23) N>>3 | [24,29) M>>4
__host__ __device__ constexpr uint32_t make_idesc(int umma_m, int umma_n, bool acc_f32, bool bf16 = false) {
  return (acc_f32 ? 1u : 0u) << 4 | (bf16 ? 1u : 0u) << 7 | (bf16 ? 1u : 0u) << 10 | (uint32_t(umma_n >> 3) << 17) |
         (uint32_t(umma_m >> 4) << 24);
}

// 64-bit shared-memory matrix descriptor: K-major tile, 128B swizzle, rows 128 B apart,
// 8-row groups 1024 B apart (SBO), LBO unused for swizzled K-major, version 1 (sm_100).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= uint64_t((smem_addr & 0x3FFFF) >> 4);
  d |= uint64_t(1024 >> 4) << 32;
  d |= uint64_t(1) << 46;
  d |= uint64_t(2) << 61;   // SWIZZLE_128B
  return d;
}

constexpr int kMaxSplitTiles = 256;   // split-K is only used when tiles * splits <= #SMs

// TMEM columns [32j, 32j + 32) of this warp's lanes as fp32, whatever the accumulator type
template <class Cfg>
__device__ __forceinline__ void tmem_load_f32_x32(uint32_t taddr0, int j, float (&f)[32]) {
  using namespace ptx;
  uint32_t v[32];
  if constexpr (Cfg::ACC_F32) {
    tmem_ld_32x32b_x32(taddr0 + j * 32, v);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
  } else {
    // fp16 accumulators: 64 columns arrive packed two per register, so 32 columns fill half of the registers
    tmem_ld_32x32b_x32_pack16(taddr0 + (j / 2) * 64, v);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const __half2 h = *reinterpret_cast<const __half2*>(&v[(j & 1) * 16 + i]);
      f[2 * i] = __low2float(h);
      f[2 * i + 1] = __high2float(h);
    }
  }
}

// Four adjacent output columns rounded once and stored to C (the split-K reductions' direct stores)
template <class Cfg>
__device__ __forceinline__ void store_out_x4(__half* __restrict__ C, int gm, int gn, int N, float4 acc) {
  uint2 out;
  out.x = ptx::pack_out_x2_rn<Cfg::BF16>(acc.x, acc.y);
  out.y = ptx::pack_out_x2_rn<Cfg::BF16>(acc.z, acc.w);
  *reinterpret_cast<uint2*>(C + size_t(gm) * N + gn) = out;
}

// Split-K epilogue (CTA_GROUP == 1, one (tile, split) unit per CTA, all units resident at once).
//   phase 1  every split writes its 128 x BN fp32 partial tile to the workspace slot (tile, split);
//   barrier  a per-tile arrival counter in global memory (release/acquire at gpu scope);
//   phase 2  split s sums a contiguous 1/splits slice of the tile's rows over ALL partials in the fixed
//            order s' = 0..splits-1 (deterministic), rounds once to fp16 and stores to C.
// The last split to finish phase 2 zeroes both counters, so the next launch on the stream starts clean.
template <class Cfg>
__device__ __forceinline__ void splitk_epilogue(uint32_t taddr0, int q, int lane, int tile, int split, int splits,
                                                int m_base, int n0, int M, int N, float* __restrict__ ws,
                                                unsigned* __restrict__ ctr, __half* __restrict__ C,
                                                uint32_t red_smem, uint32_t red_bar) {
  using namespace ptx;
  constexpr int BN = Cfg::BN;
  const int row = q * 32 + lane;
  float* slot = ws + (size_t(tile) * splits + split) * (kBlockM * BN) + size_t(row) * BN;
#pragma unroll
  for (int j = 0; j < BN / 32; ++j) {
    float f[32];
    tmem_load_f32_x32<Cfg>(taddr0, j, f);
#pragma unroll
    for (int i = 0; i < 8; ++i)
      __stcg(reinterpret_cast<float4*>(slot + j * 32) + i, make_float4(f[4 * i], f[4 * i + 1], f[4 * i + 2], f[4 * i + 3]));
  }
  // publish the partial, then wait until every split of this tile has published its own
  __threadfence();
  asm volatile("bar.sync 1, 128;" ::: "memory");
  const int e = q * 32 + lane;   // 0..127 over the four epilogue warps
  if (e == 0) {
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ctr + tile) : "memory");
    unsigned seen = 0, spins = 0;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(ctr + tile) : "memory");
      if (seen < unsigned(splits)) {
        __nanosleep(64);
        if (++spins > (1u << 24)) { printf("b200_hgemm watchdog: split-K tile %d saw %u/%d arrivals\n", tile, seen, splits); __trap(); }
      }
    } while (seen < unsigned(splits));
  }
  asm volatile("bar.sync 1, 128;" ::: "memory");
  // phase 2: rows [r0, r1) of the tile belong to this split. Their slices of all `splits` partials are pulled
  // into the (now idle) pipeline smem with 1-D bulk copies — one contiguous slice per partial — and summed there.
  const int rows_per = (kBlockM + splits - 1) / splits;
  const int r0 = split * rows_per;
  const int r1 = min(kBlockM, r0 + rows_per);
  if (r0 < r1) {
    const uint32_t slice_bytes = uint32_t(r1 - r0) * BN * 4u;
    const float* tile_ws = ws + size_t(tile) * splits * (kBlockM * BN) + size_t(r0) * BN;
    if (e == 0) {
      fence_proxy_async_all();   // the partials were written through the generic proxy by other CTAs
      mbar_arrive_expect_tx(red_bar, slice_bytes * uint32_t(splits));
      for (int sp = 0; sp < splits; ++sp)
        bulk_load_1d(red_smem + uint32_t(sp) * slice_bytes, tile_ws + size_t(sp) * (kBlockM * BN), slice_bytes, red_bar);
    }
    mbar_wait(red_bar, 0);
    constexpr int V = BN / 4;      // float4 per row
    for (int i = e; i < (r1 - r0) * V; i += 128) {
      const int r = r0 + i / V, c4 = i % V;
      const int gm = m_base + r, gn = n0 + c4 * 4;
      if (gm >= M || gn >= N) continue;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int sp = 0; sp < splits; ++sp) {   // fixed order: deterministic
        const float4 p = ld_shared_v4f(red_smem + uint32_t(sp) * slice_bytes + uint32_t(i) * 16u);
        acc.x += p.x; acc.y += p.y; acc.z += p.z; acc.w += p.w;
      }
      store_out_x4<Cfg>(C, gm, gn, N, acc);
    }
  }
  asm volatile("bar.sync 1, 128;" ::: "memory");
  if (e == 0) {
    unsigned old;
    asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;" : "=r"(old) : "l"(ctr + kMaxSplitTiles + tile) : "memory");
    if (old == unsigned(splits - 1)) {   // everyone is past the arrival wait: safe to reset for the next launch
      ctr[tile] = 0;
      ctr[kMaxSplitTiles + tile] = 0;
      __threadfence();
    }
  }
}

// Cluster split-K (CTA_GROUP == 1): the `splits` CTAs of a thread-block cluster share one output tile, each
// accumulating its own k-range. Phase 1 parks the fp32 partial tile in the CTA's own (now idle) pipeline smem;
// after a cluster barrier, CTA r sums rows [r*128/splits, (r+1)*128/splits) over all peers through distributed
// shared memory in fixed order (deterministic), rounds once and stores to C. No global workspace, no atomics.
__host__ __device__ constexpr uint32_t cluster_partial_row_bytes(int bn) { return uint32_t(bn) * 4u + 16u; }   // +16 B: conflict-free rows

template <class Cfg>
__device__ __forceinline__ void cluster_splitk_park(uint32_t taddr0, int q, int lane, uint32_t part_smem) {
  using namespace ptx;
  constexpr int BN = Cfg::BN;
  const uint32_t row_addr = part_smem + uint32_t(q * 32 + lane) * cluster_partial_row_bytes(BN);
#pragma unroll
  for (int j = 0; j < BN / 32; ++j) {
    float f[32];
    tmem_load_f32_x32<Cfg>(taddr0, j, f);
#pragma unroll
    for (int i = 0; i < 8; ++i)
      st_shared_v4f(row_addr + uint32_t(j) * 128u + uint32_t(i) * 16u, f[4 * i], f[4 * i + 1], f[4 * i + 2], f[4 * i + 3]);
  }
}

template <class Cfg>
__device__ __forceinline__ void cluster_splitk_reduce(int e, int split, int splits, int m_base, int n0, int M, int N,
                                                      uint32_t part_smem, __half* __restrict__ C) {
  using namespace ptx;
  constexpr int BN = Cfg::BN;
  constexpr int V = BN / 4;
  const int rows_per = kBlockM / splits;            // splits is 2, 4 or 8
  const int r0 = split * rows_per;
  uint32_t peer[8];
#pragma unroll
  for (int p = 0; p < 8; ++p) peer[p] = (p < splits) ? mapa(part_smem, uint32_t(p)) : 0u;
  for (int i = e; i < rows_per * V; i += 128) {
    const int r = r0 + i / V, c4 = i % V;
    const int gm = m_base + r, gn = n0 + c4 * 4;
    if (gm >= M || gn >= N) continue;
    const uint32_t off = uint32_t(r) * cluster_partial_row_bytes(BN) + uint32_t(c4) * 16u;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int p = 0; p < 8; ++p) {
      if (p < splits) {
        const float4 v = ld_dsmem_v4f(peer[p] + off);
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      }
    }
    store_out_x4<Cfg>(C, gm, gn, N, acc);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Stream-K (hgemm_schedule.cuh). Partial tiles travel through the global workspace as REGISTER IMAGES: an epilogue
// warp holds 32 rows x 64 accumulator columns of a chunk, one row per lane; the lanes write register quad i of the
// chunk to 32 consecutive uint4 and the owner's same warp reads them back the same way, so both directions are
// fully coalesced and no thread ever needs another thread's element. One flag per (CTA slot, epilogue warp):
// raised by the contributor warp after its chunks are written, polled and lowered again by the owner warp, so the
// warps stay as decoupled as in the plain epilogue and the flags are zero again when the grid ends.
constexpr int kMaxStreamKSlots = 160;   // CTAs of a launch (>= 148 SMs), one partial-tile slot each
constexpr int kStreamKFlagsPerSlot = 8; // epilogue warps

template <class Cfg>
struct StreamK {
  static constexpr int REGS = Cfg::ACC_F32 ? Cfg::EPI_N : Cfg::EPI_N / 2;   // 32-bit registers per lane per chunk
  static constexpr int R4 = REGS / 4;
  static constexpr int CHUNK_U4 = R4 * 32;                                  // one warp, one chunk
  static constexpr int SLOT_U4 = 4 * Cfg::EPI_CHUNKS * CHUNK_U4;            // one CTA: 128 rows x BN columns
  static constexpr size_t SLOT_BYTES = size_t(SLOT_U4) * 16;
  static constexpr uint32_t CHUNK_BYTES = uint32_t(CHUNK_U4) * 16;
  static constexpr int FIX_RING = Cfg::FIX_REGION_BYTES / int(CHUNK_BYTES) >= 3 ? 3 : Cfg::FIX_REGION_BYTES / int(CHUNK_BYTES);
  // The owner adds its own accumulator to the summed partials in pieces of PIECE columns, so that (sums + values in
  // flight + own accumulator) stays near the register footprint of the plain epilogue: fp32 images in two pieces of 32
  // columns, fp16 images (half the registers) in one piece of 64.
  static constexpr int PIECE = Cfg::ACC_F32 ? 32 : 64;
};

// this warp's chunk `j` of the accumulator, raw: fp32 bit patterns, or fp16 pairs (two columns per register)
template <class Cfg>
__device__ __forceinline__ void streamk_load_chunk(uint32_t taddr, uint32_t (&r)[StreamK<Cfg>::REGS]) {
  using namespace ptx;
  static_assert(Cfg::EPI_N == 64, "stream-K is wired for 64-column epilogue chunks");
  if constexpr (Cfg::ACC_F32) {
    uint32_t v0[32], v1[32];
    tmem_ld_32x32b_x32(taddr, v0);
    tmem_ld_32x32b_x32(taddr + 32, v1);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 32; ++i) { r[i] = v0[i]; r[32 + i] = v1[i]; }
  } else {
    tmem_ld_32x32b_x32_pack16(taddr, r);
    tmem_ld_wait();
  }
}

// registers -> swizzled staging buffer -> TMA store of one 32 x EPI_N chunk (shared by the plain and the owner epilogue)
template <class Cfg>
__device__ __forceinline__ void epilogue_store_chunk(const uint32_t (&packed)[Cfg::EPI_N / 2], uint32_t epi_buf,
                                                     uint32_t row_off, uint32_t sw, int lane,
                                                     const CUtensorMap* tmap_c, int nc, int m0, int M, int N) {
  using namespace ptx;
  // the previous store from this warp's staging buffer must have finished reading it
  if (lane == 0) tma_store_wait_read<0>();
  __syncwarp();
  const uint32_t dst = epi_buf + row_off;
#pragma unroll
  for (int c = 0; c < Cfg::EPI_N / 8; ++c)
    st_shared_v4(dst + ((uint32_t(c) ^ sw) << 4), packed[4 * c], packed[4 * c + 1], packed[4 * c + 2], packed[4 * c + 3]);
  fence_proxy_async_smem();
  __syncwarp();
  if (lane == 0) {
    if (m0 < M && nc < N)   // rows/cols past the edge are clipped by the tensor map
      tma_store_2d(tmap_c, epi_buf, nc, m0);
    tma_store_commit();
  }
}

struct EpilogueWarp {          // what one epilogue warp knows about itself
  int q, ew, lane;             // TMEM lane quadrant, index among the epilogue warps (0..7), lane
  int j_begin, j_end;          // its share of a tile's column chunks
  uint32_t epi_buf, row_off, sw;
};

// Contributor: spill this warp's chunks of the partial accumulator to the CTA's slot and raise the warp's flag.
// `release_tmem` hands the accumulator stage back to the MMA warp as soon as the last chunk is in registers.
template <class Cfg, class ReleaseTmem>
__device__ __forceinline__ void streamk_contribute(const EpilogueWarp& w, uint32_t taddr0, uint4* __restrict__ ws,
                                                   unsigned* __restrict__ flags, int slot, ReleaseTmem release_tmem) {
  using namespace ptx;
  using SK = StreamK<Cfg>;
  uint4* base = ws + size_t(slot) * SK::SLOT_U4 + size_t(w.q * Cfg::EPI_CHUNKS) * SK::CHUNK_U4 + w.lane;
#pragma unroll 1   // one chunk image (64 registers) at a time
  for (int j = w.j_begin; j < w.j_end; ++j) {
    uint32_t r[SK::REGS];
    streamk_load_chunk<Cfg>(taddr0 + j * Cfg::EPI_N, r);
    if (j == w.j_end - 1) release_tmem();
    uint4* dst = base + size_t(j) * SK::CHUNK_U4;
#pragma unroll
    for (int i = 0; i < SK::R4; ++i) st_global_cg_v4(dst + i * 32, r[4 * i], r[4 * i + 1], r[4 * i + 2], r[4 * i + 3]);
  }
  __threadfence();   // every lane's stores are visible at gpu scope before lane 0 publishes the flag
  __syncwarp();
  if (w.lane == 0) st_release_gpu(flags + slot * kStreamKFlagsPerSlot + w.ew, 1u);
}

// Owner, before it reads any partial: lane 0 waits until each of the `n` contributors has raised this warp's flag.
__device__ __forceinline__ void streamk_wait_contributors(const EpilogueWarp& w, const unsigned* __restrict__ flags,
                                                          int slot0, int slot_stride, int n) {
  using namespace ptx;
  if (w.lane == 0) {
    for (int p = 0; p < n; ++p) {
      const unsigned* f = flags + (slot0 + p * slot_stride) * kStreamKFlagsPerSlot + w.ew;
      unsigned spins = 0;
      while (ld_acquire_gpu(f) == 0u) {
        __nanosleep(64);
        if (++spins > (1u << 24)) { printf("b200_hgemm watchdog: stream-K slot %d never arrived\n", slot0 + p * slot_stride); __trap(); }
      }
    }
  }
  __syncwarp();
}

// Owner, done: lower the flags again. This warp is their only reader, and the next writer is a later launch.
__device__ __forceinline__ void streamk_lower_flags(const EpilogueWarp& w, unsigned* __restrict__ flags, int slot0,
                                                    int slot_stride, int n) {
  __syncwarp();
  if (w.lane == 0)
    for (int p = 0; p < n; ++p) flags[(slot0 + p * slot_stride) * kStreamKFlagsPerSlot + w.ew] = 0u;
}

// Owner: piece `h` (StreamK::PIECE columns) of the chunk at `taddr_chunk`: the own accumulator added to the summed
// partials `f` of that piece, rounded once and packed into its place in `packed`. `last`: the warp's last TMEM read,
// after which the accumulator stage goes back to the MMA warp.
template <class Cfg, class ReleaseTmem>
__device__ __forceinline__ void streamk_add_own(uint32_t taddr_chunk, int h, const float* f,
                                                uint32_t (&packed)[Cfg::EPI_N / 2], bool last, ReleaseTmem release_tmem) {
  using namespace ptx;
  if constexpr (Cfg::ACC_F32) {
    uint32_t v[32];
    tmem_ld_32x32b_x32(taddr_chunk + 32 * h, v);
    tmem_ld_wait();
    if (last) release_tmem();
#pragma unroll
    for (int i = 0; i < 16; ++i)
      packed[16 * h + i] = pack_out_x2_rn<Cfg::BF16>(f[2 * i] + __uint_as_float(v[2 * i]), f[2 * i + 1] + __uint_as_float(v[2 * i + 1]));
  } else {
    uint32_t r[StreamK<Cfg>::REGS];
    streamk_load_chunk<Cfg>(taddr_chunk, r);
    if (last) release_tmem();
#pragma unroll
    for (int i = 0; i < Cfg::EPI_N / 2; ++i) {
      const __half2 hh = *reinterpret_cast<const __half2*>(&r[i]);
      packed[i] = pack_out_x2_rn<Cfg::BF16>(f[2 * i] + __low2float(hh), f[2 * i + 1] + __high2float(hh));
    }
  }
}

// Owner: the partials of `n` contributors (slots slot0, slot0 + slot_stride, ... — increasing k) summed in fp32 in that
// fixed order, plus the own accumulator, rounded once, stored like any other tile. The partials were written long
// before (they are their workers' first units), so the first chunk's are fetched BEFORE waiting for the own
// accumulator (`wait_acc`): their L2 latency hides behind the tail of the main loop.
template <class Cfg, class WaitAcc, class ReleaseTmem>
__device__ __forceinline__ void streamk_own(const EpilogueWarp& w, uint32_t taddr0, const uint4* __restrict__ ws,
                                            unsigned* __restrict__ flags, int slot0, int slot_stride, int n,
                                            const CUtensorMap* tmap_c, int m0, int n0, int M, int N,
                                            WaitAcc wait_acc, ReleaseTmem release_tmem) {
  using namespace ptx;
  using SK = StreamK<Cfg>;
  streamk_wait_contributors(w, flags, slot0, slot_stride, n);
  const size_t warp_off = size_t(w.q * Cfg::EPI_CHUNKS) * SK::CHUNK_U4 + w.lane;
  constexpr int kPiece = SK::PIECE;                               // columns
  constexpr int kPieceQuads = SK::R4 * kPiece / Cfg::EPI_N;       // image quads per piece (8 in both cases)
  constexpr int kBatch = 4;                                       // quads in flight per lane
#pragma unroll 1
  for (int j = w.j_begin; j < w.j_end; ++j) {
    uint32_t packed[Cfg::EPI_N / 2];
#pragma unroll
    for (int h = 0; h < Cfg::EPI_N / kPiece; ++h) {
      float f[kPiece];
#pragma unroll
      for (int i = 0; i < kPiece; ++i) f[i] = 0.f;
      for (int p = 0; p < n; ++p) {
        const uint4* src = ws + size_t(slot0 + p * slot_stride) * SK::SLOT_U4 + warp_off + size_t(j) * SK::CHUNK_U4 +
                           size_t(h * kPieceQuads) * 32;
#pragma unroll
        for (int b = 0; b < kPieceQuads / kBatch; ++b) {
          uint4 v[kBatch];
#pragma unroll
          for (int i = 0; i < kBatch; ++i) v[i] = ld_global_cg_v4(src + (kBatch * b + i) * 32);
#pragma unroll
          for (int i = 0; i < kBatch; ++i) {
            const uint32_t x[4] = {v[i].x, v[i].y, v[i].z, v[i].w};
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              if constexpr (Cfg::ACC_F32) {
                f[4 * (kBatch * b + i) + c] += __uint_as_float(x[c]);
              } else {
                const __half2 hh = *reinterpret_cast<const __half2*>(&x[c]);
                f[8 * (kBatch * b + i) + 2 * c] += __low2float(hh);
                f[8 * (kBatch * b + i) + 2 * c + 1] += __high2float(hh);
              }
            }
          }
          __syncwarp();   // keeps the compiler from hoisting the next batch's loads above these sums
        }
      }
      if (j == w.j_begin && h == 0) wait_acc();
      const bool last = (j == w.j_end - 1) && (h == Cfg::EPI_N / kPiece - 1);
      streamk_add_own<Cfg>(taddr0 + j * Cfg::EPI_N, h, f, packed, last, release_tmem);
    }
    epilogue_store_chunk<Cfg>(packed, w.epi_buf, w.row_off, w.sw, w.lane, tmap_c, n0 + j * Cfg::EPI_N, m0, M, N);
  }
  streamk_lower_flags(w, flags, slot0, slot_stride, n);
}

// Owner whose unit ends the worker's schedule: nothing hides the fix-up any more, and register loads would crawl
// (one 16-byte load per lane and round trip). The pipeline shared memory is idle once the own accumulator is
// complete, so lane 0 streams this warp's chunk images of every contributor through a ring of bulk copies
// (`fix_smem`: this warp's region, `fix_bar`: its FIX_RING mbarriers, phase 0 on entry) while the warp sums them from
// shared memory — same order of additions as streamk_own, hence the same bits.
template <class Cfg, class WaitAcc, class ReleaseTmem>
__device__ __forceinline__ void streamk_own_bulk(const EpilogueWarp& w, uint32_t taddr0, const uint4* __restrict__ ws,
                                                 unsigned* __restrict__ flags, int slot0, int slot_stride, int n,
                                                 const CUtensorMap* tmap_c, int m0, int n0, int M, int N,
                                                 uint32_t fix_smem, uint32_t fix_bar, WaitAcc wait_acc,
                                                 ReleaseTmem release_tmem) {
  using namespace ptx;
  using SK = StreamK<Cfg>;
  constexpr int RING = SK::FIX_RING;
  static_assert(RING >= 2, "the fix-up ring needs two chunk images per epilogue warp");
  streamk_wait_contributors(w, flags, slot0, slot_stride, n);
  const int total = (w.j_end - w.j_begin) * n;   // items in (chunk, contributor) order
  auto issue = [&](int i) {
    if (w.lane == 0) {
      const int jj = i / n, p = i - jj * n, s = i % RING;
      const uint4* src = ws + size_t(slot0 + p * slot_stride) * SK::SLOT_U4 +
                         size_t(w.q * Cfg::EPI_CHUNKS + w.j_begin + jj) * SK::CHUNK_U4;
      mbar_arrive_expect_tx(fix_bar + 8 * s, SK::CHUNK_BYTES);
      bulk_load_1d(fix_smem + uint32_t(s) * SK::CHUNK_BYTES, src, SK::CHUNK_BYTES, fix_bar + 8 * s);
    }
  };
  wait_acc();                 // every MMA of the worker has read its operands: the pipeline shared memory is free
  fence_proxy_async_all();    // the partials were written through the generic proxy (by other CTAs, acquired above)
  for (int i = 0; i < RING && i < total; ++i) issue(i);
  int item = 0;
#pragma unroll 1
  for (int j = w.j_begin; j < w.j_end; ++j) {
    float f[Cfg::EPI_N];
#pragma unroll
    for (int i = 0; i < Cfg::EPI_N; ++i) f[i] = 0.f;
    for (int p = 0; p < n; ++p, ++item) {
      const int s = item % RING;
      mbar_wait(fix_bar + 8 * s, uint32_t(item / RING) & 1u);
      const uint32_t img = fix_smem + uint32_t(s) * SK::CHUNK_BYTES + uint32_t(w.lane) * 16u;
#pragma unroll
      for (int i = 0; i < SK::R4; ++i) {
        const uint4 v = ld_shared_v4(img + uint32_t(i) * 512u);
        const uint32_t x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if constexpr (Cfg::ACC_F32) {
            f[4 * i + c] += __uint_as_float(x[c]);
          } else {
            const __half2 hh = *reinterpret_cast<const __half2*>(&x[c]);
            f[8 * i + 2 * c] += __low2float(hh);
            f[8 * i + 2 * c + 1] += __high2float(hh);
          }
        }
      }
      __syncwarp();   // every lane is done with this ring slot
      if (item + RING < total) {
        fence_proxy_async_smem();
        issue(item + RING);
      }
    }
    uint32_t packed[Cfg::EPI_N / 2];
#pragma unroll
    for (int h = 0; h < Cfg::EPI_N / SK::PIECE; ++h) {
      const bool last = (j == w.j_end - 1) && (h == Cfg::EPI_N / SK::PIECE - 1);
      streamk_add_own<Cfg>(taddr0 + j * Cfg::EPI_N, h, f + h * SK::PIECE, packed, last, release_tmem);
    }
    epilogue_store_chunk<Cfg>(packed, w.epi_buf, w.row_off, w.sw, w.lane, tmap_c, n0 + j * Cfg::EPI_N, m0, M, N);
  }
  streamk_lower_flags(w, flags, slot0, slot_stride, n);
}

template <class Cfg, int KMODE = kPlain>
__global__ void __launch_bounds__(Cfg::NUM_THREADS, 1)
hgemm_tn_kernel(const __grid_constant__ CUtensorMap tmap_a,   // A  [M,K]  box {64, A_BOX_ROWS}
                const __grid_constant__ CUtensorMap tmap_b,   // Bt [N,K]  box {64, B_BOX_ROWS}
                const __grid_constant__ CUtensorMap tmap_c,   // C  [M,N]  box {EPI_N, 32}
                int M, int N, int K, int group_m,
                int splits_arg,                   // split-K factor (modes kWorkspaceSplitK / kClusterSplitK: one unit per CTA)
                int sk_tiles_arg,                 // mode kStreamK: the first sk_tiles tiles are cut along K across all workers
                float* __restrict__ splitk_ws,    // [units][128][BN] fp32 partial tiles (workspace split-K) / stream-K slots
                unsigned* __restrict__ splitk_ctr,   // [2][kMaxSplitTiles] split-K arrive / done counters, then the
                                                     // stream-K flags; all zero between launches
                __half* __restrict__ c_raw,       // C base pointer, used by the split-K reductions' direct stores
                uint64_t hint_a, uint64_t hint_b  /* L2 eviction priority of the A / B loads (ptx::kL2Evict*) */) {
  constexpr int BN = Cfg::BN;
  constexpr int STAGES = Cfg::STAGES;
  constexpr int CG = Cfg::CTA_GROUP;
  constexpr int CM = Cfg::CLUSTER_M;
  constexpr int CN = Cfg::CLUSTER_N;
  constexpr bool kMcast = Cfg::MCAST_CTAS > 1;
  constexpr int AS = Cfg::ACC_STAGES;
  constexpr int MR = Cfg::M_REP;
  constexpr bool kSplit = (KMODE == kWorkspaceSplitK || KMODE == kClusterSplitK);
  static_assert(!kSplit || Cfg::SPLIT_K, "this configuration has no split-K epilogues");
  static_assert(KMODE != kStreamK || Cfg::STREAM_K, "this configuration has no stream-K epilogues");
  // the schedule parameters a mode does not use are constants for it
  const int splits = kSplit ? splits_arg : 1;
  const int sk_tiles = (KMODE == kStreamK) ? sk_tiles_arg : 0;
  using namespace ptx;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t smem_a = smem_base;
  const uint32_t smem_b = smem_a + STAGES * Cfg::A_STAGE_BYTES;
  const uint32_t smem_epi = smem_b + STAGES * Cfg::B_STAGE_BYTES;
  const uint32_t smem_bar = smem_epi + Cfg::EPI_BYTES;
  const uint32_t bar_full = smem_bar;                        // [STAGES]
  const uint32_t bar_empty = bar_full + 8 * STAGES;          // [STAGES]
  const uint32_t bar_tmem_full = bar_empty + 8 * STAGES;     // [kAccStages]
  const uint32_t bar_tmem_empty = bar_tmem_full + 8 * kAccStages;
  const uint32_t bar_splitk = bar_tmem_empty + 8 * kAccStages;   // split-K: bulk loads of the partial slices
  const uint32_t tmem_slot = bar_splitk + 8;
  const uint32_t bar_fix = tmem_slot + 8;                        // [8 epilogue warps][3]: stream-K fix-up rings

  const int warp = __shfl_sync(0xffffffffu, int(threadIdx.x) >> 5, 0);
  const int lane = threadIdx.x & 31;
  B200_TRACE_ONLY(if (threadIdx.x == 64) B200_TRACE(0);)
  // Position inside the cluster: rank = (cm + CLUSTER_M * cn) * CTA_GROUP + (position inside the MMA pair).
  // (A cluster split-K launch of a plain config also has ranks, but does not use them here.)
  const uint32_t cluster_rank = (Cfg::CLUSTER_CTAS > 1) ? cluster_ctarank() : 0u;
  const uint32_t cta_rank = cluster_rank % CG;             // position inside the MMA pair (0 for single-CTA groups)
  const uint32_t group_rank = cluster_rank / CG;           // which group of the cluster
  const uint32_t leader_rank = cluster_rank - cta_rank;    // cluster rank of this group's leader CTA
  const bool is_leader = (cta_rank == 0);
  const int cm = kMcast ? int(group_rank % CM) : 0;
  const int cn = kMcast ? int(group_rank / CM) : 0;

  // The schedule is over cluster blocks of (CM x TILE_M) x (CN x BN); a plain config has 1 x 1 blocks.
  const int num_m_blocks = (M + Cfg::TILE_M * CM - 1) / (Cfg::TILE_M * CM);
  const int num_n_blocks = (N + BN * CN - 1) / (BN * CN);
  const int num_tiles = num_m_blocks * num_n_blocks;
  const int num_k_blocks = (K + kBlockK - 1) / kBlockK;
  const int num_workers = gridDim.x / Cfg::CLUSTER_CTAS;   // clusters (or single CTAs)
  const int worker = blockIdx.x / Cfg::CLUSTER_CTAS;
  // A work unit is (tile, k-block range), see hgemm_schedule.cuh. splits == 1: whole tiles walked persistently
  // (after the worker's stream-K slice, if any). splits > 1: the host launches exactly one CTA per (tile, split)
  // unit, so the sibling splits of a tile run concurrently.

  // ------------------------------------------------------------------ one-time setup
  if (warp == 0 && elect_one()) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(bar_full + 8 * s, 1);                      // the producer's arrive.expect_tx (the leader's, for a pair)
      mbar_init(bar_empty + 8 * s, kMcast ? CM + CN - 1 : 1);   // tcgen05.commit of every CTA this stage is shared with
    }
    for (int a = 0; a < AS; ++a) {
      mbar_init(bar_tmem_full + 8 * a, 1);        // tcgen05.commit after the tile's last k-block
      mbar_init(bar_tmem_empty + 8 * a, 4 * Cfg::EPI_GROUPS * CG);  // one arrive per working epilogue warp of the group
    }
    mbar_init(bar_splitk, 1);
    if constexpr (KMODE == kStreamK) {
      for (int i = 0; i < Cfg::FIX_BARS; ++i) mbar_init(bar_fix + 8 * i, 1);
    }
    fence_mbar_init();
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    tma_prefetch_desc(&tmap_c);
  }
  if (warp == 2) {
    tmem_alloc<CG>(tmem_slot, Cfg::TMEM_COLS);
    tmem_relinquish<CG>();
  }
  __syncwarp();   // reconverge after the elected-lane branches before the aligned barrier
  tc_fence_before_sync();
  if constexpr (Cfg::CLUSTER_CTAS > 1) cluster_sync_all(); else __syncthreads();
  tc_fence_after_sync();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  B200_TRACE_ONLY(if (threadIdx.x == 64) B200_TRACE(1);)

  // Programmatic dependent launch (the host sets cudaLaunchAttributeProgrammaticStreamSerialization): this grid may have
  // been started while the previous kernel of the stream was still running, so that everything above — barrier
  // initialisation, TMEM allocation, descriptor prefetch, the set-up barrier — overlaps that kernel's tail instead of
  // following it. Nothing above touches global memory; everything below may, so every thread first waits until the
  // prerequisite grids have completed and their writes are visible (a no-op for an ordinary launch). The next kernel
  // of the stream may in turn begin ITS prologue as soon as SMs free up.
  ptx::grid_dependency_launch_dependents();
  ptx::grid_dependency_wait();

  [[maybe_unused]] int ck_m_base = 0, ck_n0 = 0, ck_split = 0;   // cluster split-K: where this CTA's unit lives (set by the epilogue warps)

  // ------------------------------------------------------------------ roles
  if (warp == 0) {
    // ===== TMA producer: the warp walks the schedule, one elected lane issues =====
    // pair mode: every load of both CTAs reports its bytes to the leader's full barrier
    // (multicast in pair mode: the barrier operand is the local offset with the pair-peer bit cleared, which
    //  every destination resolves to ITS OWN pair leader — the same convention CUTLASS uses)
    const uint32_t full_uc = (CG == 2) ? mapa(bar_full, leader_rank) : bar_full;     // unicast loads
    const uint32_t full_mc = (CG == 2) ? (bar_full & 0xFEFFFFFFu) : bar_full;        // multicast loads
    // multicast masks: my A slice goes to the same-position CTAs of my cluster row (same cm), my B slice to
    // those of my cluster column (same cn)
    uint16_t mask_a = 0, mask_b = 0;
#pragma unroll
    for (int j = 0; j < CN; ++j) mask_a |= uint16_t(1u << ((cm + CM * j) * CG + int(cta_rank)));
#pragma unroll
    for (int i = 0; i < CM; ++i) mask_b |= uint16_t(1u << ((i + CM * cn) * CG + int(cta_rank)));
    const uint32_t a_slice = uint32_t(cn) * (Cfg::A_BOX_ROWS * kBlockK * 2);
    const uint32_t b_slice = uint32_t(cm) * (Cfg::B_BOX_ROWS * kBlockK * 2);
    int stage = 0; uint32_t phase = 0;
    B200_TRACE_ONLY(bool trace_first = true;)
    WorkIter work(worker, num_workers, num_tiles, num_k_blocks, splits, sk_tiles);
    WorkUnit u;
    while (work.next(u)) {
      const TileCoord tc = tile_coord(u.tile, num_m_blocks, num_n_blocks, group_m);
      const int m0 = (tc.m_blk * CM + cm) * Cfg::TILE_M + int(cta_rank) * Cfg::CTA_M + cn * Cfg::A_BOX_ROWS;
      const int n0 = (tc.n_blk * CN + cn) * BN + int(cta_rank) * Cfg::LOAD_N + cm * Cfg::B_BOX_ROWS;
      for (int kb = u.kb0; kb < u.kb1; ++kb) {
        mbar_wait(bar_empty + 8 * stage, phase ^ 1);
        if (elect_one()) {
          if (is_leader) mbar_arrive_expect_tx(bar_full + 8 * stage, Cfg::STAGE_BYTES * CG);
          const uint32_t dst_a = smem_a + stage * Cfg::A_STAGE_BYTES + a_slice;
          const uint32_t dst_b = smem_b + stage * Cfg::B_STAGE_BYTES + b_slice;
          if constexpr (CN > 1) tma_load_2d_mcast_hint<CG>(dst_a, &tmap_a, full_mc + 8 * stage, kb * kBlockK, m0, mask_a, hint_a);
          else tma_load_2d_hint<CG>(dst_a, &tmap_a, full_uc + 8 * stage, kb * kBlockK, m0, hint_a);
          if constexpr (CM > 1) tma_load_2d_mcast_hint<CG>(dst_b, &tmap_b, full_mc + 8 * stage, kb * kBlockK, n0, mask_b, hint_b);
          else tma_load_2d_hint<CG>(dst_b, &tmap_b, full_uc + 8 * stage, kb * kBlockK, n0, hint_b);
          B200_TRACE_ONLY(if (trace_first) { B200_TRACE(2); trace_first = false; })
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
    B200_TRACE_ONLY(if (lane == 0) B200_TRACE(3);)
  } else if (warp == 1) {
    // ===== MMA issuer: the whole warp of the leader CTA walks the schedule (so loop state stays in uniform
    // registers and the waits are warp-wide), one elected lane issues tcgen05.mma / tcgen05.commit =====
    if (is_leader) {
      constexpr uint32_t idesc = make_idesc(kBlockM * CG, BN, Cfg::ACC_F32, Cfg::BF16);   // one MMA covers 128 rows per CTA of the group
      const uint64_t desc_a0 = make_smem_desc(smem_a);
      const uint64_t desc_b0 = make_smem_desc(smem_b);
      // who must learn that a stage has been consumed: the pair (pair mode), or every CTA that multicasts
      // into this CTA's smem, i.e. my cluster row and column (multicast mode)
      constexpr uint16_t kGroupBits = (CG == 2) ? 0b11 : 0b1;          // every CTA of a group
      const uint16_t mask_self = uint16_t(kGroupBits << (group_rank * CG));
      uint16_t mask_free = mask_self;
      if constexpr (kMcast) {
#pragma unroll
        for (int j = 0; j < CN; ++j) mask_free |= uint16_t(kGroupBits << ((cm + CM * j) * CG));
#pragma unroll
        for (int i = 0; i < CM; ++i) mask_free |= uint16_t(kGroupBits << ((i + CM * cn) * CG));
      }
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      B200_TRACE_ONLY(bool trace_first = true; unsigned long long trace_kb = 0, trace_units = 0;)
      WorkIter work(worker, num_workers, num_tiles, num_k_blocks, splits, sk_tiles);
      WorkUnit u;
      while (work.next(u)) {
        const int kb0 = u.kb0, kb1 = u.kb1;
        mbar_wait(bar_tmem_empty + 8 * acc, acc_phase ^ 1);   // epilogue drained this accumulator
        tc_fence_after_sync();
        const uint32_t tmem_d = tmem_base + acc * Cfg::ACC_COLS;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(bar_full + 8 * stage, phase);
          tc_fence_after_sync();
          B200_TRACE_ONLY(if (trace_first) { if (lane == 0) B200_TRACE(4); trace_first = false; } ++trace_kb;)
          if (elect_one()) {
            // stage s lives (A_STAGE_BYTES >> 4) further along in the descriptor's (addr >> 4) field;
            // +32 B per K step inside the 128 B swizzle row == +2 in that field
            const uint64_t da = desc_a0 + uint64_t(stage * (Cfg::A_STAGE_BYTES >> 4));
            const uint64_t db = desc_b0 + uint64_t(stage * (Cfg::B_STAGE_BYTES >> 4));
#pragma unroll
            for (int k = 0; k < kBlockK / kUmmaK; ++k)
              umma_f16<CG>(tmem_d, da + uint64_t(2 * k), db + uint64_t(2 * k), idesc, ((kb - kb0) | k) != 0);
            if constexpr (MR == 2) {
              // the second 128-row block of this CTA's A tile (16 KB further into the stage) -> the second accumulator
              constexpr uint64_t kSecondBlock = uint64_t((kBlockM * kBlockK * 2) >> 4);
#pragma unroll
              for (int k = 0; k < kBlockK / kUmmaK; ++k)
                umma_f16<CG>(tmem_d + BN, da + kSecondBlock + uint64_t(2 * k), db + uint64_t(2 * k), idesc, ((kb - kb0) | k) != 0);
            }
            // free the smem slot everywhere it is shared once these MMAs have read it
            if constexpr (CG == 2 || kMcast) umma_commit_mcast<CG>(bar_empty + 8 * stage, mask_free);
            else umma_commit<CG>(bar_empty + 8 * stage);
            if (kb == kb1 - 1) {   // accumulator complete: wake the epilogue
              if constexpr (CG == 2) umma_commit_mcast<CG>(bar_tmem_full + 8 * acc, mask_self);
              else umma_commit<CG>(bar_tmem_full + 8 * acc);
            }
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        if (++acc == AS) { acc = 0; acc_phase ^= 1; }
        B200_TRACE_ONLY(++trace_units;)
      }
      B200_TRACE_ONLY(if (lane == 0) { B200_TRACE(5); B200_TRACE_VALUE(9, trace_kb); B200_TRACE_VALUE(11, trace_units); })
    }
  } else if (warp >= kEpiWarp0) {
    // ===== epilogue: TMEM -> registers -> (cvt) -> swizzled smem -> TMA store =====
    constexpr int EN = Cfg::EPI_N;
    const int q = (warp - kEpiWarp0) & 3;           // == warp % 4: TMEM lanes [32q, 32q+32)
    const int eg = (warp - kEpiWarp0) >> 2;         // 0: first half of the column chunks, 1: second half
    const uint32_t epi_buf = smem_epi + uint32_t(warp - kEpiWarp0) * (32 * 64 * 2);
    const uint32_t tmem_empty0 = (CG == 2) ? mapa(bar_tmem_empty, leader_rank) : bar_tmem_empty;
    const uint32_t row_off = uint32_t(lane) * uint32_t(EN * 2);
    // staging rows are EN*2 bytes: 128 B rows use the 128B swizzle (chunk ^= row % 8), 64 B rows the 64B one
    const uint32_t sw = (EN == 64) ? uint32_t(lane & 7) : uint32_t((lane >> 1) & 3);
    constexpr int CPG = Cfg::EPI_CHUNKS_PER_GROUP;
    const int j_begin = eg * CPG;
    const int j_end = min(Cfg::EPI_CHUNKS, j_begin + CPG);
    const bool working = eg < Cfg::EPI_GROUPS;      // narrow tiles keep the second set of warps idle
    int acc = 0; uint32_t acc_phase = 0;
    B200_TRACE_ONLY(bool trace_first = true;)
    const EpilogueWarp ew{q, warp - kEpiWarp0, lane, j_begin, j_end, epi_buf, row_off, sw};
    if (working) {
    WorkIter work(worker, num_workers, num_tiles, num_k_blocks, splits, sk_tiles);
    WorkUnit u;
    while (work.next(u)) {
      const int t = u.tile;
      const TileCoord tc = tile_coord(t, num_m_blocks, num_n_blocks, group_m);
      const int m_tile0 = (tc.m_blk * CM + cm) * Cfg::TILE_M + int(cta_rank) * Cfg::CTA_M;
      const int n0 = (tc.n_blk * CN + cn) * BN;
      if constexpr (kSplit) {
        if (eg != 0) break;   // the split-K reductions are written for the first four epilogue warps
      }
      const uint32_t taddr_acc = tmem_base + uint32_t(acc * Cfg::ACC_COLS) + (uint32_t(q * 32) << 16);
      // the MMA warp's commit: this unit's accumulator is complete
      auto wait_acc = [&] {
        mbar_wait(bar_tmem_full + 8 * acc, acc_phase);
        tc_fence_after_sync();
        B200_TRACE_ONLY(if (warp == kEpiWarp0 && lane == 0) { if (trace_first) { B200_TRACE(6); trace_first = false; } B200_TRACE(10); })
      };
      // this warp's share of the accumulator is in registers: hand the TMEM stage back to the MMA warp
      auto release_tmem = [&] {
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) {
          if constexpr (CG == 2) mbar_arrive_cluster(tmem_empty0 + 8 * acc);
          else mbar_arrive(tmem_empty0 + 8 * acc);
        }
      };
      [[maybe_unused]] uint4* ws4 = reinterpret_cast<uint4*>(splitk_ws);
      [[maybe_unused]] unsigned* sk_flags = splitk_ctr + 2 * kMaxSplitTiles;
      if constexpr (KMODE == kStreamK) {
        if (u.kb0 == 0 && u.kb1 < num_k_blocks) {   // the head of a tile, which owns it
          const int n = streamk_contributors(worker, num_workers, sk_tiles * num_k_blocks, t, num_k_blocks);
          if (!work.has_more())   // nothing left to hide the fix-up behind: stream it through shared memory
            streamk_own_bulk<Cfg>(ew, taddr_acc, ws4, sk_flags, (worker + 1) * CG + int(cta_rank), CG, n, &tmap_c,
                                  m_tile0 + q * 32, n0, M, N, smem_a + uint32_t(ew.ew) * Cfg::FIX_REGION_BYTES,
                                  bar_fix + 8 * 3 * ew.ew, wait_acc, release_tmem);
          else
            streamk_own<Cfg>(ew, taddr_acc, ws4, sk_flags, (worker + 1) * CG + int(cta_rank), CG, n, &tmap_c, m_tile0 + q * 32,
                             n0, M, N, wait_acc, release_tmem);
          if (++acc == AS) { acc = 0; acc_phase ^= 1; }
          continue;
        }
      }
      wait_acc();
      // (split-K modes: one unit per CTA, so no accumulator ring bookkeeping is needed after it)
      if constexpr (KMODE == kClusterSplitK) {
        cluster_splitk_park<Cfg>(taddr_acc, q, lane, smem_a);
        ck_m_base = m_tile0; ck_n0 = n0; ck_split = worker - t * splits;   // the reduction runs after the cluster barrier below
      } else if constexpr (KMODE == kWorkspaceSplitK) {
        splitk_epilogue<Cfg>(taddr_acc, q, lane, t, worker - t * splits, splits, m_tile0, n0, M, N,
                             splitk_ws, splitk_ctr, c_raw, smem_a, bar_splitk);
      } else {
      if constexpr (KMODE == kStreamK) {
        if (u.kb0 > 0) {   // a later part of a tile's k-range, handed to the tile's owner
          streamk_contribute<Cfg>(ew, taddr_acc, ws4, sk_flags, worker * CG + int(cta_rank), release_tmem);
          if (++acc == AS) { acc = 0; acc_phase ^= 1; }
          continue;
        }
      }
#pragma unroll
      for (int r = 0; r < MR; ++r) {   // the 128-row blocks of this CTA's tile, one accumulator each
      const uint32_t taddr0 = taddr_acc + uint32_t(r * BN);
      const int m0 = m_tile0 + r * kBlockM + q * 32;
      for (int j = j_begin; j < j_end; ++j) {
        uint32_t packed[EN / 2];
        if constexpr (Cfg::ACC_F32) {
          uint32_t v0[32];
          tmem_ld_32x32b_x32(taddr0 + j * EN, v0);
          if constexpr (EN == 64) {
            uint32_t v1[32];
            tmem_ld_32x32b_x32(taddr0 + j * EN + 32, v1);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i)
              packed[16 + i] = pack_out_x2_rn<Cfg::BF16>(__uint_as_float(v1[2 * i]), __uint_as_float(v1[2 * i + 1]));
          } else {
            tmem_ld_wait();
          }
#pragma unroll
          for (int i = 0; i < 16; ++i)
            packed[i] = pack_out_x2_rn<Cfg::BF16>(__uint_as_float(v0[2 * i]), __uint_as_float(v0[2 * i + 1]));
        } else {
          if constexpr (EN == 64) tmem_ld_32x32b_x32_pack16(taddr0 + j * EN, packed);
          else tmem_ld_32x32b_x16_pack16(taddr0 + j * EN, packed);
          tmem_ld_wait();
        }
        if (j == j_end - 1 && r == MR - 1) release_tmem();
        epilogue_store_chunk<Cfg>(packed, epi_buf, row_off, sw, lane, &tmap_c, n0 + j * EN, m0, M, N);
      }
      }
      if (++acc == AS) { acc = 0; acc_phase ^= 1; }
      }   // plain / stream-K modes
    }
    }
    // smem may be released once the bulk stores have READ it; their global writes complete with the grid
    if (lane == 0) tma_store_wait_read<0>();
    B200_TRACE_ONLY(if (warp == kEpiWarp0 && lane == 0) B200_TRACE(7);)
  }

  // ------------------------------------------------------------------ cluster split-K reduction
  if constexpr (KMODE == kClusterSplitK) {
    __syncwarp();
    cluster_sync_all();   // every split's partial tile is parked in its CTA's shared memory
    if (warp >= kEpiWarp0 && warp < kEpiWarp0 + 4)
      cluster_splitk_reduce<Cfg>((warp - kEpiWarp0) * 32 + lane, ck_split, splits, ck_m_base, ck_n0, M, N, smem_a, c_raw);
    __syncwarp();
    cluster_sync_all();   // no CTA leaves (and frees its smem) while a peer may still be reading it
  }

  // ------------------------------------------------------------------ teardown
  __syncwarp();   // single-lane roles rejoin their warp before the aligned barrier
  tc_fence_before_sync();
  if constexpr (Cfg::CLUSTER_CTAS > 1) cluster_sync_all(); else __syncthreads();
  B200_TRACE_ONLY(if (threadIdx.x == 64) B200_TRACE(8);)
  if (warp == 2) {
    tc_fence_after_sync();
    tmem_dealloc<CG>(tmem_base, Cfg::TMEM_COLS);
  }
}

}  // namespace b200
