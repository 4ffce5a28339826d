// One shape-specialised entry point per kernels/b200_*/<M>_<N>_<K>.cu: instantiates exactly one
// kernel configuration (the tuned choice for that shape) and exports it under the fixed C name the
// torch binding links against (pybind/b200_raw_api.h). The reference does the equivalent with a
// hand-picked tile/stage/swizzle inside each per-shape .cu (kernels/a100_F32F16F16F32/4096_4096_4096.cu:292-310).
#pragma once
#include "hgemm_host.cuh"

// The K-modes a per-shape translation unit needs compiled: its own (from the tuned split code) and the plain fallback.
#define B200_HGEMM_SHAPE_MODES(SPLITS)                                                                  \
  ((1u << b200::kPlain) | ((SPLITS) >= 100 ? (1u << b200::kStreamK)                                     \
                           : (SPLITS) > 1  ? (1u << b200::kWorkspaceSplitK)                              \
                           : (SPLITS) < -1 ? (1u << b200::kClusterSplitK) : 0u))

// Exports the launcher of one configuration; M_REP = 2 for the configurations with 256 rows per CTA.
#define B200_HGEMM_SHAPE_ENTRY_WIDE(ACC_F32, BN, STAGES, CTA_GROUP, CLUSTER_M, CLUSTER_N, M_REP, GROUP_M, SPLITS)            \
  extern "C" int b200_hgemm_shape_entry(const void* A, const void* B_kmajor, void* C, int M, int N, int K,    \
                                        void* stream) {                                                       \
    return b200::host::launch<b200::Config<BN, STAGES, CTA_GROUP, ACC_F32, CLUSTER_M, CLUSTER_N, M_REP>, B200_HGEMM_SHAPE_MODES(SPLITS)>( \
        A, B_kmajor, C, M, N, K, static_cast<cudaStream_t>(stream), GROUP_M, 0, SPLITS);                      \
  }                                                                                                           \
  extern "C" const char* b200_hgemm_shape_strerror(int status) { return b200::host::status_string(status); }

#define B200_HGEMM_SHAPE_ENTRY(ACC_F32, BN, STAGES, CTA_GROUP, CLUSTER_M, CLUSTER_N, GROUP_M, SPLITS) \
  B200_HGEMM_SHAPE_ENTRY_WIDE(ACC_F32, BN, STAGES, CTA_GROUP, CLUSTER_M, CLUSTER_N, 1, GROUP_M, SPLITS)
