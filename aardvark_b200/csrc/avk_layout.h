// avk_layout.h -- device-side data layouts shared by the warp solvers (avk_solver.cuh), the thread-per-cluster solver
// (avk_thread_solver.cuh) and the host build of the latter used by the tests.  Plain C++ (no CUDA types).
#pragma once
#include <stdint.h>
#include "../../include/aardvark_b200.h"

#if defined(__CUDACC__)
#define AVK_HD __host__ __device__
#define AVK_HD_NOINLINE __host__ __device__ __noinline__
#else
#define AVK_HD
#define AVK_HD_NOINLINE
#endif

namespace avk {

// Cluster digest written by k_prep_fill: header (64 bytes), then N VI_* records in merged processing order, then the allele
// bytes (VI_AOFF is relative to their start).
enum { PH_STATUS = 0, PH_N = 4, PH_N0 = 8, PH_N1 = 12, PH_SUM_L1 = 16, PH_B0 = 20, PH_SUM_ALLE = 24, PH_MAX_END = 28,
       PH_NSLOTS = 32, PH_SLOT_TYPE = 36, PH_SIZE = 64 };

// One variant of the cluster in merged processing order (order_variants, query_optimizer.rs:372-381): 32-byte record.
enum { VI_POS = 0, VI_L0 = 4, VI_L1 = 8, VI_AOFF = 12, VI_ALTED = 16, VI_RAW = 20, VI_GV = 24, VI_FLAGS = 28, VI_SIZE = 32 };
// flags: type | zyg << 8 | is_truth << 16 | slot << 24

enum { AL_UNSET = 0, AL_REF = 1, AL_ALT = 2 };

// Summary counters accumulated inside the solver kernels (SummaryWriter::add_comparison_benchmark,
// writers/summary.rs:146-158): TOT_SLOTS partial tables of [13][22] metric sums + {type mask, solved, errors};
// a CTA adds to slot blockIdx.x % TOT_SLOTS (u64 atomics in L2, little contention), k_fold_slots sums the slots.
enum { TOT_SLOTS = 128, TOT_COLS = AVK_N_GROUPS * AVK_N_METRICS, TOT_MASK = TOT_COLS, TOT_SOLVED = TOT_COLS + 1,
       TOT_ERRORS = TOT_COLS + 2, TOT_STRIDE = TOT_COLS + 6 };
// Per-stratum sums, added at the same places as the totals: STRAT_SLOTS partial tables [n_strata][TOT_COLS] (fewer than
// TOT_SLOTS so that 1,000 strata of the list path stay at 36 MB); a CTA adds to slot blockIdx.x % STRAT_SLOTS, k_fold_strata
// sums the slots.
enum { STRAT_SLOTS = 16 };

static AVK_HD inline bool type_supported(int t) {   // SUPPORTED_VARIANT_TYPES waffle_solver.rs:82-91
    return t == AVK_VT_SNV || t == AVK_VT_INSERTION || t == AVK_VT_DELETION || t == AVK_VT_INDEL ||
           t == AVK_VT_TR_CONTRACTION || t == AVK_VT_TR_EXPANSION || t == AVK_VT_SV_DELETION || t == AVK_VT_SV_INSERTION;
}
static AVK_HD inline uint32_t supported_type_mask() {
    return (1u << AVK_VT_SNV) | (1u << AVK_VT_INSERTION) | (1u << AVK_VT_DELETION) | (1u << AVK_VT_INDEL) |
           (1u << AVK_VT_TR_CONTRACTION) | (1u << AVK_VT_TR_EXPANSION) | (1u << AVK_VT_SV_DELETION) | (1u << AVK_VT_SV_INSERTION);
}

}  // namespace avk
