// avk_lib.cu -- kernels and the C ABI of libaardvark_b200.so (include/aardvark_b200.h).
//
// Kernels (all sm_100a, no tensor cores -- integer DP):
//   k_alt_ed       per-variant ED(allele0, allele1)           variants.rs:413-415 (alt_ed)
//   k_compare      one warp per cluster, persistent warps     waffle_solver.rs:122-284
//   k_merge        one warp per cluster                       merge_solver.rs:110-200
//   k_wfa_ed       one warp per alignment                     util/sequence_alignment.rs:9-13
//   k_reduce       sum of per-region metrics                  writers/summary.rs:146-158
//
// There is NO CPU fallback in this library: every entry point either runs the CUDA path or
// returns an error code.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <chrono>
#include <thread>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_run_length_encode.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "avk_solver.cuh"
#include "avk_thread_solver.cuh"
#include "avk_writers.h"
#include "avk_vcf.cuh"
#include "avk_inflate.cuh"

using namespace avk;

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                         \
            return (e_ == cudaErrorMemoryAllocation) ? AVK_ERR_OOM : AVK_ERR_CUDA;                 \
        }                                                                                          \
    } while (0)

// ------------------------------------------------------------------------------------ kernels

// Flush the per-warp work counters kept in an arena / scratch header (WK_* offsets) to the global totals.
template <bool SMEM>
__device__ __forceinline__ void flush_work(typename Mem<SMEM>::addr hdr, unsigned long long *out) {
    typedef Mem<SMEM> M;
    if (lane_id() == 0 && out) {
        const u64 cells = LD64(hdr + WK_CELLS), matched = LD64(hdr + WK_MATCHED);
        const u32 al = LD32(hdr + WK_ALIGN), sp = LD32(hdr + WK_SPOPS), xp = LD32(hdr + WK_XPOPS);
        if (al) atomicAdd(out + 0, (unsigned long long)al);
        if (cells) atomicAdd(out + 1, (unsigned long long)cells);
        if (matched) atomicAdd(out + 2, (unsigned long long)matched);
        if (sp) atomicAdd(out + 3, (unsigned long long)sp);
        if (xp) atomicAdd(out + 4, (unsigned long long)xp);
    }
}
template <bool SMEM>
__device__ __forceinline__ void clear_work(typename Mem<SMEM>::addr hdr) {
    typedef Mem<SMEM> M;
    const int lane = lane_id();
    if (lane < 10) ST32(hdr + 8 + 4 * lane, 0);   // WK_COOP and the counters
    __syncwarp();
}

// per-warp scratch of the two alignment kernels: [ARENA_HDR bytes header | wavefront ints]
__device__ __forceinline__ VSeq<false> plain_seq(const u8 *p, int n) {
    VSeq<false> v;
    v.data = (u64)(uintptr_t)p; v.tail = v.data + (u64)n; v.mlen = n; v.len = n;
    return v;
}

// alt_ed: 32 variants per warp pass; SNVs are answered by their lane, everything else is aligned
// warp-cooperatively (prefix shortcut for pure insertions/deletions, WFA otherwise).
// Variants [v_base, v_base + n_variants) of the caller's table are resident (a contiguous bin of regions); every per-variant
// device pointer is biased so that it is indexed with the caller's (global) variant index.
__global__ void __launch_bounds__(256) k_alt_ed(DevBatch b, u64 v_base, u64 n_variants, u32 *alt_ed, u8 *scratch, int scratch_ints,
                                                unsigned long long *work_out) {
    const int lane = lane_id();
    const u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const u64 n_warps = ((u64)gridDim.x * blockDim.x) >> 5;
    const u64 hdr = (u64)(uintptr_t)(scratch + warp * ((u64)scratch_ints * 4 + ARENA_HDR));
    clear_work<false>(hdr);
    for (u64 base = v_base + warp * 32; base < v_base + n_variants; base += n_warps * 32) {
        const u64 v = base + lane;
        bool coop = false;
        if (v < v_base + n_variants) {
            const u32 l0 = b.l0[v], l1 = b.l1[v];
            if (l0 == 1 && l1 == 1) alt_ed[v] = (b.pool[b.aoff[v]] != b.pool[b.aoff[v] + 1]) ? 1u : 0u;
            else coop = true;
        }
        unsigned m = __ballot_sync(AVK_FULL, coop);
        while (m) {
            const int src = __ffs(m) - 1;
            m &= m - 1;
            const u64 vv = base + src;
            const int l0 = (int)b.l0[vv], l1 = (int)b.l1[vv];
            const u8 *a0 = b.pool + b.aoff[vv];
            const u8 *a1 = a0 + l0;
            int ed;
            const int mn = min(l0, l1);
            if (mn == 0) ed = max(l0, l1);
            else if (2 * max(l0, l1) + 3 > scratch_ints) ed = 0;   // cannot happen: host sizes scratch by the max allele
            else {
                const int p = raw_lcp<false>((u64)(uintptr_t)a0, (u64)(uintptr_t)a1, mn);
                if (p == mn) ed = max(l0, l1) - mn;                // one allele is a prefix of the other
                else {
                    ed = wfa_ed_warp<false>(plain_seq(a0, l0), plain_seq(a1, l1), hdr + ARENA_HDR, (scratch_ints - 3) / 2, hdr);
                    if (ed < 0) ed = 0;
                }
            }
            if (lane == 0) alt_ed[vv] = (u32)ed;
        }
    }
    flush_work<false>(hdr, work_out);
}

__global__ void __launch_bounds__(256) k_wfa_ed(const u32 *list, const u32 *n_list, const u8 *pool, const u64 *a_off, const u32 *a_len,
                                                const u64 *b_off, const u32 *b_len, u32 *ed_out, u8 *scratch,
                                                int scratch_ints, u32 *counter, unsigned long long *work_out) {
    const int lane = lane_id();
    const u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const u64 hdr = (u64)(uintptr_t)(scratch + warp * ((u64)scratch_ints * 4 + ARENA_HDR));
    clear_work<false>(hdr);
    const u32 n_pairs = *n_list;
    for (;;) {
        u32 p = 0;
        if (lane == 0) p = atomicAdd(counter, 1u);
        p = __shfl_sync(AVK_FULL, p, 0);
        if (p >= n_pairs) break;
        p = list[p];
        const int ed = wfa_ed_warp<false>(plain_seq(pool + a_off[p], (int)a_len[p]), plain_seq(pool + b_off[p], (int)b_len[p]),
                                          hdr + ARENA_HDR, (scratch_ints - 3) / 2, hdr);
        if (lane == 0) ed_out[p] = (u32)ed;
    }
    flush_work<false>(hdr, work_out);
}

// Long pairs: one alignment per CTA, advanced by all COOP_THREADS threads (coop_dwfa_body: sequences staged in shared memory,
// 16-bit wavefront).  Thread 0 posts the job; if the wavefront outgrows shared memory warp 0 finishes it on the warp path.
__global__ void __launch_bounds__(COOP_THREADS, 1) k_wfa_ed_cta(const u32 *list, const u32 *n_list, const u8 *pool, const u64 *a_off, const u32 *a_len,
                                                                const u64 *b_off, const u32 *b_len, u32 *ed_out, u8 *scratch, int scratch_ints,
                                                                int cap_ints, u32 *counter, unsigned long long *work_out) {
    __shared__ u32 s_idx;
    CoopJob &J = *(CoopJob *)avk_dyn_smem;
    const u64 hdr = (u64)(uintptr_t)(scratch + (u64)blockIdx.x * ((u64)scratch_ints * 4 + ARENA_HDR));
    if (threadIdx.x < 32) clear_work<false>(hdr);
    const u32 n = *n_list;
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) s_idx = atomicAdd(counter, 1u);
        __syncthreads();
        const u32 idx = s_idx;
        if (idx >= n) break;
        const u32 p = list[idx];
        if (threadIdx.x == 0) {
            int *gw = (int *)(uintptr_t)(hdr + ARENA_HDR);
            gw[0] = 0;
            J.wf = hdr + ARENA_HDR;
            J.a_data = (u64)(uintptr_t)(pool + a_off[p]); J.a_mlen = J.a_len = (int)a_len[p]; J.a_tail = J.a_data + a_len[p];
            J.b_data = (u64)(uintptr_t)(pool + b_off[p]); J.b_mlen = J.b_len = (int)b_len[p]; J.b_tail = J.b_data + b_len[p];
            J.ed = 0; J.max_ed = 0x7ffffff0; J.to_full = 1; J.status = 0; J.exit_ = 0; J.matched = 0; J.cells = 0; J.cap_ints = cap_ints;
        }
        __threadfence();
        __syncthreads();
        coop_dwfa_body();
        int ed = J.ed;
        const int st = J.status;
        if (threadIdx.x < 32) {
            if (st == DWFA_COOP_SPILL) {                                   // wavefront outgrew shared memory: finish on the warp path
                const int rc = dwfa_run<false>(hdr + ARENA_HDR, &ed, (scratch_ints - 3) / 2, plain_seq(pool + a_off[p], (int)a_len[p]),
                                               plain_seq(pool + b_off[p], (int)b_len[p]), true, hdr);
                if (rc != DWFA_OK) ed = -1;
            }
            if (threadIdx.x == 0) {
                ed_out[p] = (u32)ed;
                *(u64 *)(uintptr_t)(hdr + WK_CELLS) += J.cells; *(u64 *)(uintptr_t)(hdr + WK_MATCHED) += J.matched; *(u32 *)(uintptr_t)(hdr + WK_ALIGN) += 1;
            }
        }
    }
    if (threadIdx.x < 32) flush_work<false>(hdr, work_out);
}

// splits the pairs of a wfa_ed batch: long pairs go to the CTA-wide kernel, the rest to one warp each
__global__ void __launch_bounds__(256) k_wfa_split(u64 n_pairs, const u32 *a_len, const u32 *b_len, u32 long_min, u32 max_sum, u32 *list_warp, u32 *n_warp,
                                                   u32 *list_cta, u32 *n_cta) {
    const u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pairs) return;
    const u32 la = a_len[p], lb = b_len[p];
    const bool cta = min(la, lb) >= long_min && (u64)la + lb + 4096 <= max_sum && max(la, lb) < 60000u;
    if (cta) list_cta[atomicAdd(n_cta, 1u)] = (u32)p; else list_warp[atomicAdd(n_warp, 1u)] = (u32)p;
}

// ---- cluster digests (compare path) -------------------------------------------------------------------------
// k_prep_size / scan / k_prep_fill turn every cluster into one contiguous, 16-byte aligned blob:
//   [PH_* header 64 B][N variant records of 32 B in merged processing order][allele bytes]
// i.e. everything RegionSolver::setup_pair derives (validation, order_variants, per-type metric slots).  The solver
// kernels then fetch a cluster with one TMA bulk copy instead of re-deriving it with dependent global loads.
__global__ void __launch_bounds__(256) k_prep_size(DevBatch b, u64 n, u64 *sizes) {
    const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r > n) return;
    if (r == n) { sizes[r] = 0; return; }
    const u64 v0 = b.var_off[r * 2], v1 = b.var_off[r * 2 + 2];
    u64 alle = 0;
    for (u64 v = v0; v < v1; ++v) alle += (u64)min(b.l0[v], 1u << 24) + (u64)min(b.l1[v], 1u << 24);
    sizes[r] = (PH_SIZE + VI_SIZE * (v1 - v0) + alle + 16 + 15) & ~15ull;
}

__global__ void __launch_bounds__(256) k_prep_fill(DevBatch b, u64 n_all, const u64 *offs, u8 *digest, const u32 *list, const u32 *n_list) {
    const int lane = lane_id();
    const u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const u64 n_warps = ((u64)gridDim.x * blockDim.x) >> 5;
    const u64 n = list ? (u64)*n_list : n_all;
    for (u64 ri = warp; ri < n; ri += n_warps) {
        const u64 r = list ? (u64)list[ri] : ri;
        u8 *dig = digest + offs[r];
        int *hdr = (int *)dig;
        const long long start = b.start[r], end = b.end[r];
        const u64 v0[2] = {b.var_off[r * 2], b.var_off[r * 2 + 1]};
        const int cnt[2] = {(int)(b.var_off[r * 2 + 1] - v0[0]), (int)(b.var_off[r * 2 + 2] - v0[1])};
        const int N = cnt[0] + cnt[1];
        // validation (same rules as the oracle's list_valid) + the sums that size the solver workspace
        bool invalid = false;
        int s_l1 = 0, s_b0 = 0, s_al = 0, mx = (int)min(start, 0x7fffffffLL);
        for (int side = 0; side < 2; ++side) {
            for (int i = lane; i < cnt[side]; i += 32) {
                const u64 gv = v0[side] + i;
                const u32 l0 = b.l0[gv], l1 = b.l1[gv], p = b.pos[gv];
                invalid = invalid || l0 == 0 || l1 == 0 || b.vtype[gv] >= AVK_N_VARIANT_TYPES || b.zyg[gv] > AVK_ZYG_HOM_ALT;
                invalid = invalid || (long long)p < start || (long long)p + l0 > end;
                if (i > 0) invalid = invalid || b.pos[gv - 1] > p;
                s_l1 += (int)min(l1, 1u << 24);
                s_b0 += (int)min(max(l0, l1), 1u << 24);
                s_al += (int)min(l0, 1u << 24) + (int)min(l1, 1u << 24);
                mx = max(mx, (int)min(p + l0, 0x7fffffffu));
            }
        }
        invalid = __any_sync(AVK_FULL, invalid);
        s_l1 = __reduce_add_sync(AVK_FULL, s_l1); s_b0 = __reduce_add_sync(AVK_FULL, s_b0);
        s_al = __reduce_add_sync(AVK_FULL, s_al); mx = __reduce_max_sync(AVK_FULL, mx);
        if (invalid) {
            if (lane < PH_SIZE / 4) hdr[lane] = lane == 0 ? AVK_ST_BAD_INPUT : 0;
            continue;
        }
        // merged order: stable, truth before query on equal positions (order_variants, query_optimizer.rs:372-381)
        u8 *recs = dig + PH_SIZE;
        for (int side = 0; side < 2; ++side) {
            const int nm = cnt[side], no = cnt[side ^ 1];
            const u64 vm = v0[side], vo = v0[side ^ 1];
            for (int i = lane; i < nm; i += 32) {
                const u64 gv = vm + i;
                const u32 p = b.pos[gv];
                int lo = 0, hi = no;
                while (lo < hi) {
                    const int m = (lo + hi) >> 1;
                    const u32 pm = b.pos[vo + m];
                    const bool before = side == 0 ? (pm < p) : (pm <= p);
                    if (before) lo = m + 1; else hi = m;
                }
                u32 *rec = (u32 *)(recs + (size_t)VI_SIZE * (i + lo));
                rec[VI_POS / 4] = p; rec[VI_L0 / 4] = b.l0[gv]; rec[VI_L1 / 4] = b.l1[gv]; rec[VI_AOFF / 4] = b.aoff[gv];
                rec[VI_ALTED / 4] = b.alt_ed[gv]; rec[VI_RAW / 4] = b.raw[gv]; rec[VI_GV / 4] = (u32)gv;
                rec[VI_FLAGS / 4] = (u32)b.vtype[gv] | ((u32)b.zyg[gv] << 8) | ((side == 0 ? 1u : 0u) << 16);
            }
        }
        __syncwarp();
        // allele bytes in merged order; VI_AOFF becomes the offset inside the digest's allele area
        u8 *alle = recs + (size_t)VI_SIZE * N;
        u32 seen = 0;
        int acc = 0;
        for (int oi = 0; oi < N; ++oi) {
            u32 *rec = (u32 *)(recs + (size_t)VI_SIZE * oi);
            const int na = (int)(rec[VI_L0 / 4] + rec[VI_L1 / 4]);
            const u8 *src = b.pool + rec[VI_AOFF / 4];
            for (int i = lane; i < na; i += 32) alle[acc + i] = src[i];
            seen |= 1u << (rec[VI_FLAGS / 4] & 0xff);
            __syncwarp();
            if (lane == 0) rec[VI_AOFF / 4] = (u32)acc;
            acc += na;
        }
        __syncwarp();
        // metric-row slots: one per distinct variant type, in type order
        for (int oi = lane; oi < N; oi += 32) {
            u32 *rec = (u32 *)(recs + (size_t)VI_SIZE * oi);
            const u32 f = rec[VI_FLAGS / 4];
            rec[VI_FLAGS / 4] = f | ((u32)__popc(seen & ((1u << (f & 0xff)) - 1)) << 24);
        }
        if (lane == 0) {
            hdr[PH_STATUS / 4] = AVK_ST_OK; hdr[PH_N / 4] = N; hdr[PH_N0 / 4] = cnt[0]; hdr[PH_N1 / 4] = cnt[1];
            hdr[PH_SUM_L1 / 4] = s_l1; hdr[PH_B0 / 4] = s_b0; hdr[PH_SUM_ALLE / 4] = s_al; hdr[PH_MAX_END / 4] = mx;
            hdr[PH_NSLOTS / 4] = __popc(seen);
            int k = 0;
            for (int t = 0; t < AVK_N_VARIANT_TYPES; ++t) if (seen & (1u << t)) dig[PH_SLOT_TYPE + (k++)] = (u8)t;
        }
    }
}

// k_prep_fill for the common small cluster, one THREAD per cluster (a warp per two-variant cluster leaves 30 lanes idle and
// serialises on its shuffles): same digest, byte for byte.  Clusters with more than PREP_SMALL_N variants are appended to
// `big` and take the warp kernel.
enum { PREP_SMALL_N = 12 };
__global__ void __launch_bounds__(256) k_prep_fill_small(DevBatch b, u64 n, const u64 *offs, u8 *digest, u32 *big, u32 *big_ctr) {
    const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const u64 v0 = b.var_off[r * 2], vq = b.var_off[r * 2 + 1], v1 = b.var_off[r * 2 + 2];
    const int nT = (int)(vq - v0), nQ = (int)(v1 - vq), N = nT + nQ;
    if (N > PREP_SMALL_N) { big[atomicAdd(big_ctr, 1u)] = (u32)r; return; }
    u8 *dig = digest + offs[r];
    const long long start = b.start[r], end = b.end[r];
    bool invalid = false;
    int s_l1 = 0, s_b0 = 0, s_al = 0, mx = (int)min(start, 0x7fffffffLL);
    u32 seen = 0;
    for (u64 gv = v0; gv < v1; ++gv) {
        const u32 l0 = b.l0[gv], l1 = b.l1[gv], p = b.pos[gv], ty = b.vtype[gv];
        invalid = invalid || l0 == 0 || l1 == 0 || ty >= AVK_N_VARIANT_TYPES || b.zyg[gv] > AVK_ZYG_HOM_ALT;
        invalid = invalid || (long long)p < start || (long long)p + l0 > end;
        if (gv != v0 && gv != vq) invalid = invalid || b.pos[gv - 1] > p;
        s_l1 += (int)min(l1, 1u << 24); s_b0 += (int)min(max(l0, l1), 1u << 24); s_al += (int)min(l0, 1u << 24) + (int)min(l1, 1u << 24);
        mx = max(mx, (int)min(p + l0, 0x7fffffffu));
        seen |= 1u << (ty & 31u);
    }
    uint4 *h4 = (uint4 *)dig;
    if (invalid) {
        h4[0] = make_uint4((u32)AVK_ST_BAD_INPUT, 0, 0, 0); h4[1] = make_uint4(0, 0, 0, 0); h4[2] = make_uint4(0, 0, 0, 0); h4[3] = make_uint4(0, 0, 0, 0);
        return;
    }
    // merged order: stable, truth before query on equal positions (order_variants, query_optimizer.rs:372-381)
    u8 *recs = dig + PH_SIZE, *alle = recs + (size_t)VI_SIZE * N;
    u64 it = v0, iq = vq;
    u32 acc = 0;
    for (int oi = 0; oi < N; ++oi) {
        const bool take_t = it < vq && (iq >= v1 || b.pos[it] <= b.pos[iq]);
        const u64 gv = take_t ? it : iq;
        if (take_t) ++it; else ++iq;
        const u32 l0 = b.l0[gv], l1 = b.l1[gv], ty = b.vtype[gv];
        uint4 *rec = (uint4 *)(recs + (size_t)VI_SIZE * oi);
        rec[0] = make_uint4(b.pos[gv], l0, l1, acc);
        rec[1] = make_uint4(b.alt_ed[gv], b.raw[gv], (u32)gv,
                            ty | ((u32)b.zyg[gv] << 8) | ((take_t ? 1u : 0u) << 16) | ((u32)__popc(seen & ((1u << ty) - 1)) << 24));
        const u8 *src = b.pool + b.aoff[gv];
        for (u32 k = 0; k < l0 + l1; ++k) alle[acc + k] = src[k];
        acc += l0 + l1;
    }
    h4[0] = make_uint4((u32)AVK_ST_OK, (u32)N, (u32)nT, (u32)nQ);
    h4[1] = make_uint4((u32)s_l1, (u32)s_b0, (u32)s_al, (u32)mx);
    u32 st[4] = {0, 0, 0, 0};
    int k = 0;
    for (int ty = 0; ty < AVK_N_VARIANT_TYPES; ++ty) if (seen & (1u << ty)) { st[k >> 2] |= (u32)ty << (8 * (k & 3)); ++k; }
    h4[2] = make_uint4((u32)__popc(seen), st[0], st[1], st[2]);
    h4[3] = make_uint4(0, 0, 0, 0);
}

__device__ __forceinline__ void zero_region_outputs(const DevBatch &b, const DevCompareOut &out, u64 r, bool metrics_only) {
    const int lane = lane_id();
    if (out.region_metrics) {
        u64 *gm = out.region_metrics + r * (u64)(AVK_N_GROUPS * AVK_N_METRICS);
        for (int i = lane; i < AVK_N_GROUPS * AVK_N_METRICS; i += 32) gm[i] = 0;
    }
    if (!metrics_only) {
        const u64 v0 = b.var_off[r * 2], v1 = b.var_off[r * 2 + 2];
        for (u64 v = v0 + lane; v < v1; v += 32) { out.vexp[v] = 0; out.vobs[v] = 0; out.vcls[v] = AVK_CLASS_UNKNOWN; }
        if (lane == 0) { out.ed1[r] = 0; out.ed2[r] = 0; out.type_mask[r] = 0; }
        if (out.seq_off && lane < 5) out.seq_len[r * 5 + lane] = 0;
    }
    __syncwarp();
}

// ---- closed form for the commonest cluster shape ------------------------------------------------------------
// One truth and one query record that are the same variant -- same position, reference span, ALT bytes, (supported) type
// label and number of ALT copies -- where the variant is a substitution that changes the base, or an anchored pure
// insertion / deletion (first ALT base == the reference base); or TWO such pairs of substitutions at increasing positions:
// ~80 % of a small-variant WGS comparison.  What solve_compare_region computes for them follows from the search itself
// (query_optimizer.rs:203-328): the orientation(s) in which both haplotypes spell identical sequences finalise with cost
// 0 -- the search tree has at most 4 (one pair) or 16 (two pairs) nodes per depth, hence max_branch_factor >= 4 / 16 so
// that the branch quota never drops one; every other orientation pairs two different strings on some haplotype and costs
// more.  So each equal-best result has ED 0, no skipped variant and expected == observed == ALT copies for every record,
// whichever of them comes first.  Metrics: gt/hap/weighted_hap TP on both sides (grouped_metrics.rs:183-227); basepair
// X = Y = ED(reference window, haplotype), Z = 0 (waffle_solver.rs:639-648), where the sum of X over the two haplotypes
// is the same for every equal-best result: 1 per copy of a substitution (a haplotype with two of them has Hamming
// distance 2 = ED 2 to the window), the length difference per copy of an anchored indel (closed forms of
// RegionSolver::build_hap_seq); record basepair 2 * copies * raw_allele_space (:455-522; needs raw >= X, else the
// general path reports the underflow).  Everything else -- including these shapes with the hidden exact shortcut or the
// sequence bundle requested -- goes to the search kernels through `work_list`.
// Clusters with at least `dense_n` variants skip the search / score pair: they go to list `dense`, which the fused
// stage starts on first (the longest searches of a batch are among them).
__global__ void __launch_bounds__(256) k_compare_simple(DevBatch b, DevCompareOut out, avk_compare_cfg cfg, u64 n, u32 *work_list,
                                                        u32 *work_ctr, u32 *dense, u32 *dense_ctr, int dense_n, u64 *work_key) {
    const int lane = lane_id();
    const u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const u64 n_warps = ((u64)gridDim.x * blockDim.x) >> 5;
    const bool enabled = !cfg.enable_exact_shortcut && !(out.seq_off && cfg.enable_sequences) && cfg.max_branch_factor >= 4;
    const u32 supported = (1u << AVK_VT_SNV) | (1u << AVK_VT_INSERTION) | (1u << AVK_VT_DELETION) | (1u << AVK_VT_INDEL) |
                          (1u << AVK_VT_TR_CONTRACTION) | (1u << AVK_VT_TR_EXPANSION) | (1u << AVK_VT_SV_DELETION) | (1u << AVK_VT_SV_INSERTION);
    for (u64 base = warp * 32; base < n; base += n_warps * 32) {
        const u64 r = base + lane;
        bool simple = false;
        int nvar = 0, npairs = 0;
        u32 gv[4] = {0, 0, 0, 0}, cp[2] = {0, 0}, vtype = 0;
        u64 s_c = 0, s_wT = 0, s_wQ = 0, s_X = 0, s_rT = 0, s_rQ = 0;   // sums over the pairs, each weighted by its ALT copies
        if (r < n) {
            const u8 *dig = b.digest + b.digest_off[r];
            const int4 h = *(const int4 *)dig;                         // status, N, nT, nQ
            const u32 c = b.contig[r];
            nvar = h.x == AVK_ST_OK ? h.y : 0;
            const int M = (h.y == 2 && h.z == 1 && h.w == 1) ? 1 : ((h.y == 4 && h.z == 2 && h.w == 2) ? 2 : 0);
            if (enabled && h.x == AVK_ST_OK && M && (M == 1 || cfg.max_branch_factor >= 16) && c < b.n_contigs && b.start[r] <= b.end[r] &&
                (u64)b.end[r] <= b.contig_len[c] && b.end[r] <= 0x7fff0000u) {
                const u8 *alle = dig + PH_SIZE + 2 * M * VI_SIZE;
                bool ok = true;
                u32 prev_pos = 0;
                for (int m = 0; m < M && ok; ++m) {
                    const u8 *rt = dig + PH_SIZE + 2 * m * VI_SIZE, *rq = rt + VI_SIZE;      // merged order: truth before query on ties
                    const uint4 t0 = *(const uint4 *)rt, t1 = *(const uint4 *)(rt + 16), q0 = *(const uint4 *)rq, q1 = *(const uint4 *)(rq + 16);
                    // t0 = {pos, l0, l1, aoff}, t1 = {alt_ed, raw, gv, flags}
                    const u32 zT = (t1.w >> 8) & 0xff, zQ = (q1.w >> 8) & 0xff;
                    const u32 cT = zT == AVK_ZYG_HOM_ALT ? 2u : (zT >= AVK_ZYG_UNPHASED_HET ? 1u : 0u);
                    const u32 cQ = zQ == AVK_ZYG_HOM_ALT ? 2u : (zQ >= AVK_ZYG_UNPHASED_HET ? 1u : 0u);
                    const u32 ty = t1.w & 0xffu;
                    // same record on both sides: position, reference span, ALT bytes, type label (a supported one), ALT copies
                    ok = (t1.w & 0x10000u) && !(q1.w & 0x10000u) && ty == (q1.w & 0xffu) && ((supported >> ty) & 1u) && t0.x == q0.x &&
                         t0.y == q0.y && t0.z == q0.z && (t0.y == 1 || t0.z == 1) && t0.y + t0.z <= 64 && cT != 0 && cT == cQ;
                    // two pairs: substitutions only, at increasing positions (the Hamming argument below needs equal lengths)
                    if (M == 2) ok = ok && t0.y == 1 && t0.z == 1 && ty == AVK_VT_SNV && (m == 0 || t0.x > prev_pos);
                    if (!ok) break;
                    const u8 *aT = alle + t0.w + t0.y, *aQ = alle + q0.w + q0.y;   // ALT alleles
                    for (u32 k = 0; k < t0.z; ++k) ok = ok && aT[k] == aQ[k];
                    const bool anchored = aT[0] == b.contig_ptr[c][t0.x];
                    // ED(reference window, ALT haplotype): a substitution that changes the base: 1 (two of them on one
                    // haplotype: Hamming 2 = ED 2); anchored pure insertion / deletion: the length difference
                    // (RegionSolver::build_hap_seq, SD_CLOSED)
                    u32 X = 0;
                    if (t0.y == 1 && t0.z == 1) X = anchored ? 0u : 1u;
                    else if (anchored) X = (t0.y == 1 ? t0.z : t0.y) - 1u;
                    ok = ok && X != 0 && t1.y >= X && q1.y >= X;
                    gv[2 * m] = t1.z; gv[2 * m + 1] = q1.z; cp[m] = cT; vtype = ty; prev_pos = t0.x;
                    s_c += cT; s_wT += (u64)cT * t1.x; s_wQ += (u64)cT * q1.x; s_X += (u64)cT * X; s_rT += (u64)cT * t1.y; s_rQ += (u64)cT * q1.y;
                }
                simple = ok;
                npairs = M;
            }
        }
        // everything else: compact list for the search / score kernels (cluster order kept inside a warp's chunk)
        const bool is_dense = r < n && !simple && nvar >= dense_n;
        const u32 rest = __ballot_sync(AVK_FULL, r < n && !simple && !is_dense);
        const u32 dn = __ballot_sync(AVK_FULL, is_dense);
        u32 pos0 = 0, pos1 = 0;
        if (lane == 0 && rest) pos0 = atomicAdd(work_ctr, (u32)__popc(rest));
        if (lane == 0 && dn) pos1 = atomicAdd(dense_ctr, (u32)__popc(dn));
        pos0 = __shfl_sync(AVK_FULL, pos0, 0);
        pos1 = __shfl_sync(AVK_FULL, pos1, 0);
        if (r < n && !simple && !is_dense) {
            const u32 slot_ = pos0 + __popc(rest & ((1u << lane) - 1));
            work_list[slot_] = (u32)r;
            if (work_key) {
                // SHAPE of the cluster: per order entry {side, zygosity, same position as the previous entry, allele-length class}.
                // Clusters of the same shape run (nearly) the same control flow in the thread-per-cluster stage; the list is
                // sorted by this key so that the 32 lanes of a warp get clusters of one shape.
                u64 key = 0;
                const int *dh = (const int *)(b.digest + b.digest_off[r]);
                // heaviest first (a thread is a slow serial machine: what takes thousands of wavefront steps must not start
                // last): weight ~ variants x (edit-distance bound + 1)^2, in powers of two
                const u32 edb = (u32)min(max(dh[PH_B0 / 4], 0), 16);
                const u32 wgt = (u32)max(nvar, 1) * (edb + 1u) * (edb + 1u);
                const u32 heavy = min(15u, (u32)(31 - __clz((int)max(wgt, 1u))));
                if (nvar > 0 && nvar <= 9) {
                    const u8 *recs = b.digest + b.digest_off[r] + PH_SIZE;
                    u32 prev = 0xffffffffu;
                    for (int oi = 0; oi < nvar; ++oi) {
                        const uint4 a = *(const uint4 *)(recs + (size_t)VI_SIZE * oi);          // pos, l0, l1, aoff
                        const u32 f = *(const u32 *)(recs + (size_t)VI_SIZE * oi + VI_FLAGS);
                        const u32 lc = (a.y == 1 && a.z == 1) ? 0u : (a.y == 1 ? 1u : (a.z == 1 ? 2u : 3u));
                        const u32 code = ((f >> 16) & 1u) | ((((f >> 8) & 0xffu) & 3u) << 1) | ((a.x == prev ? 1u : 0u) << 3) | (lc << 4);
                        key = (key << 6) | code;
                        prev = a.x;
                    }
                    key |= (u64)nvar << 54;
                } else key = (u64)min(nvar, 15) << 54;
                key |= (u64)(15u - heavy) << 58;
                work_key[slot_] = key;
            }
        }
        if (is_dense) dense[pos1 + __popc(dn & ((1u << lane) - 1))] = (u32)r;
        if (simple) {
            out.status[r] = AVK_ST_OK; out.ed1[r] = 0; out.ed2[r] = 0; out.type_mask[r] = (uint16_t)supported;   // vtype is one of them
            for (int m = 0; m < npairs; ++m) {
                out.vexp[gv[2 * m]] = (u8)cp[m]; out.vobs[gv[2 * m]] = (u8)cp[m]; out.vcls[gv[2 * m]] = AVK_CLASS_TP;
                out.vexp[gv[2 * m + 1]] = (u8)cp[m]; out.vobs[gv[2 * m + 1]] = (u8)cp[m]; out.vcls[gv[2 * m + 1]] = AVK_CLASS_TP;
            }
        }
        // summary counters (in-kernel totals): one warp reduction per variant type present among this warp's closed-form
        // clusters; the joint row of such a cluster equals its (single) type's row
        if (out.tot_slots) {
            unsigned long long *slot = out.tot_slots + (size_t)(blockIdx.x & (TOT_SLOTS - 1)) * TOT_STRIDE;
            u32 left = __ballot_sync(AVK_FULL, simple);
            while (left) {
                const u32 ty = __shfl_sync(AVK_FULL, vtype, __ffs(left) - 1);
                const bool in = simple && vtype == ty;
                const u32 same = __ballot_sync(AVK_FULL, in);
                left &= ~same;
                unsigned long long v[7] = {(unsigned long long)npairs, (unsigned long long)s_c, (unsigned long long)s_wT, (unsigned long long)s_wQ,
                                           2ull * s_X, 2ull * s_rT, 2ull * s_rQ};
#pragma unroll
                for (int k = 0; k < 7; ++k) {
                    if (!in) v[k] = 0;
#pragma unroll
                    for (int o = 16; o; o >>= 1) v[k] += __shfl_xor_sync(AVK_FULL, v[k], o);
                }
                if (lane < 2) {                                          // lane 0: joint row, lane 1: the type's row
                    unsigned long long *g = slot + (lane == 0 ? 0 : (1 + ty) * AVK_N_METRICS);
                    atomicAdd(g + AVK_M_GT, v[0]); atomicAdd(g + AVK_M_GT + 2, v[0]);
                    atomicAdd(g + AVK_M_HAP, v[1]); atomicAdd(g + AVK_M_HAP + 2, v[1]);
                    atomicAdd(g + AVK_M_WEIGHTED_HAP, v[2]); atomicAdd(g + AVK_M_WEIGHTED_HAP + 2, v[3]);
                    atomicAdd(g + AVK_M_BASEPAIR, v[4]); atomicAdd(g + AVK_M_BASEPAIR + 2, v[4]);
                    atomicAdd(g + AVK_M_RECORD_BP, v[5]); atomicAdd(g + AVK_M_RECORD_BP + 2, v[6]);
                    if (lane == 0) { atomicAdd(slot + TOT_SOLVED, (unsigned long long)__popc(same)); atomicOr(slot + TOT_MASK, (unsigned long long)supported); }
                }
            }
        }
        // metric rows [13][22] (only when the caller wants per-region rows or strata), written by the whole warp per
        // cluster: joint row == the (single) type's row, the rest zero
        u32 todo = out.region_metrics ? __ballot_sync(AVK_FULL, simple) : 0u;
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const u64 vM = (u64)__shfl_sync(AVK_FULL, npairs, src), vc = __shfl_sync(AVK_FULL, (unsigned long long)s_c, src);
            const u64 vwT = __shfl_sync(AVK_FULL, (unsigned long long)s_wT, src), vwQ = __shfl_sync(AVK_FULL, (unsigned long long)s_wQ, src);
            const u64 vrT = __shfl_sync(AVK_FULL, (unsigned long long)s_rT, src), vrQ = __shfl_sync(AVK_FULL, (unsigned long long)s_rQ, src);
            const u64 vX = __shfl_sync(AVK_FULL, (unsigned long long)s_X, src);
            const int grow = 1 + (int)__shfl_sync(AVK_FULL, vtype, src);
            u64 *dst = out.region_metrics + (base + src) * (u64)(AVK_N_GROUPS * AVK_N_METRICS);
#pragma unroll 1
            for (int i = lane; i < AVK_N_GROUPS * AVK_N_METRICS; i += 32) {
                const int g = i / AVK_N_METRICS, m = i - g * AVK_N_METRICS;
                u64 v = 0;
                if (g == 0 || g == grow) {
                    if (m == AVK_M_GT || m == AVK_M_GT + 2) v = vM;
                    else if (m == AVK_M_HAP || m == AVK_M_HAP + 2) v = vc;
                    else if (m == AVK_M_WEIGHTED_HAP) v = vwT;
                    else if (m == AVK_M_WEIGHTED_HAP + 2) v = vwQ;
                    else if (m == AVK_M_BASEPAIR || m == AVK_M_BASEPAIR + 2) v = 2 * vX;
                    else if (m == AVK_M_RECORD_BP) v = 2 * vrT;
                    else if (m == AVK_M_RECORD_BP + 2) v = 2 * vrQ;
                }
                dst[i] = v;
            }
        }
    }
}

// final status of a region that ends in an error: counted as an error block (main.rs:259-262, summary.rs:161-163)
__device__ __forceinline__ void count_error_block(const DevCompareOut &out) {
    if (out.tot_slots) atomicAdd(out.tot_slots + (size_t)(blockIdx.x & (TOT_SLOTS - 1)) * TOT_STRIDE + TOT_ERRORS, 1ull);
}

// totals[j] = sum (type mask: OR) over the partial tables; layout [13][22] sums, type mask, solved blocks, error blocks
__global__ void __launch_bounds__(320) k_fold_slots(const unsigned long long *slots, unsigned long long *totals) {
    const int j = threadIdx.x;
    if (j >= TOT_COLS + 3) return;
    unsigned long long acc = 0;
    for (int s = 0; s < TOT_SLOTS; ++s) {
        const unsigned long long v = slots[(size_t)s * TOT_STRIDE + j];
        acc = (j == TOT_MASK) ? (acc | v) : (acc + v);
    }
    totals[j] = acc;
}

// Work distribution of one stage.  work_ctr = work counter of this launch, fail_ctr = number of clusters
// that did not fit (appended to fail_list, re-run by a later stage).  n_work is read from device memory
// when n_work_ptr is set, so that stages can be chained without a host round trip.
struct TierArgs {
    const u32 *work_list;
    const u32 *n_work_ptr;
    const u32 *work_list2;   // optional second list, consumed after the first (length *n_work_ptr2)
    const u32 *n_work_ptr2;
    u32 *fail_list2;         // optional: rejected clusters with >= dense_n variants go here instead of fail_list
    u32 *fail_ctr2;
    int dense_n;
    u32 n_work;
    u32 *work_ctr;
    u32 *fail_ctr;
    u8 *arena_base;        // global tiers
    long long arena_bytes; // per warp
    u32 *fail_list;
    int last_tier;
    unsigned long long *work_out;
    u8 *blobs;             // split tier: [n_regions][RB_SIZE] search results handed to the score kernel
    int wide_b0;           // global stages: hand clusters with an edit-distance bound >= wide_b0 to the next (cooperative) stage
    u8 *spill_base;        // shared-memory stages: per-warp node spill area in global memory (may be NULL)
    u32 spill_bytes;       // per warp
    int n_lo, n_hi;        // stages that scan all regions only take clusters with n_lo <= #variants <= n_hi
    int pop_budget;        // thread stage: queue pops a thread spends on one cluster before it hands it on
    int batch_min;         // thread stage: lanes that must be waiting for a kind of bookkeeping before the warp does it (0 = TS_BATCH_MIN)
    u8 *dense_blobs;       // speculative dense search -> team stage: [dense_cap][SPB_SIZE], slot = index in the dense list
    u32 dense_cap;
};

enum { MODE_FUSED = 0, MODE_SEARCH = 1, MODE_SCORE = 2, MODE_COOP = 3 };

// Per-CTA shared state: the batch descriptor and one solver object per warp (never a local-memory frame).
template <bool SMEM>
__device__ __forceinline__ RegionSolver<SMEM> &init_solver(const DevBatch &b, const TierArgs &t, DevBatch &sb, RegionSolver<SMEM> *sol) {
    typedef typename Mem<SMEM>::addr addr;
    if (threadIdx.x == 0) sb = b;
    __syncthreads();
    RegionSolver<SMEM> &s = sol[threadIdx.x >> 5];
    addr arena;
    if (SMEM) arena = (addr)((threadIdx.x >> 5) * (u32)t.arena_bytes);
    else arena = (addr)(uintptr_t)(t.arena_base + (((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * (u64)t.arena_bytes);
    if (lane_id() == 0) {
        s.bp = &sb;
        s.tma_phase = 0;
        s.tma_pending = 0;
        s.arena_bytes = (u32)t.arena_bytes;
        s.arena = arena;
        s.spill_base = nullptr; s.spill_bytes = 0; s.team = nullptr; s.pre_scored = 0;
        s.wide_b0 = t.wide_b0;
        if (SMEM && t.spill_base) {
            s.spill_base = t.spill_base + (((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * (u64)t.spill_bytes;
            s.spill_bytes = t.spill_bytes;
        }
        if (SMEM) mbar_init((u32)arena);
    }
    clear_work<SMEM>(arena);
    return s;
}

// Persistent warps pull clusters from a global counter; one warp solves one cluster at a time.
// SMEM stages keep the warp's whole workspace (staged reference window, variants, search nodes, queue, metric
// rows) in shared memory; global stages take the clusters that do not fit.
// MODE_FUSED runs solve_compare_region end to end.  The common tier is split into MODE_SEARCH (optimize_sequences ->
// result blob) and MODE_SCORE (blob -> exact-GT, metrics, outputs): ncu shows the fused solver is bound by
// instruction fetch (its executed path does not stay resident in the SM instruction cache), and two kernels of
// half the footprint each run faster than one.
template <bool SMEM, int MIN_CTAS, int MODE>
__global__ void __launch_bounds__(256, MIN_CTAS) k_compare(DevBatch b, DevCompareOut out, avk_compare_cfg cfg, TierArgs t) {
    __shared__ DevBatch sb;
    __shared__ RegionSolver<SMEM> sol[8];
    const int lane = lane_id();
    RegionSolver<SMEM> &s = init_solver<SMEM>(b, t, sb, sol);
    const u32 n1 = t.n_work_ptr ? *t.n_work_ptr : t.n_work;
    const u32 n_work = n1 + (t.n_work_ptr2 ? *t.n_work_ptr2 : 0u);
    for (;;) {
        u32 idx = 0;
        if (lane == 0) idx = atomicAdd(t.work_ctr, 1u);
        idx = __shfl_sync(AVK_FULL, idx, 0);
        if (idx >= n_work) break;
        const u64 r = t.work_list ? (idx < n1 ? t.work_list[idx] : t.work_list2[idx - n1]) : idx;
        u8 *blob = t.blobs + r * (u64)RB_SIZE;
        int rc;
        if (MODE == MODE_SEARCH) {
            rc = s.compare_search_to_blob(r, cfg, blob);
            __syncwarp();
            if (rc == SOLVE_OK) continue;                        // the score kernel finishes this cluster
            if (lane == 0) *(int *)(blob + RB_NRES) = (rc == SOLVE_WORKSPACE) ? RB_FUSED : RB_DONE;
        } else if (MODE == MODE_SCORE) {
            if (*(const int *)(blob + RB_NRES) <= 0) continue;   // handled elsewhere
            rc = s.compare_score_from_blob(r, cfg, out, blob);
        } else {
            rc = s.solve_compare(r, cfg, out);
        }
        __syncwarp();
        if (rc == SOLVE_WORKSPACE) {
            if (!t.last_tier) {
                if (lane == 0) {
                    if (t.fail_list2 && s.N >= t.dense_n) t.fail_list2[atomicAdd(t.fail_ctr2, 1u)] = (u32)r;   // the long searches: started first
                    else t.fail_list[atomicAdd(t.fail_ctr, 1u)] = (u32)r;
                }
                continue;
            }
            rc = AVK_ST_WORKSPACE;
        }
        if (rc != AVK_ST_OK) zero_region_outputs(sb, out, r, false);
        if (lane == 0) { out.status[r] = rc; if (rc != AVK_ST_OK) count_error_block(out); }
    }
    flush_work<SMEM>(s.arena, t.work_out);
}

// SV / long-indel clusters (workspace beyond 2 MB): one cluster per CTA.  Warp 0 runs the solver on a global arena;
// the other warps wait at a named barrier and join in whenever a wavefront gets wide (avk_device.cuh, dwfa_run_coop).
__global__ void __launch_bounds__(COOP_THREADS, 1) k_compare_coop(DevBatch b, DevCompareOut out, avk_compare_cfg cfg, TierArgs t, int cap_ints) {
    __shared__ DevBatch sb;
    __shared__ RegionSolver<false> sol1;
    if (threadIdx.x == 0) { sb = b; ((CoopJob *)avk_dyn_smem)->cap_ints = cap_ints; ((CoopJob *)avk_dyn_smem)->exit_ = 0; }
    __syncthreads();
    if (threadIdx.x >= 32) { coop_helper_loop(); return; }
    const int lane = lane_id();
    RegionSolver<false> &s = sol1;
    const u64 arena = (u64)(uintptr_t)(t.arena_base + (u64)blockIdx.x * (u64)t.arena_bytes);
    if (lane == 0) {
        s.bp = &sb; s.tma_phase = 0; s.tma_pending = 0;
        s.arena_bytes = (u32)(t.arena_bytes > 0xfffffff0LL ? 0xfffffff0LL : t.arena_bytes); s.arena = arena;
        s.spill_base = nullptr; s.spill_bytes = 0; s.wide_b0 = 0; s.team = nullptr; s.pre_scored = 0;
    }
    clear_work<false>(arena);
    if (lane == 0) *(u32 *)(uintptr_t)(arena + WK_COOP) = 1u;
    __syncwarp();
    const u32 n_work = t.n_work_ptr ? *t.n_work_ptr : t.n_work;
    for (;;) {
        u32 idx = 0;
        if (lane == 0) idx = atomicAdd(t.work_ctr, 1u);
        idx = __shfl_sync(AVK_FULL, idx, 0);
        if (idx >= n_work) break;
        const u64 r = t.work_list ? t.work_list[idx] : idx;
        int rc = s.solve_compare(r, cfg, out);
        __syncwarp();
        if (rc == SOLVE_WORKSPACE) {
            if (!t.last_tier) {
                if (lane == 0) t.fail_list[atomicAdd(t.fail_ctr, 1u)] = (u32)r;
                continue;
            }
            rc = AVK_ST_WORKSPACE;
        }
        if (rc != AVK_ST_OK) zero_region_outputs(sb, out, r, false);
        if (lane == 0) { out.status[r] = rc; if (rc != AVK_ST_OK) count_error_block(out); }
    }
    flush_work<false>(arena, t.work_out);
    coop_release_helpers();
}

// Biggest first for the cooperative tiers: a cluster there can occupy its SM for seconds, so the expensive ones (edit-distance
// bound x variants, both from the digest header) must not start last.  One CTA, bitonic sort in shared memory, <= 4096 entries.
__global__ void __launch_bounds__(1024) k_sort_biggest_first(DevBatch b, u32 *list, u32 n) {
    __shared__ unsigned long long key[4096];
    u32 m = 1;
    while (m < n) m <<= 1;
    for (u32 i = threadIdx.x; i < m; i += blockDim.x) {
        unsigned long long k = 0;
        if (i < n) {
            const int *h = (const int *)(b.digest + b.digest_off[list[i]]);
            const unsigned long long cost = h[PH_STATUS / 4] == AVK_ST_OK ? (unsigned long long)(u32)h[PH_B0 / 4] * (u32)(h[PH_N / 4] + 1) : 0ull;
            k = (min(cost, 0xffffffffull) << 32) | (0xffffffffu - list[i]);     // ties: lower cluster id first
        }
        key[i] = k;
    }
    __syncthreads();
    for (u32 k2 = 2; k2 <= m; k2 <<= 1)
        for (u32 j = k2 >> 1; j > 0; j >>= 1) {
            for (u32 i = threadIdx.x; i < m; i += blockDim.x) {
                const u32 l = i ^ j;
                if (l > i) {
                    const bool desc = (i & k2) == 0;
                    const unsigned long long a = key[i], c = key[l];
                    if (desc ? a < c : a > c) { key[i] = c; key[l] = a; }
                }
            }
            __syncthreads();
        }
    for (u32 i = threadIdx.x; i < n; i += blockDim.x) list[i] = 0xffffffffu - (u32)(key[i] & 0xffffffffull);
}

// ---- warp team per dense cluster ----------------------------------------------------------------------------------------
// The clusters with many variants (list X) bound a pass: one of them is hundreds of queue pops, each of which extends up to
// four (child, haplotype) pairs -- independent of each other -- and a lone warp issues one dependent instruction every ~9
// cycles.  Here a team of four warps takes one cluster (two teams per CTA, 108 KB of shared memory each, cold nodes spill
// to HBM): warp 0 of the team runs the solver and every pop's extensions are spread over the four warps (TeamBoard,
// avk_solver.cuh).
enum { TEAMS_PER_CTA = 2 };
__global__ void __launch_bounds__(128 * TEAMS_PER_CTA, 1) k_compare_team(DevBatch b, DevCompareOut out, avk_compare_cfg cfg, TierArgs t) {
    __shared__ DevBatch sb;
    __shared__ RegionSolver<true> sol2[TEAMS_PER_CTA];
    __shared__ TeamBoard board[TEAMS_PER_CTA];
    const int lane = lane_id(), warp = (threadIdx.x >> 5) & 3, tm = threadIdx.x >> 7;   // TEAMS_PER_CTA teams of four warps per CTA
    if (threadIdx.x == 0) sb = b;
    if ((threadIdx.x & 127) == 0) { board[tm].exit_ = 0; board[tm].count = 0; board[tm].bar = 1 + tm; }
    __syncthreads();
    RegionSolver<true> &s = sol2[tm];
    TeamBoard &B = board[tm];
    if (warp != 0) {                                   // helpers: one round per barrier pair until the master says stop
        for (;;) {
            asm volatile("bar.sync %0, 128;" ::"r"(B.bar) : "memory");
            if (B.exit_) return;
            s.team_exec(warp);
            asm volatile("bar.sync %0, 128;" ::"r"(B.bar) : "memory");
        }
    }
    const u32 arena = (u32)tm * (u32)t.arena_bytes;
    if (lane == 0) {
        s.bp = &sb; s.tma_phase = 0; s.tma_pending = 0; s.arena_bytes = (u32)t.arena_bytes; s.arena = arena;
        s.spill_base = nullptr; s.spill_bytes = 0; s.wide_b0 = 0; s.team = &B; s.pre_scored = 0;
        if (t.spill_base) { s.spill_base = t.spill_base + ((u64)blockIdx.x * TEAMS_PER_CTA + tm) * (u64)t.spill_bytes; s.spill_bytes = t.spill_bytes; }
        mbar_init(arena);
    }
    clear_work<true>(arena);
    __syncwarp();
    const u32 n_work = t.n_work_ptr ? *t.n_work_ptr : t.n_work;
    for (;;) {
        u32 idx = 0;
        if (lane == 0) idx = atomicAdd(t.work_ctr, 1u);
        idx = __shfl_sync(AVK_FULL, idx, 0);
        if (idx >= n_work) break;
        const u64 r = t.work_list[idx];
        // searched (and usually scored) already by k_search_spec?  then only the metrics are left
        const u8 *blob = (t.dense_blobs && idx < t.dense_cap) ? t.dense_blobs + (size_t)idx * avk_sp::SPB_SIZE : nullptr;
        if (blob && *(const int *)(blob + avk_sp::SPB_NRES) == avk_sp::SPB_DONE) continue;   // finished by k_search_spec
        int rc;
        if (blob && *(const int *)(blob + avk_sp::SPB_NRES) > 0) rc = s.compare_score_from_dense(r, cfg, out, blob);
        else rc = s.solve_compare(r, cfg, out);
        __syncwarp();
        if (rc == SOLVE_WORKSPACE) {
            if (lane == 0) t.fail_list[atomicAdd(t.fail_ctr, 1u)] = (u32)r;
            continue;
        }
        if (rc != AVK_ST_OK) zero_region_outputs(sb, out, r, false);
        if (lane == 0) { out.status[r] = rc; if (rc != AVK_ST_OK) count_error_block(out); }
    }
    flush_work<true>(s.arena, t.work_out);
    __syncwarp();
    if (lane == 0) B.exit_ = 1;
    __syncwarp();
    asm volatile("bar.sync %0, 128;" ::"r"(B.bar) : "memory");   // releases the helpers
}

// ---- speculative search of the dense clusters ---------------------------------------------------------------------------
// One warp per cluster of the dense list X (avk_spec_search.cuh): optimize_sequences with up to 32 queue pops in flight -- one
// chain per lane, committed in the reference's order -- then optimize_gt_alleles of every equal-best result's haplotypes,
// one search per lane.  What leaves is the chosen solution and its exact-GT alleles in the cluster's slot of `dense_blobs`
// (slot = index in X); the team stage that follows computes the metrics from it.  A cluster outside the fast path's limits
// gets SPB_NONE in its slot and is solved from scratch by the team stage.
enum { SPEC_WARPS = 8 };
__device__ unsigned long long *g_spec_prof = nullptr;   // AVK_SPEC_PROFILE: per cluster {region, N, pops, load, search, score, metrics + commit} cycles
struct SpecSink {
    const avk_sp::View &V;
    const DevCompareOut &out;
    u64 *row;
    unsigned long long *slot;
    __device__ __forceinline__ void variant(int oi, int e, int o) {
        const u32 *rec = (const u32 *)(V.recs + (size_t)VI_SIZE * oi);
        const u32 gv = rec[VI_GV / 4];
        const bool tr = (rec[VI_FLAGS / 4] & 0x10000u) != 0;
        out.vexp[gv] = (u8)e; out.vobs[gv] = (u8)o;
        out.vcls[gv] = (u8)(e == o ? AVK_CLASS_TP : (tr ? AVK_CLASS_FN : AVK_CLASS_FP));
    }
    __device__ __forceinline__ void metric(int g, int m, u64 v) {
        if (row) row[g * AVK_N_METRICS + m] = v;
        if (slot) atomicAdd(slot + g * AVK_N_METRICS + m, (unsigned long long)v);
    }
};
// lane 0: outputs of a cluster the speculative path has solved completely (as the commit block of k_compare_thread)
__device__ __noinline__ void spec_commit(const avk_sp::View &V, const avk_sp::Shared &S, const DevBatch &b, const DevCompareOut &out, u32 r, unsigned long long *slot) {
    u64 *row = out.region_metrics ? out.region_metrics + (u64)r * (AVK_N_GROUPS * AVK_N_METRICS) : nullptr;
    if (row) for (int i = 0; i < AVK_N_GROUPS * AVK_N_METRICS; ++i) row[i] = 0;
    SpecSink sink{V, out, row, slot};
    u32 e1 = 0, e2 = 0;
    uint16_t tm = 0;
    const int rc = avk_sp::commit_metrics(V, S, sink, &e1, &e2, &tm);
    if (rc == AVK_ST_OK) {
        out.ed1[r] = e1; out.ed2[r] = e2; out.type_mask[r] = tm;
        if (slot) { atomicOr(slot + TOT_MASK, (unsigned long long)tm); atomicAdd(slot + TOT_SOLVED, 1ull); }
    } else {
        const u64 v0 = b.var_off[(u64)r * 2], v1 = b.var_off[(u64)r * 2 + 2];
        for (u64 v = v0; v < v1; ++v) { out.vexp[v] = 0; out.vobs[v] = 0; out.vcls[v] = AVK_CLASS_UNKNOWN; }
        out.ed1[r] = 0; out.ed2[r] = 0; out.type_mask[r] = 0;
        if (out.seq_off) for (int k = 0; k < 5; ++k) out.seq_len[(u64)r * 5 + k] = 0;
        if (slot) atomicAdd(slot + TOT_ERRORS, 1ull);
    }
    out.status[r] = rc;
}
__global__ void __launch_bounds__(32 * SPEC_WARPS, 1) k_search_spec(DevBatch b, DevCompareOut out, avk_compare_cfg cfg, TierArgs t) {
    using namespace avk_sp;
    const int lane = lane_id(), warp = threadIdx.x >> 5;
    u8 *base = avk_dyn_smem + (size_t)warp * (sizeof(Shared) + 32 * sizeof(Scratch));
    Shared &S = *(Shared *)base;
    Scratch &X = ((Scratch *)(base + sizeof(Shared)))[lane];
    Counters ctr = {0, 0, 0};
    u32 spops = 0, xpops = 0;
    const u32 n_work = min(t.n_work_ptr ? *t.n_work_ptr : t.n_work, t.dense_cap);
    const u32 xcap = cfg.exact_gt_max_expansions ? cfg.exact_gt_max_expansions : AVK_EXACT_GT_DEFAULT_MAX_EXPANSIONS;
    const bool finish_here = !(out.seq_off && cfg.enable_sequences);   // the sequence bundle is emitted by the team stage
    unsigned long long *slot = out.tot_slots ? out.tot_slots + (size_t)(blockIdx.x & (TOT_SLOTS - 1)) * TOT_STRIDE : nullptr;
    for (;;) {
        u32 idx = 0;
        if (lane == 0) idx = atomicAdd(t.work_ctr, 1u);
        idx = __shfl_sync(AVK_FULL, idx, 0);
        if (idx >= n_work) break;
        const u32 r = t.work_list[idx];
        u8 *blob = t.dense_blobs + (size_t)idx * SPB_SIZE;
        const u32 c = b.contig[r];
        bool ok = !cfg.enable_exact_shortcut && c < b.n_contigs && b.start[r] <= b.end[r] && (u64)b.end[r] <= b.contig_len[c] && b.end[r] <= 0x7fff0000u &&
                  (int)cfg.max_branch_factor > 0;
        const u8 *digest = b.digest + b.digest_off[r];
        __syncwarp();
        long long tp0 = clock64(), tp1 = tp0, tp2 = tp0, tp3 = tp0;
        if (ok) {
            if (lane == 0) ok = load_cluster(S, digest, (int)b.start[r], (int)b.end[r], (int)cfg.max_branch_factor);
            ok = __shfl_sync(AVK_FULL, ok, 0);
        }
        __syncwarp();
        int nres = SPB_NONE;
        if (ok) {
            View V;
            V.S = &S; V.ref = b.contig_ptr[c] + b.start[r]; V.recs = digest + PH_SIZE; V.alle = V.recs + (size_t)VI_SIZE * S.N;
            tp1 = clock64();
            const bool found_any = search_warp(S, X, V, ctr);
            tp2 = clock64();
            if (found_any) {
                spops += S.spops;                                   // (warp-uniform reads of the shared state)
                const int n = S.N, found = S.nres;
                const bool scored = score_warp(S, X, V, ctr, xcap);
                tp3 = clock64();
                if (scored) {
                    xpops += S.xpops;
                    if (finish_here && metrics_warp(S, X, V, ctr)) {    // metrics + every output right here: nothing is left for the team stage
                        if (lane == 0) spec_commit(V, S, b, out, r, slot);
                        nres = SPB_DONE;
                    } else if (lane == 0) {
                        store_result(blob, 0, S.res[S.best_r], n);
                        *(int *)(blob + SPB_SCORED) = 1; *(u32 *)(blob + SPB_KEEP0) = S.keep0; *(u32 *)(blob + SPB_KEEP1) = S.keep1;
                    }
                    if (nres != SPB_DONE) nres = 1;
                } else {                                            // scoring outside its limits: hand over the search results only
                    for (int i = lane; i < found; i += 32) store_result(blob, i, S.res[i], n);
                    if (lane == 0) *(int *)(blob + SPB_SCORED) = 0;
                    nres = found;
                }
            }
        }
        __syncwarp();
        if (lane == 0) *(int *)(blob + SPB_NRES) = nres;
        if (g_spec_prof && lane == 0 && idx < 65536) {
            unsigned long long *q = g_spec_prof + (size_t)idx * 8;
            const long long tp4 = clock64();
            q[0] = r; q[1] = ok ? (unsigned long long)S.N : 0ull; q[2] = S.spops; q[3] = (unsigned long long)(tp1 - tp0); q[4] = (unsigned long long)(tp2 - tp1);
            q[5] = (unsigned long long)(tp3 - tp2); q[6] = (unsigned long long)(tp4 - tp3); q[7] = (unsigned long long)nres;
        }
        __syncwarp();
    }
    if (t.work_out) {
        unsigned long long v[5] = {ctr.alignments, ctr.cells, ctr.matched, lane == 0 ? spops : 0u, lane == 0 ? xpops : 0u};
#pragma unroll
        for (int k = 0; k < 5; ++k) {
#pragma unroll
            for (int o = 16; o; o >>= 1) v[k] += __shfl_xor_sync(AVK_FULL, v[k], o);
            if (lane == 0 && v[k]) atomicAdd(t.work_out + k, v[k]);
        }
    }
}

// ---- thread per cluster -------------------------------------------------------------------------------------------------
// The common non-closed-form cluster (a few variants, a window of a few hundred bases, edit distances of a few units) is
// solved by ONE thread (avk_thread_solver.cuh): 32 clusters per warp instead of one, an 836-byte workspace per thread in
// shared memory (search nodes are 12-byte queue entries, sequences are never materialised).
// 32 threads on 32 different clusters only run together where they execute the same instructions, so the solver is a
// coroutine: advance() runs a cluster's control flow up to the next alignment it needs, exec_task() -- the one place where
// sequences are built and wavefronts advanced -- executes it.  The warp alternates the two: all lanes advance, all lanes
// execute their task side by side; lanes whose cluster is finished commit it and take the next one from the list W (one
// atomic per warp and round).  A cluster that does not fit the fixed workspace is appended to the reject list -- nothing
// has been written for it -- and goes through the warp kernels (search / score / fused stages) as before.
enum { THREAD_TPB = 256, TS_BATCH_MIN = 16 };   // (default of TierArgs::batch_min; swept 1..24 on B200: 14-16 is the flat optimum at every batch size)
struct ThreadSink {
    const avk_ts::Cluster &cl;
    const DevCompareOut &out;
    u64 *row;
    unsigned long long *slot;
    __device__ __forceinline__ void variant(int oi, int e, int o) {
        const u32 gv = avk_ts::rec32(cl, oi, VI_GV);
        const bool tr = (avk_ts::rec32(cl, oi, VI_FLAGS) & 0x10000u) != 0;
        out.vexp[gv] = (u8)e; out.vobs[gv] = (u8)o;
        out.vcls[gv] = (u8)(e == o ? AVK_CLASS_TP : (tr ? AVK_CLASS_FN : AVK_CLASS_FP));
    }
    __device__ __forceinline__ void metric(int g, int m, u64 v) {
        if (row) row[g * AVK_N_METRICS + m] = v;
        if (slot) atomicAdd(slot + g * AVK_N_METRICS + m, (unsigned long long)v);
    }
};
__global__ void __launch_bounds__(THREAD_TPB, 1) k_compare_thread(DevBatch b, DevCompareOut out, avk_compare_cfg cfg, TierArgs t) {
    using namespace avk_ts;
    const int lane = lane_id();
    Counters ctr = {0, 0, 0, 0, 0};
    Solver S;
    S.wp = &((Work *)avk_dyn_smem)[threadIdx.x];
    S.ctr = &ctr;
    S.phase = PH_FETCH;
    S.task.kind = TK_NONE;
    const u32 n_work = t.n_work_ptr ? *t.n_work_ptr : t.n_work;
    const bool enabled = !cfg.enable_exact_shortcut && !(out.seq_off && cfg.enable_sequences);
    unsigned long long *slot = out.tot_slots ? out.tot_slots + (size_t)(blockIdx.x & (TOT_SLOTS - 1)) * TOT_STRIDE : nullptr;
    const int batch_min = t.batch_min > 0 ? t.batch_min : TS_BATCH_MIN;
    u32 r = 0;
    bool more = true;                                            // warp-uniform: the list is not exhausted yet
    for (;;) {
        // Every trip: one diagonal for every lane that has a task (below).  The other kinds of work are done in batches --
        // when at least TS_BATCH_MIN lanes wait for them, or when no lane can step -- so that the code they execute runs with
        // several lanes at a time.
        const bool idle = __ballot_sync(AVK_FULL, S.task.kind != TK_NONE) == 0u;
        // ---- commit: lanes whose cluster is finished write its outputs (or hand it to the reject list)
        {
            const bool want = S.phase == PH_COMMIT;
            const int cnt = __popc(__ballot_sync(AVK_FULL, want));
            if (want && (cnt >= batch_min || idle)) {
                int rc = S.rc;
                S.phase = PH_FETCH;
                if (rc == TS_REJECT) t.fail_list[atomicAdd(t.fail_ctr, 1u)] = r;
                else {
                    u64 *row = out.region_metrics ? out.region_metrics + (u64)r * (AVK_N_GROUPS * AVK_N_METRICS) : nullptr;
                    if (row) for (int i = 0; i < AVK_N_GROUPS * AVK_N_METRICS; ++i) row[i] = 0;
                    if (rc == AVK_ST_OK) {
                        ThreadSink sink{S.c, out, row, slot};
                        u32 e1 = 0, e2 = 0;
                        uint16_t tm = 0;
                        rc = commit_solution(S, sink, &e1, &e2, &tm);
                        if (rc == AVK_ST_OK) {
                            out.ed1[r] = e1; out.ed2[r] = e2; out.type_mask[r] = tm;
                            if (slot) { atomicOr(slot + TOT_MASK, (unsigned long long)tm); atomicAdd(slot + TOT_SOLVED, 1ull); }
                        }
                    }
                    out.status[r] = rc;
                    if (rc != AVK_ST_OK) {
                        const u64 v0 = b.var_off[(u64)r * 2], v1 = b.var_off[(u64)r * 2 + 2];
                        for (u64 v = v0; v < v1; ++v) { out.vexp[v] = 0; out.vobs[v] = 0; out.vcls[v] = AVK_CLASS_UNKNOWN; }
                        out.ed1[r] = 0; out.ed2[r] = 0; out.type_mask[r] = 0;
                        if (out.seq_off) for (int k = 0; k < 5; ++k) out.seq_len[(u64)r * 5 + k] = 0;
                        if (slot) atomicAdd(slot + TOT_ERRORS, 1ull);
                    }
                }
            }
        }
        // ---- fetch: lanes without a cluster take the next ones from the list (one atomic per warp)
        {
            const bool want = S.phase == PH_FETCH;
            const u32 m = __ballot_sync(AVK_FULL, want);
            if (m && (__popc(m) >= batch_min || idle)) {
                if (more) {
                    const int leader = __ffs(m) - 1;
                    u32 base = 0;
                    if (lane == leader) base = atomicAdd(t.work_ctr, (u32)__popc(m));
                    base = __shfl_sync(AVK_FULL, base, leader);
                    if (base + (u32)__popc(m) >= n_work) more = false;
                    if (want) {
                        const u32 idx = base + (u32)__popc(m & ((1u << lane) - 1u));
                        if (idx >= n_work) S.phase = PH_DONE;
                        else {
                            r = t.work_list[idx];
                            const u32 c = b.contig[r];
                            if (!enabled) S.stop(TS_REJECT);
                            else if (c >= b.n_contigs || b.start[r] > b.end[r] || (u64)b.end[r] > b.contig_len[c] || b.end[r] > 0x7fff0000u ||
                                     (int)cfg.max_branch_factor <= 0)
                                S.stop(AVK_ST_BAD_INPUT);
                            else S.begin(b.digest + b.digest_off[r], b.contig_ptr[c], (int)b.start[r], (int)b.end[r], (int)cfg.max_branch_factor, cfg.exact_gt_max_expansions, t.pop_budget);
                        }
                    }
                } else if (want) S.phase = PH_DONE;
            }
        }
        if (__all_sync(AVK_FULL, S.phase == PH_DONE)) break;
        // ---- advance: lanes between two tasks run their cluster's control flow up to the next alignment and set it up
        {
            const bool want = S.phase == PH_RUN && S.task.kind == TK_NONE;
            const int cnt = __popc(__ballot_sync(AVK_FULL, want));
            if (want && (cnt >= batch_min || idle)) {
                S.advance();
                if (S.task.kind != TK_NONE) S.task_setup();
            }
        }
        __syncwarp();
        // ---- step: one wavefront diagonal per lane
        if (S.task.kind != TK_NONE) S.task_step();
        __syncwarp();
    }
    if (t.work_out) {   // work actually executed: one set of atomics per warp
        unsigned long long v[5] = {ctr.alignments, ctr.cells, ctr.matched, ctr.spops, ctr.xpops};
#pragma unroll
        for (int k = 0; k < 5; ++k) {
#pragma unroll
            for (int o = 16; o; o >>= 1) v[k] += __shfl_xor_sync(AVK_FULL, v[k], o);
            if (lane == 0 && v[k]) atomicAdd(t.work_out + k, v[k]);
        }
    }
}

// merge, stage 1 of 3: per cluster validation, length prefilter, identical-lists shortcut; emits the pair tasks
__global__ void __launch_bounds__(256) k_merge_front(DevBatch b, DevMergeOut out, avk_merge_cfg cfg, MergeWork w, u64 n) {
    __shared__ DevBatch sb;
    __shared__ RegionSolver<false> sol[8];
    const int lane = lane_id();
    if (threadIdx.x == 0) sb = b;
    __syncthreads();
    RegionSolver<false> &s = sol[threadIdx.x >> 5];
    if (lane == 0) s.bp = &sb;
    __syncwarp();
    const u32 K = b.n_inputs;
    const u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((u64)gridDim.x * blockDim.x) >> 5;
    for (u64 r = warp; r < n; r += n_warps) {
        const int rc = s.merge_front(r, cfg, w);
        __syncwarp();
        if (lane == 0) {
            out.status[r] = rc;
            if (rc != AVK_ST_OK) {
                out.cls[r] = AVK_MERGE_DIFFERENT; out.n_idx[r] = 0;
                for (u32 k = 0; k < K; ++k) out.idx[r * K + k] = 0xFF;
            }
        }
    }
}

// merge, stage 2 of 3: one pair search per warp (persistent warps over the task list, workspace tiers as for compare)
template <bool SMEM, int MIN_CTAS>
__global__ void __launch_bounds__(256, MIN_CTAS) k_merge_pairs(DevBatch b, avk_merge_cfg cfg, TierArgs t, MergeWork w) {
    __shared__ DevBatch sb;
    __shared__ RegionSolver<SMEM> sol[8];
    const int lane = lane_id();
    RegionSolver<SMEM> &s = init_solver<SMEM>(b, t, sb, sol);
    const u32 K = b.n_inputs;
    const u32 n_work = t.n_work_ptr ? *t.n_work_ptr : t.n_work;
    for (;;) {
        u32 idx = 0;
        if (lane == 0) idx = atomicAdd(t.work_ctr, 1u);
        idx = __shfl_sync(AVK_FULL, idx, 0);
        if (idx >= n_work) break;
        const u32 task = t.work_list ? t.work_list[idx] : idx;
        const u64 tk = w.tasks[task];
        const u64 r = tk >> 16;
        const u32 i = (u32)(tk >> 8) & 0xffu, j = (u32)tk & 0xffu;
        bool exact = false;
        int rc = s.merge_pair(r, i, j, cfg, &exact);
        __syncwarp();
        if (rc == SOLVE_WORKSPACE) {
            if (!t.last_tier) {
                if (lane == 0) t.fail_list[atomicAdd(t.fail_ctr, 1u)] = task;
                continue;
            }
            rc = AVK_ST_WORKSPACE;
        }
        if (lane == 0) {
            if (rc != AVK_ST_OK) atomicMin(w.pair_err + r, ((i * K - i * (i + 1) / 2 + (j - i - 1)) << 8) | (u32)rc);   // first failing pair in loop order
            else if (exact) { atomicOr(w.rows + r * K + i, 1u << j); atomicOr(w.rows + r * K + j, 1u << i); }
        }
    }
    flush_work<SMEM>(s.arena, t.work_out);
}

// merge, stage 3 of 3: match sets -> classification
__global__ void __launch_bounds__(256) k_merge_classify(DevBatch b, DevMergeOut out, avk_merge_cfg cfg, MergeWork w, u64 n) {
    __shared__ DevBatch sb;
    __shared__ RegionSolver<false> sol[8];
    const int lane = lane_id();
    if (threadIdx.x == 0) sb = b;
    __syncthreads();
    RegionSolver<false> &s = sol[threadIdx.x >> 5];
    if (lane == 0) s.bp = &sb;
    __syncwarp();
    const u32 K = b.n_inputs;
    const u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((u64)gridDim.x * blockDim.x) >> 5;
    for (u64 r = warp; r < n; r += n_warps) {
        if (out.status[r] != AVK_ST_OK) continue;                      // rejected by the front stage
        const int rc = s.merge_classify(r, cfg, out, w);
        __syncwarp();
        if (lane == 0 && rc != AVK_ST_OK) {
            out.status[r] = rc; out.cls[r] = AVK_MERGE_DIFFERENT; out.n_idx[r] = 0;
            for (u32 k = 0; k < K; ++k) out.idx[r * K + k] = 0xFF;
        }
    }
}

// SummaryWriter::add_comparison_benchmark (writers/summary.rs:146-158): thread j sums column j of the
// [n][286] metric rows (coalesced across the block), one atomicAdd per column per block.
#define RED_COLS (AVK_N_GROUPS * AVK_N_METRICS)
__global__ void __launch_bounds__(288) k_reduce(u64 n, const int *status, const u64 *region_metrics, const uint16_t *type_mask,
                                                unsigned long long *totals, u32 *totals_mask, unsigned long long *solved,
                                                unsigned long long *errors, const u64 *strat_off, const u32 *strat_idx,
                                                const u64 *strat_mask, unsigned long long *strat_totals) {
    const int j = threadIdx.x;
    unsigned long long acc = 0, ok = 0, bad = 0;
    u32 mask = 0;
    // four regions per trip: the status loads, then the row loads, are issued together (the loop is latency-bound otherwise)
    for (u64 r0 = blockIdx.x; r0 < n; r0 += 4ull * gridDim.x) {
        bool good[4];
        unsigned long long v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const u64 r = r0 + (u64)k * gridDim.x;
            good[k] = r < n && status[r] == AVK_ST_OK;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const u64 r = r0 + (u64)k * gridDim.x;
            v[k] = (good[k] && j < RED_COLS) ? region_metrics[r * RED_COLS + j] : 0ull;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const u64 r = r0 + (u64)k * gridDim.x;
            if (r >= n) break;
            if (j == 0) { if (good[k]) { ok += 1; mask |= type_mask[r]; } else bad += 1; }
            acc += v[k];
            if (strat_off && v[k]) {
                for (u64 s = strat_off[r]; s < strat_off[r + 1]; ++s) atomicAdd(strat_totals + (u64)strat_idx[s] * RED_COLS + j, v[k]);
            } else if (strat_mask && v[k]) {
                for (u64 m = strat_mask[r]; m; m &= m - 1) atomicAdd(strat_totals + (u64)(__ffsll((long long)m) - 1) * RED_COLS + j, v[k]);
            }
        }
    }
    if (j < RED_COLS && acc) atomicAdd(totals + j, acc);
    if (j == 0) { atomicAdd(solved, ok); atomicAdd(errors, bad); atomicOr(totals_mask, mask); }
}

// Stratifications::containments (stratifications.rs:108-118, 197-210) for every region: one thread per region.
// var_coordinates() (compare_region.rs:63-74): start = min(first truth pos, first query pos), end = max(end of the LAST truth
// variant, end of the LAST query variant) -- last(), not the furthest-reaching variant -- queried 0-based inclusive as
// (start, end - 1) (waffle_solver.rs:151-166).  The intervals of a (stratum, contig) are sorted by `first` with a running
// maximum of `last`: some interval contains [a, b] iff the running maximum at the rightmost interval with first <= a is >= b.
__global__ void __launch_bounds__(256) k_strat_contain(DevBatch b, u64 n, u32 n_strata, u32 n_contigs, const u64 *off, const u32 *first,
                                                       const u32 *pmax_last, u64 *mask_out) {
    const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const u64 t0 = b.var_off[r * 2], q0 = b.var_off[r * 2 + 1], q1 = b.var_off[r * 2 + 2];
    u64 start = ~0ull, end = 0;
    if (q0 > t0) { start = min(start, (u64)b.pos[t0]); end = max(end, (u64)b.pos[q0 - 1] + b.l0[q0 - 1]); }
    if (q1 > q0) { start = min(start, (u64)b.pos[q0]); end = max(end, (u64)b.pos[q1 - 1] + b.l0[q1 - 1]); }
    u64 mask = 0;
    const u32 c = b.contig[r];
    if (start < end && c < n_contigs) {
        const u64 a = start, z = end - 1;
        for (u32 s = 0; s < n_strata; ++s) {
            const u64 i0 = off[(u64)s * n_contigs + c], i1 = off[(u64)s * n_contigs + c + 1];
            u64 lo = i0, hi = i1;                                   // first interval with first > a
            while (lo < hi) { const u64 m = (lo + hi) >> 1; if ((u64)first[m] <= a) lo = m + 1; else hi = m; }
            if (lo > i0 && (u64)pmax_last[lo - 1] >= z) mask |= 1ull << s;
        }
    }
    mask_out[r] = mask;
}

// INT32 ALU peak probe for the integer roofline (SURVEY.md 8d): 8 independent chains of
// add / xor / max per thread, the instruction mix of the wavefront recurrence (IADD3, LOP3, IMNMX).
__global__ void __launch_bounds__(256) k_int_peak(int iters, int *sink) {
    int a0 = threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const int k = blockIdx.x | 1;
#pragma unroll 4
    for (int i = 0; i < iters; ++i) {
        a0 = max(a0 + k, a1) ^ i; a1 = max(a1 + k, a2) ^ i; a2 = max(a2 + k, a3) ^ i; a3 = max(a3 + k, a4) ^ i;
        a4 = max(a4 + k, a5) ^ i; a5 = max(a5 + k, a6) ^ i; a6 = max(a6 + k, a7) ^ i; a7 = max(a7 + k, a0) ^ i;
    }
    if ((a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7) == 0x7fffffff) sink[0] = a0;
}

// ------------------------------------------------------------------------------------ context

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};

struct avk_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    uint64_t launches = 0;
    int sm_count = 148;
    // reference
    std::vector<DevBuf> contig_bufs;
    std::vector<u64> contig_lens;
    DevBuf d_contig_ptr, d_contig_len;
    // batch buffers
    DevBuf region_id, contig, start, end, var_off, pos, vtype, zyg, raw, aoff, l0, l1, pool, alt_ed;
    // outputs
    DevBuf status, ed1, ed2, region_metrics, type_mask, vexp, vobs, vcls, totals, tot_slots, strat_off, strat_idx, strat_totals,
        seq_off, seq_len, seq_pool, m_cls, m_nidx, m_idx, m_rows, m_perr, m_tasks;
    // workspace
    DevBuf digest, digest_sizes, digest_offs, scan_tmp, blobs, scratch, arena, arena2, counters, fail_a, fail_b, fail_c, fail_d, fail_h, fail_w, fail_x, fail_t, fail_s, shape_key, work_ctr, pair_a_off, pair_b_off, pair_a_len, pair_b_len, pair_ed, pair_pool;
    DevBuf rb[24];   // region builder temporaries
    DevBuf st_off, st_first, st_pmax, st_mask;   // stratification intervals (avk_set_stratifications) and per-region containment masks
    u32 st_n = 0, st_contigs = 0;
    int dense_n = 0;    // clusters with at least this many variants go to the dense list X: speculative search + team stage
                        // (AVK_DENSE_N; 0 = 10 when the thread-per-cluster stage runs, 8 or 6 (below 250 k clusters) for the batches that go without it)
    // Resident batch: regions [lo, lo + n_regions) of the caller's batch, i.e. variants [v_base, v_base + n_variants) of its
    // variant table and bytes [p_base, ..) of its allele pool.  Per-variant device pointers are biased by these bases so
    // that kernels index them with the caller's own (global) indices: a contiguous bin needs no re-basing on the host.
    bool have_batch = false;
    bool ids_resident = false;      // the resident batch was built on the device (avk_build_regions*): its region ids are in `region_id`
    bool have_result = false, result_has_rows = false;
    bool result_has_seq = false;    // the last compare pass filled the sequence bundle (seq_off / seq_len / seq_pool, offsets biased by seq_base)
    bool have_merge = false;        // the last pass was a merge: its result (status, m_cls, m_nidx, m_idx) is resident; cleared with have_result
    bool result_has_contain = false;   // the last pass filled st_mask (a resident run never computes containment)
    u64 lo = 0, n_regions = 0, v_base = 0, n_variants = 0, p_base = 0, pool_bytes = 0;
    u64 seq_base = 0, strat_base = 0;
    u32 n_inputs = 0;
    u32 max_allele = 1;
    u64 pool_len = 0;    // allele bytes the cluster digests need
    u32 *h_pin = nullptr;   // pinned host scratch: pipeline counters read back without a blocking copy
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    float last_ms[5] = {0, 0, 0, 0, 0};
    avk_work_counters last_work = {0, 0, 0, 0, 0, 0};
    u32 tier_fail[3] = {0, 0, 0};
    cudaEvent_t tev[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaStream_t side[2] = {nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_join[2] = {nullptr, nullptr}, dbg[3] = {nullptr, nullptr, nullptr};
    float tier_ms[3] = {0, 0, 0};
    // test knobs (environment): shrink the workspace tiers so that small inputs exercise the last-resort paths
    long long coop_arena0 = 256LL << 20, coop_arena1 = 2048LL << 20;
    int coop_cap_ints = 26000;
    int wide_b0 = 256;
    DevBuf dense_blobs, dense_blobs2, spec_prof;
    bool use_spec_search = true;    // AVK_NO_SPEC_SEARCH=1: the team stage searches the dense clusters itself (A/B timing)
    int thread_batch_min = 0;       // AVK_THREAD_BATCH_MIN (0 = default)
    int thread_pop_budget = 0;      // AVK_THREAD_POP_BUDGET (0: by batch size -- a launch ends with its slowest thread, and the fewer clusters a
                                    // thread has the more that one cluster weighs: 64 pops for >= 2.5 M clusters, 48 for >= 1.2 M, else 32)
    bool use_thread_stage = true;   // AVK_NO_THREAD_STAGE=1: warp kernels only (A/B timing, tests of the warp path)
    bool sort_shapes = true;        // AVK_NO_SHAPE_SORT=1: the thread stage takes its clusters in list order
    u64 thread_min_regions = 700000; // smaller batches go to the warp kernels directly: with at most a cluster or two per thread the
                                     // thread stage is bound by its slowest cluster, not by throughput (measured at 494 k clusters: 10.1 ms
                                     // with the thread stage, 8.6 ms without; at 988 k: 11.2 vs 15.5 ms) (AVK_THREAD_MIN_REGIONS)
    // Pipelined single-GPU call: sibling contexts on the same device (own stream and buffers, the owner's reference) solve
    // alternating bins so that one bin's upload, another's kernels and a third's download overlap.
    avk_ctx *ref_owner = nullptr;   // set in a sibling: whose reference it reads
    avk_ctx *sib[2] = {nullptr, nullptr};
    int pipe_bins = 0;              // AVK_PIPELINE_BINS: bins of a streamed call (-1: one bin per pipe_bin_regions clusters; 0 or 1: off, the default:
                                    // a pass has ~10 ms of fixed cost (its longest clusters), so bins only pay for batches of many millions of clusters)
    u64 pipe_min_regions = 1500000; // batches below this are solved in one piece
    u64 pipe_bin_regions = 1000000;
    // Streamed call (compare_streamed): host->device copies go on `up`, device->host copies on `dn`; both NULL outside it
    // (copies then go on `stream`).  A sibling lane shares the owner's compute streams (own_streams == false).
    cudaStream_t up = nullptr, dn = nullptr;
    cudaStream_t copy_streams[2] = {nullptr, nullptr};   // created on first use, kept
    // Concurrent lanes (compare_lanes): a large batch is cut into contiguous bins that are solved AT THE SAME TIME by sibling
    // contexts of this device, each with its own streams and buffers and one host thread -- one bin's upload runs beside
    // another's kernels, and the kernels of different bins fill each other's tails (a pass ends with its slowest clusters).
    bool many_in_flight = false;    // this context has lanes or is one (avk_create_lane): several passes share the GPU, so what counts is the work a
                                    // pass costs, not how soon its slowest cluster ends -- the thread-per-cluster stage (the cheapest per cluster) then
                                    // takes batches from thread_min_regions_lanes clusters up (AVK_THREAD_MIN_REGIONS overrides both thresholds)
    u64 thread_min_regions_lanes = 100000;
    std::vector<avk_ctx *> lanes;   // lanes[0] == this context
    int n_lanes = 0;                // AVK_LANES (0 or 1 = off, the default: measured, the bins' passes keep their fixed cost -- DESIGN.md section 5)
    u64 lane_min_regions = 2000000; // AVK_LANE_MIN_REGIONS: smaller batches are solved in one piece
    cudaEvent_t ev_up = nullptr, ev_done = nullptr;
    bool own_streams = true;
};
static inline const avk_ctx *ref_of(const avk_ctx *ctx) { return ctx->ref_owner ? ctx->ref_owner : ctx; }

static int ensure(avk_ctx *ctx, DevBuf &b, size_t bytes) {
    if (bytes == 0) bytes = 16;
    if (b.cap >= bytes) return AVK_OK;
    if (b.p) { cudaFree(b.p); b.p = nullptr; b.cap = 0; }
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) {
        ctx->err = std::string("cudaMalloc(") + std::to_string(want) + "): " + cudaGetErrorString(e);
        cudaGetLastError();
        return AVK_ERR_OOM;
    }
    b.cap = want;
    return AVK_OK;
}
#define ENSURE(buf, bytes)                        \
    do {                                          \
        int rc_ = ensure(ctx, buf, (bytes));      \
        if (rc_ != AVK_OK) return rc_;            \
    } while (0)

static int upload(avk_ctx *ctx, DevBuf &b, const void *src, size_t bytes) {
    int rc = ensure(ctx, b, bytes);
    if (rc != AVK_OK) return rc;
    if (bytes) CK(cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, ctx->up ? ctx->up : ctx->stream));
    return AVK_OK;
}
// kernels launched on ctx->stream after this call see everything upload() has queued so far
static int uploads_done(avk_ctx *ctx) {
    if (ctx->up) {
        CK(cudaEventRecord(ctx->ev_up, ctx->up));
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_up, 0));
    }
    return AVK_OK;
}
#define UPLOAD(buf, src, bytes)                          \
    do {                                                 \
        int rc_ = upload(ctx, buf, (src), (bytes));      \
        if (rc_ != AVK_OK) return rc_;                   \
    } while (0)

enum { COOP_CAP_INTS_MAX = 26000 };   // wavefronts up to ED 12998 stay in shared memory (k_compare_coop)

// Function attributes are per DEVICE: every context sets them for its own device right after cudaSetDevice (a second
// context on another GPU of the same process needs them too).
static int configure_kernels(avk_ctx *ctx) {
    const int big = 222 * 1024;
#define SMEM_OPT_IN(k)                                                                            \
    do {                                                                                          \
        CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, big));            \
        CK(cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, 100));         \
    } while (0)
    SMEM_OPT_IN((k_compare<true, 3, MODE_SEARCH>));
    SMEM_OPT_IN((k_compare<true, 4, MODE_SCORE>));
    SMEM_OPT_IN((k_compare<true, 1, MODE_FUSED>));
    SMEM_OPT_IN(k_compare_team);
    SMEM_OPT_IN(k_compare_thread);
    SMEM_OPT_IN(k_search_spec);
    SMEM_OPT_IN(k_wfa_ed_cta);
    SMEM_OPT_IN((k_merge_pairs<true, 3>));
    SMEM_OPT_IN((k_merge_pairs<true, 1>));
#undef SMEM_OPT_IN
    CK(cudaFuncSetAttribute(k_compare_coop, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)(COOP_JOB_BYTES + 2 * sizeof(int) * (size_t)COOP_CAP_INTS_MAX)));
    return AVK_OK;
}

extern "C" int avk_create(int device, avk_ctx **out) {
    if (!out) return AVK_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) return AVK_ERR_CUDA;
    avk_ctx *ctx = new avk_ctx();
    ctx->device = device;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete ctx;
        return AVK_ERR_CUDA;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
    if (configure_kernels(ctx) != AVK_OK) {
        fprintf(stderr, "[avk] avk_create: %s\n", ctx->err.c_str());
        cudaStreamDestroy(ctx->stream);
        delete ctx;
        return AVK_ERR_CUDA;
    }
    for (auto &e : ctx->ev) cudaEventCreate(&e);
    if (const char *dn = getenv("AVK_DENSE_N")) ctx->dense_n = std::max(3, atoi(dn));
    // test knobs: tiny workspace tiers so that small inputs reach the last-resort code paths (tests/test_gpu_parity.py)
    if (const char *s = getenv("AVK_TEST_COOP_ARENA_MB")) ctx->coop_arena0 = std::max(1LL, atoll(s)) << 20;
    if (const char *s = getenv("AVK_TEST_COOP_ARENA1_MB")) ctx->coop_arena1 = std::max(1LL, atoll(s)) << 20;
    if (const char *s = getenv("AVK_TEST_COOP_CAP_INTS")) ctx->coop_cap_ints = std::min<int>(COOP_CAP_INTS_MAX, std::max(64, atoi(s)));
    if (const char *s = getenv("AVK_TEST_WIDE_B0")) ctx->wide_b0 = std::max(1, atoi(s));
    if (const char *s = getenv("AVK_NO_THREAD_STAGE")) ctx->use_thread_stage = atoi(s) == 0;
    if (const char *s = getenv("AVK_NO_SPEC_SEARCH")) ctx->use_spec_search = atoi(s) == 0;
    if (const char *s = getenv("AVK_THREAD_POP_BUDGET")) ctx->thread_pop_budget = std::max(1, atoi(s));
    if (const char *s = getenv("AVK_THREAD_BATCH_MIN")) ctx->thread_batch_min = std::min(32, std::max(1, atoi(s)));
    { const int v = getenv("AVK_PACKED_DWFA") ? atoi(getenv("AVK_PACKED_DWFA")) : 0; cudaMemcpyToSymbol(g_avk_packed_dwfa, &v, sizeof(int)); }
    {   // AVK_SPEC_PROFILE=1: k_search_spec records per-cluster phase cycles (avk_spec_profile reads them back)
        unsigned long long *pp = nullptr;
        if (getenv("AVK_SPEC_PROFILE") && ensure(ctx, ctx->spec_prof, 65536 * 64) == AVK_OK) { pp = (unsigned long long *)ctx->spec_prof.p; cudaMemset(pp, 0, 65536 * 64); }
        cudaMemcpyToSymbol(g_spec_prof, &pp, sizeof(pp));
    }
    if (const char *s = getenv("AVK_NO_SHAPE_SORT")) ctx->sort_shapes = atoi(s) == 0;
    if (const char *s = getenv("AVK_THREAD_MIN_REGIONS")) ctx->thread_min_regions = ctx->thread_min_regions_lanes = (u64)std::max(0LL, atoll(s));
    if (const char *s = getenv("AVK_LANES")) ctx->n_lanes = std::max(0, std::min(8, atoi(s)));
    if (const char *s = getenv("AVK_LANE_MIN_REGIONS")) ctx->lane_min_regions = (u64)std::max(1LL, atoll(s));
    if (const char *s = getenv("AVK_PIPELINE_BINS")) ctx->pipe_bins = std::max(-1, atoi(s));
    if (const char *s = getenv("AVK_PIPELINE_BIN_REGIONS")) ctx->pipe_bin_regions = (u64)std::max(1LL, atoll(s));
    if (const char *s = getenv("AVK_PIPELINE_MIN_REGIONS")) ctx->pipe_min_regions = (u64)std::max(1LL, atoll(s));
    for (auto &e : ctx->tev) cudaEventCreate(&e);
    {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        // side streams carry the kernel that should only fill SMs the main stream's kernel has left: lowest priority
        for (auto &st : ctx->side) cudaStreamCreateWithPriority(&st, cudaStreamNonBlocking, lo);
    }
    cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming);
    for (auto &e : ctx->ev_join) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    for (auto &e : ctx->dbg) cudaEventCreate(&e);
    cudaEventCreateWithFlags(&ctx->ev_up, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&ctx->ev_done, cudaEventDisableTiming);
    if (cudaMallocHost((void **)&ctx->h_pin, 4096) != cudaSuccess) { ctx->h_pin = nullptr; cudaGetLastError(); }
    if (!ctx->h_pin) { avk_destroy(ctx); return AVK_ERR_OOM; }
    memset(ctx->h_pin, 0, 4096);
    *out = ctx;
    return AVK_OK;
}

// A lane: a second context on the owner's device that reads the owner's reference and stratification tables and has its own
// streams and batch / result buffers.  Several batches (whole call sets) are then in flight on the one GPU, one host thread per
// context: one batch's copies run beside another's kernels, and the kernels of different batches fill each other's tails.
extern "C" int avk_create_lane(avk_ctx *owner, avk_ctx **out) {
    if (!owner || !out) return AVK_ERR_INVALID;
    if (owner->ref_owner) { owner->err = "avk_create_lane: the owner is itself a lane"; return AVK_ERR_INVALID; }
    const int rc = avk_create(owner->device, out);
    if (rc != AVK_OK) { owner->err = "avk_create_lane: could not create the context"; return rc; }
    (*out)->ref_owner = owner;
    (*out)->many_in_flight = owner->many_in_flight = true;
    return AVK_OK;
}

extern "C" void avk_destroy(avk_ctx *ctx) {
    if (!ctx) return;
    for (auto &sb : ctx->sib) if (sb) { avk_destroy(sb); sb = nullptr; }
    for (size_t i = 1; i < ctx->lanes.size(); ++i) avk_destroy(ctx->lanes[i]);
    ctx->lanes.clear();
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto &st : ctx->side) if (st) cudaStreamSynchronize(st);
    for (cudaStream_t st : ctx->copy_streams) if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
    DevBuf *bufs[] = {&ctx->d_contig_ptr, &ctx->d_contig_len, &ctx->region_id, &ctx->contig, &ctx->start, &ctx->end, &ctx->var_off,
                      &ctx->pos, &ctx->vtype, &ctx->zyg, &ctx->raw, &ctx->aoff, &ctx->l0, &ctx->l1, &ctx->pool, &ctx->alt_ed,
                      &ctx->status, &ctx->ed1, &ctx->ed2, &ctx->region_metrics, &ctx->type_mask, &ctx->vexp, &ctx->vobs, &ctx->vcls,
                      &ctx->totals, &ctx->tot_slots, &ctx->strat_off, &ctx->strat_idx, &ctx->strat_totals, &ctx->seq_off, &ctx->seq_len, &ctx->seq_pool,
                      &ctx->m_cls, &ctx->m_nidx, &ctx->m_idx, &ctx->m_rows, &ctx->m_perr, &ctx->m_tasks, &ctx->digest, &ctx->digest_sizes, &ctx->digest_offs, &ctx->scan_tmp, &ctx->blobs, &ctx->scratch, &ctx->arena, &ctx->arena2, &ctx->counters, &ctx->fail_a, &ctx->fail_b, &ctx->fail_c, &ctx->fail_d, &ctx->fail_h, &ctx->fail_w, &ctx->fail_x, &ctx->fail_t, &ctx->fail_s, &ctx->shape_key, &ctx->dense_blobs, &ctx->dense_blobs2, &ctx->spec_prof,
                      &ctx->work_ctr, &ctx->pair_a_off, &ctx->pair_b_off, &ctx->pair_a_len, &ctx->pair_b_len, &ctx->pair_ed, &ctx->pair_pool};
    for (DevBuf *b : bufs) if (b->p) cudaFree(b->p);
    for (DevBuf &b : ctx->rb) if (b.p) cudaFree(b.p);
    for (DevBuf *b : {&ctx->st_off, &ctx->st_first, &ctx->st_pmax, &ctx->st_mask}) if (b->p) cudaFree(b->p);
    for (DevBuf &b : ctx->contig_bufs) if (b.p) cudaFree(b.p);
    for (auto &e : ctx->ev) if (e) cudaEventDestroy(e);
    for (auto &e : ctx->tev) if (e) cudaEventDestroy(e);
    for (auto &e : ctx->ev_join) if (e) cudaEventDestroy(e);
    for (auto &e : ctx->dbg) if (e) cudaEventDestroy(e);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_up) cudaEventDestroy(ctx->ev_up);
    if (ctx->ev_done) cudaEventDestroy(ctx->ev_done);
    if (ctx->own_streams) {
        for (auto &st : ctx->side) if (st) cudaStreamDestroy(st);
        cudaStreamDestroy(ctx->stream);
    }
    if (ctx->h_pin) cudaFreeHost(ctx->h_pin);
    delete ctx;
}

extern "C" const char *avk_last_error(const avk_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }
extern "C" uint64_t avk_launch_count(const avk_ctx *ctx) {
    if (!ctx) return 0;
    uint64_t n = ctx->launches;
    for (const avk_ctx *sb : ctx->sib) if (sb) n += sb->launches;
    for (size_t i = 1; i < ctx->lanes.size(); ++i) n += ctx->lanes[i]->launches;
    return n;
}

extern "C" int avk_set_reference(avk_ctx *ctx, uint32_t n_contigs, const uint8_t *const *seqs, const uint64_t *lens) {
    if (ctx && ctx->ref_owner) { ctx->err = "a lane reads its owner's reference: call avk_set_reference on the owner"; return AVK_ERR_INVALID; }
    if (!ctx || (n_contigs && (!seqs || !lens))) return AVK_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    for (DevBuf &b : ctx->contig_bufs) if (b.p) cudaFree(b.p);
    ctx->contig_bufs.assign(n_contigs, DevBuf());
    ctx->contig_lens.assign(lens, lens + n_contigs);
    std::vector<const u8 *> ptrs(n_contigs);
    for (uint32_t c = 0; c < n_contigs; ++c) {
        // 64 bytes of slack so that vectorised tail reads stay inside the allocation
        ENSURE(ctx->contig_bufs[c], lens[c] + 64);
        if (lens[c]) CK(cudaMemcpyAsync(ctx->contig_bufs[c].p, seqs[c], lens[c], cudaMemcpyHostToDevice, ctx->stream));
        ptrs[c] = (const u8 *)ctx->contig_bufs[c].p;
    }
    UPLOAD(ctx->d_contig_ptr, ptrs.data(), sizeof(u8 *) * n_contigs);
    UPLOAD(ctx->d_contig_len, lens, sizeof(u64) * n_contigs);
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->have_result = ctx->have_merge = ctx->result_has_seq = false;
    return AVK_OK;
}

extern "C" int avk_set_stratifications(avk_ctx *ctx, const avk_strat_intervals *in) {
    if (ctx && ctx->ref_owner) { ctx->err = "a lane reads its owner's stratifications: call avk_set_stratifications on the owner"; return AVK_ERR_INVALID; }
    if (!ctx) return AVK_ERR_INVALID;
    if (!in || in->n_strata > 64 || (in->n_strata && in->n_contigs && !in->off)) { ctx->err = "avk_set_stratifications: at most 64 strata, non-null offsets"; return AVK_ERR_INVALID; }
    CK(cudaSetDevice(ctx->device));
    const u64 cells = (u64)in->n_strata * in->n_contigs;
    const u64 n_iv = cells ? in->off[cells] : 0;
    if (n_iv && (!in->first || !in->last)) { ctx->err = "avk_set_stratifications: null interval arrays"; return AVK_ERR_INVALID; }
    std::vector<u32> first(n_iv), pmax(n_iv);
    std::vector<std::pair<u32, u32>> iv;
    for (u64 k = 0; k < cells; ++k) {
        const u64 i0 = in->off[k], i1 = in->off[k + 1];
        if (i0 > i1 || i1 > n_iv) { ctx->err = "avk_set_stratifications: offsets are not monotone"; return AVK_ERR_INVALID; }
        iv.clear();
        for (u64 i = i0; i < i1; ++i) iv.emplace_back(in->first[i], in->last[i]);
        std::sort(iv.begin(), iv.end());
        u32 run = 0;
        for (u64 i = i0; i < i1; ++i) { run = std::max(run, iv[i - i0].second); first[i] = iv[i - i0].first; pmax[i] = run; }
    }
    std::vector<u64> off(cells + 1, 0);
    for (u64 k = 0; k <= cells && cells; ++k) off[k] = in->off[k];
    UPLOAD(ctx->st_off, off.data(), 8 * (cells + 1));
    UPLOAD(ctx->st_first, first.data(), 4 * n_iv);
    UPLOAD(ctx->st_pmax, pmax.data(), 4 * n_iv);
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->st_n = in->n_strata; ctx->st_contigs = in->n_contigs;
    return AVK_OK;           // the streamed sibling and the lanes read these tables through ref_of()
}

// ---- host-side batch validation ---------------------------------------------------------------------------------------
// Everything the kernels use as a memory offset is checked here, before anything is uploaded: var_off monotone and inside
// the variant table, allele ranges inside the pool, allele lengths <= 16 MiB (the digest and workspace sizes are 32-bit),
// stratum indices < n_strata, seq_off monotone.  A violation is a whole-batch AVK_ERR_INVALID; what the reference would
// report per region (window outside the contig, unsorted list, empty allele, bad enum code) stays a per-region
// AVK_ST_BAD_INPUT decided on the device.  The scan also yields what sizes the device workspaces (longest allele, allele
// bytes, the pool range the bin touches); it runs on a few host threads for WGS-sized tables.
struct BinScan {
    u64 lo = 0, hi = 0, v0 = 0, v1 = 0, p0 = 0, p1 = 0, sum_alle = 0;
    u32 max_allele = 1;
};

// the bin's variant range (cheap; the uploads of the region and variant arrays can start from this alone)
static int bin_range(avk_ctx *ctx, const avk_region_batch *b, u64 lo, u64 hi, BinScan &sc) {
    const u64 K = b->n_inputs;
    const avk_variant_table &t = b->variants;
    sc.lo = lo; sc.hi = hi;
    if (hi == lo) return AVK_OK;
    const u64 *vo = b->var_off;
    sc.v0 = vo[lo * K]; sc.v1 = vo[hi * K];
    if (sc.v0 > sc.v1 || sc.v1 > t.n_variants) { ctx->err = "var_off outside the variant table"; return AVK_ERR_INVALID; }
    if (sc.v1 > sc.v0 && (!t.position || !t.variant_type || !t.zygosity || !t.raw_allele_space || !t.allele_off || !t.a0_len || !t.a1_len || !t.allele_pool)) {
        ctx->err = "null variant arrays";
        return AVK_ERR_INVALID;
    }
    return AVK_OK;
}
// host-side validation of the offsets the kernels index with, and the bin's allele-pool range (after bin_range)
static int scan_bin(avk_ctx *ctx, const avk_region_batch *b, BinScan &sc) {
    const u64 K = b->n_inputs, lo = sc.lo, hi = sc.hi;
    const avk_variant_table &t = b->variants;
    if (hi == lo) return AVK_OK;
    const u64 *vo = b->var_off;
    const u64 nv = sc.v1 - sc.v0, nr = (hi - lo) * K;
    const int nt = (int)std::min<u64>(12, std::max<u64>(1, (nv + nr) / 400000));
    struct Part { u64 p0 = ~0ull, p1 = 0, sum = 0; u32 mx = 1; int bad = 0; };
    std::vector<Part> parts(nt);
    auto work = [&](int ti) {
        Part &P = parts[ti];
        for (u64 i = lo * K + nr * ti / nt, e = lo * K + nr * (ti + 1) / nt; i < e; ++i) if (vo[i] > vo[i + 1]) P.bad = 1;
        const u64 pool_len = t.allele_pool_len;
        for (u64 v = sc.v0 + nv * ti / nt, e = sc.v0 + nv * (ti + 1) / nt; v < e; ++v) {
            const u64 a = t.allele_off[v], l0 = t.a0_len[v], l1 = t.a1_len[v];
            if (l0 > (1u << 24) || l1 > (1u << 24)) { P.bad = 2; continue; }
            if (a + l0 + l1 > pool_len) { P.bad = 3; continue; }
            P.p0 = std::min(P.p0, a); P.p1 = std::max(P.p1, a + l0 + l1);
            P.sum += l0 + l1;
            P.mx = std::max(P.mx, (u32)std::max(l0, l1));
        }
    };
    if (nt == 1) work(0);
    else {
        std::vector<std::thread> th;
        for (int ti = 0; ti < nt; ++ti) th.emplace_back(work, ti);
        for (auto &x : th) x.join();
    }
    u64 p0 = ~0ull, p1 = 0;
    for (const Part &P : parts) {
        if (P.bad) {
            ctx->err = P.bad == 1 ? "var_off is not monotone" : (P.bad == 2 ? "allele longer than 16 MiB" : "allele range outside the allele pool");
            return AVK_ERR_INVALID;
        }
        p0 = std::min(p0, P.p0); p1 = std::max(p1, P.p1);
        sc.sum_alle += P.sum; sc.max_allele = std::max(sc.max_allele, P.mx);
    }
    if (p1 > p0) { sc.p0 = p0; sc.p1 = p1; }
    return AVK_OK;
}

static int validate_batch(avk_ctx *ctx, const avk_region_batch *b, bool compare) {
    if (!b) { ctx->err = "null batch"; return AVK_ERR_INVALID; }
    if (compare ? b->n_inputs != 2 : (b->n_inputs < 1 || b->n_inputs > 32)) { ctx->err = "unsupported n_inputs"; return AVK_ERR_INVALID; }
    if (b->n_regions >= (1ull << 32) - 1 || b->variants.n_variants >= (1ull << 32) || b->variants.allele_pool_len >= (1ull << 32)) {
        ctx->err = "batch too large for 32-bit indices; split it";
        return AVK_ERR_INVALID;
    }
    if (b->n_regions && (!b->region_id || !b->contig || !b->start || !b->end || !b->var_off)) { ctx->err = "null region arrays"; return AVK_ERR_INVALID; }
    if (b->n_regions && b->var_off[b->n_regions * b->n_inputs] != b->variants.n_variants) { ctx->err = "var_off does not cover the variant table"; return AVK_ERR_INVALID; }
    return AVK_OK;
}

// Upload regions [sc.lo, sc.hi) of the batch (after bin_range): a contiguous bin (the whole batch for one GPU).
static int upload_batch(avk_ctx *ctx, const avk_region_batch *b, BinScan &sc) {
    if (ref_of(ctx)->contig_bufs.empty()) { ctx->err = "avk_set_reference has not been called"; return AVK_ERR_NO_REFERENCE; }
    const u64 lo = sc.lo, n = sc.hi - sc.lo, K = b->n_inputs, v0 = sc.v0, nv = sc.v1 - sc.v0;
    const avk_variant_table &t = b->variants;
    ctx->have_batch = false; ctx->have_result = ctx->have_merge = ctx->result_has_seq = false; ctx->ids_resident = false;
    UPLOAD(ctx->contig, b->contig + lo, 4 * n);
    UPLOAD(ctx->start, b->start + lo, 4 * n);
    UPLOAD(ctx->end, b->end + lo, 4 * n);
    if (n) UPLOAD(ctx->var_off, b->var_off + lo * K, 8 * (n * K + 1));
    else { ENSURE(ctx->var_off, 8); CK(cudaMemsetAsync(ctx->var_off.p, 0, 8, ctx->stream)); }
    UPLOAD(ctx->pos, t.position + v0, 4 * nv);
    UPLOAD(ctx->vtype, t.variant_type + v0, nv);
    UPLOAD(ctx->zyg, t.zygosity + v0, nv);
    UPLOAD(ctx->raw, t.raw_allele_space + v0, 4 * nv);
    UPLOAD(ctx->aoff, t.allele_off + v0, 4 * nv);
    UPLOAD(ctx->l0, t.a0_len + v0, 4 * nv);
    UPLOAD(ctx->l1, t.a1_len + v0, 4 * nv);
    ENSURE(ctx->alt_ed, 4 * nv);
    // while those copies are under way the host validates the offsets and finds the bin's allele-pool range
    int rc = scan_bin(ctx, b, sc);
    if (rc != AVK_OK) { cudaStreamSynchronize(ctx->up ? ctx->up : ctx->stream); return rc; }
    UPLOAD(ctx->pool, t.allele_pool + sc.p0, sc.p1 - sc.p0);
    ctx->max_allele = sc.max_allele;
    ctx->pool_len = sc.sum_alle;
    ctx->lo = lo; ctx->n_regions = n; ctx->v_base = v0; ctx->n_variants = nv; ctx->p_base = sc.p0; ctx->pool_bytes = sc.p1 - sc.p0;
    ctx->n_inputs = b->n_inputs;
    ctx->have_batch = true;
    return AVK_OK;
}

// device pointer biased so that element `base` of the caller's array is the first resident element
template <class T>
static inline T *biased(const DevBuf &b, u64 base) { return (T *)((uintptr_t)b.p - (uintptr_t)(base * sizeof(T))); }

static DevBatch dev_batch(avk_ctx *ctx) {
    DevBatch d;
    const u64 vb = ctx->v_base;
    d.n_regions = ctx->n_regions; d.n_inputs = ctx->n_inputs;
    d.region_id = nullptr; d.contig = (const u32 *)ctx->contig.p;
    d.start = (const u32 *)ctx->start.p; d.end = (const u32 *)ctx->end.p; d.var_off = (const u64 *)ctx->var_off.p;
    d.pos = biased<const u32>(ctx->pos, vb); d.vtype = biased<const u8>(ctx->vtype, vb); d.zyg = biased<const u8>(ctx->zyg, vb);
    d.raw = biased<const u32>(ctx->raw, vb); d.aoff = biased<const u32>(ctx->aoff, vb); d.l0 = biased<const u32>(ctx->l0, vb);
    d.l1 = biased<const u32>(ctx->l1, vb);
    d.pool = biased<const u8>(ctx->pool, ctx->p_base);
    d.contig_ptr = (const u8 *const *)ref_of(ctx)->d_contig_ptr.p; d.contig_len = (const u64 *)ref_of(ctx)->d_contig_len.p;
    d.n_contigs = (u32)ref_of(ctx)->contig_lens.size();
    d.alt_ed = biased<const u32>(ctx->alt_ed, vb);
    d.digest = (const u8 *)ctx->digest.p;
    d.digest_off = (const u64 *)ctx->digest_offs.p;
    return d;
}

static int run_alt_ed(avk_ctx *ctx, const DevBatch &db) {
    if (ctx->n_variants == 0) return AVK_OK;
    const int blocks = ctx->sm_count * 4, threads = 256;
    const int warps = blocks * threads / 32;
    const int scratch_ints = (2 * (int)ctx->max_allele + 8 + 3) / 4 * 4;
    ENSURE(ctx->scratch, (size_t)warps * ((size_t)scratch_ints * 4 + ARENA_HDR));
    k_alt_ed<<<blocks, threads, 0, ctx->stream>>>(db, ctx->v_base, ctx->n_variants, biased<u32>(ctx->alt_ed, ctx->v_base), (u8 *)ctx->scratch.p,
                                                   scratch_ints, (unsigned long long *)ctx->work_ctr.p);
    ctx->launches += 1;
    CK(cudaGetLastError());
    return AVK_OK;
}

// Workspace stages.  The common tier keeps the per-warp workspace in shared memory; for compare it is split into a
// search kernel and a score kernel (see k_compare).  Clusters whose search does not fit go down a chain of fused
// stages: 8 warps x 27 KB of shared memory per SM, then global-memory arenas.  The first stages are launched back
// to back: each reads its work count from an earlier stage's fail counter in device memory, so the common case
// needs no host round trip.
struct Stage {
    int mode;              // MODE_*
    bool smem;
    int min_ctas;          // CTAs per SM the kernel is compiled for
    long long arena_bytes; // per warp
    int ctas;              // grid size (persistent)
    int warps;             // warps per CTA
    int in_list;           // -1: all regions; else index of the fail list to consume (0 = A, 1 = B)
    int in_ctr;            // counter index holding that list's length
    int work_ctr;          // counter index of this launch's work counter
    int fail_list;         // fail list to append to
    int fail_ctr;          // counter index of that list's length
    int stream;            // 0 main; 1, 2: side streams of the concurrent first group
    int n_lo, n_hi;        // cluster-size class (stages scanning all regions)
};

// Merge pipeline driver.  `pre(ctrs)` runs after the counters are cleared and before the first stage; when `first_ctr` >= 0
// the first stage takes its work count from that counter (written by `pre`) instead of n, which is then only an upper bound.
template <class P, class F>
static int run_stages(avk_ctx *ctx, u64 n, const std::vector<Stage> &stages, P pre, int first_ctr, F launch) {
    if (n == 0) return AVK_OK;
    const int sm = ctx->sm_count;
    ENSURE(ctx->fail_a, 4 * n);
    ENSURE(ctx->fail_b, 4 * n);
    ENSURE(ctx->counters, 256);
    u32 *ctrs = (u32 *)ctx->counters.p;
    CK(cudaMemsetAsync(ctrs, 0, 256, ctx->stream));
    u32 *fail_lists[2] = {(u32 *)ctx->fail_a.p, (u32 *)ctx->fail_b.p};
    size_t garena = 0;
    for (const Stage &st : stages) if (!st.smem) garena = std::max(garena, (size_t)st.ctas * st.warps * (size_t)st.arena_bytes);
    if (garena) ENSURE(ctx->arena, garena);
    ENSURE(ctx->arena2, (size_t)sm * 8 * (size_t)(1u << 20));
    CK(cudaEventRecord(ctx->tev[0], ctx->stream));
    pre(ctrs);
    int ev = 1;
    for (size_t i = 0; i < stages.size(); ++i) {
        const Stage &st = stages[i];
        TierArgs a = {};
        a.work_list = st.in_list < 0 ? nullptr : fail_lists[st.in_list];
        a.n_work_ptr = st.in_list < 0 ? (first_ctr >= 0 ? ctrs + first_ctr : nullptr) : ctrs + st.in_ctr;
        a.n_work = (u32)n;
        a.work_ctr = ctrs + st.work_ctr;
        a.fail_ctr = ctrs + st.fail_ctr;
        a.arena_base = (u8 *)ctx->arena.p;
        a.arena_bytes = st.arena_bytes;
        a.fail_list = fail_lists[st.fail_list];
        a.last_tier = 0;
        a.work_out = (unsigned long long *)ctx->work_ctr.p;
        a.blobs = (u8 *)ctx->blobs.p;
        a.spill_base = nullptr; a.spill_bytes = 0;
        if (st.smem && st.arena_bytes >= 16384) { a.spill_base = (u8 *)ctx->arena2.p; a.spill_bytes = 1u << 20; }   // cold search nodes spill to HBM
        a.n_lo = st.n_lo; a.n_hi = st.n_hi;
        int ctas = st.ctas;
        if (st.in_list < 0) ctas = (int)std::min<u64>((u64)ctas, (n + st.warps - 1) / st.warps);
        launch(st, a, ctas, ctx->stream);
        ctx->launches += 1;
        CK(cudaGetLastError());
        if (ev < 3 && (i + 1 < stages.size())) CK(cudaEventRecord(ctx->tev[ev++], ctx->stream));
    }
    while (ev < 4) CK(cudaEventRecord(ctx->tev[ev++], ctx->stream));
    const Stage &lastst = stages.back();
    CK(cudaMemcpyAsync(ctx->h_pin, ctrs, 64, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const u32 *host_ctrs = ctx->h_pin;
    for (int t = 0; t < 3; ++t) cudaEventElapsedTime(&ctx->tier_ms[t], ctx->tev[t], ctx->tev[t + 1]);
    {   // diagnostics: overflow counts of the (up to) three chained tiers
        int k = 0;
        for (const Stage &st : stages) if (k < 3) ctx->tier_fail[k++] = host_ctrs[st.fail_ctr];
        while (k < 3) ctx->tier_fail[k++] = 0;
    }
    u32 n_work = host_ctrs[lastst.fail_ctr];
    int cur_list = lastst.fail_list;
    // rare: pair searches that overflow 2 MB per warp; host-synchronised escalation
    const Stage big[2] = {{MODE_FUSED, false, 1, 64LL << 20, (sm + 7) / 8, 8, 0, 0, 0, 0, 0, 0, 0, 0x7fffffff}, {MODE_FUSED, false, 1, 2048LL << 20, 1, 8, 0, 0, 0, 0, 0, 0, 0, 0x7fffffff}};
    for (int t = 0; t < 2 && n_work > 0; ++t) {
        ENSURE(ctx->arena, (size_t)big[t].ctas * big[t].warps * (size_t)big[t].arena_bytes);
        CK(cudaMemsetAsync(ctrs + 32, 0, 8, ctx->stream));
        TierArgs a = {};
        a.work_list = fail_lists[cur_list];
        a.n_work_ptr = nullptr;
        a.n_work = n_work;
        a.work_ctr = ctrs + 32;
        a.fail_ctr = ctrs + 33;
        a.arena_base = (u8 *)ctx->arena.p;
        a.arena_bytes = big[t].arena_bytes;
        a.fail_list = fail_lists[cur_list ^ 1];
        a.last_tier = t == 1;
        a.work_out = (unsigned long long *)ctx->work_ctr.p;
        a.blobs = (u8 *)ctx->blobs.p;
        a.n_lo = 0; a.n_hi = 0x7fffffff;
        launch(big[t], a, big[t].ctas, ctx->stream);
        ctx->launches += 1;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(ctx->h_pin, ctrs + 32, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        n_work = ctx->h_pin[1];
        cur_list ^= 1;
    }
    return AVK_OK;
}

template <bool SMEM, int MIN_CTAS, int MODE>
static void launch_compare(const DevBatch &db, const DevCompareOut &out, const avk_compare_cfg &c, const TierArgs &a, int ctas, int warps, cudaStream_t strm) {
    const size_t smem = SMEM ? (size_t)a.arena_bytes * warps : 0;
    k_compare<SMEM, MIN_CTAS, MODE><<<ctas, 32 * warps, smem, strm>>>(db, out, c, a);
}
template <bool SMEM, int MIN_CTAS>
static void launch_merge_pairs(const DevBatch &db, const avk_merge_cfg &c, const TierArgs &a, const MergeWork &w, int ctas, int warps, cudaStream_t strm) {
    const size_t smem = SMEM ? (size_t)a.arena_bytes * warps : 0;
    k_merge_pairs<SMEM, MIN_CTAS><<<ctas, 32 * warps, smem, strm>>>(db, c, a, w);
}

static int run_prepare(avk_ctx *ctx, const DevBatch &db) {
    const u64 n = ctx->n_regions;
    if (n == 0) return AVK_OK;
    u64 *sizes = (u64 *)ctx->digest_sizes.p, *offs = (u64 *)ctx->digest_offs.p;
    k_prep_size<<<(unsigned)((n + 1 + 255) / 256), 256, 0, ctx->stream>>>(db, n, sizes);
    size_t tmp_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, sizes, offs, (int)(n + 1), ctx->stream);
    ENSURE(ctx->scan_tmp, tmp_bytes);
    cub::DeviceScan::ExclusiveSum(ctx->scan_tmp.p, tmp_bytes, sizes, offs, (int)(n + 1), ctx->stream);
    // small clusters: one thread each; the few large ones (list in fail_a, count in counters[40]) one warp each
    ENSURE(ctx->fail_a, 4 * n);
    ENSURE(ctx->counters, 256);
    u32 *big_ctr = (u32 *)ctx->counters.p + 40;
    CK(cudaMemsetAsync(big_ctr, 0, 4, ctx->stream));
    k_prep_fill_small<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(db, n, offs, (u8 *)ctx->digest.p, (u32 *)ctx->fail_a.p, big_ctr);
    k_prep_fill<<<ctx->sm_count * 2, 256, 0, ctx->stream>>>(db, n, offs, (u8 *)ctx->digest.p, (const u32 *)ctx->fail_a.p, big_ctr);
    ctx->launches += 4;
    CK(cudaGetLastError());
    return AVK_OK;
}

// strata sums are requested with a caller-provided membership list (strat_off / strat_idx) or, when strat_off is NULL, through
// the device containment lookup (avk_set_stratifications)
static inline bool strata_wanted(const avk_compare_out *out) { return out->strat_totals && out->n_strata; }

struct CompareRun {           // what one compare pass needs to know to launch, finish and (rarely) re-finish
    DevBatch db;
    DevCompareOut out;
    avk_compare_cfg cfg;
    bool strata = false;
    const u64 *strat_off = nullptr;
    const u32 *strat_idx = nullptr;
    const u64 *strat_mask = nullptr;   // device containment lookup instead of a caller-provided membership list
    bool want_contain = false;         // compute the containment masks (for the strata sums and / or out->containment)
    u32 n_strata = 0;
};

static void launch_stage(avk_ctx *ctx, const CompareRun &R, const Stage &st, const TierArgs &a, int ctas, cudaStream_t strm) {
    if (st.mode == MODE_COOP) {
        const size_t smem = COOP_JOB_BYTES + 2 * sizeof(int) * (size_t)ctx->coop_cap_ints;
        k_compare_coop<<<ctas, COOP_THREADS, smem, strm>>>(R.db, R.out, R.cfg, a, ctx->coop_cap_ints);
    }
    else if (st.mode == MODE_SEARCH) launch_compare<true, 3, MODE_SEARCH>(R.db, R.out, R.cfg, a, ctas, st.warps, strm);
    else if (st.mode == MODE_SCORE) launch_compare<true, 4, MODE_SCORE>(R.db, R.out, R.cfg, a, ctas, st.warps, strm);
    else if (st.smem) launch_compare<true, 1, MODE_FUSED>(R.db, R.out, R.cfg, a, ctas, st.warps, strm);
    else launch_compare<false, 1, MODE_FUSED>(R.db, R.out, R.cfg, a, ctas, st.warps, strm);
}

static TierArgs tier_args(avk_ctx *ctx, const u32 *list, int in_ctr, int work_ctr, u32 *fail_list, int fail_ctr, long long arena_bytes, u8 *garena) {
    u32 *ctrs = (u32 *)ctx->counters.p;
    TierArgs a = {};
    a.work_list = list; a.n_work_ptr = list ? ctrs + in_ctr : nullptr; a.n_work = (u32)ctx->n_regions;
    a.work_ctr = ctrs + work_ctr; a.fail_ctr = ctrs + fail_ctr; a.fail_list = fail_list;
    a.arena_base = garena; a.arena_bytes = arena_bytes; a.last_tier = 0;
    a.work_out = (unsigned long long *)ctx->work_ctr.p; a.blobs = (u8 *)ctx->blobs.p; a.n_lo = 0; a.n_hi = 0x7fffffff;
    a.spill_base = nullptr; a.spill_bytes = 0;
    return a;
}

// The compare pipeline.  k_compare_simple takes every cluster: closed forms are final, clusters with >= dense_n variants go
// to the dense list X, the rest to W.  Main stream: X -> speculative search + team stage.  Beside it on a lowest-priority
// side stream: W -> one thread per cluster (large batches; its rejects W2 -> speculative search + team stage), or for small
// batches W -> warp search / score kernels (the search kernel's rejects A -> speculative search + team stage).  Then on the
// main stream the fused 27 KB stage for the score kernel's rejects (A2) and the fused 2 MB global-arena stage for whatever did
// not fit a team's shared memory (B).  Every stage reads its work count from an earlier stage's counter in device memory and
// NOTHING here waits for the device: the counters travel back with the results (compare_finish), and only if list D
// (SV-sized clusters) turns out non-empty does the host launch the cooperative tiers afterwards.
// counters (u32): 12 |W| (clusters without a closed form), 17 |X| dense, 20 / 4 speculative search / team work on X, 19 thread-stage
// work, 13 |W2| (its rejects), 0 search work, 1 |A|, 2 score work, 15 |A2|, 22 / 23 speculative search / team work on W2 or A,
// 16 S1 work, 5 |B|, 9 G0 work, 7 |D|; 32.. big tiers; 40 digest builder
static int run_compare_pipeline(avk_ctx *ctx, const CompareRun &R) {
    const u64 n = ctx->n_regions;
    if (n == 0) return AVK_OK;
    const int sm = ctx->sm_count;
    ENSURE(ctx->fail_a, 4 * n); ENSURE(ctx->fail_b, 4 * n); ENSURE(ctx->fail_c, 4 * n); ENSURE(ctx->fail_d, 4 * n); ENSURE(ctx->fail_h, 4 * n); ENSURE(ctx->fail_w, 4 * n); ENSURE(ctx->fail_x, 4 * n); ENSURE(ctx->fail_t, 4 * n);
    ENSURE(ctx->counters, 256);
    ENSURE(ctx->blobs, (size_t)n * RB_SIZE);
    u32 *ctrs = (u32 *)ctx->counters.p;
    u32 *LA = (u32 *)ctx->fail_a.p, *LB = (u32 *)ctx->fail_b.p, *LD = (u32 *)ctx->fail_d.p;
    CK(cudaMemsetAsync(ctrs, 0, 256, ctx->stream));
    ENSURE(ctx->arena, (size_t)sm * 8 * (size_t)(2LL << 20));
    ENSURE(ctx->arena2, 2 * (size_t)sm * 8 * (size_t)(1u << 20));   // two fused stages may run side by side
    const Stage SEARCH = {MODE_SEARCH, true, 3, 8192, sm * 3, 8}, SCORE = {MODE_SCORE, true, 4, 5120, sm * 4, 8};
    const Stage S1 = {MODE_FUSED, true, 1, 27648, sm, 8}, G0 = {MODE_FUSED, false, 1, 2LL << 20, sm, 8};
    CK(cudaEventRecord(ctx->tev[0], ctx->stream));
    u32 *LW = (u32 *)ctx->fail_h.p, *LA2 = (u32 *)ctx->fail_w.p, *LX = (u32 *)ctx->fail_x.p;
    const bool thread_stage = ctx->use_thread_stage && n >= (ctx->many_in_flight ? ctx->thread_min_regions_lanes : ctx->thread_min_regions);
    const int dense_n = ctx->dense_n ? ctx->dense_n : (thread_stage ? 10 : (n >= 250000 ? 8 : 6));
    // closed-form clusters; >= dense_n variants -> X (dense); the rest -> W
    u64 *keys = nullptr;
    if (thread_stage && ctx->sort_shapes) {
        ENSURE(ctx->shape_key, 16 * n);                               // keys in / out
        ENSURE(ctx->fail_s, 4 * n);
        keys = (u64 *)ctx->shape_key.p;
        CK(cudaMemsetAsync(keys, 0xff, 8 * n, ctx->stream));          // unused tail sorts behind every real key
    }
    k_compare_simple<<<sm * 8, 256, 0, ctx->stream>>>(R.db, R.out, R.cfg, n, LW, ctrs + 12, LX, ctrs + 17, dense_n, keys);
    if (keys) {                                                       // W sorted by shape -> fail_s (the first |W| entries are the real ones)
        size_t need = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, need, keys, keys + n, LW, (u32 *)ctx->fail_s.p, (int)n, 0, 64, ctx->stream);
        ENSURE(ctx->scan_tmp, need);
        cub::DeviceRadixSort::SortPairs(ctx->scan_tmp.p, need, keys, keys + n, LW, (u32 *)ctx->fail_s.p, (int)n, 0, 64, ctx->stream);
        ctx->launches += 1;
    }
    const size_t spill_warp = 1u << 20, spill_half = (size_t)sm * 8 * spill_warp;
    const u32 dense_cap = (u32)std::min<u64>(n, std::max<u64>(65536, n / 16));   // slots of 3.6 KB; a list longer than this leaves its tail to the team stage
    // A list of hard clusters is solved in two launches: k_search_spec -- optimize_sequences with up to 32 queue pops in flight
    // and the exact-GT scoring of the equal-best results, one search per lane -- leaves the chosen solution in the cluster's
    // blob, and the team stage computes the metrics from it (or solves the cluster from scratch when the speculative search
    // declined it); what does not fit the team stage's 108 KB goes on to list B.
    auto spec_then_team = [&](const u32 *list, int in_ctr, int spec_ctr, int team_ctr, DevBuf &blobs, u8 *spill, cudaStream_t strm) -> int {
        TierArgs a = tier_args(ctx, list, in_ctr, team_ctr, LB, 5, 108 * 1024, nullptr);
        a.spill_base = spill; a.spill_bytes = (u32)spill_warp;
        if (ctx->use_spec_search) {
            ENSURE(blobs, (size_t)dense_cap * avk_sp::SPB_SIZE);
            TierArgs sa = tier_args(ctx, list, in_ctr, spec_ctr, nullptr, 21, 0, nullptr);
            sa.dense_blobs = (u8 *)blobs.p; sa.dense_cap = dense_cap;
            k_search_spec<<<sm, 32 * SPEC_WARPS, SPEC_WARPS * (sizeof(avk_sp::Shared) + 32 * sizeof(avk_sp::Scratch)), strm>>>(R.db, R.out, R.cfg, sa);
            ctx->launches += 1;
            a.dense_blobs = sa.dense_blobs; a.dense_cap = dense_cap;
        }
        k_compare_team<<<sm, 128 * TEAMS_PER_CTA, TEAMS_PER_CTA * (size_t)a.arena_bytes, strm>>>(R.db, R.out, R.cfg, a);
        ctx->launches += 1;
        return AVK_OK;
    };
    // The dense list X starts first on the main stream; everything else follows on a lowest-priority side stream behind an
    // event and fills the SMs the dense stage leaves free (all these kernels ask for the maximum shared-memory carveout;
    // kernels of different streams do not take over an SM otherwise: tools/overlap_probe.cu).
    CK(cudaEventRecord(ctx->ev_fork, ctx->stream));
    CK(cudaStreamWaitEvent(ctx->side[0], ctx->ev_fork, 0));
    {
        const int rc = spec_then_team(LX, 17, 20, 4, ctx->dense_blobs, (u8 *)ctx->arena2.p, ctx->stream);            // X -> B
        if (rc != AVK_OK) return rc;
    }
    CK(cudaEventRecord(ctx->tev[1], ctx->stream));
    if (thread_stage) {
        // W -> one thread per cluster; what exceeds a thread's fixed workspace (W2) is a hard cluster
        u32 *LW2 = (u32 *)ctx->fail_t.p;
        TierArgs a = tier_args(ctx, keys ? (const u32 *)ctx->fail_s.p : LW, 12, 19, LW2, 13, sizeof(avk_ts::Work), nullptr);
        a.batch_min = ctx->thread_batch_min;
        a.pop_budget = ctx->thread_pop_budget ? ctx->thread_pop_budget : (n >= 2500000 ? 64 : (n >= 1200000 ? 48 : 32));   // (the same with passes in flight: measured)
        k_compare_thread<<<(unsigned)std::min<u64>((u64)sm, (n + THREAD_TPB - 1) / THREAD_TPB), THREAD_TPB, THREAD_TPB * sizeof(avk_ts::Work), ctx->side[0]>>>(R.db, R.out, R.cfg, a);
        ctx->launches += 1;
        const int rc = spec_then_team(LW2, 13, 22, 23, ctx->dense_blobs2, (u8 *)ctx->arena2.p + spill_half, ctx->side[0]);   // W2 -> B
        if (rc != AVK_OK) return rc;
    } else {
        // small batches: W -> warp search / score kernels (8 KB / 5 KB per warp); the search kernel's rejects (A) are hard clusters
        const int small_ctas = (int)std::min<u64>((u64)SEARCH.ctas, (n + 7) / 8);
        launch_stage(ctx, R, SEARCH, tier_args(ctx, LW, 12, 0, LA, 1, SEARCH.arena_bytes, nullptr), small_ctas, ctx->side[0]);                                         // -> blobs, rejects -> A
        launch_stage(ctx, R, SCORE, tier_args(ctx, LW, 12, 2, LA2, 15, SCORE.arena_bytes, nullptr), (int)std::min<u64>((u64)SCORE.ctas, (n + 7) / 8), ctx->side[0]);    // rejects -> A2
        ctx->launches += 2;
        const int rc = spec_then_team(LA, 1, 22, 23, ctx->dense_blobs2, (u8 *)ctx->arena2.p + spill_half, ctx->side[0]);     // A -> B
        if (rc != AVK_OK) return rc;
    }
    CK(cudaEventRecord(ctx->ev_join[0], ctx->side[0]));
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[0], 0));
    CK(cudaEventRecord(ctx->tev[2], ctx->stream));
    {
        TierArgs a = tier_args(ctx, LA2, 15, 16, LB, 5, S1.arena_bytes, nullptr);
        a.spill_base = (u8 *)ctx->arena2.p; a.spill_bytes = 1u << 20;
        launch_stage(ctx, R, S1, a, S1.ctas, ctx->stream);                                   // A2 -> B  (score kernel's rejects, rare; empty with the thread stage)
    }
    {
        TierArgs a = tier_args(ctx, LB, 5, 9, LD, 7, G0.arena_bytes, (u8 *)ctx->arena.p);
        a.wide_b0 = ctx->wide_b0;                                                            // SV-sized events: cooperative tier
        launch_stage(ctx, R, G0, a, G0.ctas, ctx->stream);                                   // B -> D   (2 MB global arenas)
    }
    CK(cudaEventRecord(ctx->tev[3], ctx->stream));
    ctx->launches += 3;
    CK(cudaGetLastError());
    return AVK_OK;
}

// Rare: clusters that overflow 2 MB per warp or carry SV-sized events (list D): one cluster per CTA, wide wavefronts
// advanced by the whole CTA; 256 MB arenas, then 2 GB (last resort).  Host-synchronised.
static int run_big_tiers(avk_ctx *ctx, const CompareRun &R, u32 n_work) {
    const int sm = ctx->sm_count;
    u32 *ctrs = (u32 *)ctx->counters.p;
    Stage big[2] = {{MODE_COOP, false, 1, ctx->coop_arena0, sm, 1}, {MODE_COOP, false, 1, ctx->coop_arena1, 16, 1}};
    const u32 *cur = (u32 *)ctx->fail_d.p;
    u32 *other = (u32 *)ctx->fail_c.p;
    for (int t = 0; t < 2 && n_work > 0; ++t) {
        big[t].ctas = (int)std::min<u64>((u64)big[t].ctas, n_work);           // one cluster per CTA
        if (n_work > 1 && n_work <= 4096) { k_sort_biggest_first<<<1, 1024, 0, ctx->stream>>>(R.db, (u32 *)cur, n_work); ctx->launches += 1; }
        ENSURE(ctx->arena, (size_t)big[t].ctas * big[t].warps * (size_t)big[t].arena_bytes);
        CK(cudaMemsetAsync(ctrs + 32, 0, 8, ctx->stream));
        if (getenv("AVK_DEBUG")) cudaEventRecord(ctx->dbg[0], ctx->stream);
        TierArgs a = tier_args(ctx, cur, 0, 32, other, 33, big[t].arena_bytes, (u8 *)ctx->arena.p);
        a.n_work_ptr = nullptr; a.n_work = n_work; a.last_tier = t == 1;
        launch_stage(ctx, R, big[t], a, big[t].ctas, ctx->stream);
        ctx->launches += 1;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(ctx->h_pin + 64, ctrs + 32, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        if (getenv("AVK_DEBUG")) {
            float ms = 0;
            cudaEventRecord(ctx->dbg[1], ctx->stream); cudaEventSynchronize(ctx->dbg[1]); cudaEventElapsedTime(&ms, ctx->dbg[0], ctx->dbg[1]);
            fprintf(stderr, "[avk] big tier %d (cooperative, %lld MB): %u clusters in, %u rejected, %.1f ms\n", t, big[t].arena_bytes >> 20, n_work, ctx->h_pin[65], ms);
        }
        n_work = ctx->h_pin[65];
        const u32 *tmp = cur; cur = other; other = (u32 *)tmp;
    }
    return AVK_OK;
}

// Summary counters: fold the partial tables (in-kernel totals), or -- when strata are requested -- reduce the per-region
// rows (k_reduce also sums the strata).  Idempotent: may be run again after the cooperative tiers added their clusters.
static int run_finalize(avk_ctx *ctx, const CompareRun &R) {
    const u64 n = ctx->n_regions;
    unsigned long long *tot = (unsigned long long *)ctx->totals.p;
    if (!R.strata) {
        k_fold_slots<<<1, 320, 0, ctx->stream>>>((const unsigned long long *)ctx->tot_slots.p, tot);
        ctx->launches += 1;
    } else {
        CK(cudaMemsetAsync(tot, 0, 8 * RED_COLS + 64, ctx->stream));
        CK(cudaMemsetAsync(ctx->strat_totals.p, 0, 8ull * RED_COLS * R.n_strata, ctx->stream));
        if (n) {
            k_reduce<<<(unsigned)std::min<u64>(n, (u64)ctx->sm_count * 8), 288, 0, ctx->stream>>>(
                n, R.out.status, R.out.region_metrics, R.out.type_mask, tot, (u32 *)(tot + RED_COLS), tot + RED_COLS + 1, tot + RED_COLS + 2,
                R.strat_off, R.strat_idx, R.strat_mask, (unsigned long long *)ctx->strat_totals.p);
            ctx->launches += 1;
        }
    }
    CK(cudaGetLastError());
    return AVK_OK;
}

// pipeline counters + work counters travel back behind the kernels (pinned scratch: the copies do not block); ev_done marks
// the point where the pass and these copies are complete
static int queue_counter_copies(avk_ctx *ctx) {
    CK(cudaMemcpyAsync(ctx->h_pin, ctx->counters.p, 128, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_pin + 128, ctx->work_ctr.p, 40, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaEventRecord(ctx->ev_done, ctx->stream));
    return AVK_OK;
}

// Launches one compare pass over the resident batch; nothing waits for the device.
static int compare_launch(avk_ctx *ctx, const avk_compare_cfg *cfg, bool want_seq, bool want_rows, bool strata, u32 n_strata, bool strat_dev, bool want_contain, CompareRun &R) {
    const u64 n = ctx->n_regions, nv = ctx->n_variants;
    const bool rows = want_rows || strata;
    if (strat_dev || want_contain) ENSURE(ctx->st_mask, 8 * n);
    ENSURE(ctx->status, 4 * n); ENSURE(ctx->ed1, 4 * n); ENSURE(ctx->ed2, 4 * n);
    if (rows) ENSURE(ctx->region_metrics, 8ull * RED_COLS * n);
    ENSURE(ctx->type_mask, 2 * n);
    ENSURE(ctx->vexp, nv); ENSURE(ctx->vobs, nv); ENSURE(ctx->vcls, nv);
    ENSURE(ctx->totals, 8 * RED_COLS + 64);
    ENSURE(ctx->tot_slots, 8ull * TOT_SLOTS * TOT_STRIDE);
    ENSURE(ctx->counters, 256);
    ENSURE(ctx->work_ctr, 64);
    if (strata) ENSURE(ctx->strat_totals, 8ull * RED_COLS * n_strata);
    CK(cudaMemsetAsync(ctx->work_ctr.p, 0, 64, ctx->stream));
    CK(cudaMemsetAsync(ctx->tot_slots.p, 0, 8ull * TOT_SLOTS * TOT_STRIDE, ctx->stream));
    // digest buffers are sized from a host-side upper bound, so no device round trip is needed
    ENSURE(ctx->digest, (size_t)n * (PH_SIZE + 32) + (size_t)VI_SIZE * nv + (size_t)ctx->pool_len + 256);
    ENSURE(ctx->digest_sizes, 8 * (n + 1));
    ENSURE(ctx->digest_offs, 8 * (n + 1));
    R.db = dev_batch(ctx);
    DevCompareOut &out = R.out;
    out.status = (int *)ctx->status.p; out.ed1 = (u32 *)ctx->ed1.p; out.ed2 = (u32 *)ctx->ed2.p;
    out.region_metrics = rows ? (u64 *)ctx->region_metrics.p : nullptr;
    out.tot_slots = strata ? nullptr : (unsigned long long *)ctx->tot_slots.p;
    out.type_mask = (uint16_t *)ctx->type_mask.p;
    out.vexp = biased<u8>(ctx->vexp, ctx->v_base); out.vobs = biased<u8>(ctx->vobs, ctx->v_base); out.vcls = biased<u8>(ctx->vcls, ctx->v_base);
    out.seq_off = want_seq ? (const u64 *)ctx->seq_off.p : nullptr;
    out.seq_len = (u32 *)ctx->seq_len.p; out.seq_pool = biased<u8>(ctx->seq_pool, ctx->seq_base);
    R.cfg = *cfg;
    R.strata = strata; R.n_strata = n_strata;
    R.strat_off = (strata && !strat_dev) ? (const u64 *)ctx->strat_off.p : nullptr;
    R.strat_idx = (strata && !strat_dev) ? biased<const u32>(ctx->strat_idx, ctx->strat_base) : nullptr;
    R.strat_mask = (strata && strat_dev) ? (const u64 *)ctx->st_mask.p : nullptr;
    R.want_contain = strat_dev || want_contain;
    ctx->have_result = ctx->have_merge = ctx->result_has_seq = false;

    CK(cudaEventRecord(ctx->ev[0], ctx->stream));
    int rc = run_alt_ed(ctx, R.db);
    if (rc != AVK_OK) return rc;
    rc = run_prepare(ctx, R.db);
    if (rc != AVK_OK) return rc;
    CK(cudaEventRecord(ctx->ev[1], ctx->stream));
    if (R.want_contain && n) {
        const avk_ctx *so = ref_of(ctx);        // a lane reads its owner's interval tables
        k_strat_contain<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(R.db, n, so->st_n, so->st_contigs, (const u64 *)so->st_off.p,
                                                                              (const u32 *)so->st_first.p, (const u32 *)so->st_pmax.p, (u64 *)ctx->st_mask.p);
        ctx->launches += 1;
    }
    rc = run_compare_pipeline(ctx, R);
    if (rc != AVK_OK) return rc;
    CK(cudaEventRecord(ctx->ev[2], ctx->stream));
    CK(cudaEventRecord(ctx->ev[3], ctx->stream));
    rc = run_finalize(ctx, R);
    if (rc != AVK_OK) return rc;
    CK(cudaEventRecord(ctx->ev[4], ctx->stream));
    ctx->result_has_rows = rows;
    ctx->result_has_seq = want_seq && cfg->enable_sequences;   // (the kernels emit the bundle only under enable_sequences)
    ctx->result_has_contain = R.want_contain;
    return queue_counter_copies(ctx);
}

// Waits for the pass; if SV-sized clusters were left for the cooperative tiers, runs them and the summary again.
// *redo is set when outputs copied to the host before this call are stale.
static int compare_finish(avk_ctx *ctx, const CompareRun &R, bool *redo) {
    if (redo) *redo = false;
    CK(cudaEventSynchronize(ctx->ev_done));          // (not the stream: in a streamed call the next bin's kernels are queued behind)
    const u32 *h = ctx->h_pin;
    if (ctx->n_regions) {
        for (int t = 0; t < 3; ++t) cudaEventElapsedTime(&ctx->tier_ms[t], ctx->tev[t], ctx->tev[t + 1]);
        ctx->tier_fail[0] = h[1]; ctx->tier_fail[1] = h[5]; ctx->tier_fail[2] = h[7];
        if (h[7] > 0) {
            int rc = run_big_tiers(ctx, R, h[7]);
            if (rc != AVK_OK) return rc;
            CK(cudaEventRecord(ctx->ev[2], ctx->stream));
            CK(cudaEventRecord(ctx->ev[3], ctx->stream));
            rc = run_finalize(ctx, R);
            if (rc != AVK_OK) return rc;
            CK(cudaEventRecord(ctx->ev[4], ctx->stream));
            rc = queue_counter_copies(ctx);
            if (rc != AVK_OK) return rc;
            CK(cudaEventSynchronize(ctx->ev_done));
            if (redo) *redo = true;
        }
    } else {
        for (int t = 0; t < 3; ++t) { ctx->tier_ms[t] = 0; ctx->tier_fail[t] = 0; }
    }
    ctx->have_result = true;
    return AVK_OK;
}

static int fetch_timings(avk_ctx *ctx) {
    CK(cudaEventSynchronize(ctx->ev[4]));
    cudaEventElapsedTime(&ctx->last_ms[0], ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&ctx->last_ms[1], ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&ctx->last_ms[2], ctx->ev[2], ctx->ev[3]);
    cudaEventElapsedTime(&ctx->last_ms[3], ctx->ev[3], ctx->ev[4]);
    cudaEventElapsedTime(&ctx->last_ms[4], ctx->ev[0], ctx->ev[4]);
    CK(cudaEventSynchronize(ctx->ev_done));
    const unsigned long long *w = (const unsigned long long *)(ctx->h_pin + 128);
    ctx->last_work.alignments = w[0]; ctx->last_work.cells = w[1]; ctx->last_work.matched_bases = w[2];
    ctx->last_work.search_pops = w[3]; ctx->last_work.exact_pops = w[4];
    return AVK_OK;
}

#define DL(dst, buf, bytes)                                                                                     \
    do {                                                                                                        \
        if ((dst) && (bytes)) CK(cudaMemcpyAsync((dst), (buf).p, (bytes), cudaMemcpyDeviceToHost, ds)); \
    } while (0)

// Partial results of one bin: what the host adds up over bins (wrapping u64, like the reference's AddAssign).
struct BinTotals {
    unsigned long long tot[RED_COLS + 8];
    std::vector<u64> strat;
};

// Queues the device->host copies of the resident bin's results INTO THE CALLER'S ARRAYS AT THE BIN'S OFFSETS (regions from
// ctx->lo, variants from ctx->v_base); totals go to `bt` (pinned scratch first).  No synchronisation here.
static int download_compare_async(avk_ctx *ctx, avk_compare_out *out, bool want_seq, u64 seq_bytes) {
    const u64 n = ctx->n_regions, nv = ctx->n_variants, lo = ctx->lo, vb = ctx->v_base;
    const cudaStream_t ds = ctx->dn ? ctx->dn : ctx->stream;
    // st_mask holds whatever an earlier pass left there, possibly for a smaller batch
    if (out->containment && n && !ctx->result_has_contain) {
        ctx->err = "containment masks were not computed by this run (avk_compare_run_resident never computes them)";
        return AVK_ERR_INVALID;
    }
    if (ctx->dn) CK(cudaStreamWaitEvent(ctx->dn, ctx->ev_done, 0));
    DL(out->status ? out->status + lo : nullptr, ctx->status, 4 * n);
    DL(out->ed1 ? out->ed1 + lo : nullptr, ctx->ed1, 4 * n);
    DL(out->ed2 ? out->ed2 + lo : nullptr, ctx->ed2, 4 * n);
    if (out->region_metrics && n) {
        if (!ctx->result_has_rows) { ctx->err = "per-region metric rows were not kept by this run (AVK_CMP_KEEP_REGION_ROWS)"; return AVK_ERR_INVALID; }
        DL(out->region_metrics + lo * RED_COLS, ctx->region_metrics, 8ull * RED_COLS * n);
    }
    DL(out->type_mask ? out->type_mask + lo : nullptr, ctx->type_mask, 2 * n);
    DL(out->var_expected ? out->var_expected + vb : nullptr, ctx->vexp, nv);
    DL(out->var_observed ? out->var_observed + vb : nullptr, ctx->vobs, nv);
    DL(out->var_class ? out->var_class + vb : nullptr, ctx->vcls, nv);
    CK(cudaMemcpyAsync(ctx->h_pin + 256, ctx->totals.p, 8 * RED_COLS + 64, cudaMemcpyDeviceToHost, ds));
    if (out->containment) DL(out->containment + lo, ctx->st_mask, 8 * n);
    if (want_seq) {
        DL(out->seq_len + lo * 5, ctx->seq_len, 4 * 5 * n);
        DL(out->seq_pool + ctx->seq_base, ctx->seq_pool, seq_bytes);
    }
    return AVK_OK;
}

// after the download stream has been synchronised: collect totals (+ strata) of this bin
static int collect_totals(avk_ctx *ctx, const avk_compare_out *out, bool strata, BinTotals &bt) {
    memcpy(bt.tot, ctx->h_pin + 256, 8 * RED_COLS + 64);
    bt.strat.clear();
    if (strata) {
        bt.strat.resize((size_t)RED_COLS * out->n_strata);
        const cudaStream_t ds = ctx->dn ? ctx->dn : ctx->stream;
        CK(cudaMemcpyAsync(bt.strat.data(), ctx->strat_totals.p, 8ull * RED_COLS * out->n_strata, cudaMemcpyDeviceToHost, ds));
        CK(cudaStreamSynchronize(ds));
    }
    return AVK_OK;
}

static void store_totals(avk_compare_out *out, const BinTotals &bt, bool strata, bool accumulate) {
    if (out->totals) for (int j = 0; j < RED_COLS; ++j) out->totals[j] = (accumulate ? out->totals[j] : 0) + bt.tot[j];
    if (out->totals_mask) *out->totals_mask = (uint16_t)((accumulate ? *out->totals_mask : 0) | (bt.tot[RED_COLS] & 0xffff));
    if (out->solved_blocks) *out->solved_blocks = (accumulate ? *out->solved_blocks : 0) + bt.tot[RED_COLS + 1];
    if (out->error_blocks) *out->error_blocks = (accumulate ? *out->error_blocks : 0) + bt.tot[RED_COLS + 2];
    if (strata && out->strat_totals)
        for (size_t j = 0; j < bt.strat.size(); ++j) out->strat_totals[j] = (accumulate ? out->strat_totals[j] : 0) + bt.strat[j];
}

// optional inputs that travel with the outputs struct: sequence-bundle layout and stratum membership of the bin
static int prepare_outputs_on_device(avk_ctx *ctx, const avk_compare_out *out, u64 n_total, bool &want_seq, u64 &seq_bytes, bool &strata, bool &strat_dev) {
    const u64 n = ctx->n_regions, lo = ctx->lo;
    want_seq = out->seq_off && out->seq_len && out->seq_pool;
    seq_bytes = 0;
    ctx->seq_base = 0; ctx->strat_base = 0;
    if (want_seq) {
        for (u64 i = lo * 5; i < (lo + n) * 5; ++i) if (out->seq_off[i] > out->seq_off[i + 1]) { ctx->err = "seq_off is not monotone"; return AVK_ERR_INVALID; }
        ctx->seq_base = out->seq_off[lo * 5];
        seq_bytes = out->seq_off[(lo + n) * 5] - ctx->seq_base;
        UPLOAD(ctx->seq_off, out->seq_off + lo * 5, 8 * (n * 5 + 1));
        ENSURE(ctx->seq_len, 4 * 5 * n + 4);
        ENSURE(ctx->seq_pool, seq_bytes);
        CK(cudaMemsetAsync(ctx->seq_len.p, 0, 4 * 5 * n + 4, ctx->stream));
    }
    strata = strata_wanted(out);
    strat_dev = strata && !out->strat_off;
    if ((strat_dev || out->containment) && (ref_of(ctx)->st_n == 0 || (strat_dev && ref_of(ctx)->st_n != out->n_strata) || ref_of(ctx)->st_contigs != (u32)ref_of(ctx)->contig_lens.size())) {
        ctx->err = "the device containment lookup needs avk_set_stratifications (same number of strata as n_strata, contigs as the reference)";
        return AVK_ERR_INVALID;
    }
    if (strata && !strat_dev) {
        const u64 s0 = out->strat_off[lo], s1 = out->strat_off[lo + n];
        bool bad = s0 > s1 || (s1 > s0 && !out->strat_idx);
        for (u64 r = lo; r < lo + n && !bad; ++r) bad = out->strat_off[r] > out->strat_off[r + 1];
        for (u64 s = s0; s < s1 && !bad; ++s) bad = out->strat_idx[s] >= out->n_strata;
        if (bad) { ctx->err = "strat_off / strat_idx are inconsistent (not monotone, or a stratum index >= n_strata)"; return AVK_ERR_INVALID; }
        ctx->strat_base = s0;
        UPLOAD(ctx->strat_off, out->strat_off + lo, 8 * (n + 1));
        UPLOAD(ctx->strat_idx, out->strat_idx + s0, 4 * (s1 - s0));
    }
    (void)n_total;
    return AVK_OK;
}

// One contiguous bin [lo, hi) of the batch on this context's GPU; results land in the caller's arrays at the bin's
// offsets, the bin's summary counters in `bt`.  bin_enqueue queues upload, kernels and download without waiting for the
// device; bin_finish waits for them (and runs the cooperative tiers if SV-sized clusters were left over).
static inline double host_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
struct BinPending {
    CompareRun R;
    bool want_seq = false, strata = false;
    u64 seq_bytes = 0;
};
static int bin_enqueue(avk_ctx *ctx, const avk_region_batch *batch, u64 lo, u64 hi, const avk_compare_cfg *cfg, avk_compare_out *out, BinPending &P) {
    CK(cudaSetDevice(ctx->device));
    const bool timing = getenv("AVK_TIMING") != nullptr;
    const double t0 = timing ? host_ms() : 0;
    BinScan sc;
    int rc = bin_range(ctx, batch, lo, hi, sc);
    if (rc != AVK_OK) return rc;
    const double t1 = timing ? host_ms() : 0;
    rc = upload_batch(ctx, batch, sc);
    if (rc != AVK_OK) return rc;
    if (timing) fprintf(stderr, "[avk]   enqueue: queueing the uploads + host scan beside them %.2f ms\n", host_ms() - t1);
    (void)t0;
    bool strat_dev;
    rc = prepare_outputs_on_device(ctx, out, batch->n_regions, P.want_seq, P.seq_bytes, P.strata, strat_dev);
    if (rc != AVK_OK) return rc;
    rc = uploads_done(ctx);
    if (rc != AVK_OK) return rc;
    const bool want_rows = out->region_metrics != nullptr || (cfg->flags & AVK_CMP_KEEP_REGION_ROWS);
    rc = compare_launch(ctx, cfg, P.want_seq, want_rows, P.strata, P.strata ? out->n_strata : 0, strat_dev, out->containment != nullptr, P.R);
    if (rc != AVK_OK) return rc;
    return download_compare_async(ctx, out, P.want_seq, P.seq_bytes);
}
static int bin_finish(avk_ctx *ctx, avk_compare_out *out, const BinPending &P, BinTotals &bt) {
    CK(cudaSetDevice(ctx->device));
    bool redo = false;
    int rc = compare_finish(ctx, P.R, &redo);
    if (rc != AVK_OK) return rc;
    if (redo) {
        rc = download_compare_async(ctx, out, P.want_seq, P.seq_bytes);
        if (rc != AVK_OK) return rc;
    }
    CK(cudaStreamSynchronize(ctx->dn ? ctx->dn : ctx->stream));
    rc = collect_totals(ctx, out, P.strata, bt);
    if (rc != AVK_OK) return rc;
    return fetch_timings(ctx);
}
static int compare_bin(avk_ctx *ctx, const avk_region_batch *batch, u64 lo, u64 hi, const avk_compare_cfg *cfg, avk_compare_out *out, BinTotals &bt) {
    BinPending P;
    const bool timing = getenv("AVK_TIMING") != nullptr;
    const double t0 = timing ? host_ms() : 0;
    int rc = bin_enqueue(ctx, batch, lo, hi, cfg, out, P);
    if (rc != AVK_OK) { cudaStreamSynchronize(ctx->stream); return rc; }
    const double t1 = timing ? host_ms() : 0;
    rc = bin_finish(ctx, out, P, bt);
    if (timing) fprintf(stderr, "[avk] one bin: %llu regions, host enqueue %.2f ms (scan + async copies + launches), wait %.2f ms, device pass %.2f ms\n",
                        (unsigned long long)(hi - lo), t1 - t0, host_ms() - t1, ctx->last_ms[4]);
    return rc;
}

extern "C" int avk_compare_batch_range(avk_ctx *ctx, const avk_region_batch *batch, uint64_t lo, uint64_t hi,
                                       const avk_compare_cfg *cfg, avk_compare_out *out) {
    if (!ctx) return AVK_ERR_INVALID;
    if (!cfg || !out || !out->status) { ctx->err = "null cfg/out/status"; return AVK_ERR_INVALID; }
    int rc = validate_batch(ctx, batch, true);
    if (rc != AVK_OK) return rc;
    if (lo > hi || hi > batch->n_regions) { ctx->err = "region range outside the batch"; return AVK_ERR_INVALID; }
    BinTotals bt;
    rc = compare_bin(ctx, batch, lo, hi, cfg, out, bt);
    if (rc != AVK_OK) return rc;
    store_totals(out, bt, strata_wanted(out), false);
    return AVK_OK;
}

// Large batches on one GPU are STREAMED: the batch is cut into contiguous bins (avk_partition_regions) that go through
// the device one after the other on this context's compute streams, alternating between two sets of buffers (this context
// and a sibling lane that shares its streams and reads its reference).  A bin's host->device copies run on its lane's
// `up` stream, its device->host copies on the lane's `dn` stream, so bin k+1 is uploaded (and scanned on the host) while
// bin k is being solved and bin k-1 is travelling back; results land in the caller's arrays at the bins' offsets and the
// bins' counters are added up, exactly as avk_compare_batch_multi does across GPUs.  One host thread; the host waits for
// bin k-2 before it re-uses that lane for bin k, so at most two bins are in flight.
static int streamed_lane(avk_ctx *ctx, avk_ctx **lane) {
    if (!ctx->sib[0]) {
        avk_ctx *sb = nullptr;
        const int rc = avk_create(ctx->device, &sb);
        if (rc != AVK_OK) { ctx->err = "streamed compare: could not create the second lane"; return rc; }
        // the lane launches on the owner's compute streams: bins stay in order and never compete for the SMs
        for (auto &st : sb->side) if (st) cudaStreamDestroy(st);
        cudaStreamDestroy(sb->stream);
        sb->stream = ctx->stream; sb->side[0] = ctx->side[0]; sb->side[1] = ctx->side[1];
        sb->own_streams = false;
        sb->ref_owner = ctx;
        sb->pipe_bins = 0;
        ctx->sib[0] = sb;
    }
    *lane = ctx->sib[0];
    return AVK_OK;
}
static int compare_streamed(avk_ctx *ctx, const avk_region_batch *batch, const avk_compare_cfg *cfg, avk_compare_out *out, u32 n_bins) {
    avk_ctx *lanes[2] = {ctx, nullptr};
    int rc = streamed_lane(ctx, &lanes[1]);
    if (rc != AVK_OK) return rc;
    CK(cudaSetDevice(ctx->device));
    for (avk_ctx *l : lanes) {
        l->dense_n = ctx->dense_n; l->thread_pop_budget = ctx->thread_pop_budget; l->thread_batch_min = ctx->thread_batch_min; l->use_spec_search = ctx->use_spec_search; l->use_thread_stage = ctx->use_thread_stage; l->sort_shapes = ctx->sort_shapes; l->thread_min_regions = ctx->thread_min_regions;
        l->coop_arena0 = ctx->coop_arena0; l->coop_arena1 = ctx->coop_arena1; l->coop_cap_ints = ctx->coop_cap_ints; l->wide_b0 = ctx->wide_b0;
        for (auto &st : l->copy_streams) if (!st) CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        l->up = l->copy_streams[0]; l->dn = l->copy_streams[1];
    }
    std::vector<u64> cuts(n_bins + 1);
    avk_partition_regions(batch, n_bins, cuts.data());
    std::vector<BinTotals> bts(n_bins);
    BinPending pend[2];
    rc = AVK_OK;
    avk_ctx *failed = nullptr;
    const bool timing = getenv("AVK_TIMING") != nullptr;
    const double t0 = timing ? host_ms() : 0;
    for (u32 k = 0; k < n_bins + 2 && rc == AVK_OK; ++k) {
        const double ta = timing ? host_ms() : 0;
        if (k >= 2) { rc = bin_finish(lanes[k & 1], out, pend[k & 1], bts[k - 2]); if (rc != AVK_OK) failed = lanes[k & 1]; }
        const double tb = timing ? host_ms() : 0;
        if (rc == AVK_OK && k < n_bins) { rc = bin_enqueue(lanes[k & 1], batch, cuts[k], cuts[k + 1], cfg, out, pend[k & 1]); if (rc != AVK_OK) failed = lanes[k & 1]; }
        if (timing) fprintf(stderr, "[avk] streamed step %u at %.2f ms: wait for bin k-2 %.2f ms (its device pass %.2f ms), enqueue bin k %.2f ms\n", k, ta - t0, tb - ta,
                            k >= 2 ? lanes[k & 1]->last_ms[4] : 0.f, host_ms() - tb);
    }
    // leave the streamed mode (the resident entry points copy on the compute stream); on an error nothing may stay in flight
    cudaStreamSynchronize(ctx->stream);
    for (avk_ctx *l : lanes) {
        cudaStreamSynchronize(l->up); cudaStreamSynchronize(l->dn);
        l->up = l->dn = nullptr;
    }
    if (rc != AVK_OK) { if (failed && failed != ctx) ctx->err = failed->err; return rc; }
    const bool strata = strata_wanted(out);
    for (u32 k = 0; k < n_bins; ++k) store_totals(out, bts[k], strata, k > 0);
    return AVK_OK;
}

static int compare_lanes(avk_ctx *ctx, const avk_region_batch *batch, const avk_compare_cfg *cfg, avk_compare_out *out, int n);
extern "C" int avk_compare_batch(avk_ctx *ctx, const avk_region_batch *batch, const avk_compare_cfg *cfg, avk_compare_out *out) {
    if (!ctx) return AVK_ERR_INVALID;
    if (!batch) { ctx->err = "null batch"; return AVK_ERR_INVALID; }
    const int want_lanes = ctx->n_lanes;
    if (want_lanes > 1 && batch->n_regions >= ctx->lane_min_regions && !ctx->ref_owner && (ctx->pipe_bins == 0 || ctx->pipe_bins == 1)) {
        if (!cfg || !out || !out->status) { ctx->err = "null cfg/out/status"; return AVK_ERR_INVALID; }
        const int rc = validate_batch(ctx, batch, true);
        if (rc != AVK_OK) return rc;
        return compare_lanes(ctx, batch, cfg, out, want_lanes);
    }
    if (ctx->pipe_bins != 0 && ctx->pipe_bins != 1 && batch->n_regions >= ctx->pipe_min_regions && !ctx->ref_owner) {
        const u64 n_bins = ctx->pipe_bins > 1 ? (u64)ctx->pipe_bins : std::min<u64>(16, (batch->n_regions + ctx->pipe_bin_regions / 2) / ctx->pipe_bin_regions);
        if (n_bins >= 2) {
            if (!cfg || !out || !out->status) { ctx->err = "null cfg/out/status"; return AVK_ERR_INVALID; }
            const int rc = validate_batch(ctx, batch, true);
            if (rc != AVK_OK) return rc;
            return compare_streamed(ctx, batch, cfg, out, (u32)n_bins);
        }
    }
    return avk_compare_batch_range(ctx, batch, 0, batch->n_regions, cfg, out);
}

// ---- multi-GPU behind the C ABI (SURVEY 8e) ---------------------------------------------------------------------------
// Cost proxy per region: (variants + 1) * window + sum over variants of max(|allele0|, |allele1|)^2 (the SV tail is quadratic).
// cuts[k] = first region of bin k: the first index whose cumulative cost reaches k/n of the total (bins are contiguous in
// region_id order, so concatenating the bins' results restores the reference's output order, src/main.rs:271).
static inline u64 region_cost(const avk_region_batch *b, u64 r) {
    const u64 K = b->n_inputs, v0 = b->var_off[r * K], v1 = b->var_off[(r + 1) * K];
    u64 c = (v1 - v0 + 1) * (u64)(b->end[r] > b->start[r] ? b->end[r] - b->start[r] : 0);
    for (u64 v = v0; v < v1; ++v) { const u64 m = std::max(b->variants.a0_len[v], b->variants.a1_len[v]); c += m * m; }
    return c;
}
// The sums are taken per chunk of 16 Ki regions (by several host threads when the batch is large: this runs inside the timed
// call of the lane / multi-GPU entry points); a cut is then looked up in the chunk that holds it.
extern "C" int avk_partition_regions(const avk_region_batch *b, uint32_t n_bins, uint64_t *cuts) {
    if (!b || !cuts || n_bins == 0) return AVK_ERR_INVALID;
    const u64 n = b->n_regions, CH = 16384, n_ch = (n + CH - 1) / CH;
    std::vector<u64> chunk(n_ch + 1, 0);
    auto sum_chunks = [&](u64 c0, u64 c1) {
        for (u64 c = c0; c < c1; ++c) {
            u64 t = 0;
            for (u64 r = c * CH, e = std::min(n, r + CH); r < e; ++r) t += region_cost(b, r);
            chunk[c + 1] = t;
        }
    };
    const u64 n_thr = n >= 500000 ? std::min<u64>(8, std::max(1u, std::thread::hardware_concurrency())) : 1;
    if (n_thr > 1) {
        std::vector<std::thread> th;
        for (u64 t = 0; t < n_thr; ++t) th.emplace_back(sum_chunks, n_ch * t / n_thr, n_ch * (t + 1) / n_thr);
        for (auto &t : th) t.join();
    } else sum_chunks(0, n_ch);
    for (u64 c = 0; c < n_ch; ++c) chunk[c + 1] += chunk[c];
    const unsigned __int128 total = chunk[n_ch];
    cuts[0] = 0;
    for (uint32_t k = 1; k < n_bins; ++k) {
        // first r with cum[r + 1] * n_bins >= total * k, cum[r + 1] = cost of regions [0, r]
        u64 lo = 0, hi = n_ch;
        while (lo < hi) {                                   // first chunk whose inclusive sum reaches the target
            const u64 m = (lo + hi) >> 1;
            if ((unsigned __int128)chunk[m + 1] * n_bins < total * k) lo = m + 1; else hi = m;
        }
        u64 r = n;
        if (lo < n_ch) {
            u64 cum = chunk[lo];
            for (r = lo * CH; r < n; ++r) { cum += region_cost(b, r); if ((unsigned __int128)cum * n_bins >= total * k) break; }
        }
        cuts[k] = std::max(std::min(r, n), cuts[k - 1]);
    }
    cuts[n_bins] = n;
    return AVK_OK;
}

// One host thread per context (= per GPU); bin k goes to ctxs[k].  Every device copies its slice of the results straight into
// the caller's arrays at its bin offset -- the bins are contiguous, so on one node the "gather" is those copies -- and the
// summary counters of the bins are added on the host.  Every context must hold the reference (avk_set_reference).
static int compare_bins_concurrent(avk_ctx *const *ctxs, uint32_t n_ctx, const avk_region_batch *batch, const avk_compare_cfg *cfg, avk_compare_out *out) {
    avk_ctx *ctx = ctxs[0];
    std::vector<u64> cuts(n_ctx + 1);
    if (batch->n_regions && (!batch->variants.a0_len || !batch->variants.a1_len) && batch->variants.n_variants) { ctx->err = "null variant arrays"; return AVK_ERR_INVALID; }
    avk_partition_regions(batch, n_ctx, cuts.data());
    std::vector<BinTotals> bts(n_ctx);
    std::vector<int> rcs(n_ctx, AVK_OK);
    std::vector<std::thread> th;
    auto work = [&](uint32_t k) {
        if (!ctxs[k]) { rcs[k] = AVK_ERR_INVALID; return; }
        rcs[k] = compare_bin(ctxs[k], batch, cuts[k], cuts[k + 1], cfg, out, bts[k]);
    };
    for (uint32_t k = 1; k < n_ctx; ++k) th.emplace_back(work, k);
    work(0);                                                // the caller's thread takes the first bin
    for (auto &t : th) t.join();
    for (uint32_t k = 0; k < n_ctx; ++k)
        if (rcs[k] != AVK_OK) { if (k && ctxs[k]) ctx->err = "bin " + std::to_string(k) + ": " + ctxs[k]->err; return rcs[k]; }
    const bool strata = strata_wanted(out);
    for (uint32_t k = 0; k < n_ctx; ++k) store_totals(out, bts[k], strata, k > 0);
    return AVK_OK;
}
extern "C" int avk_compare_batch_multi(avk_ctx *const *ctxs, uint32_t n_ctx, const avk_region_batch *batch,
                                       const avk_compare_cfg *cfg, avk_compare_out *out) {
    if (!ctxs || n_ctx == 0 || !ctxs[0]) return AVK_ERR_INVALID;
    avk_ctx *ctx = ctxs[0];
    if (!cfg || !out || !out->status) { ctx->err = "null cfg/out/status"; return AVK_ERR_INVALID; }
    int rc = validate_batch(ctx, batch, true);
    if (rc != AVK_OK) return rc;
    return compare_bins_concurrent(ctxs, n_ctx, batch, cfg, out);
}

// One large batch on ONE GPU, as concurrent lanes: sibling contexts of this device (own streams and buffers, this context's
// reference and stratification tables) take one contiguous bin each.  Measured on the whole-genome batch (3.95 M clusters):
// see DESIGN.md section 5.
static int ensure_lanes(avk_ctx *ctx, int n) {
    if (ctx->lanes.empty()) ctx->lanes.push_back(ctx);
    while ((int)ctx->lanes.size() < n) {
        avk_ctx *l = nullptr;
        const int rc = avk_create(ctx->device, &l);
        if (rc != AVK_OK) { ctx->err = "compare lanes: could not create a sibling context"; return rc; }
        l->ref_owner = ctx;
        l->n_lanes = 1;
        l->pipe_bins = 0;
        ctx->lanes.push_back(l);
    }
    for (size_t i = 1; i < ctx->lanes.size(); ++i) {
        avk_ctx *l = ctx->lanes[i];
        l->dense_n = ctx->dense_n; l->thread_pop_budget = ctx->thread_pop_budget; l->thread_batch_min = ctx->thread_batch_min; l->use_spec_search = ctx->use_spec_search;
        l->use_thread_stage = ctx->use_thread_stage; l->sort_shapes = ctx->sort_shapes; l->thread_min_regions = ctx->thread_min_regions;
        l->coop_arena0 = ctx->coop_arena0; l->coop_arena1 = ctx->coop_arena1; l->coop_cap_ints = ctx->coop_cap_ints; l->wide_b0 = ctx->wide_b0;
    }
    return AVK_OK;
}
static int compare_lanes(avk_ctx *ctx, const avk_region_batch *batch, const avk_compare_cfg *cfg, avk_compare_out *out, int n) {
    int rc = ensure_lanes(ctx, n);
    if (rc != AVK_OK) return rc;
    rc = compare_bins_concurrent(ctx->lanes.data(), (uint32_t)n, batch, cfg, out);
    ctx->have_batch = ctx->have_result = ctx->have_merge = ctx->result_has_seq = false;   // the owner holds one bin only: nothing "resident" to re-run or download
    // the owner's timings describe the call: the longest device pass of the lanes
    for (int i = 1; i < n; ++i) if (ctx->lanes[i]->last_ms[4] > ctx->last_ms[4]) for (int k = 0; k < 5; ++k) ctx->last_ms[k] = ctx->lanes[i]->last_ms[k];
    return rc;
}

// ------------------------------------------------------------------------------------ region builder (SURVEY 8f N1)
// src/parsing/region_generation.rs:352-469 as sorts, scans and gathers; see include/aardvark_b200.h.
// A variant closes the open cluster iff its position reaches the running maximum of (pos + ref_len + flank) -- and the
// maximum over ALL earlier variants equals the maximum inside the open cluster whenever that comparison matters (every
// earlier cluster ended at or before the position that opened this one), so one exclusive max-scan gives the breaks.
struct MaxOp64 { __device__ __forceinline__ u64 operator()(u64 a, u64 b) const { return a > b ? a : b; } };

// Sort key (contig << 32 | position) of every variant that lies fully inside one BED interval of its contig (0-based half-open,
// sorted, non-overlapping): get_variant_containment (:796-812) against the first interval that ends behind the variant's
// start -- for every earlier interval the variant is After, and Before / Overlapping variants are consumed without being used
// (:388-391, :438-442).  Everything else gets the key ~0 and sorts to the end.  ivl[i] = 1 + global index of the interval.
__global__ void __launch_bounds__(256) k_rb_keys(u64 nv, const u32 *pos, const u32 *l0, const u32 *vcontig, u32 contig0, const u64 *contig_len, u32 n_contigs,
                                                 const u64 *ifirst, const u32 *istart, const u32 *iend, u64 *key, u32 *idx, u32 *ivl) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nv) return;
    idx[i] = (u32)i;
    const u32 c = vcontig ? vcontig[i] : contig0;
    u64 k = ~0ull;
    u32 tag = 0;
    if (c < n_contigs && (u64)pos[i] + l0[i] <= contig_len[c]) {              // fully inside the contig (:551 against the full region)
        if (!ifirst) { k = ((u64)c << 32) | pos[i]; tag = 1 + c; }            // no BED: one interval spanning each contig
        else {
            u64 lo = ifirst[c], hi = ifirst[c + 1];
            const u64 end_c = hi;
            while (lo < hi) { const u64 m = (lo + hi) >> 1; if (iend[m] <= pos[i]) lo = m + 1; else hi = m; }   // first interval with end > pos
            if (lo < end_c && pos[i] >= istart[lo] && (u64)pos[i] + l0[i] <= iend[lo]) { k = ((u64)c << 32) | pos[i]; tag = 1 + (u32)lo; }
        }
    }
    key[i] = k; ivl[i] = tag;
}
// per sorted variant: (interval tag << 32 | window end it asks for); the exclusive running maximum of these is, inside one
// interval, the open cluster's window end (intervals come in increasing tag order, so a later interval's entries always win)
__global__ void __launch_bounds__(256) k_rb_vend(u64 nv, const u64 *key, const u32 *idx, const u32 *l0, const u32 *ivl, const u64 *contig_len, u32 flank,
                                                 u64 *vend, unsigned long long *n_valid) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nv) return;
    const bool valid = key[i] != ~0ull;
    const u32 p = (u32)key[i], c = (u32)(key[i] >> 32);
    vend[i] = valid ? (((u64)ivl[idx[i]] << 32) | (u32)min((u64)p + l0[idx[i]] + flank, contig_len[c])) : 0ull;   // :411-429
    if (valid && (i + 1 == nv || key[i + 1] == ~0ull)) *n_valid = i + 1;
    if (i == 0 && !valid) *n_valid = 0;
}
__global__ void __launch_bounds__(256) k_rb_flags(u64 nv, const u64 *key, const u64 *vend, const u64 *pmax, u32 *flag) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nv) return;
    // a new cluster: first variant of its interval (:379-383 fresh window per interval), or pos >= window_end (:396-409)
    flag[i] = (key[i] != ~0ull && ((pmax[i] >> 32) != (vend[i] >> 32) || (u32)key[i] >= (u32)pmax[i])) ? 1u : 0u;
}
// per sorted variant: cluster id, grouping key (cluster, input); per cluster: window and ids
__global__ void __launch_bounds__(256) k_rb_clusters(u64 nvalid, const u64 *key, const u32 *idx, const u32 *cid1, const u32 *flag,
                                                     const u64 *pmax, const u64 *vend, const u64 *input_off, u32 K, u32 flank,
                                                     u64 first_region_id, u64 *key2, u64 *region_id, u32 *rcontig, u32 *start, u32 *end) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nvalid) return;
    const u32 c = cid1[i] - 1;                                                // inclusive sum of the break flags
    u32 k = 0;
    while (k + 1 < K && input_off[k + 1] <= idx[i]) ++k;
    key2[i] = (u64)c * K + k;
    const u32 p = (u32)key[i];
    if (flag[i]) { start[c] = p > flank ? p - flank : 0u; region_id[c] = first_region_id + c; rcontig[c] = (u32)(key[i] >> 32); }
    if (i + 1 == nvalid || flag[i + 1]) {                                     // running maximum at the cluster's last variant (same interval only)
        const u32 own = (u32)vend[i], before = (pmax[i] >> 32) == (vend[i] >> 32) ? (u32)pmax[i] : 0u;
        end[c] = max(own, before);
    }
}
__global__ void __launch_bounds__(256) k_rb_varoff(u64 n_seg, u64 nvalid, const u64 *key2_sorted, u64 *var_off) {
    const u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (s > n_seg) return;
    u64 lo = 0, hi = nvalid;                                                  // first sorted variant with key2 >= s
    while (lo < hi) { const u64 m = (lo + hi) >> 1; if (key2_sorted[m] < s) lo = m + 1; else hi = m; }
    var_off[s] = lo;
}
__global__ void __launch_bounds__(256) k_rb_gather(u64 nvalid, const u32 *perm, const u32 *pos, const u8 *vt, const u8 *zy, const u32 *raw,
                                                   const u32 *l0, const u32 *l1, u32 *opos, u8 *ovt, u8 *ozy, u32 *oraw, u32 *ol0, u32 *ol1, u32 *alen) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nvalid) return;
    const u32 j = perm[i];
    opos[i] = pos[j]; ovt[i] = vt[j]; ozy[i] = zy[j]; oraw[i] = raw[j]; ol0[i] = l0[j]; ol1[i] = l1[j];
    alen[i] = l0[j] + l1[j];
}
__global__ void __launch_bounds__(256) k_rb_alleles(u64 nvalid, const u32 *perm, const u32 *aoff_in, const u32 *alen, const u32 *aoff_out,
                                                    const u8 *pool_in, u8 *pool_out) {
    const int lane = lane_id();
    const u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((u64)gridDim.x * blockDim.x) >> 5;
    for (u64 i = warp; i < nvalid; i += n_warps) {
        const u8 *src = pool_in + aoff_in[perm[i]];
        u8 *dst = pool_out + aoff_out[i];
        for (u32 t = lane; t < alen[i]; t += 32) dst[t] = src[t];
    }
}

static int build_regions_impl(avk_ctx *ctx, const avk_callsets *in, const uint32_t *variant_contig, uint32_t contig, const avk_bed_intervals *bed,
                              uint32_t flank, uint64_t first_region_id, uint64_t *n_regions_out, uint64_t *n_variants_out);
extern "C" int avk_build_regions(avk_ctx *ctx, const avk_callsets *in, uint32_t contig, uint32_t flank, uint64_t first_region_id,
                                 uint64_t *n_regions_out, uint64_t *n_variants_out) {
    if (!ctx) return AVK_ERR_INVALID;
    if (contig >= ctx->contig_lens.size()) { ctx->err = "avk_build_regions: unknown contig (call avk_set_reference first)"; return AVK_ERR_INVALID; }
    return build_regions_impl(ctx, in, nullptr, contig, nullptr, flank, first_region_id, n_regions_out, n_variants_out);
}
extern "C" int avk_build_regions_bed(avk_ctx *ctx, const avk_callsets *in, const uint32_t *variant_contig, const avk_bed_intervals *bed,
                                     uint32_t flank, uint64_t first_region_id, uint64_t *n_regions_out, uint64_t *n_variants_out) {
    if (!ctx) return AVK_ERR_INVALID;
    if (!variant_contig) { ctx->err = "avk_build_regions_bed: null variant_contig"; return AVK_ERR_INVALID; }
    if (bed) {
        if (bed->n_contigs != ctx->contig_lens.size() || !bed->first || (bed->first[bed->n_contigs] && (!bed->start || !bed->end))) {
            ctx->err = "avk_build_regions_bed: the interval table must cover the reference's contigs";
            return AVK_ERR_INVALID;
        }
        for (uint32_t c = 0; c < bed->n_contigs; ++c) {
            if (bed->first[c] > bed->first[c + 1]) { ctx->err = "avk_build_regions_bed: interval offsets are not monotone"; return AVK_ERR_INVALID; }
            for (uint64_t j = bed->first[c]; j < bed->first[c + 1]; ++j)
                if (bed->start[j] > bed->end[j] || (j > bed->first[c] && bed->start[j] < bed->end[j - 1])) {
                    ctx->err = "avk_build_regions_bed: intervals must be sorted and non-overlapping within a contig";
                    return AVK_ERR_INVALID;
                }
        }
        if (bed->first[bed->n_contigs] >= 0xfffffffeull) { ctx->err = "avk_build_regions_bed: too many intervals"; return AVK_ERR_INVALID; }
    }
    return build_regions_impl(ctx, in, variant_contig, 0, bed, flank, first_region_id, n_regions_out, n_variants_out);
}
static int build_regions_impl(avk_ctx *ctx, const avk_callsets *in, const uint32_t *variant_contig, uint32_t contig, const avk_bed_intervals *bed,
                              uint32_t flank, uint64_t first_region_id, uint64_t *n_regions_out, uint64_t *n_variants_out) {
    if (!ctx || !in || !n_regions_out || !n_variants_out || in->n_inputs == 0 || !in->input_off) return AVK_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    if (ctx->contig_lens.empty()) { ctx->err = "avk_build_regions: avk_set_reference has not been called"; return AVK_ERR_NO_REFERENCE; }
    const avk_variant_table &t = in->variants;
    const u64 nv = t.n_variants, K = in->n_inputs;
    const u32 n_contigs = (u32)ctx->contig_lens.size();
    if (in->input_off[K] != nv || nv >= 0xffffffffull || t.allele_pool_len >= 0xffffffffull) { ctx->err = "avk_build_regions: bad call-set table"; return AVK_ERR_INVALID; }
    for (u64 len : ctx->contig_lens) if (len > 0xffffffffull) { ctx->err = "avk_build_regions: contig longer than 2^32 - 1 bases"; return AVK_ERR_INVALID; }
    enum { T_POS, T_VT, T_ZY, T_RAW, T_AOFF, T_L0, T_L1, T_POOL, T_KEY, T_IDX, T_KEY_S, T_IDX_S, T_VEND, T_PMAX, T_FLAG, T_CID, T_KEY2, T_KEY2_S, T_PERM, T_MISC, T_VCONTIG, T_IVL, T_IFIRST, T_ISTART };
    DevBuf *rb = ctx->rb;
    UPLOAD(rb[T_POS], t.position, 4 * nv); UPLOAD(rb[T_VT], t.variant_type, nv); UPLOAD(rb[T_ZY], t.zygosity, nv);
    UPLOAD(rb[T_RAW], t.raw_allele_space, 4 * nv); UPLOAD(rb[T_AOFF], t.allele_off, 4 * nv); UPLOAD(rb[T_L0], t.a0_len, 4 * nv);
    UPLOAD(rb[T_L1], t.a1_len, 4 * nv); UPLOAD(rb[T_POOL], t.allele_pool, t.allele_pool_len);
    for (int b : {T_IDX, T_IDX_S, T_FLAG, T_CID, T_PERM, T_IVL}) ENSURE(rb[b], 4 * nv);
    for (int b : {T_KEY, T_KEY_S, T_VEND, T_PMAX, T_KEY2, T_KEY2_S}) ENSURE(rb[b], 8 * nv);
    if (variant_contig) UPLOAD(rb[T_VCONTIG], variant_contig, 4 * nv);
    const u64 n_ivl = bed ? bed->first[bed->n_contigs] : 0;
    if (bed) {
        UPLOAD(rb[T_IFIRST], bed->first, 8 * ((u64)n_contigs + 1));
        ENSURE(rb[T_ISTART], 8 * n_ivl + 16);
        if (n_ivl) {
            CK(cudaMemcpyAsync(rb[T_ISTART].p, bed->start, 4 * n_ivl, cudaMemcpyHostToDevice, ctx->stream));
            CK(cudaMemcpyAsync((u32 *)rb[T_ISTART].p + n_ivl, bed->end, 4 * n_ivl, cudaMemcpyHostToDevice, ctx->stream));
        }
    }
    ENSURE(rb[T_MISC], 8 * (K + 1) + 64);
    u64 *d_input_off = (u64 *)rb[T_MISC].p;
    unsigned long long *d_nvalid = (unsigned long long *)((u8 *)rb[T_MISC].p + 8 * (K + 1));
    CK(cudaMemcpyAsync(d_input_off, in->input_off, 8 * (K + 1), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(d_nvalid, 0, 8, ctx->stream));
    u32 mx = 1;
    u64 sum_alle = 0;
    for (u64 i = 0; i < nv; ++i) {
        mx = std::max(mx, std::max(t.a0_len[i], t.a1_len[i])); sum_alle += (u64)t.a0_len[i] + t.a1_len[i];
        if ((u64)t.allele_off[i] + t.a0_len[i] + t.a1_len[i] > t.allele_pool_len || t.a0_len[i] > (1u << 24) || t.a1_len[i] > (1u << 24)) {
            ctx->err = "avk_build_regions: allele range outside the pool (or longer than 16 MiB)";
            return AVK_ERR_INVALID;
        }
    }
    if (sum_alle >= 0xffffffffull) { ctx->err = "avk_build_regions: allele bytes exceed 4 GiB"; return AVK_ERR_INVALID; }
    ctx->have_batch = false; ctx->have_result = ctx->have_merge = ctx->result_has_seq = false; ctx->ids_resident = false;
    ctx->lo = 0; ctx->v_base = 0; ctx->p_base = 0; ctx->pool_bytes = 0;
    *n_regions_out = 0; *n_variants_out = 0;
    if (nv == 0) { ctx->n_regions = 0; ctx->n_variants = 0; ctx->n_inputs = (u32)K; ctx->max_allele = 1; ctx->pool_len = 0; ctx->have_batch = ctx->ids_resident = true; ENSURE(ctx->var_off, 8); CK(cudaMemsetAsync(ctx->var_off.p, 0, 8, ctx->stream)); return AVK_OK; }
    const unsigned g = (unsigned)((nv + 255) / 256);
    u64 *key = (u64 *)rb[T_KEY].p, *key_s = (u64 *)rb[T_KEY_S].p, *vend = (u64 *)rb[T_VEND].p, *pmax = (u64 *)rb[T_PMAX].p;
    u32 *idx = (u32 *)rb[T_IDX].p, *idx_s = (u32 *)rb[T_IDX_S].p, *flag = (u32 *)rb[T_FLAG].p, *cid = (u32 *)rb[T_CID].p, *perm = (u32 *)rb[T_PERM].p, *ivl = (u32 *)rb[T_IVL].p;
    const u64 *d_clen = (const u64 *)ctx->d_contig_len.p;
    int key_bits = 33;
    while (key_bits < 64 && (1ull << (key_bits - 32)) < (u64)n_contigs + 1) ++key_bits;     // (contig << 32 | pos); ~0 keys sort last within these bits
    u64 *key2 = (u64 *)rb[T_KEY2].p, *key2_s = (u64 *)rb[T_KEY2_S].p;
    const u32 *pos = (const u32 *)rb[T_POS].p, *l0 = (const u32 *)rb[T_L0].p;
    size_t tmp = 0, need = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, need, key, key_s, idx, idx_s, (int)nv, 0, 64, ctx->stream); tmp = std::max(tmp, need);
    cub::DeviceRadixSort::SortPairs(nullptr, need, key2, key2_s, idx_s, perm, (int)nv, 0, 64, ctx->stream); tmp = std::max(tmp, need);
    cub::DeviceScan::ExclusiveScan(nullptr, need, vend, pmax, MaxOp64(), 0ull, (int)nv, ctx->stream); tmp = std::max(tmp, need);
    cub::DeviceScan::InclusiveSum(nullptr, need, flag, cid, (int)nv, ctx->stream); tmp = std::max(tmp, need);
    ENSURE(ctx->scan_tmp, tmp);
    k_rb_keys<<<g, 256, 0, ctx->stream>>>(nv, pos, l0, variant_contig ? (const u32 *)rb[T_VCONTIG].p : nullptr, contig, d_clen, n_contigs,
                                          bed ? (const u64 *)rb[T_IFIRST].p : nullptr, (const u32 *)rb[T_ISTART].p, (const u32 *)rb[T_ISTART].p + n_ivl, key, idx, ivl);
    (void)key_bits;
    need = tmp; cub::DeviceRadixSort::SortPairs(ctx->scan_tmp.p, need, key, key_s, idx, idx_s, (int)nv, 0, 64, ctx->stream);   // stable: ties keep input then list order (:352-373)
    k_rb_vend<<<g, 256, 0, ctx->stream>>>(nv, key_s, idx_s, l0, ivl, d_clen, flank, vend, d_nvalid);
    need = tmp; cub::DeviceScan::ExclusiveScan(ctx->scan_tmp.p, need, vend, pmax, MaxOp64(), 0ull, (int)nv, ctx->stream);
    k_rb_flags<<<g, 256, 0, ctx->stream>>>(nv, key_s, vend, pmax, flag);
    need = tmp; cub::DeviceScan::InclusiveSum(ctx->scan_tmp.p, need, flag, cid, (int)nv, ctx->stream);
    unsigned long long nvalid = 0;
    CK(cudaMemcpyAsync(&nvalid, d_nvalid, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    u32 n_reg = 0;
    if (nvalid) CK(cudaMemcpy(&n_reg, cid + (nvalid - 1), 4, cudaMemcpyDeviceToHost));
    const u64 n = n_reg;
    ENSURE(ctx->region_id, 8 * n); ENSURE(ctx->contig, 4 * n); ENSURE(ctx->start, 4 * n); ENSURE(ctx->end, 4 * n);
    ENSURE(ctx->var_off, 8 * (n * K + 1));
    ENSURE(ctx->pos, 4 * nvalid); ENSURE(ctx->vtype, nvalid); ENSURE(ctx->zyg, nvalid); ENSURE(ctx->raw, 4 * nvalid);
    ENSURE(ctx->aoff, 4 * nvalid); ENSURE(ctx->l0, 4 * nvalid); ENSURE(ctx->l1, 4 * nvalid); ENSURE(ctx->pool, sum_alle + 16);
    ENSURE(ctx->alt_ed, 4 * nvalid);
    if (nvalid) {
        const unsigned gv = (unsigned)((nvalid + 255) / 256);
        k_rb_clusters<<<gv, 256, 0, ctx->stream>>>(nvalid, key_s, idx_s, cid, flag, pmax, vend, d_input_off, (u32)K, flank, first_region_id,
                                                   key2, (u64 *)ctx->region_id.p, (u32 *)ctx->contig.p, (u32 *)ctx->start.p, (u32 *)ctx->end.p);
        need = tmp; cub::DeviceRadixSort::SortPairs(ctx->scan_tmp.p, need, key2, key2_s, idx_s, perm, (int)nvalid, 0, 64, ctx->stream);   // stable regroup: (cluster, input)
        k_rb_varoff<<<(unsigned)((n * K + 1 + 255) / 256), 256, 0, ctx->stream>>>(n * K, nvalid, key2_s, (u64 *)ctx->var_off.p);
        u32 *alen = (u32 *)vend;   // reuse
        k_rb_gather<<<gv, 256, 0, ctx->stream>>>(nvalid, perm, pos, (const u8 *)rb[T_VT].p, (const u8 *)rb[T_ZY].p, (const u32 *)rb[T_RAW].p, l0,
                                                 (const u32 *)rb[T_L1].p, (u32 *)ctx->pos.p, (u8 *)ctx->vtype.p, (u8 *)ctx->zyg.p, (u32 *)ctx->raw.p,
                                                 (u32 *)ctx->l0.p, (u32 *)ctx->l1.p, alen);
        need = tmp; cub::DeviceScan::ExclusiveSum(ctx->scan_tmp.p, need, alen, (u32 *)ctx->aoff.p, (int)nvalid, ctx->stream);
        k_rb_alleles<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(nvalid, perm, (const u32 *)rb[T_AOFF].p, alen, (const u32 *)ctx->aoff.p,
                                                                 (const u8 *)rb[T_POOL].p, (u8 *)ctx->pool.p);
        ctx->launches += 12;
    } else {
        CK(cudaMemsetAsync(ctx->var_off.p, 0, 8, ctx->stream));
    }
    CK(cudaGetLastError());
    u64 kept_bytes = 0;                                           // allele bytes of the variants that were kept
    if (nvalid) {
        u32 last[2] = {0, 0};
        CK(cudaMemcpyAsync(&last[0], (u32 *)ctx->aoff.p + (nvalid - 1), 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(&last[1], (u32 *)vend + (nvalid - 1), 4, cudaMemcpyDeviceToHost, ctx->stream));   // alen (vend reused)
        CK(cudaStreamSynchronize(ctx->stream));
        kept_bytes = (u64)last[0] + last[1];
    }
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->n_regions = n; ctx->n_variants = nvalid; ctx->n_inputs = (u32)K; ctx->max_allele = mx; ctx->pool_len = kept_bytes; ctx->pool_bytes = kept_bytes;
    ctx->have_batch = ctx->ids_resident = true;
    *n_regions_out = n; *n_variants_out = nvalid;
    return AVK_OK;
}

extern "C" int avk_regions_download(avk_ctx *ctx, avk_region_batch *out) {
    if (!ctx || !out) return AVK_ERR_INVALID;
    if (!ctx->have_batch || ctx->lo != 0 || ctx->v_base != 0) { ctx->err = "avk_regions_download: no device-built batch is resident"; return AVK_ERR_INVALID; }
    CK(cudaSetDevice(ctx->device));
    const u64 n = ctx->n_regions, nv = ctx->n_variants, K = ctx->n_inputs;
    avk_variant_table &t = out->variants;
#define RBDL(dst, buf, bytes) do { if ((bytes) && (dst)) CK(cudaMemcpyAsync((void *)(dst), (buf).p, (bytes), cudaMemcpyDeviceToHost, ctx->stream)); } while (0)
    RBDL(out->region_id, ctx->region_id, 8 * n); RBDL(out->contig, ctx->contig, 4 * n); RBDL(out->start, ctx->start, 4 * n); RBDL(out->end, ctx->end, 4 * n);
    RBDL(out->var_off, ctx->var_off, 8 * (n * K + 1));
    RBDL(t.position, ctx->pos, 4 * nv); RBDL(t.variant_type, ctx->vtype, nv); RBDL(t.zygosity, ctx->zyg, nv); RBDL(t.raw_allele_space, ctx->raw, 4 * nv);
    RBDL(t.allele_off, ctx->aoff, 4 * nv); RBDL(t.a0_len, ctx->l0, 4 * nv); RBDL(t.a1_len, ctx->l1, 4 * nv); RBDL(t.allele_pool, ctx->pool, ctx->pool_bytes);
#undef RBDL
    CK(cudaStreamSynchronize(ctx->stream));
    out->n_regions = n; out->n_inputs = (uint32_t)K; t.n_variants = nv; t.allele_pool_len = ctx->pool_bytes;
    return AVK_OK;
}

extern "C" int avk_compare_upload_range(avk_ctx *ctx, const avk_region_batch *batch, uint64_t lo, uint64_t hi) {
    if (!ctx) return AVK_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    int rc = validate_batch(ctx, batch, true);
    if (rc != AVK_OK) return rc;
    if (lo > hi || hi > batch->n_regions) { ctx->err = "region range outside the batch"; return AVK_ERR_INVALID; }
    BinScan sc;
    rc = bin_range(ctx, batch, lo, hi, sc);
    if (rc != AVK_OK) return rc;
    rc = upload_batch(ctx, batch, sc);
    if (rc != AVK_OK) return rc;
    ctx->seq_base = 0; ctx->strat_base = 0;
    CK(cudaStreamSynchronize(ctx->stream));
    return AVK_OK;
}

extern "C" int avk_compare_upload(avk_ctx *ctx, const avk_region_batch *batch) {
    if (!ctx) return AVK_ERR_INVALID;
    if (!batch) { ctx->err = "null batch"; return AVK_ERR_INVALID; }
    return avk_compare_upload_range(ctx, batch, 0, batch->n_regions);
}

// AVK_CMP_KEEP_SEQUENCES: the layout avk_compare_seq_offsets gives the resident bin (offsets from 0), built on the device --
// per region the sizes {win, win + alt0, win + alt0, win + alt1, win + alt1} (k_seq_sizes), an exclusive scan into seq_off,
// and the pool sized from the scan's total
__global__ void __launch_bounds__(256) k_seq_sizes(DevBatch b, u64 n, u64 *sizes) {
    const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r > n) return;
    if (r == n) { sizes[n * 5] = 0; return; }
    const u64 win = b.end[r] > b.start[r] ? b.end[r] - b.start[r] : 0;
    u64 alt[2] = {0, 0};
    for (int k = 0; k < 2; ++k)
        for (u64 v = b.var_off[r * 2 + k]; v < b.var_off[r * 2 + k + 1]; ++v) alt[k] += b.l1[v];
    u64 *o = sizes + r * 5;
    o[0] = win; o[1] = o[2] = win + alt[0]; o[3] = o[4] = win + alt[1];
}
static int resident_seq_layout(avk_ctx *ctx) {
    const u64 n = ctx->n_regions, m = n * 5 + 1;
    ctx->result_has_seq = false;                                  // the buffers below are overwritten from here on
    ENSURE(ctx->seq_off, 8 * m);
    ENSURE(ctx->seq_len, 4 * 5 * n + 4);
    u64 *off = (u64 *)ctx->seq_off.p;
    size_t need = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, need, off, off, m, ctx->stream);
    ENSURE(ctx->scan_tmp, need);
    k_seq_sizes<<<(unsigned)((n + 1 + 255) / 256), 256, 0, ctx->stream>>>(dev_batch(ctx), n, off);
    CK(cub::DeviceScan::ExclusiveSum(ctx->scan_tmp.p, need, off, off, m, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_pin, off + n * 5, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->launches += 2;
    CK(cudaGetLastError());
    u64 pool = 0;
    memcpy(&pool, ctx->h_pin, 8);
    ENSURE(ctx->seq_pool, pool);
    CK(cudaMemsetAsync(ctx->seq_len.p, 0, 4 * 5 * n + 4, ctx->stream));
    ctx->seq_base = 0;
    return AVK_OK;
}

extern "C" int avk_compare_run_resident(avk_ctx *ctx, const avk_compare_cfg *cfg) {
    if (!ctx) return AVK_ERR_INVALID;
    if (!cfg || !ctx->have_batch || ctx->n_inputs != 2) { ctx->err = "no resident compare batch"; return AVK_ERR_INVALID; }
    const bool keep_seq = (cfg->flags & AVK_CMP_KEEP_SEQUENCES) != 0;
    if (keep_seq && !cfg->enable_sequences) { ctx->err = "AVK_CMP_KEEP_SEQUENCES needs enable_sequences"; return AVK_ERR_INVALID; }
    CK(cudaSetDevice(ctx->device));
    CompareRun R;
    int rc = keep_seq ? resident_seq_layout(ctx) : AVK_OK;
    if (rc != AVK_OK) return rc;
    rc = compare_launch(ctx, cfg, keep_seq, (cfg->flags & AVK_CMP_KEEP_REGION_ROWS) != 0, false, 0, false, false, R);
    if (rc != AVK_OK) return rc;
    rc = compare_finish(ctx, R, nullptr);
    if (rc != AVK_OK) return rc;
    return fetch_timings(ctx);
}

// Results of the last run, copied into the caller's arrays at the resident bin's offsets.
extern "C" int avk_compare_download(avk_ctx *ctx, avk_compare_out *out) {
    if (!ctx) return AVK_ERR_INVALID;
    if (!out || !ctx->have_batch || !ctx->have_result) { ctx->err = "no compare result is resident (run avk_compare_run_resident first)"; return AVK_ERR_INVALID; }
    if (strata_wanted(out)) { ctx->err = "avk_compare_download returns no stratified sums: request them from avk_compare_batch*"; return AVK_ERR_INVALID; }
    CK(cudaSetDevice(ctx->device));
    int rc = download_compare_async(ctx, out, false, 0);
    if (rc != AVK_OK) return rc;
    CK(cudaStreamSynchronize(ctx->stream));
    BinTotals bt;
    rc = collect_totals(ctx, out, false, bt);
    if (rc != AVK_OK) return rc;
    store_totals(out, bt, false, false);
    return AVK_OK;
}

// Device addresses of the last run's results (the single gather of a one-process-per-GPU run sends them to the root
// GPU over NVLink without a host round trip).  The arrays stay valid until the next call on this context.
extern "C" int avk_compare_result_device(avk_ctx *ctx, avk_compare_dev_view *v) {
    if (!ctx || !v) return AVK_ERR_INVALID;
    if (!ctx->have_batch || !ctx->have_result) { ctx->err = "no compare result is resident"; return AVK_ERR_INVALID; }
    v->lo = ctx->lo; v->n_regions = ctx->n_regions; v->v_base = ctx->v_base; v->n_variants = ctx->n_variants;
    v->status = ctx->status.p; v->ed1 = ctx->ed1.p; v->ed2 = ctx->ed2.p; v->type_mask = ctx->type_mask.p;
    v->var_expected = ctx->vexp.p; v->var_observed = ctx->vobs.p; v->var_class = ctx->vcls.p; v->totals = ctx->totals.p;
    return AVK_OK;
}

// Measured INT32 throughput in integer ops per second (3 ops per chain step: add, max, xor).
extern "C" int avk_int_peak(avk_ctx *ctx, double *ops_per_s) {
    if (!ctx || !ops_per_s) return AVK_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    ENSURE(ctx->counters, 64);
    const int iters = 1 << 13, blocks = ctx->sm_count * 16, threads = 256;
    float best = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {
        CK(cudaEventRecord(ctx->ev[0], ctx->stream));
        k_int_peak<<<blocks, threads, 0, ctx->stream>>>(iters, (int *)ctx->counters.p);
        CK(cudaEventRecord(ctx->ev[1], ctx->stream));
        CK(cudaEventSynchronize(ctx->ev[1]));
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
        if (rep > 0 && ms < best) best = ms;
    }
    ctx->launches += 4;
    CK(cudaGetLastError());
    *ops_per_s = (double)blocks * threads * (double)iters * 8.0 * 3.0 / (best * 1e-3);
    return AVK_OK;
}

extern "C" int avk_last_timings(avk_ctx *ctx, float *ms5) {
    if (!ctx || !ms5) return AVK_ERR_INVALID;
    memcpy(ms5, ctx->last_ms, sizeof(ctx->last_ms));
    return AVK_OK;
}
// Diagnostics: how many clusters overflowed workspace tiers 0, 1, 2 in the last run.
extern "C" int avk_last_tier_overflow(avk_ctx *ctx, uint32_t *out3) {
    if (!ctx || !out3) return AVK_ERR_INVALID;
    for (int i = 0; i < 3; ++i) out3[i] = ctx->tier_fail[i];
    return AVK_OK;
}
// Diagnostics: device milliseconds of workspace tiers 0, 1, 2 in the last run.
extern "C" int avk_last_tier_ms(avk_ctx *ctx, float *out3) {
    if (!ctx || !out3) return AVK_ERR_INVALID;
    for (int i = 0; i < 3; ++i) out3[i] = ctx->tier_ms[i];
    return AVK_OK;
}
extern "C" int avk_last_work(avk_ctx *ctx, avk_work_counters *out) {
    if (!ctx || !out) return AVK_ERR_INVALID;
    *out = ctx->last_work;
    return AVK_OK;
}

// solve_merge_region over the resident batch: front stage, pair tasks and classification are queued on ctx->stream; the
// result stays in status / m_cls / m_nidx / m_idx (merge_finish marks it resident)
static int merge_launch(avk_ctx *ctx, const avk_merge_cfg *cfg) {
    const u64 n = ctx->n_regions;
    const u32 K = ctx->n_inputs;
    ctx->have_result = ctx->have_merge = ctx->result_has_seq = false;                 // the pass overwrites `status`, which a compare result owns too
    ENSURE(ctx->status, 4 * n); ENSURE(ctx->m_cls, n); ENSURE(ctx->m_nidx, n); ENSURE(ctx->m_idx, n * K);
    ENSURE(ctx->counters, 64); ENSURE(ctx->work_ctr, 64);
    CK(cudaMemsetAsync(ctx->work_ctr.p, 0, 64, ctx->stream));
    DevBatch db = dev_batch(ctx);
    DevMergeOut mo;
    mo.status = (int *)ctx->status.p; mo.cls = (u8 *)ctx->m_cls.p; mo.n_idx = (u8 *)ctx->m_nidx.p; mo.idx = (u8 *)ctx->m_idx.p;
    avk_merge_cfg c = *cfg;
    CK(cudaEventRecord(ctx->ev[0], ctx->stream));
    int rc = run_alt_ed(ctx, db);
    if (rc != AVK_OK) return rc;
    CK(cudaEventRecord(ctx->ev[1], ctx->stream));
    const int sm = ctx->sm_count;
    const int INF = 0x7fffffff;
    // front stage (per cluster) -> pair tasks (per pair, three workspace tiers) -> classification (per cluster)
    const u64 pairs = (u64)K * (K - 1) / 2, max_tasks = n * pairs;
    if (max_tasks >= 0xffffffffull || n >= (1ull << 47)) { ctx->err = "avk_merge_batch: too many pair tasks"; return AVK_ERR_INVALID; }
    ENSURE(ctx->m_rows, 4 * n * K); ENSURE(ctx->m_perr, 4 * n); ENSURE(ctx->m_tasks, 8 * max_tasks);
    MergeWork mw;
    mw.rows = (u32 *)ctx->m_rows.p; mw.pair_err = (u32 *)ctx->m_perr.p; mw.tasks = (u64 *)ctx->m_tasks.p; mw.task_ctr = nullptr;
    const std::vector<Stage> stages = {
        {MODE_FUSED, true, 3, 8192, sm * 3, 8, -1, 0, 0, 0, 1, 0, 0, INF},
        {MODE_FUSED, true, 1, 27648, sm, 8, 0, 1, 3, 1, 4, 0, 0, INF},
        {MODE_FUSED, false, 1, 2LL << 20, sm, 8, 1, 4, 5, 0, 6, 0, 0, INF},
    };
    const unsigned cgrid = (unsigned)std::min<u64>((u64)sm * 8, (n + 7) / 8);
    rc = run_stages(ctx, std::max<u64>(max_tasks, 1), stages, [&](u32 *ctrs) {   // (an upper bound; the task count is produced on the device)
        mw.task_ctr = ctrs + 20;
        if (n) k_merge_front<<<cgrid, 256, 0, ctx->stream>>>(db, mo, c, mw, n);
        ctx->launches += 1;
    }, 20, [&](const Stage &st, const TierArgs &a, int ctas, cudaStream_t strm) {
        if (st.smem && st.min_ctas == 3) launch_merge_pairs<true, 3>(db, c, a, mw, ctas, st.warps, strm);
        else if (st.smem) launch_merge_pairs<true, 1>(db, c, a, mw, ctas, st.warps, strm);
        else launch_merge_pairs<false, 1>(db, c, a, mw, ctas, st.warps, strm);
    });
    if (rc != AVK_OK) return rc;
    if (n) {
        k_merge_classify<<<cgrid, 256, 0, ctx->stream>>>(db, mo, c, mw, n);
        ctx->launches += 1;
        CK(cudaGetLastError());
    }
    CK(cudaEventRecord(ctx->ev[2], ctx->stream));
    CK(cudaEventRecord(ctx->ev[3], ctx->stream));
    CK(cudaEventRecord(ctx->ev[4], ctx->stream));
    return AVK_OK;
}
// the resident bin's merge result -> the caller's arrays at the bin's offsets (queued on ctx->stream)
static int merge_queue_download(avk_ctx *ctx, avk_merge_out *out) {
    const u64 n = ctx->n_regions, lo = ctx->lo, K = ctx->n_inputs;
    const cudaStream_t ds = ctx->stream;
    DL(out->status + lo, ctx->status, 4 * n);
    DL(out->classification ? out->classification + lo : nullptr, ctx->m_cls, n);
    DL(out->n_indices ? out->n_indices + lo : nullptr, ctx->m_nidx, n);
    DL(out->indices ? out->indices + lo * K : nullptr, ctx->m_idx, n * K);
    return AVK_OK;
}
// waits for the pass (and any queued download) and reads its timings and work counters; the result is then resident
static int merge_finish(avk_ctx *ctx) {
    CK(cudaMemcpyAsync(ctx->h_pin + 128, ctx->work_ctr.p, 40, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaEventRecord(ctx->ev_done, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const int rc = fetch_timings(ctx);
    if (rc != AVK_OK) return rc;
    ctx->have_merge = true;
    return AVK_OK;
}

// solve_merge_region over one contiguous bin [lo, hi) of the batch; results land in the caller's arrays at the bin's offsets
// and stay resident on the context
static int merge_bin(avk_ctx *ctx, const avk_region_batch *batch, u64 lo, u64 hi, const avk_merge_cfg *cfg, avk_merge_out *out) {
    CK(cudaSetDevice(ctx->device));
    BinScan sc;
    int rc = bin_range(ctx, batch, lo, hi, sc);
    if (rc != AVK_OK) return rc;
    rc = upload_batch(ctx, batch, sc);
    if (rc != AVK_OK) return rc;
    rc = merge_launch(ctx, cfg);
    if (rc != AVK_OK) return rc;
    rc = merge_queue_download(ctx, out);
    if (rc != AVK_OK) return rc;
    return merge_finish(ctx);
}

extern "C" int avk_merge_upload_range(avk_ctx *ctx, const avk_region_batch *batch, uint64_t lo, uint64_t hi) {
    if (!ctx) return AVK_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    int rc = validate_batch(ctx, batch, false);
    if (rc != AVK_OK) return rc;
    if (lo > hi || hi > batch->n_regions) { ctx->err = "region range outside the batch"; return AVK_ERR_INVALID; }
    BinScan sc;
    rc = bin_range(ctx, batch, lo, hi, sc);
    if (rc != AVK_OK) return rc;
    rc = upload_batch(ctx, batch, sc);
    if (rc != AVK_OK) return rc;
    CK(cudaStreamSynchronize(ctx->stream));
    return AVK_OK;
}

extern "C" int avk_merge_run_resident(avk_ctx *ctx, const avk_merge_cfg *cfg) {
    if (!ctx) return AVK_ERR_INVALID;
    if (!cfg || !ctx->have_batch) { ctx->err = "avk_merge_run_resident: no resident batch (avk_merge_upload_range or avk_build_regions[_bed] first)"; return AVK_ERR_INVALID; }
    if (ctx->n_inputs < 1 || ctx->n_inputs > 32) { ctx->err = "avk_merge_run_resident: unsupported n_inputs (1 .. 32)"; return AVK_ERR_INVALID; }
    CK(cudaSetDevice(ctx->device));
    const int rc = merge_launch(ctx, cfg);
    if (rc != AVK_OK) return rc;
    return merge_finish(ctx);
}

extern "C" int avk_merge_download(avk_ctx *ctx, avk_merge_out *out) {
    if (!ctx) return AVK_ERR_INVALID;
    if (!ctx->have_batch || !ctx->have_merge) { ctx->err = "avk_merge_download: no merge result is resident (run avk_merge_run_resident first)"; return AVK_ERR_INVALID; }
    if (!out || !out->status) { ctx->err = "avk_merge_download: null out/status"; return AVK_ERR_INVALID; }
    CK(cudaSetDevice(ctx->device));
    const int rc = merge_queue_download(ctx, out);
    if (rc != AVK_OK) return rc;
    CK(cudaStreamSynchronize(ctx->stream));
    return AVK_OK;
}

extern "C" int avk_merge_batch(avk_ctx *ctx, const avk_region_batch *batch, const avk_merge_cfg *cfg, avk_merge_out *out) {
    if (!ctx) return AVK_ERR_INVALID;
    if (!cfg || !out || !out->status) { ctx->err = "null cfg/out/status"; return AVK_ERR_INVALID; }
    int rc = validate_batch(ctx, batch, false);
    if (rc != AVK_OK) return rc;
    return merge_bin(ctx, batch, 0, batch->n_regions, cfg, out);
}

// Multi-GPU merge: contiguous bins, one host thread per context, results written at the bins' offsets (see
// avk_compare_batch_multi).
extern "C" int avk_merge_batch_multi(avk_ctx *const *ctxs, uint32_t n_ctx, const avk_region_batch *batch,
                                     const avk_merge_cfg *cfg, avk_merge_out *out) {
    if (!ctxs || n_ctx == 0 || !ctxs[0]) return AVK_ERR_INVALID;
    avk_ctx *ctx = ctxs[0];
    if (!cfg || !out || !out->status) { ctx->err = "null cfg/out/status"; return AVK_ERR_INVALID; }
    int rc = validate_batch(ctx, batch, false);
    if (rc != AVK_OK) return rc;
    std::vector<u64> cuts(n_ctx + 1);
    avk_partition_regions(batch, n_ctx, cuts.data());
    std::vector<int> rcs(n_ctx, AVK_OK);
    std::vector<std::thread> th;
    for (uint32_t k = 0; k < n_ctx; ++k)
        th.emplace_back([&, k]() { rcs[k] = ctxs[k] ? merge_bin(ctxs[k], batch, cuts[k], cuts[k + 1], cfg, out) : AVK_ERR_INVALID; });
    for (auto &t : th) t.join();
    for (uint32_t k = 0; k < n_ctx; ++k)
        if (rcs[k] != AVK_OK) { if (k && ctxs[k]) ctx->err = "device " + std::to_string(k) + ": " + ctxs[k]->err; return rcs[k]; }
    return AVK_OK;
}


extern "C" int avk_wfa_ed_batch(avk_ctx *ctx, uint64_t n_pairs, const uint8_t *pool, uint64_t pool_len, const uint64_t *a_off,
                                const uint32_t *a_len, const uint64_t *b_off, const uint32_t *b_len, uint32_t *ed_out) {
    if (!ctx) return AVK_ERR_INVALID;
    if (n_pairs && (!pool || !a_off || !a_len || !b_off || !b_len || !ed_out)) { ctx->err = "null argument"; return AVK_ERR_INVALID; }
    if (n_pairs >= (1ull << 32) - 1) { ctx->err = "too many pairs"; return AVK_ERR_INVALID; }
    CK(cudaSetDevice(ctx->device));
    if (n_pairs == 0) return AVK_OK;
    u32 mx = 1;
    for (u64 i = 0; i < n_pairs; ++i) {
        if (a_off[i] + a_len[i] > pool_len || b_off[i] + b_len[i] > pool_len) { ctx->err = "pair outside pool"; return AVK_ERR_INVALID; }
        mx = std::max(mx, std::max(a_len[i], b_len[i]));
    }
    UPLOAD(ctx->pair_pool, pool, pool_len);
    UPLOAD(ctx->pair_a_off, a_off, 8 * n_pairs);
    UPLOAD(ctx->pair_b_off, b_off, 8 * n_pairs);
    UPLOAD(ctx->pair_a_len, a_len, 4 * n_pairs);
    UPLOAD(ctx->pair_b_len, b_len, 4 * n_pairs);
    ENSURE(ctx->pair_ed, 4 * n_pairs);
    ENSURE(ctx->counters, 64); ENSURE(ctx->work_ctr, 64);
    CK(cudaMemsetAsync(ctx->counters.p, 0, 64, ctx->stream));
    CK(cudaMemsetAsync(ctx->work_ctr.p, 0, 64, ctx->stream));
    const int scratch_ints = (2 * (int)mx + 8 + 3) / 4 * 4;
    int warps = (int)std::min<u64>((u64)ctx->sm_count * 32, (n_pairs + 7) / 8 * 8);
    warps = (warps + 7) / 8 * 8;
    const int ctas = (int)std::min<u64>((u64)ctx->sm_count, n_pairs);
    ENSURE(ctx->scratch, (size_t)(warps + ctas) * ((size_t)scratch_ints * 4 + ARENA_HDR));
    ENSURE(ctx->fail_a, 4 * n_pairs); ENSURE(ctx->fail_b, 4 * n_pairs);
    u32 *ctrs = (u32 *)ctx->counters.p;          // [0] warp work, [1] cta work, [2] |warp list|, [3] |cta list|
    const int cap_ints = ctx->coop_cap_ints;
    CK(cudaEventRecord(ctx->ev[0], ctx->stream));
    k_wfa_split<<<(unsigned)((n_pairs + 255) / 256), 256, 0, ctx->stream>>>(n_pairs, (const u32 *)ctx->pair_a_len.p, (const u32 *)ctx->pair_b_len.p, 512u,
                                                                          (u32)(8 * cap_ints), (u32 *)ctx->fail_a.p, ctrs + 2, (u32 *)ctx->fail_b.p, ctrs + 3);
    CK(cudaEventRecord(ctx->ev[1], ctx->stream));
    // long pairs first: one CTA each, the whole CTA on one wavefront
    k_wfa_ed_cta<<<ctas, COOP_THREADS, COOP_JOB_BYTES + 2 * sizeof(int) * (size_t)cap_ints, ctx->stream>>>(
        (const u32 *)ctx->fail_b.p, ctrs + 3, (const u8 *)ctx->pair_pool.p, (const u64 *)ctx->pair_a_off.p, (const u32 *)ctx->pair_a_len.p,
        (const u64 *)ctx->pair_b_off.p, (const u32 *)ctx->pair_b_len.p, (u32 *)ctx->pair_ed.p,
        (u8 *)ctx->scratch.p + (size_t)warps * ((size_t)scratch_ints * 4 + ARENA_HDR), scratch_ints, cap_ints, ctrs + 1, (unsigned long long *)ctx->work_ctr.p);
    k_wfa_ed<<<warps / 8, 256, 0, ctx->stream>>>((const u32 *)ctx->fail_a.p, ctrs + 2, (const u8 *)ctx->pair_pool.p, (const u64 *)ctx->pair_a_off.p,
                                                  (const u32 *)ctx->pair_a_len.p, (const u64 *)ctx->pair_b_off.p,
                                                  (const u32 *)ctx->pair_b_len.p, (u32 *)ctx->pair_ed.p, (u8 *)ctx->scratch.p,
                                                  scratch_ints, ctrs, (unsigned long long *)ctx->work_ctr.p);
    ctx->launches += 2;
    ctx->launches += 1;
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->ev[2], ctx->stream));
    CK(cudaEventRecord(ctx->ev[3], ctx->stream));
    CK(cudaEventRecord(ctx->ev[4], ctx->stream));
    ctx->have_result = ctx->have_merge = ctx->result_has_seq = false;
    CK(cudaMemcpyAsync(ed_out, ctx->pair_ed.p, 4 * n_pairs, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_pin + 128, ctx->work_ctr.p, 40, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaEventRecord(ctx->ev_done, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return fetch_timings(ctx);
}

// Host-only: upper-bound layout of the sequence bundle (ref = window; haplotype <= window + sum of ALT lengths of its side).
extern "C" int avk_compare_seq_offsets(const avk_region_batch *b, uint64_t *seq_off, uint64_t *pool_len) {
    if (!b || !seq_off || b->n_inputs != 2) return AVK_ERR_INVALID;
    u64 off = 0;
    for (u64 r = 0; r < b->n_regions; ++r) {
        const u64 win = b->end[r] > b->start[r] ? b->end[r] - b->start[r] : 0;
        u64 alt[2] = {0, 0};
        for (int k = 0; k < 2; ++k)
            for (u64 v = b->var_off[r * 2 + k]; v < b->var_off[r * 2 + k + 1]; ++v) alt[k] += b->variants.a1_len[v];
        const u64 sizes[5] = {win, win + alt[0], win + alt[0], win + alt[1], win + alt[1]};
        for (int s = 0; s < 5; ++s) { seq_off[r * 5 + s] = off; off += sizes[s]; }
    }
    seq_off[b->n_regions * 5] = off;
    if (pool_len) *pool_len = off;
    return AVK_OK;
}

// ---- writers (SURVEY 8f N3): host-side formatting of what the kernels counted -----------------------------------------
static int copy_text(const std::string &txt, char *buf, uint64_t cap, uint64_t *len) {
    if (len) *len = txt.size();
    if (!buf) return AVK_OK;                                        // size query
    if (cap < txt.size()) return AVK_ERR_INVALID;
    memcpy(buf, txt.data(), txt.size());
    return AVK_OK;
}
extern "C" int avk_summary_write(const uint64_t *totals, const uint8_t *metrics, uint32_t n_metrics, const char *compare_label, const char *region_label,
                                 int csv, int header, char *buf, uint64_t cap, uint64_t *len) {
    if (!totals || (!metrics && n_metrics) || !compare_label || !region_label) return AVK_ERR_INVALID;
    return copy_text(avk_writers::summary_text(totals, metrics, n_metrics, compare_label, region_label, csv ? ',' : '\t', header != 0), buf, cap, len);
}
extern "C" int avk_vcf_records_write(const avk_region_batch *batch, uint32_t side, const char *const *contig_names, uint32_t n_contigs,
                                     const uint8_t *var_class, const uint8_t *var_expected, const uint8_t *var_observed, uint64_t lo, uint64_t hi,
                                     char *buf, uint64_t cap, uint64_t *len) {
    if (!batch || !contig_names || !var_class || !var_expected || !var_observed || side >= batch->n_inputs || lo > hi || hi > batch->n_regions) return AVK_ERR_INVALID;
    for (uint64_t r = lo; r < hi; ++r) if (batch->contig[r] >= n_contigs) return AVK_ERR_INVALID;
    return copy_text(avk_writers::vcf_records_text(batch, side, contig_names, var_class, var_expected, var_observed, lo, hi), buf, cap, len);
}

// the argument checks both debug writers share, host and device: names present and printable without quoting
static bool debug_names_ok(const char *const *contig_names, uint32_t n_contigs) {
    if (!contig_names && n_contigs) return false;
    for (uint32_t c = 0; c < n_contigs; ++c) if (!contig_names[c] || !avk_writers::plain_name(contig_names[c])) return false;
    return true;
}
static bool debug_range_ok(const avk_region_batch *batch, const int32_t *status, uint32_t n_contigs, uint64_t lo, uint64_t hi) {
    if (!batch || !status || lo > hi || hi > batch->n_regions) return false;
    for (uint64_t r = lo; r < hi; ++r) if (batch->contig[r] >= n_contigs) return false;
    return true;
}
extern "C" int avk_region_summary_write(const avk_region_batch *batch, const int32_t *status, const uint64_t *region_metrics,
                                        const char *const *contig_names, uint32_t n_contigs, const uint8_t *metrics, uint32_t n_metrics, int header,
                                        uint64_t lo, uint64_t hi, char *buf, uint64_t cap, uint64_t *len) {
    if (!region_metrics || (!metrics && n_metrics) || !debug_names_ok(contig_names, n_contigs) || !debug_range_ok(batch, status, n_contigs, lo, hi)) return AVK_ERR_INVALID;
    for (uint32_t q = 0; q < n_metrics; ++q) if (metrics[q] > 4) return AVK_ERR_INVALID;
    return copy_text(avk_writers::region_summary_text(batch, status, region_metrics, contig_names, metrics, n_metrics, header != 0, lo, hi), buf, cap, len);
}
extern "C" int avk_region_sequences_write(const avk_region_batch *batch, const int32_t *status, const uint64_t *seq_off, const uint32_t *seq_len,
                                          const uint8_t *seq_pool, const char *const *contig_names, uint32_t n_contigs, int header,
                                          uint64_t lo, uint64_t hi, char *buf, uint64_t cap, uint64_t *len) {
    if (!seq_off || !seq_len || !seq_pool || !debug_names_ok(contig_names, n_contigs) || !debug_range_ok(batch, status, n_contigs, lo, hi)) return AVK_ERR_INVALID;
    return copy_text(avk_writers::region_sequences_text(batch, status, seq_off, seq_len, seq_pool, contig_names, header != 0, lo, hi), buf, cap, len);
}

static int merge_view(const avk_region_batch *batch, const avk_merge_out *res, uint32_t n_contigs, bool need_contigs, avk_writers::MergeView &m) {
    if (!batch || !res || !res->classification || !res->n_indices || !res->indices || batch->n_inputs == 0 || batch->n_inputs > 255) return AVK_ERR_INVALID;
    m = {res->status, res->classification, res->n_indices, res->indices};
    for (uint64_t r = 0; r < batch->n_regions; ++r) {
        if (need_contigs && batch->contig[r] >= n_contigs) return AVK_ERR_INVALID;
        if (res->n_indices[r] > batch->n_inputs) return AVK_ERR_INVALID;
        for (uint8_t k = 0; k < res->n_indices[r]; ++k) if (res->indices[r * batch->n_inputs + k] >= batch->n_inputs) return AVK_ERR_INVALID;
    }
    return AVK_OK;
}
extern "C" int avk_merge_records_write(const avk_region_batch *batch, const avk_merge_out *result, const char *const *contig_names, uint32_t n_contigs,
                                       const char *const *input_labels, uint64_t lo, uint64_t hi, char *buf, uint64_t cap, uint64_t *len) {
    avk_writers::MergeView m;
    if (!contig_names || !input_labels || merge_view(batch, result, n_contigs, true, m) != AVK_OK || lo > hi || hi > batch->n_regions) return AVK_ERR_INVALID;
    return copy_text(avk_writers::merge_records_text(batch, contig_names, input_labels, m, lo, hi), buf, cap, len);
}
extern "C" int avk_merge_regions_write(const avk_region_batch *batch, const avk_merge_out *result, const char *const *contig_names, uint32_t n_contigs,
                                       int passing, uint64_t lo, uint64_t hi, char *buf, uint64_t cap, uint64_t *len) {
    avk_writers::MergeView m;
    if (!contig_names || merge_view(batch, result, n_contigs, true, m) != AVK_OK || lo > hi || hi > batch->n_regions) return AVK_ERR_INVALID;
    return copy_text(avk_writers::merge_regions_text(batch, contig_names, m, lo, hi, passing != 0), buf, cap, len);
}
extern "C" int avk_merge_summary_write(const avk_region_batch *batch, const avk_merge_out *result, const char *const *input_labels, int csv, int header,
                                       char *buf, uint64_t cap, uint64_t *len) {
    avk_writers::MergeView m;
    if (!input_labels || merge_view(batch, result, 0, false, m) != AVK_OK) return AVK_ERR_INVALID;
    return copy_text(avk_writers::merge_summary_text(batch, input_labels, m, csv ? ',' : '\t', header != 0), buf, cap, len);
}
extern "C" int avk_merge_summary_rows_write(const avk_merge_summary_row *rows, uint64_t n_rows, uint32_t n_inputs, const char *const *input_labels,
                                            int csv, int header, char *buf, uint64_t cap, uint64_t *len) {
    if ((!rows && n_rows) || !input_labels || n_inputs == 0 || n_inputs > 32) return AVK_ERR_INVALID;
    for (uint64_t i = 0; i < n_rows; ++i)
        if (rows[i].input >= n_inputs || !input_labels[rows[i].input] || (n_inputs < 32 && (rows[i].indices >> n_inputs))) return AVK_ERR_INVALID;
    avk_writers::MergeSummaryCounts counts;
    avk_writers::merge_summary_count_rows(counts, rows, n_rows);
    return copy_text(avk_writers::merge_summary_format(counts, input_labels, csv ? ',' : '\t', header != 0), buf, cap, len);
}

// ---- VCF body text -> call-set table (SURVEY 8f N2, avk_vcf.cuh) -----------------------------------------------------------
struct LineStart {
    const u8 *t;
    u64 len;
    __device__ __forceinline__ bool operator()(const u64 &i) const { return i < len && (i == 0 || t[i - 1] == '\n'); }
};
// per line: number of variants it yields, their allele bytes, or an error (the first failing line wins, like the `?` of the loop)
__global__ void __launch_bounds__(256) k_vcf_scan(const u8 *t, u64 len, const u64 *starts, u64 n_lines, const char *names, u32 n_contigs, u32 name_stride,
                                                  u32 sample_index, int trim, u32 *n_out, u32 *n_bytes, unsigned long long *first_err) {
    const u64 li = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (li >= n_lines) return;
    u64 b = starts[li], e = li + 1 < n_lines ? starts[li + 1] : len;
    while (e > b && (t[e - 1] == '\n' || t[e - 1] == '\r')) --e;
    avk_vcf::LineInfo L;
    avk_vcf::parse_line(t, b, e, names, n_contigs, name_stride, sample_index, trim != 0, L);
    u32 bytes = 0;
    for (int q = 0; q < L.n; ++q) bytes += L.v[q].l0 + L.v[q].l1;
    n_out[li] = L.err ? 0u : (u32)L.n; n_bytes[li] = L.err ? 0u : bytes;
    if (L.err) atomicMin(first_err, (unsigned long long)((li << 8) | (u64)L.err));
}
__global__ void __launch_bounds__(256) k_vcf_emit(const u8 *t, u64 len, const u64 *starts, u64 n_lines, const char *names, u32 n_contigs, u32 name_stride,
                                                  u32 sample_index, int trim, const u32 *v_off, const u32 *b_off, u32 *contig, u32 *pos, u8 *vt, u8 *zy,
                                                  u32 *raw, u32 *aoff, u32 *l0, u32 *l1, u8 *pool) {
    const u64 li = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (li >= n_lines) return;
    u64 b = starts[li], e = li + 1 < n_lines ? starts[li + 1] : len;
    while (e > b && (t[e - 1] == '\n' || t[e - 1] == '\r')) --e;
    avk_vcf::LineInfo L;
    avk_vcf::parse_line(t, b, e, names, n_contigs, name_stride, sample_index, trim != 0, L);
    if (L.err) return;
    u32 v = v_off[li], o = b_off[li];
    for (int q = 0; q < L.n; ++q, ++v) {
        const avk_vcf::Var &V = L.v[q];
        contig[v] = L.contig; pos[v] = L.pos; vt[v] = V.type; zy[v] = V.zyg; raw[v] = V.raw; aoff[v] = o; l0[v] = V.l0; l1[v] = V.l1;
        for (u32 k = 0; k < V.l0; ++k) pool[o + k] = t[L.ref.b + k];
        for (u32 k = 0; k < V.l1; ++k) pool[o + V.l0 + k] = t[b + V.alt_b + k];
        o += V.l0 + V.l1;
    }
}
enum { V_TEXT, V_STARTS, V_NOUT, V_NBYTES, V_VOFF, V_BOFF, V_NAMES, V_MISC, V_C, V_POS, V_VT, V_ZY, V_RAW, V_AOFF, V_L0, V_L1, V_POOL, V_GZ, V_MEMBERS, V_MSTATUS };
// `text` on the host (uploaded into rb[V_TEXT]) or, with text == NULL and len > 0, already in rb[V_TEXT] on the device
static int vcf_parse_impl(avk_ctx *ctx, const uint8_t *text, uint64_t len, const char *const *contig_names, uint32_t n_contigs, uint32_t sample_index,
                          int enable_trimming, avk_vcf_out *out, uint64_t *error_line, int32_t *error_code) {
    if (!out || !contig_names || n_contigs == 0 || len >= 0xfffffff0ull) { ctx->err = "avk_vcf_parse: bad arguments (text up to 4 GiB per call)"; return AVK_ERR_INVALID; }
    CK(cudaSetDevice(ctx->device));
    if (error_line) *error_line = 0;
    if (error_code) *error_code = 0;
    out->n_variants = 0; out->allele_pool_len = 0;
    if (len == 0) return AVK_OK;
    DevBuf *rb = ctx->rb;   // the region builder's temporaries are free between its calls
    u32 stride = 1;
    for (u32 c = 0; c < n_contigs; ++c) { if (!contig_names[c]) { ctx->err = "avk_vcf_parse: null contig name"; return AVK_ERR_INVALID; } stride = std::max<u32>(stride, (u32)strlen(contig_names[c]) + 1); }
    std::vector<char> names((size_t)stride * n_contigs, 0);
    for (u32 c = 0; c < n_contigs; ++c) strcpy(names.data() + (size_t)c * stride, contig_names[c]);
    if (text) UPLOAD(rb[V_TEXT], text, len);
    UPLOAD(rb[V_NAMES], names.data(), names.size());
    ENSURE(rb[V_STARTS], 8 * (len / 2 + 2));                      // a line is at least one byte and its newline
    ENSURE(rb[V_MISC], 64);
    const u8 *d_text = (const u8 *)rb[V_TEXT].p;
    u64 *d_starts = (u64 *)rb[V_STARTS].p;
    unsigned long long *d_misc = (unsigned long long *)rb[V_MISC].p;   // [0] number of lines, [1] first error
    size_t need = 0, tmp = 0;
    thrust::counting_iterator<u64> it(0);
    LineStart pred{d_text, len};
    cub::DeviceSelect::If(nullptr, need, it, d_starts, d_misc, (int)len, pred, ctx->stream); tmp = std::max(tmp, need);
    ENSURE(ctx->scan_tmp, tmp);
    need = tmp; cub::DeviceSelect::If(ctx->scan_tmp.p, need, it, d_starts, d_misc, (int)len, pred, ctx->stream);
    const unsigned long long no_err = ~0ull;
    CK(cudaMemcpyAsync(d_misc + 1, &no_err, 8, cudaMemcpyHostToDevice, ctx->stream));
    unsigned long long n_lines = 0;
    CK(cudaMemcpyAsync(&n_lines, d_misc, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->launches += 1;
    if (n_lines == 0) return AVK_OK;
    for (int b : {V_NOUT, V_NBYTES, V_VOFF, V_BOFF}) ENSURE(rb[b], 4 * (n_lines + 1));
    u32 *n_out = (u32 *)rb[V_NOUT].p, *n_bytes = (u32 *)rb[V_NBYTES].p, *v_off = (u32 *)rb[V_VOFF].p, *b_off = (u32 *)rb[V_BOFF].p;
    cub::DeviceScan::ExclusiveSum(nullptr, need, n_out, v_off, (int)n_lines + 1, ctx->stream); tmp = std::max(tmp, need);
    ENSURE(ctx->scan_tmp, tmp);
    CK(cudaMemsetAsync(n_out + n_lines, 0, 4, ctx->stream)); CK(cudaMemsetAsync(n_bytes + n_lines, 0, 4, ctx->stream));
    const unsigned g = (unsigned)((n_lines + 255) / 256);
    k_vcf_scan<<<g, 256, 0, ctx->stream>>>(d_text, len, d_starts, n_lines, (const char *)rb[V_NAMES].p, n_contigs, stride, sample_index, enable_trimming, n_out, n_bytes, d_misc + 1);
    need = tmp; cub::DeviceScan::ExclusiveSum(ctx->scan_tmp.p, need, n_out, v_off, (int)n_lines + 1, ctx->stream);
    need = tmp; cub::DeviceScan::ExclusiveSum(ctx->scan_tmp.p, need, n_bytes, b_off, (int)n_lines + 1, ctx->stream);
    unsigned long long first_err = 0;
    u32 totals[2] = {0, 0};
    CK(cudaMemcpyAsync(&first_err, d_misc + 1, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&totals[0], v_off + n_lines, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&totals[1], b_off + n_lines, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->launches += 3;
    if (first_err != no_err) {                                    // Err(..) of the first failing record (region_generation.rs:533-541)
        if (error_line) *error_line = first_err >> 8;
        if (error_code) *error_code = (int32_t)(first_err & 0xff);
        ctx->err = "avk_vcf_parse: record " + std::to_string(first_err >> 8) + " cannot be parsed (code " + std::to_string(first_err & 0xff) + ")";
        return AVK_ERR_INVALID;
    }
    const u64 nv = totals[0], nb = totals[1];
    if (nv > out->cap_variants || nb > out->cap_pool) {
        out->n_variants = nv; out->allele_pool_len = nb;          // what the caller must provide
        ctx->err = "avk_vcf_parse: output capacity too small";
        return AVK_ERR_OOM;
    }
    for (int b : {V_C, V_POS, V_RAW, V_AOFF, V_L0, V_L1}) ENSURE(rb[b], 4 * nv);
    ENSURE(rb[V_VT], nv); ENSURE(rb[V_ZY], nv); ENSURE(rb[V_POOL], nb);
    k_vcf_emit<<<g, 256, 0, ctx->stream>>>(d_text, len, d_starts, n_lines, (const char *)rb[V_NAMES].p, n_contigs, stride, sample_index, enable_trimming, v_off, b_off,
                                           (u32 *)rb[V_C].p, (u32 *)rb[V_POS].p, (u8 *)rb[V_VT].p, (u8 *)rb[V_ZY].p, (u32 *)rb[V_RAW].p, (u32 *)rb[V_AOFF].p,
                                           (u32 *)rb[V_L0].p, (u32 *)rb[V_L1].p, (u8 *)rb[V_POOL].p);
    ctx->launches += 1;
    CK(cudaGetLastError());
#define VDL(dst, buf, bytes) do { if ((bytes) && (dst)) CK(cudaMemcpyAsync((void *)(dst), (buf).p, (bytes), cudaMemcpyDeviceToHost, ctx->stream)); } while (0)
    VDL(out->contig, rb[V_C], 4 * nv); VDL(out->position, rb[V_POS], 4 * nv); VDL(out->variant_type, rb[V_VT], nv); VDL(out->zygosity, rb[V_ZY], nv);
    VDL(out->raw_allele_space, rb[V_RAW], 4 * nv); VDL(out->allele_off, rb[V_AOFF], 4 * nv); VDL(out->a0_len, rb[V_L0], 4 * nv); VDL(out->a1_len, rb[V_L1], 4 * nv);
    VDL(out->allele_pool, rb[V_POOL], nb);
#undef VDL
    CK(cudaStreamSynchronize(ctx->stream));
    out->n_variants = nv; out->allele_pool_len = nb;
    return AVK_OK;
}
extern "C" int avk_vcf_parse(avk_ctx *ctx, const uint8_t *text, uint64_t len, const char *const *contig_names, uint32_t n_contigs, uint32_t sample_index,
                             int enable_trimming, avk_vcf_out *out, uint64_t *error_line, int32_t *error_code) {
    if (!ctx) return AVK_ERR_INVALID;
    if (!text && len) { ctx->err = "avk_vcf_parse: null text"; return AVK_ERR_INVALID; }
    return vcf_parse_impl(ctx, text, len, contig_names, n_contigs, sample_index, enable_trimming, out, error_line, error_code);
}

// ---- BGZF inflate (SURVEY 8f N2, avk_inflate.cuh): one thread per member ------------------------------------------------------
// One warp per member: lane 0 decodes into a 64 KiB window in shared memory (Huffman tables and the CRC tables beside it: a
// decoder is a chain of dependent loads, ~30 cycles each there against ~600 in global memory, where a match would read bytes the
// same thread has just written), then the warp copies the window out with 16-byte stores.  The window starts at the output's
// offset modulo 16 so that both sides of that copy are aligned.  Members that declare more than 64 KiB (legal gzip, not BGZF)
// are decoded straight into global memory.
enum { BGZF_WIN = 65536, BGZF_SMEM = BGZF_WIN + 16 + ((sizeof(avk_inflate::Tables) + 15) & ~15) + 4 * 256 * 4 };
__global__ void __launch_bounds__(32) k_bgzf_inflate(const u8 *gz, const avk_inflate::Member *mem, u32 n_members, u8 *out, int verify_crc, u32 *status) {
    u8 *win = avk_dyn_smem;
    avk_inflate::Tables &tab = *(avk_inflate::Tables *)(avk_dyn_smem + BGZF_WIN + 16);
    u32 *crc_t = (u32 *)(avk_dyn_smem + BGZF_WIN + 16 + ((sizeof(avk_inflate::Tables) + 15) & ~15));      // slicing by 4: T0..T3
    const int lane = threadIdx.x;
    for (u32 i = lane; i < 256; i += 32) crc_t[i] = avk_inflate::crc_entry(i);
    __syncwarp();
    for (int t = 1; t < 4; ++t) {
        for (u32 i = lane; i < 256; i += 32) { const u32 p = crc_t[(t - 1) * 256 + i]; crc_t[t * 256 + i] = (p >> 8) ^ crc_t[p & 0xffu]; }
        __syncwarp();
    }
    for (u32 k = blockIdx.x; k < n_members; k += gridDim.x) {
        const avk_inflate::Member m = mem[k];
        u8 *dst = out + m.o_off;
        const bool windowed = m.isize <= BGZF_WIN;
        const u32 pad = (u32)((uintptr_t)dst & 15u);
        u8 *buf = windowed ? win + pad : dst;
        int rc = 0;
        uint64_t got = 0;
        if (lane == 0) {
            rc = avk_inflate::inflate(gz + m.c_off, m.c_len, buf, m.isize, &got, tab);
            if (rc == avk_inflate::INF_OK && got != m.isize) rc = avk_inflate::INF_E_SIZE;
            if (rc == avk_inflate::INF_OK && verify_crc) {
                u32 c = 0xffffffffu;
                u32 i = 0;
                const u32 n = (u32)got;
                while (i < n && ((uintptr_t)(buf + i) & 3u)) { c = crc_t[(c ^ buf[i]) & 0xffu] ^ (c >> 8); ++i; }
                for (; i + 4 <= n; i += 4) {
                    c ^= *(const u32 *)(buf + i);
                    c = crc_t[768 + (c & 0xffu)] ^ crc_t[512 + ((c >> 8) & 0xffu)] ^ crc_t[256 + ((c >> 16) & 0xffu)] ^ crc_t[c >> 24];
                }
                for (; i < n; ++i) c = crc_t[(c ^ buf[i]) & 0xffu] ^ (c >> 8);
                if ((c ^ 0xffffffffu) != m.crc) rc = avk_inflate::INF_E_CRC;
            }
            status[k] = (u32)rc;
        }
        rc = __shfl_sync(AVK_FULL, rc, 0);
        __syncwarp();
        if (rc == avk_inflate::INF_OK && windowed) {
            const u32 n = m.isize;
            const u32 head = min(n, (16u - pad) & 15u);
            for (u32 i = lane; i < head; i += 32) dst[i] = buf[i];
            const u32 body = (n - head) >> 4;
            const uint4 *s4 = (const uint4 *)(buf + head);
            uint4 *d4 = (uint4 *)(dst + head);
            for (u32 i = lane; i < body; i += 32) d4[i] = s4[i];
            for (u32 i = head + (body << 4) + lane; i < n; i += 32) dst[i] = buf[i];
        }
        __syncwarp();
    }
}
// Walks the members on the host, uploads the file and inflates every member on the device into rb[V_TEXT]; *total = bytes.
static int bgzf_inflate_device(avk_ctx *ctx, const uint8_t *gz, uint64_t gz_len, int verify_crc, uint64_t *total, std::vector<avk_inflate::Member> *members_out) {
    std::vector<avk_inflate::Member> mem;
    uint64_t at = 0, o = 0;
    while (at < gz_len) {
        avk_inflate::Member m;
        uint64_t next = 0;
        const int rc = avk_inflate::member_at(gz, gz_len, at, m, next);
        if (rc != 0) {
            ctx->err = "BGZF member " + std::to_string(mem.size()) + " at byte " + std::to_string(at) +
                       (rc == -1 ? ": truncated" : rc == -2 ? ": not a gzip member with an extra field (plain gzip is not BGZF)" : ": no BC subfield / inconsistent sizes");
            return AVK_ERR_INVALID;
        }
        m.o_off = o; o += m.isize;
        if (m.isize) mem.push_back(m);                       // (empty members -- the EOF marker -- produce nothing)
        at = next;
    }
    *total = o;
    if (members_out) { *members_out = mem; return AVK_OK; }
    if (o == 0) return AVK_OK;
    CK(cudaSetDevice(ctx->device));
    DevBuf *rb = ctx->rb;
    UPLOAD(rb[V_GZ], gz, gz_len);
    UPLOAD(rb[V_MEMBERS], mem.data(), mem.size() * sizeof(avk_inflate::Member));
    ENSURE(rb[V_MSTATUS], 4 * mem.size());
    ENSURE(rb[V_TEXT], o);
    const u32 n = (u32)mem.size();
    CK(cudaFuncSetAttribute(k_bgzf_inflate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BGZF_SMEM));      // (per device; cheap)
    k_bgzf_inflate<<<std::min<u32>(n, 3u * (u32)ctx->sm_count), 32, BGZF_SMEM, ctx->stream>>>((const u8 *)rb[V_GZ].p, (const avk_inflate::Member *)rb[V_MEMBERS].p, n, (u8 *)rb[V_TEXT].p, verify_crc,
                                                          (u32 *)rb[V_MSTATUS].p);
    ctx->launches += 1;
    CK(cudaGetLastError());
    std::vector<u32> st(n);
    CK(cudaMemcpyAsync(st.data(), rb[V_MSTATUS].p, 4 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (u32 k = 0; k < n; ++k)
        if (st[k] != 0) { ctx->err = "BGZF member with payload at byte " + std::to_string(mem[k].c_off) + " does not inflate (code " + std::to_string(st[k]) + ")"; return AVK_ERR_INVALID; }
    return AVK_OK;
}
extern "C" int avk_bgzf_inflate(avk_ctx *ctx, const uint8_t *gz, uint64_t gz_len, int verify_crc, uint8_t *out, uint64_t out_cap, uint64_t *out_len) {
    if (!ctx) return AVK_ERR_INVALID;
    if ((!gz && gz_len) || !out_len) { ctx->err = "avk_bgzf_inflate: bad arguments"; return AVK_ERR_INVALID; }
    uint64_t total = 0;
    if (!out) {                                              // size query: the host walk only
        std::vector<avk_inflate::Member> mem;
        const int rc = bgzf_inflate_device(ctx, gz, gz_len, verify_crc, &total, &mem);
        *out_len = total;
        return rc;
    }
    int rc = bgzf_inflate_device(ctx, gz, gz_len, verify_crc, &total, nullptr);
    *out_len = total;
    if (rc != AVK_OK) return rc;
    if (total > out_cap) { ctx->err = "avk_bgzf_inflate: output capacity too small"; return AVK_ERR_OOM; }
    if (total) CK(cudaMemcpyAsync(out, ctx->rb[V_TEXT].p, total, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return AVK_OK;
}
// ---- BGZF compression of the text outputs (SURVEY 8f N3, avk_inflate.cuh::deflate_member): one warp per 0xff00-byte chunk ---------
// The chunk is staged in shared memory by the whole warp; lane 0 runs the two LZ77 passes over it (hash table, symbol counts and
// Huffman codes are in shared memory too) and writes the payload into the chunk's slot of a scratch buffer; k_bgzf_pack then lays header, payload and trailer of
// every member end to end (the offsets are the prefix sums of the payload lengths, taken on the host).
enum { BGZF_DEF_WORK = (sizeof(avk_inflate::DeflateWork) + 15) & ~15, BGZF_DEF_SMEM = avk_inflate::DEFLATE_CHUNK + BGZF_DEF_WORK + 4 * 256 * 4, BGZF_PAY_STRIDE = 65536 };
__global__ void __launch_bounds__(32) k_bgzf_deflate(const u8 *text, u64 len, u32 n_chunks, u8 *pay, u32 *c_len, u32 *crc) {
    u8 *win = avk_dyn_smem;
    avk_inflate::DeflateWork &work = *(avk_inflate::DeflateWork *)(avk_dyn_smem + avk_inflate::DEFLATE_CHUNK);      // hash table, symbol counts, codes
    u32 *crc_t = (u32 *)(avk_dyn_smem + avk_inflate::DEFLATE_CHUNK + BGZF_DEF_WORK);
    const int lane = threadIdx.x;
    for (u32 i = lane; i < 256; i += 32) crc_t[i] = avk_inflate::crc_entry(i);
    __syncwarp();
    for (int t = 1; t < 4; ++t) {
        for (u32 i = lane; i < 256; i += 32) { const u32 p = crc_t[(t - 1) * 256 + i]; crc_t[t * 256 + i] = (p >> 8) ^ crc_t[p & 0xffu]; }
        __syncwarp();
    }
    for (u32 k = blockIdx.x; k < n_chunks; k += gridDim.x) {
        const u64 at = (u64)k * avk_inflate::DEFLATE_CHUNK;
        const u32 n = (u32)min((u64)avk_inflate::DEFLATE_CHUNK, len - at);
        const u8 *src = text + at;                               // chunk starts are multiples of 0xff00: 16-byte aligned in a cudaMalloc'd buffer
        const u32 body = n >> 4;
        for (u32 i = lane; i < body; i += 32) ((uint4 *)win)[i] = ((const uint4 *)src)[i];
        for (u32 i = (body << 4) + lane; i < n; i += 32) win[i] = src[i];
        __syncwarp();
        if (lane == 0) {
            c_len[k] = avk_inflate::deflate_member(win, n, pay + (u64)k * BGZF_PAY_STRIDE, work);
            crc[k] = avk_inflate::crc32_4(crc_t, win, n);
        }
        __syncwarp();
    }
}
__global__ void __launch_bounds__(128) k_bgzf_pack(const u8 *pay, const u32 *c_len, const u32 *crc, const u64 *m_off, u64 len, u32 n_chunks, u8 *out) {
    const u32 k = blockIdx.x;                                    // member k; member n_chunks is the EOF marker
    u8 *dst = out + m_off[k];
    if (k == n_chunks) {
        if (threadIdx.x == 0) { avk_inflate::member_header(dst, 2); dst[18] = 3; dst[19] = 0; avk_inflate::member_trailer(dst + 20, 0, 0); }
        return;
    }
    const u32 c = c_len[k];
    const u64 at = (u64)k * avk_inflate::DEFLATE_CHUNK;
    if (threadIdx.x == 0) {
        avk_inflate::member_header(dst, c);
        avk_inflate::member_trailer(dst + 18 + c, crc[k], (u32)min((u64)avk_inflate::DEFLATE_CHUNK, len - at));
    }
    const u8 *src = pay + (u64)k * BGZF_PAY_STRIDE;
    for (u32 i = threadIdx.x; i < c; i += blockDim.x) dst[18 + i] = src[i];
}
static u64 bgzf_chunks(u64 len) { return (len + avk_inflate::DEFLATE_CHUNK - 1) / avk_inflate::DEFLATE_CHUNK; }
static u64 bgzf_bound(u64 len) { return len + 31 * bgzf_chunks(len) + 28; }         // upper bound: every chunk stored, EOF marker
enum { C_TEXT = V_TEXT, C_PAY = V_GZ, C_LEN = V_NOUT, C_CRC = V_NBYTES, C_OFF = V_STARTS, C_OUT = V_POOL };   // the compressor's rb slots
// The `len` bytes of text already in rb[V_TEXT] -> BGZF members of 0xff00 input bytes (+ the EOF marker when eof) in `out`.
static int bgzf_compress_device(avk_ctx *ctx, u64 len, bool eof, uint8_t *out, uint64_t cap, uint64_t *out_len) {
    DevBuf *rb = ctx->rb;
    const u64 n_chunks = bgzf_chunks(len);
    std::vector<u64> m_off(n_chunks + 2, 0);
    std::vector<u32> c_len(n_chunks);
    if (n_chunks) {
        ENSURE(rb[C_PAY], n_chunks * (u64)BGZF_PAY_STRIDE);
        ENSURE(rb[C_LEN], 4 * n_chunks); ENSURE(rb[C_CRC], 4 * n_chunks);
        CK(cudaFuncSetAttribute(k_bgzf_deflate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BGZF_DEF_SMEM));
        k_bgzf_deflate<<<(unsigned)std::min<u64>(n_chunks, 2ull * ctx->sm_count), 32, BGZF_DEF_SMEM, ctx->stream>>>((const u8 *)rb[C_TEXT].p, len, (u32)n_chunks, (u8 *)rb[C_PAY].p,
                                                                                                                   (u32 *)rb[C_LEN].p, (u32 *)rb[C_CRC].p);
        ctx->launches += 1;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(c_len.data(), rb[C_LEN].p, 4 * n_chunks, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    for (u64 k = 0; k < n_chunks; ++k) m_off[k + 1] = m_off[k] + 18 + c_len[k] + 8;
    m_off[n_chunks + 1] = m_off[n_chunks] + 28;
    const u64 total = m_off[n_chunks + (eof ? 1 : 0)];
    *out_len = total;
    if (total > cap) { ctx->err = "BGZF output capacity too small"; return AVK_ERR_OOM; }
    if (total == 0) return AVK_OK;
    UPLOAD(rb[C_OFF], m_off.data(), 8 * m_off.size());
    ENSURE(rb[C_OUT], total);
    k_bgzf_pack<<<(unsigned)(n_chunks + (eof ? 1 : 0)), 128, 0, ctx->stream>>>((const u8 *)rb[C_PAY].p, (const u32 *)rb[C_LEN].p, (const u32 *)rb[C_CRC].p,
                                                                                (const u64 *)rb[C_OFF].p, len, (u32)n_chunks, (u8 *)rb[C_OUT].p);
    ctx->launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, rb[C_OUT].p, total, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return AVK_OK;
}
extern "C" int avk_bgzf_compress(avk_ctx *ctx, const uint8_t *text, uint64_t len, uint8_t *out, uint64_t cap, uint64_t *out_len) {
    if (!ctx) return AVK_ERR_INVALID;
    if ((!text && len) || !out_len) { ctx->err = "avk_bgzf_compress: bad arguments"; return AVK_ERR_INVALID; }
    if (bgzf_chunks(len) >= 0x7fffffffull) { ctx->err = "avk_bgzf_compress: text too long for one call"; return AVK_ERR_INVALID; }
    if (!out) { *out_len = bgzf_bound(len); return AVK_OK; }
    CK(cudaSetDevice(ctx->device));
    if (len) UPLOAD(ctx->rb[C_TEXT], text, len);
    return bgzf_compress_device(ctx, len, true, out, cap, out_len);
}

// ---- labelled VCF records of the resident compare, formatted on the device (avk_writers.h::vcf_records_text) ----------------
// Count pass (one thread per region: records of the side, contig check) -> 64-bit scan -> length pass (one thread per record)
// -> 64-bit scan -> write pass into rb[V_TEXT] after the header -> bgzf_compress_device.  Alleles longer than RW_LONG bytes
// are copied by the whole warp, so an SV allele (or one of the 16 MiB scan_bin admits) does not hold up its warp's other lines.
enum { W_CNT = V_VOFF, W_LEN = V_BOFF, W_NAMES = V_NAMES, W_MISC = V_MISC, W_REG = V_C, W_RID = V_POS };   // off the compressor's slots
enum { RW_LONG = 32 };
// The contig names (and, for the merge records, the input labels) of a device writer, packed into rb[W_NAMES]: the
// [n_contigs + 1] name offsets, the [n_labels + 1] label offsets (from the first label), then the names and the labels.
// plain: refuse a name the debug writers would have to quote (avk_writers.h::plain_name).
struct NameTable {
    const u64 *name_off, *label_off;
    const char *names, *labels;
};
static int upload_names(avk_ctx *ctx, const char *who, const char *const *contig_names, u32 n_contigs, const char *const *labels, u64 n_labels,
                        bool plain, NameTable &t) {
    std::vector<u64> tab(n_contigs + 1 + (labels ? n_labels + 1 : 0), 0);
    std::string packed;
    for (u32 c = 0; c < n_contigs; ++c) {
        if (!contig_names[c]) { ctx->err = std::string(who) + ": null contig name"; return AVK_ERR_INVALID; }
        if (plain && !avk_writers::plain_name(contig_names[c])) {
            ctx->err = std::string(who) + ": a contig name contains a tab, '\"', CR or LF";
            return AVK_ERR_INVALID;
        }
        packed += contig_names[c];
        tab[c + 1] = packed.size();
    }
    const u64 names_len = packed.size();
    if (labels) {
        u64 *lt = tab.data() + n_contigs + 1;
        for (u64 k = 0; k < n_labels; ++k) {
            if (!labels[k]) { ctx->err = std::string(who) + ": null input label"; return AVK_ERR_INVALID; }
            packed += labels[k];
            lt[k + 1] = packed.size() - names_len;
        }
    }
    DevBuf *rb = ctx->rb;
    const size_t tab_bytes = 8 * tab.size();
    ENSURE(rb[W_NAMES], tab_bytes + packed.size());
    CK(cudaMemcpyAsync(rb[W_NAMES].p, tab.data(), tab_bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (!packed.empty()) CK(cudaMemcpyAsync((u8 *)rb[W_NAMES].p + tab_bytes, packed.data(), packed.size(), cudaMemcpyHostToDevice, ctx->stream));
    t.name_off = (const u64 *)rb[W_NAMES].p; t.label_off = t.name_off + n_contigs + 1;
    t.names = (const char *)rb[W_NAMES].p + tab_bytes; t.labels = t.names + names_len;
    return AVK_OK;
}
struct RecView {
    const u64 *var_off, *rid;
    const u32 *contig, *pos, *aoff, *l0, *l1;
    const u8 *zyg, *pool, *cls, *exp, *obs;
    const u64 *name_off;                 // [n_contigs + 1], the packed names follow
    const char *names;
    u32 K, side;
};
__device__ __forceinline__ u32 rw_digits(u64 x) { u32 d = 1; while (x >= 10) { x /= 10; ++d; } return d; }
__device__ __forceinline__ u8 *rw_put_u64(u8 *o, u64 x, u32 d) { for (u32 k = d; k-- > 0; x /= 10) o[k] = (u8)('0' + x % 10); return o + d; }
__device__ __forceinline__ u8 *rw_put_str(u8 *o, const char *s, u32 n) { for (u32 k = 0; k < n; ++k) o[k] = (u8)s[k]; return o + n; }
// GT string (PhasedZygosity, variant_categorizer.rs:190-197) and BD label (Classification) of a record, as the host writer picks them
__device__ __forceinline__ const char *rw_gt(u8 z, u32 &n) {
    const char *s = z == 1 ? "0/0" : z == 2 ? "0/1" : z == 3 ? "0|1" : z == 4 ? "1|0" : z == 5 ? "1/1" : ".";
    n = z >= 1 && z <= AVK_ZYG_HOM_ALT ? 3 : 1;
    return s;
}
__device__ __forceinline__ const char *rw_bd(u8 c, u32 &n) {
    n = c == 1 || c == 2 || c == 3 ? 2 : 3;
    return c == 1 ? "TP" : c == 2 ? "FN" : c == AVK_CLASS_FP ? "FP" : "UNK";
}
// one allele copied by the whole warp, eight loads in flight per lane (the source and the text never overlap)
__device__ __forceinline__ void rw_warp_copy(u8 *__restrict__ dst, const u8 *__restrict__ src, u32 n, int lane) {
    for (u32 k = lane; k < n; k += 256) {
        u8 b[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) b[j] = k + 32 * j < n ? src[k + 32 * j] : 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) if (k + 32 * j < n) dst[k + 32 * j] = b[j];
    }
}
static __device__ const char RW_MID[] ="\t.\t.\t.\tGT:BD:EA:OA:RI\t";       // ALT | QUAL FILTER INFO FORMAT | sample
enum { RW_MID_LEN = 22 };

__global__ void __launch_bounds__(256) k_rw_count(RecView w, u64 n, u32 n_contigs, u64 *cnt, unsigned long long *bad) {
    const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r > n) return;
    if (r == n) { cnt[n] = 0; return; }
    cnt[r] = w.var_off[r * w.K + w.side + 1] - w.var_off[r * w.K + w.side];
    if (w.contig[r] >= n_contigs) atomicMax(bad, 1ull);
}
// record i of the side -> (region r, variant v); rec_off = exclusive scan of the per-region counts, [n + 1]
__device__ __forceinline__ u64 rw_region(const u64 *rec_off, u64 n, u64 i) {
    u64 lo = 0, hi = n;                                          // last r with rec_off[r] <= i (empty regions share offsets)
    while (hi - lo > 1) { const u64 m = (lo + hi) >> 1; if (rec_off[m] <= i) lo = m; else hi = m; }
    return lo;
}
__global__ void __launch_bounds__(256) k_rw_len(RecView w, u64 n, u64 n_rec, const u64 *rec_off, u32 *reg, u64 *len) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n_rec) return;
    if (i == n_rec) { len[n_rec] = 0; return; }
    const u64 r = rw_region(rec_off, n, i);
    const u64 v = w.var_off[r * w.K + w.side] + (i - rec_off[r]);
    const u32 c = w.contig[r];
    const int32_t ri = (int32_t)(u32)w.rid[r];
    u32 ng, nb;
    rw_gt(w.zyg[v], ng); rw_bd(w.cls[v], nb);
    reg[i] = (u32)r;
    len[i] = (w.name_off[c + 1] - w.name_off[c]) + 1 + rw_digits((u64)w.pos[v] + 1) + 3 + w.l0[v] + 1 + w.l1[v] + RW_MID_LEN + ng + 1 + nb + 1 +
             rw_digits(w.exp[v]) + 1 + rw_digits(w.obs[v]) + 1 + (ri < 0 ? 1 : 0) + rw_digits(ri < 0 ? (u64)(-(int64_t)ri) : (u64)ri) + 1;
}
// off = exclusive scan of the line lengths; line i starts at text + base + off[i]
__global__ void __launch_bounds__(256) k_rw_write(RecView w, u64 n_rec, const u32 *reg, const u64 *rec_off, const u64 *off, u64 base, u8 *text) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const bool act = i < n_rec;
    u64 a0_at = 0, a1_at = 0, src = 0;
    u32 l0 = 0, l1 = 0;
    if (act) {
        const u64 r = reg[i];
        const u64 v = w.var_off[r * w.K + w.side] + (i - rec_off[r]);
        const u32 c = w.contig[r];
        u8 *o = text + base + off[i];
        o = rw_put_str(o, w.names + w.name_off[c], (u32)(w.name_off[c + 1] - w.name_off[c]));
        *o++ = '\t';
        const u64 p = (u64)w.pos[v] + 1;
        o = rw_put_u64(o, p, rw_digits(p));
        *o++ = '\t'; *o++ = '.'; *o++ = '\t';
        l0 = w.l0[v]; l1 = w.l1[v];
        src = (u64)(uintptr_t)(w.pool + w.aoff[v]);
        a0_at = (u64)(o - text);
        if (l0 <= RW_LONG) rw_put_str(o, (const char *)src, l0);
        o += l0;
        *o++ = '\t';
        a1_at = (u64)(o - text);
        if (l1 <= RW_LONG) rw_put_str(o, (const char *)src + l0, l1);
        o += l1;
        o = rw_put_str(o, RW_MID, RW_MID_LEN);
        u32 ng, nb;
        const char *gt = rw_gt(w.zyg[v], ng), *bd = rw_bd(w.cls[v], nb);
        o = rw_put_str(o, gt, ng); *o++ = ':';
        o = rw_put_str(o, bd, nb); *o++ = ':';
        o = rw_put_u64(o, w.exp[v], rw_digits(w.exp[v])); *o++ = ':';
        o = rw_put_u64(o, w.obs[v], rw_digits(w.obs[v])); *o++ = ':';
        const int32_t ri = (int32_t)(u32)w.rid[r];                   // `region_id as i32` (:214)
        if (ri < 0) *o++ = '-';
        const u64 ra = ri < 0 ? (u64)(-(int64_t)ri) : (u64)ri;
        o = rw_put_u64(o, ra, rw_digits(ra));
        *o = '\n';
    }
    const int lane = lane_id();
    for (u32 m = __ballot_sync(AVK_FULL, act && (l0 > RW_LONG || l1 > RW_LONG)); m; m &= m - 1) {
        const int s = __ffs(m) - 1;
        const u8 *sp = (const u8 *)(uintptr_t)__shfl_sync(AVK_FULL, src, s);
        const u32 n0 = __shfl_sync(AVK_FULL, l0, s), n1 = __shfl_sync(AVK_FULL, l1, s);
        const u64 d0 = __shfl_sync(AVK_FULL, a0_at, s), d1 = __shfl_sync(AVK_FULL, a1_at, s);
        if (n0 > RW_LONG) rw_warp_copy(text + d0, sp, n0, lane);
        if (n1 > RW_LONG) rw_warp_copy(text + d1, sp + n0, n1, lane);
    }
}

extern "C" int avk_compare_records_bgzf(avk_ctx *ctx, uint32_t side, const char *const *contig_names, uint32_t n_contigs, const uint64_t *region_id,
                                        const uint8_t *header, uint64_t header_len, int eof, uint8_t *out, uint64_t cap, uint64_t *out_len) {
    if (!ctx) return AVK_ERR_INVALID;
    if (!ctx->have_batch || !ctx->have_result) { ctx->err = "avk_compare_records_bgzf: no compare result is resident (run avk_compare_run_resident first)"; return AVK_ERR_INVALID; }
    if (side >= ctx->n_inputs || (!contig_names && n_contigs) || (!header && header_len) || !out_len) { ctx->err = "avk_compare_records_bgzf: bad arguments"; return AVK_ERR_INVALID; }
    if (!region_id && !ctx->ids_resident) { ctx->err = "avk_compare_records_bgzf: the batch was uploaded, so its region ids must be given"; return AVK_ERR_INVALID; }
    CK(cudaSetDevice(ctx->device));
    DevBuf *rb = ctx->rb;
    const u64 n = ctx->n_regions, K = ctx->n_inputs;
    NameTable nt;
    int rc = upload_names(ctx, "avk_compare_records_bgzf", contig_names, n_contigs, nullptr, 0, false, nt);
    if (rc != AVK_OK) return rc;
    const DevBatch db = dev_batch(ctx);
    RecView w;
    w.var_off = db.var_off; w.contig = db.contig; w.pos = db.pos; w.aoff = db.aoff; w.l0 = db.l0; w.l1 = db.l1; w.zyg = db.zyg; w.pool = db.pool;
    w.cls = biased<const u8>(ctx->vcls, ctx->v_base); w.exp = biased<const u8>(ctx->vexp, ctx->v_base); w.obs = biased<const u8>(ctx->vobs, ctx->v_base);
    w.name_off = nt.name_off; w.names = nt.names;
    w.K = (u32)K; w.side = side;
    if (region_id) {                                              // the caller's ids of the resident bin [lo, lo + n)
        UPLOAD(rb[W_RID], region_id + ctx->lo, 8 * n);
        w.rid = (const u64 *)rb[W_RID].p;
    } else {
        w.rid = (const u64 *)ctx->region_id.p;
    }
    // count pass and the scan of the per-region record counts
    ENSURE(rb[W_MISC], 64);
    unsigned long long *d_misc = (unsigned long long *)rb[W_MISC].p;     // [0] contig out of range
    ENSURE(rb[W_CNT], 8 * (n + 1));
    u64 *rec_off = (u64 *)rb[W_CNT].p;
    CK(cudaMemsetAsync(d_misc, 0, 8, ctx->stream));
    size_t need = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, need, rec_off, rec_off, n + 1, ctx->stream);
    ENSURE(ctx->scan_tmp, need);
    k_rw_count<<<(unsigned)((n + 1 + 255) / 256), 256, 0, ctx->stream>>>(w, n, n_contigs, rec_off, d_misc);
    CK(cub::DeviceScan::ExclusiveSum(ctx->scan_tmp.p, need, rec_off, rec_off, n + 1, ctx->stream));
    unsigned long long h[2] = {0, 0};
    CK(cudaMemcpyAsync(&h[0], d_misc, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&h[1], rec_off + n, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->launches += 2;
    CK(cudaGetLastError());
    if (h[0]) { ctx->err = "avk_compare_records_bgzf: a region's contig is not below n_contigs"; return AVK_ERR_INVALID; }
    const u64 n_rec = h[1];
    // length pass and the scan of the line lengths (64-bit counts and offsets throughout)
    ENSURE(rb[W_LEN], 8 * (n_rec + 1));
    ENSURE(rb[W_REG], 4 * n_rec);
    u64 *off = (u64 *)rb[W_LEN].p;
    u32 *reg = (u32 *)rb[W_REG].p;
    need = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, need, off, off, n_rec + 1, ctx->stream);
    ENSURE(ctx->scan_tmp, need);
    k_rw_len<<<(unsigned)((n_rec + 1 + 255) / 256), 256, 0, ctx->stream>>>(w, n, n_rec, rec_off, reg, off);
    CK(cub::DeviceScan::ExclusiveSum(ctx->scan_tmp.p, need, off, off, n_rec + 1, ctx->stream));
    u64 body = 0;
    CK(cudaMemcpyAsync(&body, off + n_rec, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->launches += 2;
    CK(cudaGetLastError());
    const u64 len = header_len + body;
    if (bgzf_chunks(len) >= 0x7fffffffull) { ctx->err = "avk_compare_records_bgzf: text too long for one call"; return AVK_ERR_INVALID; }
    if (!out) { *out_len = bgzf_bound(len); return AVK_OK; }
    // header + lines into rb[V_TEXT], then the compressor
    ENSURE(rb[C_TEXT], len);
    u8 *text = (u8 *)rb[C_TEXT].p;
    if (header_len) CK(cudaMemcpyAsync(text, header, header_len, cudaMemcpyHostToDevice, ctx->stream));
    if (n_rec) {
        k_rw_write<<<(unsigned)((n_rec + 255) / 256), 256, 0, ctx->stream>>>(w, n_rec, reg, rec_off, off, header_len, text);
        ctx->launches += 1;
        CK(cudaGetLastError());
    }
    return bgzf_compress_device(ctx, len, eof != 0, out, cap, out_len);
}

// ---- the debug folder of the resident compare, formatted on the device (avk_writers.h::region_summary_text and
// region_sequences_text) ----------------------------------------------------------------------------------------------------
// region_summary.tsv: count pass (one thread per region: n_metrics lines when solved, contig check) -> 64-bit scan -> length
// pass (one thread per line; a line is a (solved region, metric) pair) -> scan -> write pass -> bgzf_compress_device.
// region_sequences.tsv: length pass (one thread per region) -> scan -> write pass.  Strings longer than RW_LONG bytes are
// copied by the whole warp: SV windows reach 64 kbp and more, so one line can be longer than a BGZF member.
struct RegionView {
    const u64 *rid;
    const u32 *contig, *start, *end;
    const int *status;
    const u64 *rows;                     // [n][RED_COLS] per-region metric rows
    const u64 *seq_off;                  // [n * 5 + 1], values biased by seq_base
    const u32 *seq_len;                  // [n * 5]
    const u8 *seq_pool;                  // biased by seq_base: string s of region r starts at seq_pool + seq_off[r * 5 + s]
    const u8 *metrics;
    u32 n_metrics;
    NameTable nt;
};
__device__ __forceinline__ u32 rv_name_len(const RegionView &w, u32 c) { return (u32)(w.nt.name_off[c + 1] - w.nt.name_off[c]); }
// "region_id \t chrom:start+1-end" (avk_writers.h::region_key)
__device__ __forceinline__ u64 rv_key_len(const RegionView &w, u64 r) {
    return rw_digits(w.rid[r]) + 1 + rv_name_len(w, w.contig[r]) + 1 + rw_digits((u64)w.start[r] + 1) + 1 + rw_digits(w.end[r]);
}
__device__ __forceinline__ u8 *rv_put_key(const RegionView &w, u64 r, u8 *o) {
    o = rw_put_u64(o, w.rid[r], rw_digits(w.rid[r])); *o++ = '\t';
    const u32 c = w.contig[r];
    o = rw_put_str(o, w.nt.names + w.nt.name_off[c], rv_name_len(w, c)); *o++ = ':';
    const u64 s = (u64)w.start[r] + 1;
    o = rw_put_u64(o, s, rw_digits(s)); *o++ = '-';
    return rw_put_u64(o, w.end[r], rw_digits(w.end[r]));
}
// avk_writers.h::METRIC_NAMES / METRIC_COL
__device__ __forceinline__ const char *rs_metric(u32 m, u32 &n, u32 &col) {
    switch (m) {
        case 0: n = 2; col = AVK_M_GT; return "GT";
        case 1: n = 3; col = AVK_M_HAP; return "HAP";
        case 2: n = 12; col = AVK_M_WEIGHTED_HAP; return "WEIGHTED_HAP";
        case 3: n = 8; col = AVK_M_BASEPAIR; return "BASEPAIR";
        default: n = 9; col = AVK_M_RECORD_BP; return "RECORD_BP";
    }
}
__global__ void __launch_bounds__(256) k_rs_count(RegionView w, u64 n, u32 n_contigs, u64 *cnt, unsigned long long *bad) {
    const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r > n) return;
    if (r == n) { cnt[n] = 0; return; }
    cnt[r] = w.status[r] == 0 ? w.n_metrics : 0;
    if (w.contig[r] >= n_contigs) atomicMax(bad, 1ull);
}
__global__ void __launch_bounds__(256) k_rs_len(RegionView w, u64 n, u64 n_lines, const u64 *line_off, u32 *reg, u64 *len) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n_lines) return;
    if (i == n_lines) { len[n_lines] = 0; return; }
    const u64 r = rw_region(line_off, n, i);
    u32 nm, col;
    const u32 m = w.metrics[i - line_off[r]];
    rs_metric(m, nm, col);
    const u64 *row = w.rows + r * RED_COLS;                       // the joint group
    u64 l = rv_key_len(w, r) + 1 + nm + 4 + rw_digits(row[col]) + rw_digits(row[col + 1]) + rw_digits(row[col + 2]) + rw_digits(row[col + 3]) + 3;
    if (m == 0) l += rw_digits(row[AVK_M_GT_TRUTH_FN_GT]) + rw_digits(row[AVK_M_GT_QUERY_FP_GT]);
    reg[i] = (u32)r;
    len[i] = l;
}
// off = exclusive scan of the line lengths; line i starts at text + base + off[i]
__global__ void __launch_bounds__(256) k_rs_write(RegionView w, u64 n_lines, const u32 *reg, const u64 *line_off, const u64 *off, u64 base, u8 *text) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_lines) return;
    const u64 r = reg[i];
    u32 nm, col;
    const u32 m = w.metrics[i - line_off[r]];
    const char *name = rs_metric(m, nm, col);
    const u64 *row = w.rows + r * RED_COLS;
    u8 *o = rv_put_key(w, r, text + base + off[i]);
    *o++ = '\t';
    o = rw_put_str(o, name, nm);
    for (u32 k = 0; k < 4; ++k) { *o++ = '\t'; o = rw_put_u64(o, row[col + k], rw_digits(row[col + k])); }
    *o++ = '\t';
    if (m == 0) o = rw_put_u64(o, row[AVK_M_GT_TRUTH_FN_GT], rw_digits(row[AVK_M_GT_TRUTH_FN_GT]));
    *o++ = '\t';
    if (m == 0) o = rw_put_u64(o, row[AVK_M_GT_QUERY_FP_GT], rw_digits(row[AVK_M_GT_QUERY_FP_GT]));
    *o = '\n';
}
__global__ void __launch_bounds__(256) k_rq_len(RegionView w, u64 n, u32 n_contigs, u64 *len, unsigned long long *bad) {
    const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r > n) return;
    if (r == n) { len[n] = 0; return; }
    if (w.contig[r] >= n_contigs) { atomicMax(bad, 1ull); len[r] = 0; return; }
    u64 l = 0;
    if (w.status[r] == 0) {
        l = rv_key_len(w, r) + 5 + 1;
        for (int s = 0; s < 5; ++s) l += w.seq_len[r * 5 + s];
    }
    len[r] = l;
}
__global__ void __launch_bounds__(256) k_rq_write(RegionView w, u64 n, const u64 *off, u64 base, u8 *text) {
    const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const bool act = r < n && off[r + 1] > off[r];
    u64 at[5] = {0, 0, 0, 0, 0};
    bool any_long = false;
    if (act) {
        u8 *o = rv_put_key(w, r, text + base + off[r]);
#pragma unroll
        for (int s = 0; s < 5; ++s) {
            *o++ = '\t';
            const u32 l = w.seq_len[r * 5 + s];
            at[s] = (u64)(o - text);
            if (l <= RW_LONG) rw_put_str(o, (const char *)w.seq_pool + w.seq_off[r * 5 + s], l);
            else any_long = true;
            o += l;
        }
        *o = '\n';
    }
    const int lane = lane_id();
    for (u32 m = __ballot_sync(AVK_FULL, any_long); m; m &= m - 1) {
        const int src_lane = __ffs(m) - 1;
        const u64 rr = __shfl_sync(AVK_FULL, r, src_lane);
#pragma unroll
        for (int s = 0; s < 5; ++s) {
            const u64 d = __shfl_sync(AVK_FULL, at[s], src_lane);
            const u32 l = w.seq_len[rr * 5 + s];
            if (l > RW_LONG) rw_warp_copy(text + d, w.seq_pool + w.seq_off[rr * 5 + s], l, lane);
        }
    }
}

// The resident compare result as the debug writers read it; names uploaded into rb[W_NAMES], ids as in avk_compare_records_bgzf
static int region_view_device(avk_ctx *ctx, const char *who, const char *const *contig_names, uint32_t n_contigs, const uint64_t *region_id,
                              const uint64_t *out_len, RegionView &w) {
    std::string &err = ctx->err;
    if (!ctx->have_batch || !ctx->have_result) {
        err = std::string(who) + (ctx->have_merge ? ": the resident result is a merge result, not a compare result" : ": no compare result is resident (run avk_compare_run_resident first)");
        return AVK_ERR_INVALID;
    }
    if ((!contig_names && n_contigs) || !out_len) { err = std::string(who) + ": bad arguments"; return AVK_ERR_INVALID; }
    if (!region_id && !ctx->ids_resident) { err = std::string(who) + ": the batch was uploaded, so its region ids must be given"; return AVK_ERR_INVALID; }
    const int rc = upload_names(ctx, who, contig_names, n_contigs, nullptr, 0, true, w.nt);
    if (rc != AVK_OK) return rc;
    DevBuf *rb = ctx->rb;
    const DevBatch db = dev_batch(ctx);
    w.contig = db.contig; w.start = db.start; w.end = db.end;
    w.status = (const int *)ctx->status.p;
    w.rows = (const u64 *)ctx->region_metrics.p;
    w.seq_off = (const u64 *)ctx->seq_off.p; w.seq_len = (const u32 *)ctx->seq_len.p; w.seq_pool = biased<const u8>(ctx->seq_pool, ctx->seq_base);
    w.metrics = nullptr; w.n_metrics = 0;
    if (region_id) {                                              // the caller's ids of the resident bin [lo, lo + n)
        UPLOAD(rb[W_RID], region_id + ctx->lo, 8 * ctx->n_regions);
        w.rid = (const u64 *)rb[W_RID].p;
    } else {
        w.rid = (const u64 *)ctx->region_id.p;
    }
    return AVK_OK;
}
// out == NULL: *out_len = the size bound of (header line + `body` bytes); else *text = rb[V_TEXT] with the header line copied in
// front, for the write pass to fill behind it
static int debug_finish(avk_ctx *ctx, const char *who, const char *header, u64 body, const uint8_t *out, uint64_t *out_len, u8 **text) {
    const u64 hl = header ? strlen(header) : 0, len = hl + body;
    *text = nullptr;
    if (bgzf_chunks(len) >= 0x7fffffffull) { ctx->err = std::string(who) + ": text too long for one call"; return AVK_ERR_INVALID; }
    if (!out) { *out_len = bgzf_bound(len); return AVK_OK; }
    ENSURE(ctx->rb[C_TEXT], len);
    *text = (u8 *)ctx->rb[C_TEXT].p;
    if (hl) CK(cudaMemcpyAsync(*text, header, hl, cudaMemcpyHostToDevice, ctx->stream));
    return AVK_OK;
}

extern "C" int avk_compare_region_summary_bgzf(avk_ctx *ctx, const char *const *contig_names, uint32_t n_contigs, const uint8_t *metrics, uint32_t n_metrics,
                                               const uint64_t *region_id, int header, int eof, uint8_t *out, uint64_t cap, uint64_t *out_len) {
    static const char *who = "avk_compare_region_summary_bgzf";
    if (!ctx) return AVK_ERR_INVALID;
    if (!metrics && n_metrics) { ctx->err = std::string(who) + ": bad arguments"; return AVK_ERR_INVALID; }
    for (uint32_t q = 0; q < n_metrics; ++q)
        if (metrics[q] > 4) { ctx->err = std::string(who) + ": metric code " + std::to_string(metrics[q]) + " (0 GT .. 4 RECORD_BP)"; return AVK_ERR_INVALID; }
    CK(cudaSetDevice(ctx->device));
    RegionView w;
    int rc = region_view_device(ctx, who, contig_names, n_contigs, region_id, out_len, w);
    if (rc != AVK_OK) return rc;
    if (!ctx->result_has_rows) { ctx->err = std::string(who) + ": per-region metric rows were not kept by the last pass (AVK_CMP_KEEP_REGION_ROWS)"; return AVK_ERR_INVALID; }
    DevBuf *rb = ctx->rb;
    const u64 n = ctx->n_regions;
    ENSURE(rb[W_MISC], 64 + n_metrics);
    unsigned long long *d_misc = (unsigned long long *)rb[W_MISC].p;     // [0] contig out of range, then the metric list
    if (n_metrics) CK(cudaMemcpyAsync((u8 *)rb[W_MISC].p + 64, metrics, n_metrics, cudaMemcpyHostToDevice, ctx->stream));
    w.metrics = (const u8 *)rb[W_MISC].p + 64; w.n_metrics = n_metrics;
    // count pass and the scan of the per-region line counts
    ENSURE(rb[W_CNT], 8 * (n + 1));
    u64 *line_off = (u64 *)rb[W_CNT].p;
    CK(cudaMemsetAsync(d_misc, 0, 8, ctx->stream));
    size_t need = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, need, line_off, line_off, n + 1, ctx->stream);
    ENSURE(ctx->scan_tmp, need);
    k_rs_count<<<(unsigned)((n + 1 + 255) / 256), 256, 0, ctx->stream>>>(w, n, n_contigs, line_off, d_misc);
    CK(cub::DeviceScan::ExclusiveSum(ctx->scan_tmp.p, need, line_off, line_off, n + 1, ctx->stream));
    unsigned long long h[2] = {0, 0};
    CK(cudaMemcpyAsync(&h[0], d_misc, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&h[1], line_off + n, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->launches += 2;
    CK(cudaGetLastError());
    if (h[0]) { ctx->err = std::string(who) + ": a region's contig is not below n_contigs"; return AVK_ERR_INVALID; }
    const u64 n_lines = h[1];
    // length pass and the scan of the line lengths
    ENSURE(rb[W_LEN], 8 * (n_lines + 1));
    ENSURE(rb[W_REG], 4 * n_lines);
    u64 *off = (u64 *)rb[W_LEN].p;
    u32 *reg = (u32 *)rb[W_REG].p;
    need = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, need, off, off, n_lines + 1, ctx->stream);
    ENSURE(ctx->scan_tmp, need);
    k_rs_len<<<(unsigned)((n_lines + 1 + 255) / 256), 256, 0, ctx->stream>>>(w, n, n_lines, line_off, reg, off);
    CK(cub::DeviceScan::ExclusiveSum(ctx->scan_tmp.p, need, off, off, n_lines + 1, ctx->stream));
    u64 body = 0;
    CK(cudaMemcpyAsync(&body, off + n_lines, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->launches += 2;
    CK(cudaGetLastError());
    const char *hdr = header ? avk_writers::REGION_SUMMARY_HEADER : nullptr;
    u8 *text = nullptr;
    rc = debug_finish(ctx, who, hdr, body, out, out_len, &text);
    if (rc != AVK_OK || !text) return rc;
    if (n_lines) {
        k_rs_write<<<(unsigned)((n_lines + 255) / 256), 256, 0, ctx->stream>>>(w, n_lines, reg, line_off, off, hdr ? strlen(hdr) : 0, text);
        ctx->launches += 1;
        CK(cudaGetLastError());
    }
    return bgzf_compress_device(ctx, (hdr ? strlen(hdr) : 0) + body, eof != 0, out, cap, out_len);
}

extern "C" int avk_compare_region_sequences_bgzf(avk_ctx *ctx, const char *const *contig_names, uint32_t n_contigs, const uint64_t *region_id,
                                                 int header, int eof, uint8_t *out, uint64_t cap, uint64_t *out_len) {
    static const char *who = "avk_compare_region_sequences_bgzf";
    if (!ctx) return AVK_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    RegionView w;
    int rc = region_view_device(ctx, who, contig_names, n_contigs, region_id, out_len, w);
    if (rc != AVK_OK) return rc;
    if (!ctx->result_has_seq) {
        ctx->err = std::string(who) + ": the last pass kept no sequence bundle (AVK_CMP_KEEP_SEQUENCES, or enable_sequences with the seq_* outputs)";
        return AVK_ERR_INVALID;
    }
    DevBuf *rb = ctx->rb;
    const u64 n = ctx->n_regions;
    ENSURE(rb[W_MISC], 64);
    unsigned long long *d_misc = (unsigned long long *)rb[W_MISC].p;     // [0] contig out of range
    ENSURE(rb[W_LEN], 8 * (n + 1));
    u64 *off = (u64 *)rb[W_LEN].p;
    CK(cudaMemsetAsync(d_misc, 0, 8, ctx->stream));
    size_t need = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, need, off, off, n + 1, ctx->stream);
    ENSURE(ctx->scan_tmp, need);
    k_rq_len<<<(unsigned)((n + 1 + 255) / 256), 256, 0, ctx->stream>>>(w, n, n_contigs, off, d_misc);
    CK(cub::DeviceScan::ExclusiveSum(ctx->scan_tmp.p, need, off, off, n + 1, ctx->stream));
    unsigned long long h[2] = {0, 0};
    CK(cudaMemcpyAsync(&h[0], d_misc, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&h[1], off + n, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->launches += 2;
    CK(cudaGetLastError());
    if (h[0]) { ctx->err = std::string(who) + ": a region's contig is not below n_contigs"; return AVK_ERR_INVALID; }
    const u64 body = h[1];
    const char *hdr = header ? avk_writers::REGION_SEQUENCES_HEADER : nullptr;
    u8 *text = nullptr;
    rc = debug_finish(ctx, who, hdr, body, out, out_len, &text);
    if (rc != AVK_OK || !text) return rc;
    if (body) {
        k_rq_write<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(w, n, off, hdr ? strlen(hdr) : 0, text);
        ctx->launches += 1;
        CK(cudaGetLastError());
    }
    return bgzf_compress_device(ctx, (hdr ? strlen(hdr) : 0) + body, eof != 0, out, cap, out_len);
}

// ---- outputs of the resident merge, formatted on the device (avk_writers.h::merge_records_text / merge_regions_text and the
// keys of merge_summary_count_batch) --------------------------------------------------------------------------------------
// passing.vcf.gz: count pass (one thread per region: records of the source input, length of the region's INFO text, checks)
// -> scans of the record counts and of the INFO lengths -> the INFO text of every passing region into rb[M_INFO], built once
// -> length pass (one thread per record) -> scan -> write pass, which copies the region's INFO into each of its lines ->
// bgzf_compress_device.  INFO strings and alleles longer than RW_LONG bytes are copied by the whole warp, as in k_rw_write.
// regions.bed / failed_regions.bed: one line per region, a length pass, a scan and a write pass.
enum { M_IOFF = V_VT, M_INFO = V_ZY, M_KEY = V_RAW, M_KEY_S = V_AOFF, M_UNIQ = V_L0, M_RUNS = V_L1 };    // beside the compare writer's slots
enum { MW_BAD_CONTIG = 1, MW_BAD_INDEX = 2 };
struct MergeRecView {
    const u64 *var_off, *rid;
    const u32 *contig, *start, *end, *pos, *aoff, *l0, *l1;
    const u8 *zyg, *vtype, *pool;
    const int *status;
    const u8 *cls, *n_idx, *idx;
    const u64 *name_off, *label_off;     // [n_contigs + 1] and [K + 1] offsets into the packed names / labels
    const char *names, *labels;
    u32 K;
};
// avk_writers.h::merge_simple and merge_source
__device__ __forceinline__ const char *mw_simple(u8 c, u32 &n) {
    switch (c) {
        case AVK_MERGE_NO_CONFLICT: n = 11; return "no_conflict";
        case AVK_MERGE_MAJORITY_AGREE: n = 8; return "majority";
        case AVK_MERGE_CONFLICT_SELECTION: n = 15; return "conflict_select";
        case AVK_MERGE_BASEPAIR_IDENTICAL: n = 9; return "identical";
        default: n = 9; return "different";
    }
}
__device__ __forceinline__ int mw_source(const MergeRecView &w, u64 r) {
    const u8 c = w.cls[r];
    if (c == AVK_MERGE_BASEPAIR_IDENTICAL) return 0;
    if (c == AVK_MERGE_DIFFERENT || w.n_idx[r] == 0) return -1;
    return w.idx[r * w.K];
}
// the checks of avk_lib.cu::merge_view on one region: its contig has a name, its index list lies inside the inputs
__device__ __forceinline__ u32 mw_check(const MergeRecView &w, u64 r, u32 n_contigs) {
    u32 bad = w.contig[r] >= n_contigs ? (u32)MW_BAD_CONTIG : 0u;
    const u32 ni = w.n_idx[r];
    if (ni > w.K) bad |= MW_BAD_INDEX;
    else for (u32 k = 0; k < ni; ++k) if (w.idx[r * w.K + k] >= w.K) bad |= MW_BAD_INDEX;
    return bad;
}
__device__ __forceinline__ u32 mw_label_len(const MergeRecView &w, u32 k) { return (u32)(w.label_off[k + 1] - w.label_off[k]); }

__global__ void __launch_bounds__(256) k_mw_count(MergeRecView w, u64 n, u32 n_contigs, u64 *cnt, u64 *ilen, unsigned long long *bad) {
    const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r > n) return;
    if (r == n) { cnt[n] = 0; ilen[n] = 0; return; }
    const u32 b = mw_check(w, r, n_contigs);
    if (b) atomicOr(bad, (unsigned long long)b);
    u64 c = 0, il = 0;
    const int src = b || w.status[r] != 0 ? -1 : mw_source(w, r);
    if (src >= 0) c = w.var_off[r * w.K + src + 1] - w.var_off[r * w.K + src];
    if (c) {                                                      // SOURCES=<labels>;MR=<reason>
        u32 ns;
        mw_simple(w.cls[r], ns);
        il = 8 + 4 + ns;
        if (w.cls[r] == AVK_MERGE_BASEPAIR_IDENTICAL) for (u32 k = 0; k < w.K; ++k) il += (k ? 1 : 0) + mw_label_len(w, k);
        else for (u32 k = 0; k < w.n_idx[r]; ++k) il += (k ? 1 : 0) + mw_label_len(w, w.idx[r * w.K + k]);
    }
    cnt[r] = c;
    ilen[r] = il;
}
// the INFO text of each region with records, at info + ioff[r] (ioff = exclusive scan of the INFO lengths)
__global__ void __launch_bounds__(256) k_mw_info(MergeRecView w, u64 n, const u64 *ioff, u8 *info) {
    const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n || ioff[r + 1] == ioff[r]) return;
    u8 *o = info + ioff[r];
    o = rw_put_str(o, "SOURCES=", 8);
    const bool all = w.cls[r] == AVK_MERGE_BASEPAIR_IDENTICAL;
    const u32 m = all ? w.K : w.n_idx[r];
    for (u32 k = 0; k < m; ++k) {
        if (k) *o++ = ',';
        const u32 in = all ? k : w.idx[r * w.K + k];
        o = rw_put_str(o, w.labels + w.label_off[in], mw_label_len(w, in));
    }
    o = rw_put_str(o, ";MR=", 4);
    u32 ns;
    const char *s = mw_simple(w.cls[r], ns);
    rw_put_str(o, s, ns);
}
__global__ void __launch_bounds__(256) k_mw_len(MergeRecView w, u64 n, u64 n_rec, const u64 *rec_off, const u64 *ioff, u32 *reg, u64 *len) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n_rec) return;
    if (i == n_rec) { len[n_rec] = 0; return; }
    const u64 r = rw_region(rec_off, n, i);
    const u64 v = w.var_off[r * w.K + mw_source(w, r)] + (i - rec_off[r]);
    const u32 c = w.contig[r];
    const int32_t ri = (int32_t)(u32)w.rid[r];
    u32 ng;
    rw_gt(w.zyg[v], ng);
    reg[i] = (u32)r;
    len[i] = (w.name_off[c + 1] - w.name_off[c]) + 1 + rw_digits((u64)w.pos[v] + 1) + 3 + w.l0[v] + 1 + w.l1[v] + 5 + (ioff[r + 1] - ioff[r]) + 7 +
             ng + 1 + (ri < 0 ? 1 : 0) + rw_digits(ri < 0 ? (u64)(-(int64_t)ri) : (u64)ri) + 1;
}
// off = exclusive scan of the line lengths; line i starts at text + base + off[i]
__global__ void __launch_bounds__(256) k_mw_write(MergeRecView w, u64 n_rec, const u32 *reg, const u64 *rec_off, const u64 *ioff, const u8 *info,
                                                  const u64 *off, u64 base, u8 *text) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const bool act = i < n_rec;
    u64 a0_at = 0, a1_at = 0, in_at = 0, src = 0, isrc = 0;
    u32 l0 = 0, l1 = 0, li = 0;
    if (act) {
        const u64 r = reg[i];
        const u64 v = w.var_off[r * w.K + mw_source(w, r)] + (i - rec_off[r]);
        const u32 c = w.contig[r];
        u8 *o = text + base + off[i];
        o = rw_put_str(o, w.names + w.name_off[c], (u32)(w.name_off[c + 1] - w.name_off[c]));
        *o++ = '\t';
        const u64 p = (u64)w.pos[v] + 1;
        o = rw_put_u64(o, p, rw_digits(p));
        *o++ = '\t'; *o++ = '.'; *o++ = '\t';
        l0 = w.l0[v]; l1 = w.l1[v];
        src = (u64)(uintptr_t)(w.pool + w.aoff[v]);
        a0_at = (u64)(o - text);
        if (l0 <= RW_LONG) rw_put_str(o, (const char *)src, l0);
        o += l0;
        *o++ = '\t';
        a1_at = (u64)(o - text);
        if (l1 <= RW_LONG) rw_put_str(o, (const char *)src + l0, l1);
        o += l1;
        o = rw_put_str(o, "\t.\t.\t", 5);
        li = (u32)(ioff[r + 1] - ioff[r]);
        isrc = (u64)(uintptr_t)(info + ioff[r]);
        in_at = (u64)(o - text);
        if (li <= RW_LONG) rw_put_str(o, (const char *)isrc, li);
        o += li;
        o = rw_put_str(o, "\tGT:RI\t", 7);
        u32 ng;
        const char *gt = rw_gt(w.zyg[v], ng);
        o = rw_put_str(o, gt, ng); *o++ = ':';
        const int32_t ri = (int32_t)(u32)w.rid[r];                   // `region_id as i32`
        if (ri < 0) *o++ = '-';
        const u64 ra = ri < 0 ? (u64)(-(int64_t)ri) : (u64)ri;
        o = rw_put_u64(o, ra, rw_digits(ra));
        *o = '\n';
    }
    const int lane = lane_id();
    for (u32 m = __ballot_sync(AVK_FULL, act && (l0 > RW_LONG || l1 > RW_LONG || li > RW_LONG)); m; m &= m - 1) {
        const int s = __ffs(m) - 1;
        const u8 *sp = (const u8 *)(uintptr_t)__shfl_sync(AVK_FULL, src, s), *ip = (const u8 *)(uintptr_t)__shfl_sync(AVK_FULL, isrc, s);
        const u32 n0 = __shfl_sync(AVK_FULL, l0, s), n1 = __shfl_sync(AVK_FULL, l1, s), ni = __shfl_sync(AVK_FULL, li, s);
        const u64 d0 = __shfl_sync(AVK_FULL, a0_at, s), d1 = __shfl_sync(AVK_FULL, a1_at, s), di = __shfl_sync(AVK_FULL, in_at, s);
        if (n0 > RW_LONG) rw_warp_copy(text + d0, sp, n0, lane);
        if (n1 > RW_LONG) rw_warp_copy(text + d1, sp + n0, n1, lane);
        if (ni > RW_LONG) rw_warp_copy(text + di, ip, ni, lane);
    }
}
// BED4 line of a solved region whose pass / fail state is `passing`: chrom, start, end, {reason}_{region id as u64}
__global__ void __launch_bounds__(256) k_mr_len(MergeRecView w, u64 n, u32 n_contigs, int passing, u64 *len, unsigned long long *bad) {
    const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r > n) return;
    if (r == n) { len[n] = 0; return; }
    const u32 b = mw_check(w, r, n_contigs);
    if (b) atomicOr(bad, (unsigned long long)b);
    u64 l = 0;
    if (!b && w.status[r] == 0 && (mw_source(w, r) >= 0) == (passing != 0)) {
        const u32 c = w.contig[r];
        u32 ns;
        mw_simple(w.cls[r], ns);
        l = (w.name_off[c + 1] - w.name_off[c]) + 1 + rw_digits(w.start[r]) + 1 + rw_digits(w.end[r]) + 1 + ns + 1 + rw_digits(w.rid[r]) + 1;
    }
    len[r] = l;
}
__global__ void __launch_bounds__(256) k_mr_write(MergeRecView w, u64 n, const u64 *off, u8 *text) {
    const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n || off[r + 1] == off[r]) return;
    const u32 c = w.contig[r];
    u8 *o = text + off[r];
    o = rw_put_str(o, w.names + w.name_off[c], (u32)(w.name_off[c + 1] - w.name_off[c]));
    *o++ = '\t';
    o = rw_put_u64(o, w.start[r], rw_digits(w.start[r])); *o++ = '\t';
    o = rw_put_u64(o, w.end[r], rw_digits(w.end[r])); *o++ = '\t';
    u32 ns;
    const char *s = mw_simple(w.cls[r], ns);
    o = rw_put_str(o, s, ns); *o++ = '_';
    o = rw_put_u64(o, w.rid[r], rw_digits(w.rid[r]));
    *o = '\n';
}
// the summary key of every variant of the bin (avk_writers.h::merge_summary_count_batch): class << 56 | variant type << 48 |
// input << 40 | index-list mask; ~0 for a variant of an unsolved region (it sorts last and is dropped)
__global__ void __launch_bounds__(256) k_ms_keys(MergeRecView w, u64 n, u64 v_base, u64 nv, u64 *key, unsigned long long *bad) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nv) return;
    const u64 v = v_base + i, nl = n * w.K;
    u64 lo = 0, hi = nl;                                          // list j = r * K + k holds v: the last j with var_off[j] <= v
    while (hi - lo > 1) { const u64 m = (lo + hi) >> 1; if (w.var_off[m] <= v) lo = m; else hi = m; }
    const u64 r = lo / w.K, k = lo % w.K;
    if (w.status[r] != 0) { key[i] = ~0ull; return; }
    if (mw_check(w, r, 0xffffffffu)) atomicOr(bad, (unsigned long long)MW_BAD_INDEX);
    const u8 c = w.cls[r];
    const u8 *ix = w.idx + r * w.K;
    u32 mask = 0;
    if (c == AVK_MERGE_NO_CONFLICT || c == AVK_MERGE_MAJORITY_AGREE) { for (u32 j = 0; j < w.n_idx[r] && j < w.K; ++j) mask |= 1u << (ix[j] & 31); }
    else if (c == AVK_MERGE_CONFLICT_SELECTION) mask = 1u << (ix[0] & 31);
    key[i] = (u64)c << 56 | (u64)w.vtype[v] << 48 | k << 40 | mask;
}

// the resident merge result and batch as the writers read them; names and labels (when given) uploaded into rb[W_NAMES]
static int merge_view_device(avk_ctx *ctx, const char *who, const char *const *contig_names, uint32_t n_contigs, const char *const *labels,
                             const uint64_t *region_id, bool need_ids, MergeRecView &w) {
    std::string &err = ctx->err;
    if (!ctx->have_batch || !ctx->have_merge) { err = std::string(who) + ": no merge result is resident (run avk_merge_run_resident first)"; return AVK_ERR_INVALID; }
    if (!contig_names && n_contigs) { err = std::string(who) + ": bad arguments"; return AVK_ERR_INVALID; }
    if (need_ids && !region_id && !ctx->ids_resident) { err = std::string(who) + ": the batch was uploaded, so its region ids must be given"; return AVK_ERR_INVALID; }
    const u64 n = ctx->n_regions, K = ctx->n_inputs;
    NameTable nt;
    const int rc = upload_names(ctx, who, contig_names, n_contigs, labels, K, false, nt);
    if (rc != AVK_OK) return rc;
    DevBuf *rb = ctx->rb;
    const DevBatch db = dev_batch(ctx);
    w.var_off = db.var_off; w.contig = db.contig; w.start = db.start; w.end = db.end; w.pos = db.pos; w.aoff = db.aoff; w.l0 = db.l0; w.l1 = db.l1;
    w.zyg = db.zyg; w.vtype = db.vtype; w.pool = db.pool;
    w.status = (const int *)ctx->status.p; w.cls = (const u8 *)ctx->m_cls.p; w.n_idx = (const u8 *)ctx->m_nidx.p; w.idx = (const u8 *)ctx->m_idx.p;
    w.name_off = nt.name_off; w.label_off = nt.label_off; w.names = nt.names; w.labels = nt.labels;
    w.K = (u32)K;
    w.rid = nullptr;
    if (need_ids) {
        if (region_id) {                                          // the caller's ids of the resident bin [lo, lo + n)
            UPLOAD(rb[W_RID], region_id + ctx->lo, 8 * n);
            w.rid = (const u64 *)rb[W_RID].p;
        } else {
            w.rid = (const u64 *)ctx->region_id.p;
        }
    }
    return AVK_OK;
}
static int merge_bad(avk_ctx *ctx, const char *who, unsigned long long bad) {
    if (bad & MW_BAD_CONTIG) { ctx->err = std::string(who) + ": a region's contig is not below n_contigs"; return AVK_ERR_INVALID; }
    if (bad & MW_BAD_INDEX) { ctx->err = std::string(who) + ": a merge result's index list lies outside the inputs"; return AVK_ERR_INVALID; }
    return AVK_OK;
}

extern "C" int avk_merge_records_bgzf(avk_ctx *ctx, const char *const *contig_names, uint32_t n_contigs, const char *const *input_labels,
                                      const uint64_t *region_id, const uint8_t *header, uint64_t header_len, int eof,
                                      uint8_t *out, uint64_t cap, uint64_t *out_len) {
    static const char *who = "avk_merge_records_bgzf";
    if (!ctx) return AVK_ERR_INVALID;
    if (!input_labels || (!header && header_len) || !out_len) { ctx->err = std::string(who) + ": bad arguments"; return AVK_ERR_INVALID; }
    CK(cudaSetDevice(ctx->device));
    MergeRecView w;
    int rc = merge_view_device(ctx, who, contig_names, n_contigs, input_labels, region_id, true, w);
    if (rc != AVK_OK) return rc;
    DevBuf *rb = ctx->rb;
    const u64 n = ctx->n_regions;
    // count pass and the scans of the per-region record counts and INFO lengths
    ENSURE(rb[W_MISC], 64);
    unsigned long long *d_misc = (unsigned long long *)rb[W_MISC].p;     // [0] MW_BAD_* flags
    ENSURE(rb[W_CNT], 8 * (n + 1)); ENSURE(rb[M_IOFF], 8 * (n + 1));
    u64 *rec_off = (u64 *)rb[W_CNT].p, *ioff = (u64 *)rb[M_IOFF].p;
    CK(cudaMemsetAsync(d_misc, 0, 8, ctx->stream));
    size_t need = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, need, rec_off, rec_off, n + 1, ctx->stream);
    ENSURE(ctx->scan_tmp, need);
    k_mw_count<<<(unsigned)((n + 1 + 255) / 256), 256, 0, ctx->stream>>>(w, n, n_contigs, rec_off, ioff, d_misc);
    CK(cub::DeviceScan::ExclusiveSum(ctx->scan_tmp.p, need, rec_off, rec_off, n + 1, ctx->stream));
    CK(cub::DeviceScan::ExclusiveSum(ctx->scan_tmp.p, need, ioff, ioff, n + 1, ctx->stream));
    unsigned long long h[3] = {0, 0, 0};
    CK(cudaMemcpyAsync(&h[0], d_misc, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&h[1], rec_off + n, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&h[2], ioff + n, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->launches += 3;
    CK(cudaGetLastError());
    if ((rc = merge_bad(ctx, who, h[0])) != AVK_OK) return rc;
    const u64 n_rec = h[1], info_bytes = h[2];
    // the INFO texts, then the length pass and the scan of the line lengths (64-bit counts and offsets throughout)
    ENSURE(rb[M_INFO], info_bytes);
    u8 *info = (u8 *)rb[M_INFO].p;
    if (info_bytes) {
        k_mw_info<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(w, n, ioff, info);
        ctx->launches += 1;
    }
    ENSURE(rb[W_LEN], 8 * (n_rec + 1));
    ENSURE(rb[W_REG], 4 * n_rec);
    u64 *off = (u64 *)rb[W_LEN].p;
    u32 *reg = (u32 *)rb[W_REG].p;
    need = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, need, off, off, n_rec + 1, ctx->stream);
    ENSURE(ctx->scan_tmp, need);
    k_mw_len<<<(unsigned)((n_rec + 1 + 255) / 256), 256, 0, ctx->stream>>>(w, n, n_rec, rec_off, ioff, reg, off);
    CK(cub::DeviceScan::ExclusiveSum(ctx->scan_tmp.p, need, off, off, n_rec + 1, ctx->stream));
    u64 body = 0;
    CK(cudaMemcpyAsync(&body, off + n_rec, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->launches += 2;
    CK(cudaGetLastError());
    const u64 len = header_len + body;
    if (bgzf_chunks(len) >= 0x7fffffffull) { ctx->err = std::string(who) + ": text too long for one call"; return AVK_ERR_INVALID; }
    if (!out) { *out_len = bgzf_bound(len); return AVK_OK; }
    // header + lines into rb[V_TEXT], then the compressor
    ENSURE(rb[C_TEXT], len);
    u8 *text = (u8 *)rb[C_TEXT].p;
    if (header_len) CK(cudaMemcpyAsync(text, header, header_len, cudaMemcpyHostToDevice, ctx->stream));
    if (n_rec) {
        k_mw_write<<<(unsigned)((n_rec + 255) / 256), 256, 0, ctx->stream>>>(w, n_rec, reg, rec_off, ioff, info, off, header_len, text);
        ctx->launches += 1;
        CK(cudaGetLastError());
    }
    return bgzf_compress_device(ctx, len, eof != 0, out, cap, out_len);
}

extern "C" int avk_merge_regions_bgzf(avk_ctx *ctx, const char *const *contig_names, uint32_t n_contigs, int passing,
                                      const uint64_t *region_id, int eof, uint8_t *out, uint64_t cap, uint64_t *out_len) {
    static const char *who = "avk_merge_regions_bgzf";
    if (!ctx) return AVK_ERR_INVALID;
    if (!out_len) { ctx->err = std::string(who) + ": bad arguments"; return AVK_ERR_INVALID; }
    CK(cudaSetDevice(ctx->device));
    MergeRecView w;
    int rc = merge_view_device(ctx, who, contig_names, n_contigs, nullptr, region_id, true, w);
    if (rc != AVK_OK) return rc;
    DevBuf *rb = ctx->rb;
    const u64 n = ctx->n_regions;
    ENSURE(rb[W_MISC], 64);
    unsigned long long *d_misc = (unsigned long long *)rb[W_MISC].p;
    ENSURE(rb[W_LEN], 8 * (n + 1));
    u64 *off = (u64 *)rb[W_LEN].p;
    CK(cudaMemsetAsync(d_misc, 0, 8, ctx->stream));
    size_t need = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, need, off, off, n + 1, ctx->stream);
    ENSURE(ctx->scan_tmp, need);
    k_mr_len<<<(unsigned)((n + 1 + 255) / 256), 256, 0, ctx->stream>>>(w, n, n_contigs, passing, off, d_misc);
    CK(cub::DeviceScan::ExclusiveSum(ctx->scan_tmp.p, need, off, off, n + 1, ctx->stream));
    unsigned long long h[2] = {0, 0};
    CK(cudaMemcpyAsync(&h[0], d_misc, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&h[1], off + n, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->launches += 2;
    CK(cudaGetLastError());
    if ((rc = merge_bad(ctx, who, h[0])) != AVK_OK) return rc;
    const u64 len = h[1];
    if (bgzf_chunks(len) >= 0x7fffffffull) { ctx->err = std::string(who) + ": text too long for one call"; return AVK_ERR_INVALID; }
    if (!out) { *out_len = bgzf_bound(len); return AVK_OK; }
    ENSURE(rb[C_TEXT], len);
    if (len) {
        k_mr_write<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(w, n, off, (u8 *)rb[C_TEXT].p);
        ctx->launches += 1;
        CK(cudaGetLastError());
    }
    return bgzf_compress_device(ctx, len, eof != 0, out, cap, out_len);
}

// The summary's keys of the resident bin counted on the device: one key per variant (k_ms_keys), radix sort, run-length
// encoding; only the distinct keys and their counts are copied to the host.
extern "C" int avk_merge_summary_counts(avk_ctx *ctx, avk_merge_summary_row *rows, uint64_t cap, uint64_t *n_rows) {
    static const char *who = "avk_merge_summary_counts";
    if (!ctx) return AVK_ERR_INVALID;
    if (!n_rows) { ctx->err = std::string(who) + ": bad arguments"; return AVK_ERR_INVALID; }
    CK(cudaSetDevice(ctx->device));
    MergeRecView w;
    int rc = merge_view_device(ctx, who, nullptr, 0, nullptr, nullptr, false, w);
    if (rc != AVK_OK) return rc;
    DevBuf *rb = ctx->rb;
    const u64 n = ctx->n_regions, nv = ctx->n_variants;
    *n_rows = 0;
    if (nv == 0) return AVK_OK;
    ENSURE(rb[W_MISC], 64);
    unsigned long long *d_misc = (unsigned long long *)rb[W_MISC].p;     // [0] MW_BAD_* flags, [1] number of runs
    ENSURE(rb[M_KEY], 8 * nv); ENSURE(rb[M_KEY_S], 8 * nv); ENSURE(rb[M_UNIQ], 8 * nv); ENSURE(rb[M_RUNS], 4 * nv);
    u64 *key = (u64 *)rb[M_KEY].p, *key_s = (u64 *)rb[M_KEY_S].p, *uniq = (u64 *)rb[M_UNIQ].p;
    u32 *runs = (u32 *)rb[M_RUNS].p;
    u32 *n_runs = (u32 *)(d_misc + 1);
    size_t tmp = 0, need = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, need, key, key_s, (int)nv, 0, 64, ctx->stream); tmp = std::max(tmp, need);
    cub::DeviceRunLengthEncode::Encode(nullptr, need, key_s, uniq, runs, n_runs, (int)nv, ctx->stream); tmp = std::max(tmp, need);
    ENSURE(ctx->scan_tmp, tmp);
    CK(cudaMemsetAsync(d_misc, 0, 16, ctx->stream));
    k_ms_keys<<<(unsigned)((nv + 255) / 256), 256, 0, ctx->stream>>>(w, n, ctx->v_base, nv, key, d_misc);
    need = tmp; CK(cub::DeviceRadixSort::SortKeys(ctx->scan_tmp.p, need, key, key_s, (int)nv, 0, 64, ctx->stream));
    need = tmp; CK(cub::DeviceRunLengthEncode::Encode(ctx->scan_tmp.p, need, key_s, uniq, runs, n_runs, (int)nv, ctx->stream));
    unsigned long long h[2] = {0, 0};
    CK(cudaMemcpyAsync(h, d_misc, 16, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->launches += 3;
    CK(cudaGetLastError());
    if ((rc = merge_bad(ctx, who, h[0])) != AVK_OK) return rc;
    u64 m = (u32)h[1];
    std::vector<u64> hk(m);
    std::vector<u32> hc(m);
    if (m) {
        CK(cudaMemcpyAsync(hk.data(), uniq, 8 * m, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(hc.data(), runs, 4 * m, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    if (m && hk[m - 1] == ~0ull) --m;                             // the variants of unsolved regions
    *n_rows = m;
    if (!rows) return AVK_OK;
    if (cap < m) { ctx->err = std::string(who) + ": row capacity too small"; return AVK_ERR_OOM; }
    for (u64 i = 0; i < m; ++i) {
        avk_merge_summary_row &o = rows[i];
        const u64 k = hk[i];
        o.indices = (u32)k; o.classification = (u8)(k >> 56); o.variant_type = (u8)(k >> 48); o.input = (u8)(k >> 40); o.pad = 0;
        const bool pass = o.classification == AVK_MERGE_BASEPAIR_IDENTICAL || (o.indices >> o.input & 1u);
        o.pass_variants = pass ? hc[i] : 0; o.fail_variants = pass ? 0 : hc[i];
    }
    return AVK_OK;
}

extern "C" int avk_vcf_parse_bgzf(avk_ctx *ctx, const uint8_t *gz, uint64_t gz_len, int verify_crc, const char *const *contig_names, uint32_t n_contigs,
                                  uint32_t sample_index, int enable_trimming, avk_vcf_out *out, uint64_t *error_line, int32_t *error_code) {
    if (!ctx) return AVK_ERR_INVALID;
    if (!gz && gz_len) { ctx->err = "avk_vcf_parse_bgzf: null input"; return AVK_ERR_INVALID; }
    uint64_t total = 0;
    const int rc = bgzf_inflate_device(ctx, gz, gz_len, verify_crc, &total, nullptr);
    if (rc != AVK_OK) return rc;
    return vcf_parse_impl(ctx, nullptr, total, contig_names, n_contigs, sample_index, enable_trimming, out, error_line, error_code);   // the text never leaves the device
}

// diagnostics: per-cluster phase cycles of the LAST k_search_spec launches (AVK_SPEC_PROFILE=1); out = [n][8] u64
extern "C" int avk_spec_profile(avk_ctx *ctx, unsigned long long *out, uint32_t n) {
    if (!ctx || !out || !ctx->spec_prof.p) return AVK_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaMemcpy(out, ctx->spec_prof.p, (size_t)std::min<uint32_t>(n, 65536) * 64, cudaMemcpyDeviceToHost));
    return AVK_OK;
}
