// avk_solver.cuh -- per-cluster solvers, one warp per cluster.
//
//   RegionSolver::optimize()       <- optimize_sequences      src/query_optimizer.rs:166-365
//   RegionSolver::exact_gt()       <- optimize_gt_alleles     src/exact_gt_optimizer.rs:108-357
//   RegionSolver::solve_compare()  <- solve_compare_region    src/waffle_solver.rs:122-284
//                                     compare_expected_observed :296-327, add_basepair_stats :335-449,
//                                     add_record_basepair_stats :455-522, generate_allele_sequence :726-778
//   RegionSolver::solve_merge()    <- solve_merge_region      src/merge_solver.rs:110-223
//
// The sequential best-first searches of the reference are replayed exactly: the same (unique)
// priority keys, the same node-id assignment, the same quotas and prunes, so the same equal-cost
// solution is reported.  What differs is the machine mapping: a warp keeps the whole problem of one
// cluster in a private workspace ("arena": shared memory in the common tiers, global memory for the
// rare oversized cluster):
//   * the reference window, staged once with a TMA bulk copy,
//   * the cluster's variants in merged processing order and their allele bytes,
//   * the search nodes (materialised haplotype prefixes + wavefronts) and the key array of the queue,
//   * the metric rows being accumulated.
// Pops are a warp-wide scan + REDUX min over the unsorted key array, clones are warp-wide copies,
// scoring is the warp-cooperative DWFA of avk_device.cuh over virtual sequences.  The solver object
// lives in shared memory (one per warp); all arena accesses use Mem<SMEM> addresses.
#pragma once
#include "avk_device.cuh"
#include "avk_spec_search.cuh"
#include "avk_layout.h"

namespace avk {

struct DevBatch {
    u64 n_regions;
    u32 n_inputs;
    const u64 *region_id;
    const u32 *contig, *start, *end;
    const u64 *var_off;
    const u32 *pos;
    const u8 *vtype, *zyg;
    const u32 *raw, *aoff, *l0, *l1;
    const u8 *pool;
    const u8 *const *contig_ptr;
    const u64 *contig_len;
    u32 n_contigs;
    const u32 *alt_ed;   // per variant, filled by k_alt_ed
    // compare only: per-cluster "digest" written by k_prep_fill (header + variant records in merged order + alleles)
    const u8 *digest;
    const u64 *digest_off;   // [n_regions + 1]
};

struct DevCompareOut {
    int *status;
    u32 *ed1, *ed2;
    u64 *region_metrics;   // [n][13][22], or NULL when the caller wants no per-region rows
    unsigned long long *tot_slots;   // [TOT_SLOTS][TOT_STRIDE]
    uint16_t *type_mask;
    u8 *vexp, *vobs, *vcls;
    const u64 *seq_off;    // may be NULL
    u32 *seq_len;
    u8 *seq_pool;
    const struct DevStrata *strata;   // per-stratum sums (device memory), or NULL when no strata are requested
};

// Per-stratum sums of a pass: partial tables [STRAT_SLOTS][n_strata][TOT_COLS].  Region r belongs to the strata of its
// containment mask st_mask[r] (device lookup) when st_mask is set, else to strat_idx[strat_off[r] .. strat_off[r + 1]) (the
// caller's list; strat_idx is biased so that the caller's offsets index it).  Kept behind one pointer in device memory so that
// the solver kernels' parameter block (copied to the stack where its address is taken) does not grow.
struct DevStrata {
    unsigned long long *slots;
    const u64 *st_mask;
    const u64 *strat_off;
    const u32 *strat_idx;
    u32 n_strata;

    // adds v to column `col` of every stratum region r belongs to, in this CTA's partial table (out of line: the solver
    // kernels of a pass without strata keep their own code)
    __device__ __noinline__ void add(u64 r, int col, unsigned long long v) const {
        unsigned long long *t = slots + (size_t)(blockIdx.x & (STRAT_SLOTS - 1)) * n_strata * TOT_COLS + col;
        if (st_mask) for (u64 m = st_mask[r]; m; m &= m - 1) atomicAdd(t + (size_t)(__ffsll((long long)m) - 1) * TOT_COLS, v);
        else for (u64 s = strat_off[r], e = strat_off[r + 1]; s < e; ++s) atomicAdd(t + (size_t)strat_idx[s] * TOT_COLS, v);
    }
};

struct DevMergeOut {
    int *status;
    u8 *cls, *n_idx, *idx;
};

enum { SOLVE_OK = 0, SOLVE_WORKSPACE = -1 };   // internal; positive values are AVK_ST_*

__device__ __forceinline__ int align_up(int x, int a) { return (x + a - 1) / a * a; }

// The solver object is shared by the 32 lanes of its warp.  Convention (checked with compute-sanitizer racecheck): every
// lane may read a field, lane 0 alone writes it, with a __syncwarp() on either side of the write.
#define SOLVER_WRITE(...) do { __syncwarp(); if (lane_id() == 0) { __VA_ARGS__; } __syncwarp(); } while (0)

// optimize node: ints {id, depth, hap0[9], hap1[9]}; hap = {t_ref_pos, q_ref_pos, t_mlen, q_mlen, t_mref, q_mref, t_skip, q_skip, ed}
enum { ON_ID = 0, ON_DEPTH = 4, ON_HAP = 8, ON_HAPSZ = 36, ON_HDR = 80 };
enum { H_TRP = 0, H_QRP = 4, H_TML = 8, H_QML = 12, H_TMR = 16, H_QMR = 20, H_TSK = 24, H_QSK = 28, H_ED = 32 };
// exact node: ints {id, errors, depth, t_ref_pos, q_ref_pos, t_mlen, q_mlen, t_mref, q_mref, d}
enum { XN_ID = 0, XN_ERR = 4, XN_DEPTH = 8, XN_TRP = 12, XN_QRP = 16, XN_TML = 20, XN_QML = 24, XN_TMR = 28, XN_QMR = 32, XN_D = 36, XN_HDR = 48 };
// sequence descriptors written by build_hap_seq: {mlen, cur, failed, n_alt}
enum { SD_MLEN = 0, SD_CUR = 4, SD_FAILED = 8, SD_NALT = 12, SD_CLOSED = 16, SD_MAT = 20, SD_ARGS = 24, SD_SIZE = 32 };
// SD_CLOSED: ED(reference window, this haplotype) when it is known without aligning, else -1; SD_MAT: bytes materialised;
// SD_ARGS: (side, hap, result, type filter) the buffer was described from, for materialising it later


// Job board of a warp team (k_compare_team): the master warp runs the solver; the independent pieces of one queue pop --
// the two haplotypes of each child node (optimize_sequences), the two children (optimize_gt_alleles) -- are executed by
// up to four warps at once, a named barrier on either side of a round.
struct TeamBoard {
    int kind;        // 0: opt_extend_hap(nb, h, rec, alt, sync, finalize); 1: ex_extend(nb, oi, alt, err, finalize)
    int count, exit_, finalize, sync, oi;
    int bar;         // named barrier of this team (128 threads)
    unsigned rec;
    unsigned nb[4];
    int h[4], alt[4], err[4], rc[4];
};

template <bool SMEM>
struct RegionSolver {
    typedef Mem<SMEM> M;
    typedef typename M::addr addr;
    typedef VSeq<SMEM> VS;

    // ---- problem (warp-uniform) ----
    const DevBatch *bp;
    addr arena;           // this warp's workspace (shared-memory offset or global address)
    u32 arena_bytes;
    TeamBoard *team;      // set: this warp is the master of a warp team (shared-memory tiers only)
    int wide_b0;          // global tiers: clusters whose edit-distance bound reaches this go on to the cooperative tier (0 = keep)
    addr ref_base;        // byte of absolute contig position p is at ref_base + p (staged window or global contig)
    addr alle_base;       // allele bytes (staged copy or the global pool)
    int start, end;       // region window
    int nv[2];
    int N;
    int mbf;
    u32 tma_phase;        // mbarrier parity of the next window load
    int tma_pending;      // a window load has been issued and not yet waited for
    // ---- arena layout ----
    addr vinfo;           // [N] VI_* records
    addr bucket;          // [N+1] int
    addr res_alle;        // [res_cap][Npad] bit0 hap1 ALT, bit1 hap2 ALT (by order index)
    addr res_num;         // [res_cap][6] int: ed1 ed2 tvs1 tvs2 qvs1 qvs2
    addr hap_alle;        // [Npad] input alleles of exact_gt by order index
    addr cur_obs;         // [2][Npad]
    addr best_obs;        // [2][Npad]
    addr mrows;           // [1 + n_slots][22] u64 metric rows: joint, then one per distinct variant type
    addr slot_cnt;        // [n_slots][2] u32 number of truth / query variants of that type
    addr slot_tot;        // [n_slots][2] u64 zygosity-weighted raw allele space of that type (RECORD_BP)
    addr sdesc;           // [3] SD_* sequence descriptors (T, Q, F)
    addr dyn;             // start of the re-partitionable part
    u32 dyn_bytes;
    int Npad, seq_cap, wf_cap;
    int n_res, res_cap, n_slots;
    int pre_scored;       // the results come from the speculative dense search WITH their exact-GT scoring: result 0 is the solution
    u32 pre_keep[2];      //   and these are its exact-GT alleles per haplotype (bit = order entry keeps its ALT)
    int region_off;       // first arena byte after the header (+ staged window)
    int ed_overflow;
    u8 slot_type[AVK_N_VARIANT_TYPES];
    // queue + node slots (partitioned per phase)
    addr qkeys, qslot, freel, nodes;
    int stride, max_slots, qn, nfree, qcap;
    // node spill area in global memory (shared-memory tiers; 0 bytes = none)
    u8 *spill_base;
    u32 spill_bytes;
    int spill_cap, spill_used, spill_nfree;

    // ------------------------------------------------------------------ helpers
    __device__ __forceinline__ addr vi(int oi) const { return vinfo + (u32)(VI_SIZE * oi); }
    __device__ __forceinline__ int sync_pos(int oi) const {   // query_optimizer.rs:258-265
        return (oi == N - 1) ? end : (int)LD32(vi(oi + 1) + VI_POS);
    }
    __device__ __forceinline__ addr wk() const { return arena; }   // work counters live in the arena header

    // Start of a region: in shared-memory tiers the reference window is staged into the arena with a TMA
    // bulk copy (cp.async.bulk, 16-byte aligned superset of [start, end)), and ref_base is set so that
    // ref_base + pos still addresses absolute contig positions.
    __device__ __noinline__ bool begin_region(const u8 *contig) {
        if (!SMEM) { SOLVER_WRITE(region_off = ARENA_HDR; ref_base = (addr)(uintptr_t)contig); return true; }
        const int a0 = start & ~15;
        const int bytes = align_up(end - a0 + 16, 16);        // >= 16 bytes of slack for ld4u
        if ((u32)(ARENA_HDR + bytes + 2048) > arena_bytes) { SOLVER_WRITE(region_off = ARENA_HDR); return false; }
        tma_window_issue((u32)arena + ARENA_HDR, contig + a0, (u32)bytes, (u32)arena);   // waited for at the end of setup_pair
        SOLVER_WRITE(tma_pending = 1; ref_base = arena + ARENA_HDR - (u32)a0; region_off = ARENA_HDR + bytes);
        return true;
    }

    // wait for the window load issued by begin_region (every issued load must be waited for exactly once: the
    // mbarrier's parity is tracked in tma_phase)
    __device__ __forceinline__ void drain_window() {
        if (SMEM && tma_pending) {
            const u32 ph = tma_phase;
            tma_window_wait((u32)arena, ph);
            __syncwarp();
            if (lane_id() == 0) { tma_phase = ph ^ 1u; tma_pending = 0; }
            __syncwarp();
        }
    }

    // per-lane partial validation of one variant list (same rules as the oracle's list_valid)
    __device__ __noinline__ bool validate_list(u64 v0, int n, int *sums) const {
        const DevBatch &b = *bp;
        bool invalid = false;
        int s_l1 = 0, s_b0 = 0, s_al = 0, mx = 0;
#pragma unroll 1
        for (int i = lane_id(); i < n; i += 32) {
            const u64 gv = v0 + i;
            const u32 l0 = b.l0[gv], l1 = b.l1[gv], p = b.pos[gv];
            invalid = invalid || l0 == 0 || l1 == 0 || b.vtype[gv] >= AVK_N_VARIANT_TYPES || b.zyg[gv] > AVK_ZYG_HOM_ALT;
            invalid = invalid || (long long)p < start || (long long)p + l0 > (long long)end;
            if (i > 0) invalid = invalid || b.pos[gv - 1] > p;
            s_l1 += (int)min(l1, 1u << 24);
            s_b0 += (int)min(max(l0, l1), 1u << 24);
            s_al += (int)min(l0, 1u << 24) + (int)min(l1, 1u << 24);
            mx = max(mx, (int)min(p + l0, 0x7fffffffu));
        }
        sums[0] += s_l1; sums[1] += s_b0; sums[2] += s_al; sums[3] = max(sums[3], mx);
        return invalid;
    }

    // Validate and load one (truth list, query list) pair of region r: lays out the arena, fills the
    // variant records in merged order, stages the allele bytes, assigns metric-row slots.
    __device__ __noinline__ int setup_pair(u64 r, u32 ki, u32 kj, bool want_metrics) {
        const DevBatch &b = *bp;
        const int lane = lane_id();
        const u32 K = b.n_inputs;
        const u64 v0[2] = {b.var_off[r * K + ki], b.var_off[r * K + kj]};
        const int n0 = (int)(b.var_off[r * K + ki + 1] - v0[0]), n1 = (int)(b.var_off[r * K + kj + 1] - v0[1]);
        const int n = n0 + n1;
        SOLVER_WRITE(nv[0] = n0; nv[1] = n1; N = n);
        int sums[4] = {0, 0, 0, start};
        bool invalid = validate_list(v0[0], n0, sums);
        invalid = validate_list(v0[1], n1, sums) || invalid;
        if (__any_sync(AVK_FULL, invalid)) return AVK_ST_BAD_INPUT;
        const int sum_l1 = __reduce_add_sync(AVK_FULL, sums[0]);
        const int b0 = __reduce_add_sync(AVK_FULL, sums[1]);
        const int sum_alle = __reduce_add_sync(AVK_FULL, sums[2]);
        const int max_end = __reduce_max_sync(AVK_FULL, sums[3]);

        // ---- layout of the fixed part
        const int npad = align_up(max(n, 1), 16);
        // room for equal-best results: all of them (<= max_branch_factor) when the arena is large,
        // a handful in the small shared-memory tiers (more than that escalates to the next tier)
        const int rcap = (arena_bytes >= (16u << 10)) ? mbf : min(mbf, 8);
        u32 off = (u32)region_off;
        const addr L_vinfo = arena + off; off += (u32)(VI_SIZE * max(n, 1));
        const addr alle_buf = arena + off;
        if (SMEM) off += (u32)align_up(sum_alle + 16, 16);
        const addr L_bucket = arena + off; off += (u32)align_up(4 * (n + 1), 16);
        const addr L_res_alle = arena + off; off += (u32)(rcap * npad);
        const addr L_res_num = arena + off; off += (u32)align_up(rcap * 24, 16);
        // (16 bytes between the arrays: the word-wise copies between them read up to 7 bytes past their source)
        const addr L_hap_alle = arena + off; off += (u32)npad + 16;
        const addr L_cur_obs = arena + off; off += (u32)(2 * npad) + 16;
        const addr L_best_obs = arena + off; off += (u32)(2 * npad) + 16;
        const addr L_sdesc = arena + off; off += 3 * SD_SIZE;
        SOLVER_WRITE(Npad = npad;
                     seq_cap = align_up((max_end - start) + sum_l1 + 16, 16);   // materialised prefix: up to the last variant end + all ALTs
                     wf_cap = align_up(2 * b0 + 3, 4); res_cap = rcap;
                     vinfo = L_vinfo; bucket = L_bucket; res_alle = L_res_alle; res_num = L_res_num; hap_alle = L_hap_alle;
                     cur_obs = L_cur_obs; best_obs = L_best_obs; sdesc = L_sdesc;
                     alle_base = SMEM ? alle_buf : (addr)(uintptr_t)b.pool);
        if (off + 1024 > arena_bytes) return SOLVE_WORKSPACE;

        // ---- merged order: stable, truth before query on equal positions
#pragma unroll 1
        for (int side = 0; side < 2; ++side) {
            const int nm = side ? n1 : n0, no = side ? n0 : n1;
            const u64 vm = v0[side], vo = v0[side ^ 1];
#pragma unroll 1
            for (int i = lane; i < nm; i += 32) {
                const u64 gv = vm + i;
                const u32 p = b.pos[gv];
                int lo = 0, hi = no;
#pragma unroll 1
                while (lo < hi) {
                    const int m = (lo + hi) >> 1;
                    const u32 pm = b.pos[vo + m];
                    const bool before = side == 0 ? (pm < p) : (pm <= p);
                    if (before) lo = m + 1; else hi = m;
                }
                const addr rec = vi(i + lo);
                ST32(rec + VI_POS, p); ST32(rec + VI_L0, b.l0[gv]); ST32(rec + VI_L1, b.l1[gv]); ST32(rec + VI_AOFF, b.aoff[gv]);
                ST32(rec + VI_ALTED, b.alt_ed[gv]); ST32(rec + VI_RAW, b.raw[gv]); ST32(rec + VI_GV, (u32)gv);
                ST32(rec + VI_FLAGS, (u32)b.vtype[gv] | ((u32)b.zyg[gv] << 8) | ((side == 0 ? 1u : 0u) << 16));
            }
        }
        __syncwarp();
        // ---- stage allele bytes (shared-memory tiers)
        if (SMEM) {
            int acc = 0;
#pragma unroll 1
            for (int oi = 0; oi < n; ++oi) {
                const int na = (int)(LD32(vi(oi) + VI_L0) + LD32(vi(oi) + VI_L1));
                const u8 *src = b.pool + LD32(vi(oi) + VI_AOFF);
#pragma unroll 1
                for (int i = lane; i < na; i += 32) ST8(alle_buf + acc + i, src[i]);
                __syncwarp();
                if (lane == 0) ST32(vi(oi) + VI_AOFF, acc);
                acc += na;
            }
        }
        int ns = 0;
        if (want_metrics) {
            u32 seen = 0;
#pragma unroll 1
            for (int oi = 0; oi < n; ++oi) seen |= 1u << (LD32(vi(oi) + VI_FLAGS) & 0xff);
            ns = __popc(seen);
            __syncwarp();
            if (lane == 0) {
                int k = 0;
#pragma unroll 1
                for (int t = 0; t < AVK_N_VARIANT_TYPES; ++t) if (seen & (1u << t)) slot_type[k++] = (u8)t;
            }
#pragma unroll 1
            for (int oi = lane; oi < n; oi += 32) {
                const u32 f = LD32(vi(oi) + VI_FLAGS);
                ST32(vi(oi) + VI_FLAGS, f | ((u32)__popc(seen & ((1u << (f & 0xff)) - 1)) << 24));
            }
            off = (off + 7u) & ~7u;
            const addr L_mrows = arena + off; off += (u32)(8 * AVK_N_METRICS * (1 + ns));
            const addr L_slot_tot = arena + off; off += (u32)(16 * max(ns, 1));
            const addr L_slot_cnt = arena + off; off += (u32)(16 * max(ns, 1));
            SOLVER_WRITE(mrows = L_mrows; slot_tot = L_slot_tot; slot_cnt = L_slot_cnt);
            if (off + 512 > arena_bytes) return SOLVE_WORKSPACE;
#pragma unroll 1
            for (int i = lane; i < AVK_N_METRICS * (1 + ns); i += 32) ST64(L_mrows + 8 * i, 0);
#pragma unroll 1
            for (int i = lane; i < 2 * ns; i += 32) { ST32(L_slot_cnt + 4 * i, 0); ST64(L_slot_tot + 8 * i, 0); }
        }
        off = (off + 15u) & ~15u;
        SOLVER_WRITE(n_slots = ns; dyn = arena + off; dyn_bytes = arena_bytes - off);
        drain_window();
        __syncwarp();
        return SOLVE_OK;
    }

    // Compare path: load the cluster digest prepared by k_prep_fill (one TMA bulk copy in shared-memory tiers; read in
    // place from global memory otherwise) and lay out the rest of the arena.  Replaces setup_pair() + begin_region()
    // for solve_compare_region; the digest holds exactly what setup_pair computes.
    __device__ __noinline__ int load_cluster(u64 r, const u8 *contig, bool want_metrics) {
        const DevBatch &b = *bp;
        const int lane = lane_id();
        const u64 d0 = b.digest_off[r];
        const u32 dbytes = (u32)(b.digest_off[r + 1] - d0);
        const u8 *dig = b.digest + d0;
        u32 off = ARENA_HDR;
        addr hdr, L_ref_base;
        if (SMEM) {
            const int a0 = start & ~15;
            const u32 wbytes = (u32)align_up(end - a0 + 16, 16);        // >= 16 bytes of slack for ld4u
            if (ARENA_HDR + wbytes + dbytes + 1024 > arena_bytes) return SOLVE_WORKSPACE;
            const u32 ph = tma_phase;
            tma_issue2((u32)arena + ARENA_HDR, contig + a0, wbytes, (u32)arena + ARENA_HDR + wbytes, dig, dbytes, (u32)arena);
            tma_window_wait((u32)arena, ph);
            SOLVER_WRITE(tma_phase = ph ^ 1u);
            L_ref_base = arena + ARENA_HDR - (u32)a0;
            hdr = arena + ARENA_HDR + wbytes;
            off = ARENA_HDR + wbytes + dbytes;
        } else {
            L_ref_base = (addr)(uintptr_t)contig;
            hdr = (addr)(uintptr_t)dig;
        }
        const int st = LDI(hdr + PH_STATUS);
        if (st) return st;
        if (!SMEM && wide_b0 && LDI(hdr + PH_B0) >= wide_b0) return SOLVE_WORKSPACE;   // wide wavefronts: cooperative tier
        const int n = LDI(hdr + PH_N);
        const int npad = align_up(max(n, 1), 16);
        const int rcap = (arena_bytes >= (16u << 10)) ? mbf : min(mbf, 8);
        const addr L_vinfo = hdr + PH_SIZE;
        const addr L_bucket = arena + off; off += (u32)align_up(4 * (n + 1), 16);
        const addr L_res_alle = arena + off; off += (u32)(rcap * npad);
        const addr L_res_num = arena + off; off += (u32)align_up(rcap * 24, 16);
        // (16 bytes between the arrays: the word-wise copies between them read up to 7 bytes past their source)
        const addr L_hap_alle = arena + off; off += (u32)npad + 16;
        const addr L_cur_obs = arena + off; off += (u32)(2 * npad) + 16;
        const addr L_best_obs = arena + off; off += (u32)(2 * npad) + 16;
        const addr L_sdesc = arena + off; off += 3 * SD_SIZE;
        int ns = 0;
        addr L_mrows = 0, L_slot_tot = 0, L_slot_cnt = 0;
        if (want_metrics) {
            ns = LDI(hdr + PH_NSLOTS);
            off = (off + 7u) & ~7u;
            L_mrows = arena + off; off += (u32)(8 * AVK_N_METRICS * (1 + ns));
            L_slot_tot = arena + off; off += (u32)(16 * max(ns, 1));
            L_slot_cnt = arena + off; off += (u32)(16 * max(ns, 1));
        }
        const u32 fixed_end = off;
        off = (off + 15u) & ~15u;
        SOLVER_WRITE(ref_base = L_ref_base; N = n; nv[0] = LDI(hdr + PH_N0); nv[1] = LDI(hdr + PH_N1); Npad = npad;
                     seq_cap = align_up((LDI(hdr + PH_MAX_END) - start) + LDI(hdr + PH_SUM_L1) + 16, 16);
                     wf_cap = align_up(2 * LDI(hdr + PH_B0) + 3, 4); res_cap = rcap;
                     vinfo = L_vinfo; alle_base = L_vinfo + (u32)(VI_SIZE * n);
                     bucket = L_bucket; res_alle = L_res_alle; res_num = L_res_num; hap_alle = L_hap_alle;
                     cur_obs = L_cur_obs; best_obs = L_best_obs; sdesc = L_sdesc;
                     mrows = L_mrows; slot_tot = L_slot_tot; slot_cnt = L_slot_cnt; n_slots = ns;
                     dyn = arena + off; dyn_bytes = arena_bytes > off ? arena_bytes - off : 0;
                     for (int k = 0; k < ns && k < AVK_N_VARIANT_TYPES; ++k) slot_type[k] = LD8(hdr + PH_SLOT_TYPE + k));
        if (fixed_end + 512 > arena_bytes) return SOLVE_WORKSPACE;
        if (want_metrics) {
#pragma unroll 1
            for (int i = lane; i < AVK_N_METRICS * (1 + ns); i += 32) ST64(L_mrows + 8 * i, 0);
#pragma unroll 1
            for (int i = lane; i < 2 * ns; i += 32) { ST32(L_slot_cnt + 4 * i, 0); ST64(L_slot_tot + 8 * i, 0); }
        }
        __syncwarp();
        return SOLVE_OK;
    }

    // Partition the dynamic part into queue arrays + node slots of `stride_` bytes.  When the warp has a spill area
    // in global memory (shared-memory tiers), the queue may hold more entries than there are node slots: nodes that
    // are far down the queue are evicted to the spill area and brought back when they are popped.
    __device__ __noinline__ bool partition(int stride_, int min_slots) {
        const int scap = (spill_bytes > 32768u) ? (int)min((spill_bytes - 16384u) / (u32)stride_, 4096u) : 0;   // spillable nodes (after the id free list)
        const int extra = min(scap, 384);                       // queue entries beyond the resident slots
        const u32 per = (u32)stride_ + 16u;
        if (dyn_bytes < 12u * (u32)extra + 64u) return false;
        int ms = (int)min((dyn_bytes - 12u * (u32)extra - 16u) / per, 60000u);
        if (ms < min_slots) return false;
        const int qc = ms + extra;
        u32 off = 0;
        const addr qk = dyn + off; off += (u32)qc * 8;
        const addr qs = dyn + off; off += (u32)qc * 4;
        const addr fl = dyn + off; off += (u32)ms * 4;
        off = (off + 15u) & ~15u;
        if (off + (u32)ms * (u32)stride_ > dyn_bytes) ms = (int)((dyn_bytes - off) / (u32)stride_);
        if (ms < min_slots) return false;
        __syncwarp();
        if (lane_id() == 0) {
            stride = stride_; qkeys = qk; qslot = qs; freel = fl;
            max_slots = ms; qcap = qc; nodes = dyn + off; nfree = ms; qn = 0;
            spill_cap = scap; spill_used = 0; spill_nfree = 0;
        }
        __syncwarp();
#pragma unroll 1
        for (int i = lane_id(); i < ms; i += 32) ST32(freel + 4 * i, ms - 1 - i);
        __syncwarp();
        return true;
    }
    __device__ __forceinline__ addr node(int s) const { return nodes + (u32)s * (u32)stride; }
    // spill area layout (global, per warp): [u32 free_ids[4096]] [nodes of `stride` bytes]
    __device__ __forceinline__ u8 *spill_node(u32 id) const { return spill_base + 16384 + (size_t)id * (size_t)stride; }
    // field of a queued node that may be resident (slot < 0x80000000) or spilled
    __device__ __forceinline__ u32 qnode_ld32(u32 v, int off) const {
        return (v & 0x80000000u) ? *(const u32 *)(spill_node(v & 0x7fffffffu) + off) : LD32(node((int)v) + off);
    }
    __device__ __forceinline__ u32 qnode_ld8(u32 v, int off) const {
        return (v & 0x80000000u) ? (u32)spill_node(v & 0x7fffffffu)[off] : (u32)LD8(node((int)v) + off);
    }
    // The solver object is shared by the 32 lanes of its warp: every lane reads a field, lane 0 alone writes it,
    // with __syncwarp() between the reads and the write (no lane may observe a half-updated counter).
    __device__ __forceinline__ void free_slot(int s) {
        const int nf = nfree;
        __syncwarp();
        if (lane_id() == 0) { ST32(freel + 4 * nf, s); nfree = nf + 1; }
        __syncwarp();
    }
    __device__ __forceinline__ void free_spill(u32 id) {
        const int nf = spill_nfree;
        __syncwarp();
        if (lane_id() == 0) { ((u32 *)spill_base)[nf] = id; spill_nfree = nf + 1; }
        __syncwarp();
    }
    // release whatever a queue entry refers to
    __device__ __forceinline__ void free_entry(u32 v) {
        if (v & 0x80000000u) free_spill(v & 0x7fffffffu); else free_slot((int)v);
    }
    // Evict the queued resident node with the LARGEST key (popped last) to the spill area; returns its slot or -1.
    __device__ __noinline__ int evict_one() {
        const int lane = lane_id();
        const int n = qn;
        if (spill_cap == 0) return -1;
        u64 worst = 0;
        int wi = -1;
#pragma unroll 1
        for (int i = lane; i < n; i += 32) {
            if (LD32(qslot + 4 * i) & 0x80000000u) continue;
            const u64 k = LD64(qkeys + 8 * i);
            if (wi < 0 || k > worst) { worst = k; wi = i; }
        }
        const u32 hi = wi < 0 ? 0u : (u32)(worst >> 32), lo = wi < 0 ? 0u : (u32)worst;
        if (!__any_sync(AVK_FULL, wi >= 0)) return -1;
        const u32 mhi = __reduce_max_sync(AVK_FULL, hi);
        const u32 mlo = __reduce_max_sync(AVK_FULL, (wi >= 0 && hi == mhi) ? lo : 0u);
        const int owner = __ffs(__ballot_sync(AVK_FULL, wi >= 0 && hi == mhi && lo == mlo)) - 1;
        wi = __shfl_sync(AVK_FULL, wi, owner);
        u32 id;
        const int nf = spill_nfree;
        if (nf > 0) id = ((const u32 *)spill_base)[nf - 1];
        else if (spill_used < spill_cap) id = (u32)spill_used;
        else return -1;
        const int slot = (int)LD32(qslot + 4 * wi);
        u32 *dst = (u32 *)spill_node(id);
        const addr src = node(slot);
        const int words = stride >> 2;
#pragma unroll 1
        for (int i = lane; i < words; i += 32) dst[i] = LD32(src + 4 * i);
        __syncwarp();
        if (lane == 0) {
            ST32(qslot + 4 * wi, 0x80000000u | id);
            if (nf > 0) spill_nfree = nf - 1; else spill_used = spill_used + 1;
        }
        __syncwarp();
        return slot;
    }
    __device__ __noinline__ int alloc_slot() {   // warp-uniform; -1 when exhausted
        const int nf = nfree;
        if (nf == 0) return evict_one();
        const int s = (int)LD32(freel + 4 * (nf - 1));
        __syncwarp();
        if (lane_id() == 0) nfree = nf - 1;
        __syncwarp();
        return s;
    }
    __device__ __forceinline__ bool push(u64 key, int slot) {
        const int n = qn;
        if (n >= qcap) return false;
        __syncwarp();
        if (lane_id() == 0) { ST64(qkeys + 8 * n, key); ST32(qslot + 4 * n, slot); qn = n + 1; }
        __syncwarp();
        return true;
    }
    // pop the minimum key: warp-parallel scan, then two REDUX min-reductions (high word, low word) and a ballot to
    // locate the owner -- keys are unique, so exactly one lane matches.  A spilled node is brought back into a slot.
    // returns the slot, or -1 if no slot could be made available.
    __device__ __noinline__ int pop(u32 *key_hi) {
        const int lane = lane_id();
        const int n = qn;
        u64 best = ~0ull;
        int bi = 0;
#pragma unroll 1
        for (int i = lane; i < n; i += 32) { const u64 k = LD64(qkeys + 8 * i); if (k < best) { best = k; bi = i; } }
        const u32 hi = (u32)(best >> 32), lo = (u32)best;
        const u32 mhi = __reduce_min_sync(AVK_FULL, hi);
        const u32 mlo = __reduce_min_sync(AVK_FULL, hi == mhi ? lo : 0xffffffffu);
        const int owner = __ffs(__ballot_sync(AVK_FULL, hi == mhi && lo == mlo)) - 1;
        bi = __shfl_sync(AVK_FULL, bi, owner);
        const u32 v = LD32(qslot + 4 * bi);
        __syncwarp();
        if (lane == 0) { ST64(qkeys + 8 * bi, LD64(qkeys + 8 * (n - 1))); ST32(qslot + 4 * bi, LD32(qslot + 4 * (n - 1))); qn = n - 1; }
        __syncwarp();
        *key_hi = mhi;
        if (!(v & 0x80000000u)) return (int)v;
        const int slot = alloc_slot();
        if (slot < 0) return -1;
        const u32 id = v & 0x7fffffffu;
        const u32 *src = (const u32 *)spill_node(id);
        const addr dst = node(slot);
        const int words = stride >> 2;
#pragma unroll 1
        for (int i = lane; i < words; i += 32) ST32(dst + 4 * i, src[i]);
        __syncwarp();
        free_spill(id);
        return slot;
    }

    // ------------------------------------------------------------------ tracker
    // HaplotypeTracker::extend_variant() (haplotype_dwfa.rs:175-212) on one side of one haplotype.
    // copy_reference (:218-227) only moves ref_pos; bytes are materialised when an ALT is spliced.
    // returns 1 success / 0 incompatible (skipped) / -1 capacity overflow
    __device__ __forceinline__ int track(addr data, int &ref_pos, int &mlen, int &mref, int &skip, addr rec, bool alt, int sync) {
        const int vpos = (int)LD32(rec + VI_POS);
        if (ref_pos < vpos) ref_pos = vpos;
        int success = 1;
        if (alt) {
            if (ref_pos <= vpos) {
                const int l0 = (int)LD32(rec + VI_L0), l1 = (int)LD32(rec + VI_L1);
                const int nref = vpos - mref;
                if (mlen + nref + l1 > seq_cap) return -1;
                if (nref > 0) warp_copy<SMEM>(data + mlen, ref_base + mref, nref);
                warp_copy<SMEM>(data + mlen + nref, alle_base + LD32(rec + VI_AOFF) + l0, l1);
                mlen += nref + l1;
                ref_pos = vpos + l0;
                mref = ref_pos;
            } else {
                skip += (int)LD32(rec + VI_ALTED);   // edit_distance(allele0, allele1) :199
                success = 0;
            }
        }
        if (ref_pos < sync) ref_pos = sync;
        return success;
    }
    __device__ __forceinline__ VS make_vs(addr data, int mlen, int mref, int ref_pos) const {
        VS v;
        v.data = data; v.tail = ref_base + mref; v.mlen = mlen; v.len = mlen + (ref_pos - mref);
        return v;
    }

    // Queue garbage collection, used when no node slot is free.  It removes exactly the nodes the search would
    // discard WITHOUT side effects the moment they are popped, so the replayed search is unchanged:
    //   optimize_sequences : cost > best            (query_optimizer.rs:204, checked before the bucket quota)
    //   optimize_gt_alleles: errors >= best         (exact_gt_optimizer.rs:169, first check after the pop), or
    //                        depth < min_allele_sync for unfinished nodes (:194-197; finished nodes are handled
    //                        before that check and are kept)
    // key_hi of an optimize entry is its cost; an exact entry carries errors in key bits 48..63.
    __device__ __noinline__ int gc_queue(bool exact, u32 best, int min_sync, int n_total) {
        int w = 0;
        const int cnt = qn;
#pragma unroll 1
        for (int i = 0; i < cnt; ++i) {
            const u64 key = LD64(qkeys + 8 * i);
            const u32 sl = LD32(qslot + 4 * i);
            bool dead;
            if (!exact) dead = (u32)(key >> 32) > best;
            else {
                const int depth = (int)qnode_ld32(sl, XN_DEPTH);
                dead = (u32)(key >> 48) >= best || (depth != n_total && depth < min_sync);
            }
            if (!dead) {
                __syncwarp();
                if (lane_id() == 0 && w != i) { ST64(qkeys + 8 * w, key); ST32(qslot + 4 * w, sl); }
                w += 1;
            } else {
                free_entry(sl);
            }
            __syncwarp();
        }
        __syncwarp();
        if (lane_id() == 0) qn = w;
        __syncwarp();
        return cnt - w;
    }

    // ================================================================== optimize_sequences
    // node: hdr[80] | alle[Npad] | seq[4][seq_cap] (h0 truth, h0 query, h1 truth, h1 query) | wf[2][wf_cap] ints
    __device__ __forceinline__ int opt_stride() const { return ON_HDR + Npad + 4 * seq_cap + 8 * wf_cap; }
    __device__ __forceinline__ addr n_seq(addr nb, int k) const { return nb + (u32)(ON_HDR + Npad + k * seq_cap); }
    __device__ __forceinline__ addr n_wf(addr nb, int h) const { return nb + (u32)(ON_HDR + Npad + 4 * seq_cap + h * 4 * wf_cap); }

    __device__ __noinline__ void opt_clone(addr dst, addr src) {
        const int lane = lane_id();
        const int depth = LDI(src + ON_DEPTH);
        __syncwarp();
        if (lane < 20) ST32(dst + 4 * lane, LD32(src + 4 * lane));
        warp_copy<SMEM>(dst + ON_HDR, src + ON_HDR, depth);
#pragma unroll 1
        for (int h = 0; h < 2; ++h) {
            const addr hb = src + ON_HAP + ON_HAPSZ * h;
            warp_copy<SMEM>(n_seq(dst, 2 * h), n_seq(src, 2 * h), LDI(hb + H_TML));
            warp_copy<SMEM>(n_seq(dst, 2 * h + 1), n_seq(src, 2 * h + 1), LDI(hb + H_QML));
            const int nwf = 2 * LDI(hb + H_ED) + 1;
            const addr ws = n_wf(src, h), wd = n_wf(dst, h);
#pragma unroll 1
            for (int i = lane; i < nwf; i += 32) ST32(wd + 4 * i, LD32(ws + 4 * i));
        }
        __syncwarp();
    }

    // HaplotypeDWFA::extend_variant (haplotype_dwfa.rs:46-67) on hap h of node nb; finalize_dwfa (:84-95) when rec == 0.
    __device__ __noinline__ int opt_extend_hap(addr nb, int h, addr rec, bool alt, int sync, bool finalize) {
        const addr hb = nb + ON_HAP + ON_HAPSZ * h;
        int t_rp = LDI(hb + H_TRP), q_rp = LDI(hb + H_QRP), t_ml = LDI(hb + H_TML), q_ml = LDI(hb + H_QML);
        int t_mr = LDI(hb + H_TMR), q_mr = LDI(hb + H_QMR), t_sk = LDI(hb + H_TSK), q_sk = LDI(hb + H_QSK), ed = LDI(hb + H_ED);
        if (finalize) {
            t_rp = max(t_rp, end); q_rp = max(q_rp, end);
        } else if (LD32(rec + VI_FLAGS) & 0x10000u) {   // truth variant: query first copies reference to the sync point
            q_rp = max(q_rp, sync);
            if (track(n_seq(nb, 2 * h), t_rp, t_ml, t_mr, t_sk, rec, alt, sync) < 0) return SOLVE_WORKSPACE;
        } else {
            t_rp = max(t_rp, sync);
            if (track(n_seq(nb, 2 * h + 1), q_rp, q_ml, q_mr, q_sk, rec, alt, sync) < 0) return SOLVE_WORKSPACE;
        }
        __syncwarp();
        const VS T = make_vs(n_seq(nb, 2 * h), t_ml, t_mr, t_rp), Q = make_vs(n_seq(nb, 2 * h + 1), q_ml, q_mr, q_rp);
        const int cap = (wf_cap - 3) / 2;
        int rc = DWFA_OK;
        bool done = false;
        if (ed == 0) {
            // Fast path of DWFALite::update for the single diagonal: both sequences are reading the SAME reference
            // bytes from offset d on (aligned implicit tails), so the run extends to the end of the shorter one.
            const int d = LDI(n_wf(nb, h));
            if (d >= t_ml && d >= q_ml && T.tail + (u32)(d - t_ml) == Q.tail + (u32)(d - q_ml)) {
                const int nd = max(d, min(T.len, Q.len));
                __syncwarp();
                if (lane_id() == 0) {
                    ST32(n_wf(nb, h), nd);
                    wk_add64<SMEM>(wk() + WK_CELLS, 1); wk_add64<SMEM>(wk() + WK_MATCHED, (u64)(nd - d));
                }
                __syncwarp();
                done = !finalize || T.len == Q.len;     // finalize: the diagonal is at the end of both <=> equal lengths
                if (done && finalize && lane_id() == 0) wk_add64<SMEM>(wk() + WK_CELLS, 1);
            }
        }
        if (!done) {
            rc = dwfa_run<SMEM>(n_wf(nb, h), &ed, cap, T, Q, false, wk());
            if (rc == DWFA_OK && finalize) rc = dwfa_run<SMEM>(n_wf(nb, h), &ed, cap, T, Q, true, wk());
        }
        if (rc != DWFA_OK) return SOLVE_WORKSPACE;   // ED bound exceeded: never expected (DESIGN.md)
        __syncwarp();
        if (lane_id() == 0) {
            ST32(hb + H_TRP, t_rp); ST32(hb + H_QRP, q_rp); ST32(hb + H_TML, t_ml); ST32(hb + H_QML, q_ml);
            ST32(hb + H_TMR, t_mr); ST32(hb + H_QMR, q_mr); ST32(hb + H_TSK, t_sk); ST32(hb + H_QSK, q_sk); ST32(hb + H_ED, ed);
            if (finalize) wk_add32<SMEM>(wk() + WK_ALIGN, 1);
        }
        __syncwarp();
        return SOLVE_OK;
    }
    // ---- warp team ------------------------------------------------------------------------------------------------
    // executed by every warp of the team between the two barriers of a round; warp w takes job w
    __device__ __forceinline__ void team_exec(int w) {
        TeamBoard &B = *team;
        if (w < B.count) {
            const int rc = B.kind == 0 ? opt_extend_hap((addr)B.nb[w], B.h[w], (addr)B.rec, B.alt[w] != 0, B.sync, B.finalize != 0)
                                       : ex_extend((addr)B.nb[w], B.oi, B.alt[w] != 0, B.err[w] != 0, B.finalize != 0);
            if (lane_id() == 0) B.rc[w] = rc;
        }
    }
    // master warp: the board is filled (by lane 0, before); run one round
    __device__ __forceinline__ void team_sync() const { asm volatile("bar.sync %0, 128;" ::"r"(team->bar) : "memory"); }
    __device__ __noinline__ void team_round() {
        __syncwarp();
        team_sync();
        team_exec(0);
        team_sync();
    }
    // second half of opt_extend: record the alleles, return the node's new cost
    __device__ __forceinline__ u32 opt_commit(addr nb, int oi, bool a1_alt, bool a2_alt) {
        __syncwarp();
        if (lane_id() == 0) { ST8(nb + ON_HDR + oi, (a1_alt ? 1 : 0) | (a2_alt ? 2 : 0)); ST32(nb + ON_DEPTH, oi + 1); }
        __syncwarp();
        return opt_cost(nb);
    }
    // ComparisonNode::extend_variant :443-451 followed by the push; returns the node's new cost via *cost
    __device__ __noinline__ int opt_extend(addr nb, int oi, bool a1_alt, bool a2_alt, u32 *cost) {
        const addr rec = vi(oi);
        const int sync = sync_pos(oi);
        int rc = opt_extend_hap(nb, 0, rec, a1_alt, sync, false);
        if (rc) return rc;
        rc = opt_extend_hap(nb, 1, rec, a2_alt, sync, false);
        if (rc) return rc;
        __syncwarp();
        if (lane_id() == 0) { ST8(nb + ON_HDR + oi, (a1_alt ? 1 : 0) | (a2_alt ? 2 : 0)); ST32(nb + ON_DEPTH, oi + 1); }
        __syncwarp();
        *cost = opt_cost(nb);
        return SOLVE_OK;
    }
    __device__ __forceinline__ u32 opt_cost(addr nb) const {
        const addr h0 = nb + ON_HAP, h1 = nb + ON_HAP + ON_HAPSZ;
        return (u32)(LDI(h0 + H_ED) + LDI(h0 + H_TSK) + LDI(h0 + H_QSK) + LDI(h1 + H_ED) + LDI(h1 + H_TSK) + LDI(h1 + H_QSK));
    }

    // Runs the best-first search.  Results (all equal-best, in finalisation order) go to res_alle/res_num.
    // stop_at_nonzero: merge only needs "is the minimum cost zero" (merge_solver.rs:142-143); costs never
    // decrease along a path, so the search may stop at the first popped node whose cost is > 0.
    __device__ __noinline__ int optimize(bool stop_at_nonzero) {
        const int lane = lane_id();
        const int n = N;
        // without a spill area: cheap early escalation when the search obviously will not fit
        if (!partition(opt_stride(), spill_bytes ? 6 : min(n + 3, 48))) return SOLVE_WORKSPACE;
#pragma unroll 1
        for (int i = lane; i <= n; i += 32) ST32(bucket + 4 * i, 0);
        SOLVER_WRITE(n_res = 0);
        int nres = 0;
        u32 best = 0xffffffffu;
        u32 next_id = 1;
        {   // root (query_optimizer.rs:184-192): id 0, both haplotypes at region start, wavefront [0]
            const int s = alloc_slot();
            const addr nb = node(s);
            __syncwarp();
            if (lane < 20) {
                const int k = lane - 2;   // hap field index (0..17) once past id/depth
                const bool at_start = lane >= 2 && ((k % 9) == 0 || (k % 9) == 1 || (k % 9) == 4 || (k % 9) == 5);
                ST32(nb + 4 * lane, at_start ? start : 0);
            }
            __syncwarp();
            if (lane == 0) { ST32(n_wf(nb, 0), 0); ST32(n_wf(nb, 1), 0); }
            __syncwarp();
            if (!push(0ull, s)) return SOLVE_WORKSPACE;
        }
#pragma unroll 1
        while (qn > 0) {
            u32 cost;
            const int s = pop(&cost);
            if (s < 0) return SOLVE_WORKSPACE;
            __syncwarp();
            if (lane == 0) ST32(wk() + WK_SPOPS, LD32(wk() + WK_SPOPS) + 1);
            if (stop_at_nonzero && cost > 0) break;        // nothing cheaper is left; n_res tells if a zero-cost result exists
            if (cost > best) { free_slot(s); continue; }                       // :204 strict
            const addr nb = node(s);
            const int oi = LDI(nb + ON_DEPTH);
            const int bc = LDI(bucket + 4 * oi);
            if (bc >= mbf) { free_slot(s); continue; }                         // :222
            __syncwarp();
            if (lane == 0) ST32(bucket + 4 * oi, bc + 1);
            __syncwarp();
            if (oi == n) {                                                     // :227-247
                if (SMEM && team) {                                            // both haplotypes at once
                    if (lane == 0) {
                        TeamBoard &B = *team;
                        B.kind = 0; B.count = 2; B.finalize = 1; B.rec = 0; B.sync = 0;
                        B.nb[0] = B.nb[1] = (unsigned)nb; B.h[0] = 0; B.h[1] = 1; B.alt[0] = B.alt[1] = 0;
                    }
                    team_round();
                    if (team->rc[0]) return team->rc[0];
                    if (team->rc[1]) return team->rc[1];
                } else {
                int rc = opt_extend_hap(nb, 0, 0, false, 0, true);
                if (rc) return rc;
                rc = opt_extend_hap(nb, 1, 0, false, 0, true);
                if (rc) return rc;
                }
                const u32 c = opt_cost(nb);
                if (c < best) { best = c; nres = 0; }
                if (c == best) {
                    if (nres >= res_cap) return SOLVE_WORKSPACE;
                    warp_copy<SMEM>(res_alle + (u32)(nres * Npad), nb + ON_HDR, n);
                    if (lane < 6) {   // ed1 ed2 tvs1 tvs2 qvs1 qvs2
                        const int fld = lane < 2 ? H_ED : (lane < 4 ? H_TSK : H_QSK);
                        ST32(res_num + (u32)(nres * 24 + 4 * lane), LD32(nb + ON_HAP + ON_HAPSZ * (lane & 1) + fld));
                    }
                    __syncwarp();
                    nres += 1;
                }
                free_slot(s);
                continue;
            }
            const u32 flags = LD32(vi(oi) + VI_FLAGS);
            const int z = (flags >> 8) & 0xff;
            const bool is_truth = (flags & 0x10000u) != 0;
            const bool het = (z == AVK_ZYG_UNPHASED_HET || z == AVK_ZYG_PHASED_HET01 || z == AVK_ZYG_PHASED_HET10);
            if (!het && z != AVK_ZYG_HOM_ALT) return AVK_ST_BAD_ZYGOSITY;      // assert_eq! :315
            const bool two = het && (!is_truth || z == AVK_ZYG_UNPHASED_HET);  // :269: both orientations, new ids
            int s2 = -1;
            if (two) {
                s2 = alloc_slot();
                if (s2 < 0 && gc_queue(false, best, 0, n) > 0) s2 = alloc_slot();
                if (s2 < 0) return SOLVE_WORKSPACE;
                opt_clone(node(s2), nb);
                // first child (REF, ALT) gets the lower id, second (ALT, REF) the next one
                __syncwarp();
                if (lane == 0) { ST32(node(s2) + ON_ID, next_id); ST32(nb + ON_ID, next_id + 1); }
                __syncwarp();
                next_id += 2;
            }
            // child order: (REF, ALT) then (ALT, REF) for a split; the single fixed orientation otherwise
            // (phased truth het :294-312, hom-alt :313-327) keeps the node id.
            if (SMEM && team) {                                                // all haplotype extensions of this pop at once
                const int nk = two ? 2 : 1;
                if (lane == 0) {
                    TeamBoard &B = *team;
                    B.kind = 0; B.count = 2 * nk; B.finalize = 0; B.rec = (unsigned)vi(oi); B.sync = sync_pos(oi);
                    for (int k = two ? 0 : 1, q = 0; k < 2; ++k, ++q) {
                        const int sl = (two && k == 0) ? s2 : s;
                        bool a1, a2;
                        if (two) { a1 = k == 1; a2 = k == 0; }
                        else if (het) { a1 = (z == AVK_ZYG_PHASED_HET10); a2 = !a1; }
                        else { a1 = true; a2 = true; }
                        B.nb[2 * q] = B.nb[2 * q + 1] = (unsigned)node(sl);
                        B.h[2 * q] = 0; B.h[2 * q + 1] = 1; B.alt[2 * q] = a1; B.alt[2 * q + 1] = a2;
                    }
                }
                team_round();
#pragma unroll 1
                for (int q = 0; q < 2 * nk; ++q) if (team->rc[q]) return team->rc[q];
#pragma unroll 1
                for (int k = two ? 0 : 1, q = 0; k < 2; ++k, ++q) {
                    const int sl = (two && k == 0) ? s2 : s;
                    const u32 c = opt_commit(node(sl), oi, team->alt[2 * q] != 0, team->alt[2 * q + 1] != 0);
                    if (!push(((u64)c << 32) | LD32(node(sl) + ON_ID), sl)) return SOLVE_WORKSPACE;
                }
            } else {
#pragma unroll 1
            for (int k = two ? 0 : 1; k < 2; ++k) {
                const int sl = (two && k == 0) ? s2 : s;
                bool a1, a2;
                if (two) { a1 = k == 1; a2 = k == 0; }
                else if (het) { a1 = (z == AVK_ZYG_PHASED_HET10); a2 = !a1; }
                else { a1 = true; a2 = true; }
                u32 c;
                const int rc = opt_extend(node(sl), oi, a1, a2, &c);
                if (rc) return rc;
                if (!push(((u64)c << 32) | LD32(node(sl) + ON_ID), sl)) return SOLVE_WORKSPACE;
            }
            }
        }
        SOLVER_WRITE(n_res = nres);
        if (nres == 0 && !stop_at_nonzero) return AVK_ST_NO_RESULT;            // :331
        return SOLVE_OK;
    }

    // ================================================================== optimize_gt_alleles
    // node: hdr[48] | alle[Npad] | seq[2][seq_cap].  DWFA max ED is 0 (exact_gt_optimizer.rs:380), so the wavefront
    // is the single matched length d and "alive" means one sequence is a prefix of the other.
    __device__ __forceinline__ int ex_stride() const { return XN_HDR + Npad + 2 * seq_cap; }
    __device__ __forceinline__ addr x_seq(addr nb, int k) const { return nb + (u32)(XN_HDR + Npad + k * seq_cap); }

    __device__ __noinline__ void ex_clone(addr dst, addr src) {
        const int lane = lane_id();
        __syncwarp();
        if (lane < 10) ST32(dst + 4 * lane, LD32(src + 4 * lane));
        warp_copy<SMEM>(dst + XN_HDR, src + XN_HDR, LDI(src + XN_DEPTH));
        warp_copy<SMEM>(x_seq(dst, 0), x_seq(src, 0), LDI(src + XN_TML));
        warp_copy<SMEM>(x_seq(dst, 1), x_seq(src, 1), LDI(src + XN_QML));
        __syncwarp();
    }
    // ExactMatchNode::extend_variant (exact_gt_optimizer.rs:395-414), or finalize_dwfas (:421-434) when finalize.
    // returns 1 keep (alive / exact) / 0 drop / <0 error
    __device__ __noinline__ int ex_extend(addr nb, int oi, bool alt, bool is_error, bool finalize) {
        int t_rp = LDI(nb + XN_TRP), q_rp = LDI(nb + XN_QRP), t_ml = LDI(nb + XN_TML), q_ml = LDI(nb + XN_QML);
        int t_mr = LDI(nb + XN_TMR), q_mr = LDI(nb + XN_QMR), d = LDI(nb + XN_D);
        int skip = 0, success = 1;
        if (finalize) {
            t_rp = max(t_rp, end); q_rp = max(q_rp, end);
        } else {
            const addr rec = vi(oi);
            const int sync = sync_pos(oi);
            if (LD32(rec + VI_FLAGS) & 0x10000u) {
                q_rp = max(q_rp, sync);
                success = track(x_seq(nb, 0), t_rp, t_ml, t_mr, skip, rec, alt, sync);
            } else {
                t_rp = max(t_rp, sync);
                success = track(x_seq(nb, 1), q_rp, q_ml, q_mr, skip, rec, alt, sync);
            }
            if (success < 0) return SOLVE_WORKSPACE;
        }
        __syncwarp();
        // DWFA update with max ED 0: extend the single diagonal, then require an end to be reached
        const VS T = make_vs(x_seq(nb, 0), t_ml, t_mr, t_rp), Q = make_vs(x_seq(nb, 1), q_ml, q_mr, q_rp);
        int ext = 0;
        if (d < T.len && d < Q.len) {
            if (d >= t_ml && d >= q_ml && T.tail + (u32)(d - t_ml) == Q.tail + (u32)(d - q_ml)) ext = min(T.len, Q.len) - d;   // aligned tails
            else ext = vs_lcp<SMEM>(T, d, Q, d);
        }
        d += ext;
        const bool alive = finalize ? ((d >= T.len) && (d >= Q.len))    // update ok + finalize ok <=> sequences equal
                                    : ((d >= T.len) || (d >= Q.len));
        __syncwarp();
        if (lane_id() == 0) {
            wk_add64<SMEM>(wk() + WK_CELLS, 1); wk_add64<SMEM>(wk() + WK_MATCHED, (u64)ext);
            if (finalize) wk_add32<SMEM>(wk() + WK_ALIGN, 1);
            else {
                if (is_error) ST32(nb + XN_ERR, LD32(nb + XN_ERR) + 1);
                ST32(nb + XN_DEPTH, oi + 1);
                ST8(nb + XN_HDR + oi, alt ? AL_ALT : AL_REF);
            }
            ST32(nb + XN_TRP, t_rp); ST32(nb + XN_QRP, q_rp); ST32(nb + XN_TML, t_ml); ST32(nb + XN_QML, q_ml);
            ST32(nb + XN_TMR, t_mr); ST32(nb + XN_QMR, q_mr); ST32(nb + XN_D, d);
        }
        __syncwarp();
        return (success && alive) ? 1 : 0;
    }
    __device__ __forceinline__ u64 ex_key(addr nb) const {   // (Reverse(errors), set - errors, Reverse(id)) :372,452-458
        const u64 errors = (u64)LD32(nb + XN_ERR);
        const u64 good = (u64)(LD32(nb + XN_DEPTH) - LD32(nb + XN_ERR));
        return (errors << 48) | ((0xffffull - good) << 32) | LD32(nb + XN_ID);
    }

    // in: hap_alle[oi] (AL_REF / AL_ALT by order index).  out: obs[oi], *errors.
    // `budget`: the caller only cares about results with fewer than `budget` errors.  Nodes are popped in
    // non-decreasing error order, so the search stops at the first popped node that reaches the budget and reports
    // *errors_out = budget ("at least").
    __device__ __noinline__ int exact_gt(addr obs, int *errors_out, int budget, u32 max_expansions) {
        u32 expansions = 0;
        const int lane = lane_id();
        const int n = N;
        if (n >= 0xffff) return SOLVE_WORKSPACE;
        if (!partition(ex_stride(), spill_bytes ? 6 : min(n + 3, 48))) return SOLVE_WORKSPACE;
        u32 next_id = 1;
        int best_err = 0x7fffffff;
        bool have_best = false;
        int min_sync = 0, af_index = 0, af_counts = 0;
        {
            const int s = alloc_slot();
            const addr nb = node(s);
            __syncwarp();
            if (lane < 10) ST32(nb + 4 * lane, (lane == 3 || lane == 4 || lane == 7 || lane == 8) ? start : 0);
            __syncwarp();
            if (!push(ex_key(nb), s)) return SOLVE_WORKSPACE;
        }
#pragma unroll 1
        while (qn > 0) {
            u32 khi;
            const int s = pop(&khi);
            if (s < 0) return SOLVE_WORKSPACE;
            __syncwarp();
            if (lane == 0) ST32(wk() + WK_XPOPS, LD32(wk() + WK_XPOPS) + 1);
            const addr nb = node(s);
            const int errors = LDI(nb + XN_ERR);
            if (errors >= budget && !have_best) { *errors_out = budget; return SOLVE_OK; }
            if (errors >= best_err) { free_slot(s); continue; }                // :169 non-strict
            if (++expansions > max_expansions) return AVK_ST_TIMEOUT;          // stand-in for the 300 s bail (:174-176)
            const int oi = LDI(nb + XN_DEPTH);
            if (oi == n) {                                                     // :180-192
                const int exact = ex_extend(nb, oi, false, false, true);
                if (exact < 0) return exact;
                if (exact && errors < best_err) {
                    best_err = errors;
                    have_best = true;
                    warp_copy<SMEM>(obs, nb + XN_HDR, n);
                    __syncwarp();
                }
                free_slot(s);
                continue;
            }
            if (oi < min_sync) { free_slot(s); continue; }                     // :194-197
            {   // is_synchronized (:206-217): alive => ed == 0; equal logical lengths and reference positions
                const int t_rp = LDI(nb + XN_TRP), q_rp = LDI(nb + XN_QRP);
                const int tl = LDI(nb + XN_TML) + (t_rp - LDI(nb + XN_TMR)), ql = LDI(nb + XN_QML) + (q_rp - LDI(nb + XN_QMR));
                if (tl == ql && t_rp == q_rp) { min_sync = oi; af_counts = 0; af_index = oi; }
            }
            const bool is_alt = LD8(hap_alle + oi) == AL_ALT;
            // REF allele: move, id kept (:257-273).  ALT allele: (REF, error) with id next_id, then (ALT, no error)
            // with the following id unless auto-failed (:274-306).
            const bool do_alt = is_alt && !(oi < af_index);
            int s_alt = -1;
            if (do_alt) {
                s_alt = alloc_slot();
                if (s_alt < 0 && gc_queue(true, (u32)min(best_err, 0xffff), min_sync, n) > 0) s_alt = alloc_slot();
                if (s_alt < 0) return SOLVE_WORKSPACE;
                ex_clone(node(s_alt), nb);
            }
            if (is_alt) {
                __syncwarp();
                if (lane == 0) { ST32(nb + XN_ID, next_id); if (do_alt) ST32(node(s_alt) + XN_ID, next_id + 1); }
                __syncwarp();
                next_id += do_alt ? 2 : 1;
            }
            if (SMEM && team && do_alt) {                                      // both children at once
                if (lane == 0) {
                    TeamBoard &B = *team;
                    B.kind = 1; B.count = 2; B.finalize = 0; B.oi = oi;
                    B.nb[0] = (unsigned)node(s); B.alt[0] = 0; B.err[0] = is_alt;
                    B.nb[1] = (unsigned)node(s_alt); B.alt[1] = 1; B.err[1] = 0;
                }
                team_round();
            }
#pragma unroll 1
            for (int k = 0; k < (do_alt ? 2 : 1); ++k) {
                const int sl = k ? s_alt : s;
                const int keep = (SMEM && team && do_alt) ? team->rc[k] : ex_extend(node(sl), oi, k == 1, is_alt && k == 0, false);
                if (keep < 0) return keep;
                if (keep) { if (!push(ex_key(node(sl)), sl)) return SOLVE_WORKSPACE; } else free_slot(sl);
            }
            af_counts += 1;                                                    // :310-339
            if (af_counts >= 500) {
                if (af_index >= n) return AVK_ST_NO_RESULT;   // the reference would index out of bounds here
                int w = 0;
                const int cnt = qn;
#pragma unroll 1
                for (int i = 0; i < cnt; ++i) {
                    const u32 sl = LD32(qslot + 4 * i);
                    const bool set = (int)qnode_ld32(sl, XN_DEPTH) > af_index;
                    if (!set || qnode_ld8(sl, XN_HDR + af_index) == AL_REF) {
                        if (lane == 0 && w != i) { ST64(qkeys + 8 * w, LD64(qkeys + 8 * i)); ST32(qslot + 4 * w, sl); }
                        w += 1;
                    } else {
                        free_entry(sl);
                    }
                    __syncwarp();
                }
                __syncwarp();
                if (lane == 0) qn = w;
                __syncwarp();
                af_index += 1;
                af_counts = 0;
            }
        }
        if (!have_best) return AVK_ST_NO_RESULT;                               // :345-348
        *errors_out = best_err;
        return SOLVE_OK;
    }

    // ================================================================== waffle solver
    // generate_allele_sequence(): waffle_solver.rs:726-778 as a virtual sequence in buffer `k` (0 T, 1 Q, 2 F).
    // side 0 truth / 1 query, hap 0/1, alleles from result r; type_filter < 0 keeps every variant.
    // Fills sdesc[k] = {mlen, cur, failed ED, #ALT spliced}; returns 0, -1 (capacity) or -2 (variant past the window).
    // With copy == false only the description is computed; materialise(k) writes the bytes when an alignment needs them.
    //
    // ED(reference window, haplotype) is known without aligning in two cases (SD_CLOSED):
    //  (1) every spliced ALT is a single-base substitution and at most two of them differ from the reference base:
    //      the haplotype has the window's length and Hamming distance d <= 2 to it, and for equal lengths ED = 1 iff the
    //      Hamming distance is 1, so ED = d;
    //  (2) no substitution changes a base and every other spliced ALT is an anchored pure insertion (1 -> L, first base
    //      == the reference base), or every one an anchored pure deletion (L -> 1): the window is obtained from the
    //      haplotype (or the reverse) by deleting exactly D bases, D = the length difference, so D <= ED <= D.
    __device__ __noinline__ int build_hap_seq(int k, int side, int hap, int r, int type_filter, bool copy) {
        const addr dst = dyn + (u32)(k * seq_cap);
        const addr ra = res_alle + (u32)(r * Npad);
        int cur = start, mlen = 0, failed = 0, n_alt = 0;
        int subm = 0, ins = 0, del = 0;
        bool open = false;
        const int n = N;
#pragma unroll 1
        for (int oi = 0; oi < n; ++oi) {
            const addr rec = vi(oi);
            const u32 f = LD32(rec + VI_FLAGS);
            if ((int)((f >> 16) & 1) == side) continue;           // is_truth == 1 <=> side 0
            if (!((LD8(ra + oi) >> hap) & 1)) continue;           // REF allele: skipped entirely (:738-741)
            if (type_filter >= 0 && (int)(f & 0xff) != type_filter) continue;
            const int vpos = (int)LD32(rec + VI_POS);
            if (vpos < cur) { failed += (int)LD32(rec + VI_ALTED); continue; }   // :745-753
            const int l0 = (int)LD32(rec + VI_L0), l1 = (int)LD32(rec + VI_L1);
            const int nref = vpos - cur;
            if (mlen + nref + l1 > seq_cap) return -1;
            const addr a1 = alle_base + LD32(rec + VI_AOFF) + l0;
            if (copy) {
                if (nref > 0) warp_copy<SMEM>(dst + mlen, ref_base + cur, nref);
                warp_copy<SMEM>(dst + mlen + nref, a1, l1);
            }
            const bool anchored = LD8(a1) == LD8(ref_base + vpos);
            if (l0 == 1 && l1 == 1) subm += anchored ? 0 : 1;
            else if (l0 == 1 && anchored) ins += l1 - 1;
            else if (l1 == 1 && anchored) del += l0 - 1;
            else open = true;
            mlen += nref + l1;
            cur = vpos + l0;
            n_alt += 1;
        }
        if (cur > end) return -2;
        int closed = -1;
        if (!open) {
            if (ins == 0 && del == 0) { if (subm <= 2) closed = subm; }
            else if (subm == 0 && (ins == 0 || del == 0)) closed = ins + del;
        }
        __syncwarp();
        if (lane_id() == 0) {
            const addr sd = sdesc + (u32)(k * SD_SIZE);
            ST32(sd + SD_MLEN, mlen); ST32(sd + SD_CUR, cur); ST32(sd + SD_FAILED, failed); ST32(sd + SD_NALT, n_alt);
            ST32(sd + SD_CLOSED, closed); ST32(sd + SD_MAT, copy ? 1 : 0);
            ST32(sd + SD_ARGS, side | (hap << 1) | ((type_filter + 1) << 2) | (r << 8));
        }
        __syncwarp();
        return 0;
    }
    // make sure buffer k holds its bytes (no-op for the reference window, k < 0)
    __device__ __forceinline__ void materialise(int k) {
        if (k < 0) return;
        const addr sd = sdesc + (u32)(k * SD_SIZE);
        if (LDI(sd + SD_MAT)) return;
        const int a = LDI(sd + SD_ARGS);
        build_hap_seq(k, a & 1, (a >> 1) & 1, a >> 8, ((a >> 2) & 63) - 1, true);   // same walk as before: cannot fail
    }
    // virtual sequence of buffer k (k < 0: the reference window itself)
    __device__ __forceinline__ VS seq_vs(int k) const {
        VS v;
        if (k < 0) { v.data = 0; v.tail = ref_base + start; v.mlen = 0; v.len = end - start; return v; }
        const addr sd = sdesc + (u32)(k * SD_SIZE);
        const int mlen = LDI(sd + SD_MLEN), cur = LDI(sd + SD_CUR);
        v.data = dyn + (u32)(k * seq_cap); v.tail = ref_base + cur; v.mlen = mlen; v.len = mlen + (end - cur);
        return v;
    }
    // ED(reference window, buffer k): closed form when build_hap_seq found one, otherwise a global alignment
    __device__ __forceinline__ u64 ed_to_ref(int k) {
        const int closed = LDI(sdesc + (u32)(k * SD_SIZE) + SD_CLOSED);
        if (closed >= 0) {
            __syncwarp();
            if (lane_id() == 0) {
                ST32(wk() + WK_ALIGN, LD32(wk() + WK_ALIGN) + 1);
                ST64(wk() + WK_CELLS, LD64(wk() + WK_CELLS) + 1);
            }
            return (u64)closed;
        }
        return ed_between(-1, k);
    }
    // global edit distance between two sequence buffers, with overflow trap
    __device__ __noinline__ u64 ed_between(int ka, int kb) {
        materialise(ka); materialise(kb);
        const int e = wfa_ed_warp<SMEM>(seq_vs(ka), seq_vs(kb), dyn + (u32)(3 * seq_cap), (wf_cap - 3) / 2, wk());
        if (e < 0) { SOLVER_WRITE(ed_overflow = 1); return 0; }
        return (u64)e;
    }
    // copy a sequence buffer to the optional sequence-bundle output
    __device__ __noinline__ void emit_seq(const DevCompareOut &out, u64 r, int s, int k) {
        materialise(k);
        const VS v = seq_vs(k);
        u8 *dst = out.seq_pool + out.seq_off[r * 5 + s];
#pragma unroll 1
        for (int i = lane_id(); i < v.len; i += 32) dst[i] = LD8(v.at(i));
        if (lane_id() == 0) out.seq_len[r * 5 + s] = (u32)v.len;
    }

    // GroupMetrics::add_truth_zygosity (grouped_metrics.rs:183-227) on row g; col 0 = truth columns, 2 = query
    // columns (the query pass lands in the query columns through add_swap_benchmark, :268-277).  lane 0 only.
    __device__ __noinline__ void gm_add(addr g, int col, u64 w, int exp, int obs) {
        const int mn = min(exp, obs);
        ST64(g + 8 * (AVK_M_HAP + col), LD64(g + 8 * (AVK_M_HAP + col)) + (u64)mn);
        ST64(g + 8 * (AVK_M_WEIGHTED_HAP + col), LD64(g + 8 * (AVK_M_WEIGHTED_HAP + col)) + (u64)mn * w);
        if (exp == obs) {
            ST64(g + 8 * (AVK_M_GT + col), LD64(g + 8 * (AVK_M_GT + col)) + 1);
        } else {
            ST64(g + 8 * (AVK_M_HAP + col + 1), LD64(g + 8 * (AVK_M_HAP + col + 1)) + (u64)(exp - obs));
            ST64(g + 8 * (AVK_M_WEIGHTED_HAP + col + 1), LD64(g + 8 * (AVK_M_WEIGHTED_HAP + col + 1)) + (u64)(exp - obs) * w);
            ST64(g + 8 * (AVK_M_GT + col + 1), LD64(g + 8 * (AVK_M_GT + col + 1)) + 1);
            const int gt = (col == 0) ? AVK_M_GT_TRUTH_FN_GT : AVK_M_GT_QUERY_FP_GT;
            if (obs > 0) ST64(g + 8 * gt, LD64(g + 8 * gt) + 1);
        }
    }
    __device__ __forceinline__ void add4(addr g, u64 a, u64 b2, u64 c, u64 d) {   // lane 0 only
        ST64(g, LD64(g) + a); ST64(g + 8, LD64(g + 8) + b2); ST64(g + 16, LD64(g + 16) + c); ST64(g + 24, LD64(g + 24) + d);
    }

    // Merge shortcut: inputs i and j of cluster r carry the same variants (position, both alleles) with the same number
    // of ALT copies each, no two of them overlap, and the search tree (2 orientations per heterozygous variant, both
    // lists) cannot reach the branch quota.  Then optimize_sequences explores every orientation pair, the pair that
    // assigns each query variant to its truth twin's haplotype spells identical sequences without a skipped variant,
    // and the minimum cost is 0: is_exact_match() (query_optimizer.rs:96-98) holds without running the search.
    __device__ __noinline__ bool merge_pair_identical(u64 r, u32 i, u32 j) {
        const DevBatch &b = *bp;
        const u32 K = b.n_inputs;
        const u64 vi0 = b.var_off[r * K + i], vj0 = b.var_off[r * K + j];
        const int ni = (int)(b.var_off[r * K + i + 1] - vi0), nj = (int)(b.var_off[r * K + j + 1] - vj0);
        if (ni != nj) return false;
        bool ok = true;
        int hets = 0;
#pragma unroll 1
        for (int k = lane_id(); k < ni; k += 32) {
            const u64 gi = vi0 + k, gj = vj0 + k;
            const u32 l0 = b.l0[gi], l1 = b.l1[gi];
            const int zi = b.zyg[gi], zj = b.zyg[gj];
            const int ci = zi == AVK_ZYG_HOM_ALT ? 2 : (zi >= AVK_ZYG_UNPHASED_HET ? 1 : 0);
            const int cj = zj == AVK_ZYG_HOM_ALT ? 2 : (zj >= AVK_ZYG_UNPHASED_HET ? 1 : 0);
            ok = ok && b.pos[gi] == b.pos[gj] && l0 == b.l0[gj] && l1 == b.l1[gj] && l0 + l1 <= 64 && ci == cj && ci > 0;
            if (k > 0) ok = ok && b.pos[gi] >= b.pos[gi - 1] + b.l0[gi - 1];
            if (ok) {
                const u8 *pa = b.pool + b.aoff[gi], *pb = b.pool + b.aoff[gj];
#pragma unroll 1
                for (u32 t = 0; t < l0 + l1; ++t) ok = ok && pa[t] == pb[t];
            }
            hets += ci == 1 ? 1 : 0;
        }
        ok = __all_sync(AVK_FULL, ok);
        hets = __reduce_add_sync(AVK_FULL, hets);
        return ok && hets <= 12 && (1 << (2 * hets)) <= mbf;
    }

    __device__ int solve_compare(u64 r, const avk_compare_cfg &cfg, const DevCompareOut &out);
    __device__ int compare_prepare(u64 r, const avk_compare_cfg &cfg, bool want_metrics);
    __device__ int compare_search_to_blob(u64 r, const avk_compare_cfg &cfg, u8 *blob);
    __device__ int compare_score_from_blob(u64 r, const avk_compare_cfg &cfg, const DevCompareOut &out, const u8 *blob);
    __device__ int compare_score_from_dense(u64 r, const avk_compare_cfg &cfg, const DevCompareOut &out, const u8 *blob);
    __device__ int compare_score(u64 r, const avk_compare_cfg &cfg, const DevCompareOut &out);
    __device__ int merge_front(u64 r, const avk_merge_cfg &cfg, const struct MergeWork &w);
    __device__ int merge_pair(u64 r, u32 i, u32 j, const avk_merge_cfg &cfg, bool *exact);
    __device__ int merge_classify(u64 r, const avk_merge_cfg &cfg, const DevMergeOut &out, const struct MergeWork &w);
};

// Hand-off record between the search kernel and the score kernel of the common tier (N <= 16, <= 8 results).
enum { RB_NRES = 0, RB_ALLE = 16, RB_NUM = 16 + 8 * 16, RB_SIZE = 16 + 8 * 16 + 8 * 24 };
enum { RB_FUSED = -1, RB_DONE = -2 };   // n_res values: handled by a fused tier / already final (error status written)

// Loads region r and lays out the arena (first half of solve_compare_region, waffle_solver.rs:122-148).
template <bool SMEM>
__device__ int RegionSolver<SMEM>::compare_prepare(u64 r, const avk_compare_cfg &cfg, bool want_metrics) {
    const DevBatch &b = *bp;
    const u32 c = b.contig[r];
    SOLVER_WRITE(start = (int)b.start[r]; end = (int)b.end[r]; mbf = (int)cfg.max_branch_factor);
    if (c >= b.n_contigs || b.start[r] > b.end[r] || (u64)b.end[r] > b.contig_len[c] || b.end[r] > 0x7fff0000u) return AVK_ST_BAD_INPUT;
    if (mbf <= 0) return AVK_ST_BAD_INPUT;
    return load_cluster(r, b.contig_ptr[c], want_metrics);
}

// Search phase -> result blob (split tier).  Returns SOLVE_OK with the blob filled, or a status.
template <bool SMEM>
__device__ int RegionSolver<SMEM>::compare_search_to_blob(u64 r, const avk_compare_cfg &cfg, u8 *blob) {
    int rc = compare_prepare(r, cfg, false);
    if (rc) return rc;
    if (N > 16) return SOLVE_WORKSPACE;
    rc = optimize(false);
    if (rc) return rc;
    const int lane = lane_id();
    const int nres = n_res;
#pragma unroll 1
    for (int i = lane; i < nres * 16; i += 32) blob[RB_ALLE + i] = LD8(res_alle + (u32)((i >> 4) * Npad + (i & 15)));
#pragma unroll 1
    for (int i = lane; i < nres * 6; i += 32) ((int *)(blob + RB_NUM))[i] = LDI(res_num + 4 * i);
    if (lane == 0) *(int *)(blob + RB_NRES) = nres;
    return SOLVE_OK;
}

// Score phase from a result blob (split tier).
template <bool SMEM>
__device__ int RegionSolver<SMEM>::compare_score_from_blob(u64 r, const avk_compare_cfg &cfg, const DevCompareOut &out, const u8 *blob) {
    int rc = compare_prepare(r, cfg, true);
    if (rc) return rc;
    const int lane = lane_id();
    const int nres = *(const int *)(blob + RB_NRES);
    if (nres > res_cap) return SOLVE_WORKSPACE;
#pragma unroll 1
    for (int i = lane; i < nres * 16; i += 32) ST8(res_alle + (u32)((i >> 4) * Npad + (i & 15)), blob[RB_ALLE + i]);
#pragma unroll 1
    for (int i = lane; i < nres * 6; i += 32) ST32(res_num + 4 * i, ((const int *)(blob + RB_NUM))[i]);
    SOLVER_WRITE(n_res = nres);
    return compare_score(r, cfg, out);
}

// Score phase from the speculative dense search's blob (avk_spec_search.cuh: SPB_* layout): the equal-best results, or -- when
// the blob says `scored` -- the one chosen solution with its exact-GT alleles, in which case compare_score goes straight to
// the metrics.
template <bool SMEM>
__device__ int RegionSolver<SMEM>::compare_score_from_dense(u64 r, const avk_compare_cfg &cfg, const DevCompareOut &out, const u8 *blob) {
    int rc = compare_prepare(r, cfg, true);
    if (rc) return rc;
    const int lane = lane_id();
    const int nres = *(const int *)(blob + avk_sp::SPB_NRES);
    if (nres > res_cap || N > avk_sp::SP_MAXN) return SOLVE_WORKSPACE;
    const int n = N, npad = Npad;
#pragma unroll 1
    for (int i = lane; i < nres * n; i += 32) { const int ri = i / n, oi = i - ri * n; ST8(res_alle + (u32)(ri * npad + oi), blob[avk_sp::SPB_RES + ri * avk_sp::SPB_RES_STRIDE + oi]); }
#pragma unroll 1
    for (int i = lane; i < nres * 6; i += 32) { const int ri = i / 6, k = i - ri * 6; ST32(res_num + (u32)(ri * 24 + 4 * k), ((const int *)(blob + avk_sp::SPB_RES + ri * avk_sp::SPB_RES_STRIDE + avk_sp::SPB_ALLE))[k]); }
    SOLVER_WRITE(n_res = nres; pre_scored = *(const int *)(blob + avk_sp::SPB_SCORED); pre_keep[0] = *(const u32 *)(blob + avk_sp::SPB_KEEP0); pre_keep[1] = *(const u32 *)(blob + avk_sp::SPB_KEEP1));
    rc = compare_score(r, cfg, out);
    SOLVER_WRITE(pre_scored = 0);
    return rc;
}

// solve_compare_region(): returns AVK_ST_* (>= 0) or SOLVE_WORKSPACE
template <bool SMEM>
__device__ int RegionSolver<SMEM>::solve_compare(u64 r, const avk_compare_cfg &cfg, const DevCompareOut &out) {
    int rc = compare_prepare(r, cfg, true);
    if (rc) return rc;
    rc = optimize(false);
    if (rc) return rc;
    return compare_score(r, cfg, out);
}

// Second half of solve_compare_region (waffle_solver.rs:168-284): the equal-best results are in res_alle/res_num.
template <bool SMEM>
__device__ __noinline__ int RegionSolver<SMEM>::compare_score(u64 r, const avk_compare_cfg &cfg, const DevCompareOut &out) {
    const int lane = lane_id();
    const int n = N, npad = Npad;
    int rc;

    int best_r = 0;
    bool shortcut = false;
    if (cfg.enable_exact_shortcut) {                                       // :171
        int s = 0;
#pragma unroll 1
        for (int k = 0; k < 6; ++k) s += LDI(res_num + 4 * k);
        shortcut = s == 0;
    }
    if (!shortcut && pre_scored) {                                          // scored by the speculative dense search: result 0 with these alleles
#pragma unroll 1
        for (int i = lane; i < 2 * n; i += 32) { const int h = i >= n ? 1 : 0, oi = i - h * n; ST8(best_obs + (u32)(h * npad + oi), ((pre_keep[h] >> oi) & 1u) ? AL_ALT : AL_REF); }
        __syncwarp();
    } else if (!shortcut) {
        // ---- exact-GT scoring of every equal-best solution; first minimum wins (:169-265).
        // A haplotype with ED 0 and nothing skipped scores 0 errors: the zero-flip path of optimize_gt_alleles replays
        // exactly the optimizer's tracker steps, stays alive, is popped first (fewest errors, most set alleles) and
        // finalises with 0 errors, after which every other node is pruned (exact_gt_optimizer.rs:169).  Any other
        // haplotype scores at least 1: its zero-flip path ends in unequal sequences or a skipped variant.  Only a
        // strictly smaller total replaces the current first minimum, so a solution whose lower bound already reaches
        // it is not searched at all, and a search stops once it has used up what is left of the budget.
        // A solution with both haplotypes at 0 totals 0, which nothing later can beat and nothing earlier (>= 1) reaches:
        // the first such solution is the answer and no search is needed at all.
        // "Nothing skipped" is read off the skipped variants' summed edit distance, which says nothing about a skipped variant
        // whose ALT equals its REF (distance 0): in a cluster that holds such a record the zero-flip shortcuts are off (an
        // incompatible no-op ALT cannot be kept, optimize_gt_alleles drops that child: exact_gt_optimizer.rs:293-305) and only
        // the lower bound "ED or skip distance > 0 costs at least one flip" is used.
        bool noop = false;
#pragma unroll 1
        for (int oi = lane; oi < n; oi += 32) noop = noop || LD32(vi(oi) + VI_ALTED) == 0u;
        noop = __any_sync(AVK_FULL, noop);
        int best_total = 0x7fffffff;
        int lo = 0, hi = n_res;
#pragma unroll 1
        for (int ri = 0; ri < n_res && !noop; ++ri) {
            int sum = 0;
#pragma unroll 1
            for (int k = 0; k < 6; ++k) sum += LDI(res_num + (u32)(ri * 24 + 4 * k));
            if (sum == 0) { lo = ri; hi = ri + 1; break; }
        }
#pragma unroll 1
        for (int ri = lo; ri < hi; ++ri) {
            const addr ra = res_alle + (u32)(ri * npad);
            const addr rnum = res_num + (u32)(ri * 24);
            const int lb0 = LDI(rnum) + LDI(rnum + 8) + LDI(rnum + 16) == 0 ? 0 : 1;       // flips this haplotype costs at least
            const int lb1 = LDI(rnum + 4) + LDI(rnum + 12) + LDI(rnum + 20) == 0 ? 0 : 1;
            const bool zero0 = lb0 == 0 && !noop, zero1 = lb1 == 0 && !noop;                // ... and known to cost exactly none
            if (lb0 + lb1 >= best_total) continue;
            int total = 0;
            bool lost = false;
#pragma unroll 1
            for (int h = 0; h < 2 && !lost; ++h) {
#pragma unroll 1
                for (int i = lane; i < n; i += 32) ST8(hap_alle + i, ((LD8(ra + i) >> h) & 1) ? AL_ALT : AL_REF);
                __syncwarp();
                int errs = 0;
                if (h ? zero1 : zero0) {
                    warp_copy<SMEM>(cur_obs + (u32)(h * npad), hap_alle, n);
                    __syncwarp();
                } else {
                    const int budget = best_total - total - (h == 0 ? lb1 : 0);
                    rc = exact_gt(cur_obs + (u32)(h * npad), &errs, budget, cfg.exact_gt_max_expansions ? cfg.exact_gt_max_expansions : AVK_EXACT_GT_DEFAULT_MAX_EXPANSIONS);
                    if (rc) return rc;
                    lost = errs >= budget;
                }
                total += errs;
            }
            if (!lost && total < best_total) {
                best_total = total;
                best_r = ri;
                warp_copy<SMEM>(best_obs, cur_obs, 2 * npad);
                __syncwarp();
            }
        }
    }
    const addr ra = res_alle + (u32)(best_r * npad);
    const addr rnb = res_num + (u32)(best_r * 24);
    const addr gm = mrows;   // joint row; type rows follow at gm + 176 * (1 + slot)

    // ---- per-variant expected/observed (:226-258); lanes across variants
#pragma unroll 1
    for (int oi = lane; oi < n; oi += 32) {
        const u32 f = LD32(vi(oi) + VI_FLAGS);
        const bool is_truth = (f & 0x10000u) != 0;
        int exp_, obs_;
        if (shortcut) {   // generate_exact_match(): counts come from the RAW zygosities (:544-557)
            exp_ = (((f >> 8) & 0xff) == AVK_ZYG_HOM_ALT) ? 2 : 1;
            obs_ = exp_;
        } else {
            const int a = LD8(ra + oi);
            exp_ = (a & 1) + ((a >> 1) & 1);
            obs_ = (LD8(best_obs + oi) == AL_ALT ? 1 : 0) + (LD8(best_obs + npad + oi) == AL_ALT ? 1 : 0);
        }
        const int cls = (exp_ == obs_) ? AVK_CLASS_TP : (is_truth ? AVK_CLASS_FN : AVK_CLASS_FP);
        const u32 gv = LD32(vi(oi) + VI_GV);
        out.vexp[gv] = (u8)(is_truth ? exp_ : obs_);     // query entries are toggled (compare_benchmark.rs:109-123)
        out.vobs[gv] = (u8)(is_truth ? obs_ : exp_);
        out.vcls[gv] = (u8)cls;
        ST8(hap_alle + oi, exp_ | (obs_ << 4));          // scratch for the metric pass below
    }
    __syncwarp();
    // ---- GT / HAP / WEIGHTED_HAP (+ add_swap_benchmark :269) and RECORD_BP totals, accumulated by lane 0
    __syncwarp();
    if (lane == 0) {
#pragma unroll 1
        for (int oi = 0; oi < n; ++oi) {
            const addr rec = vi(oi);
            const u32 f = LD32(rec + VI_FLAGS);
            const int exp_ = LD8(hap_alle + oi) & 15, obs_ = LD8(hap_alle + oi) >> 4;
            const int side = (f & 0x10000u) ? 0 : 1, slot = (int)(f >> 24);
            const u64 w = LD32(rec + VI_ALTED);
            gm_add(gm, 2 * side, w, exp_, obs_);
            gm_add(gm + (u32)(8 * AVK_N_METRICS * (1 + slot)), 2 * side, w, exp_, obs_);
            const addr cnt = slot_cnt + (u32)(4 * (2 * slot + side));
            ST32(cnt, LD32(cnt) + 1);
            const addr tot = slot_tot + (u32)(8 * (2 * slot + side));
            ST64(tot, LD64(tot) + (u64)((((f >> 8) & 0xff) == AVK_ZYG_HOM_ALT) ? 2 : 1) * LD32(rec + VI_RAW));
        }
    }
    __syncwarp();

    // ---- basepair metrics: three sequence buffers + one wavefront in the dynamic part
    if ((u32)(3 * seq_cap + 4 * wf_cap + 16) > dyn_bytes) return SOLVE_WORKSPACE;
    const bool want_seq = out.seq_off && cfg.enable_sequences;
    SOLVER_WRITE(ed_overflow = 0);
    u32 mask = 0;
#pragma unroll 1
    for (int k = 0; k < n_slots; ++k) mask |= 1u << slot_type[k];

    int status = AVK_ST_OK;
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {
        const int rsel = shortcut ? 0 : best_r;
        // truth / query haplotypes (buffers 0 / 1)
#pragma unroll 1
        for (int side = 0; side < 2; ++side) {
            const int brc = build_hap_seq(side, side, h, rsel, -1, false);
            if (brc) return brc == -1 ? SOLVE_WORKSPACE : AVK_ST_BAD_INPUT;
            if (want_seq) emit_seq(out, r, 1 + 2 * side + h, side);
        }
        const int altT = LDI(sdesc + SD_NALT), altQ = LDI(sdesc + SD_SIZE + SD_NALT);
        const u64 failT = (u64)LDI(sdesc + SD_FAILED), failQ = (u64)LDI(sdesc + SD_SIZE + SD_FAILED);
        // X = ED(ref, truth), Y = ED(ref, query), Z = ED(truth, query).  A haplotype without a spliced ALT IS the
        // reference window; Z is the optimizer's finalised (exact Levenshtein) distance of this haplotype pair.
        const u64 X = altT ? ed_to_ref(0) : 0;
        if (shortcut) {   // generate_exact_match(): :559-598 -- joint gets 2 * ED(ref, truth) on both sides
            if (lane == 0) add4(gm + 8 * AVK_M_BASEPAIR, 2 * X, 0, 2 * X, 0);
            continue;
        }
        const u64 Z = (u64)LDI(rnb + 4 * h);
        const u64 Y = (Z == 0) ? X : (altQ ? ed_to_ref(1) : 0);
        const u64 tp = X + Y - Z;                    // (2X + 2Y - 2Z) / 2  :644
        if (lane == 0) add4(gm + 8 * AVK_M_BASEPAIR, tp, 2 * X - tp + 2 * failT, tp, 2 * Y - tp + 2 * failQ);
        // per supported type that occurs in the cluster (absent types only ever receive zeros, :395-444)
#pragma unroll 1
        for (int k = 0; k < n_slots; ++k) {
            const int ft = slot_type[k];
            if (!type_supported(ft)) continue;
#pragma unroll 1
            for (int side = 1; side >= 0; --side) {   // query filter (:395-410) then truth filter (:422-437)
                const int nf = (int)LD32(slot_cnt + (u32)(4 * (2 * k + side)));
                if (nf == 0) continue;
                u64 f_tp, f_bad;
                if (nf == nv[side]) {                 // filtered == full haplotype
                    f_tp = tp; f_bad = side ? (2 * Y - tp + 2 * failQ) : (2 * X - tp + 2 * failT);
                } else {
                    const int brc = build_hap_seq(2, side, h, best_r, ft, false);
                    if (brc) return brc == -1 ? SOLVE_WORKSPACE : AVK_ST_BAD_INPUT;
                    const bool altF = LDI(sdesc + 2 * SD_SIZE + SD_NALT) != 0;
                    const u64 failF = (u64)LDI(sdesc + 2 * SD_SIZE + SD_FAILED);
                    // side 1: (ref, truth, F): Xa = X, Yf = ED(ref, F), Zf = ED(truth, F); side 0 mirrored
                    const u64 other_ref = side ? X : Y;          // ED(ref, unfiltered other haplotype)
                    const bool alt_other = side ? (altT != 0) : (altQ != 0);
                    u64 Ef = 0, Zf = other_ref;
                    if (altF) {
                        Ef = ed_to_ref(2);
                        Zf = alt_other ? (side ? ed_between(0, 2) : ed_between(2, 1)) : Ef;
                    }
                    f_tp = other_ref + Ef - Zf;
                    f_bad = 2 * Ef - f_tp + 2 * failF;
                }
                __syncwarp();
                if (lane == 0) {
                    const addr g = gm + (u32)(8 * (AVK_N_METRICS * (1 + k) + AVK_M_BASEPAIR + 2 * side));
                    ST64(g, LD64(g) + f_tp); ST64(g + 8, LD64(g + 8) + f_bad);
                }
            }
        }
    }
    __syncwarp();
    if (shortcut) {
        // generate_exact_match(): per-variant basepair credit (:573-598); no RECORD_BP, no all-8-types fill
        __syncwarp();
        if (lane == 0) {
#pragma unroll 1
            for (int oi = 0; oi < n; ++oi) {
                const addr rec = vi(oi);
                const u32 f = LD32(rec + VI_FLAGS);
                const u64 dd = 2ull * LD32(rec + VI_ALTED) * (u64)((((f >> 8) & 0xff) == AVK_ZYG_HOM_ALT) ? 2 : 1);
                const addr g = gm + (u32)(8 * (AVK_N_METRICS * (1 + (f >> 24)) + AVK_M_BASEPAIR + ((f & 0x10000u) ? 0 : 2)));
                ST64(g, LD64(g) + dd);
            }
        }
    } else {
        // every supported type gets a (possibly all-zero) entry (:444)
        mask |= (1u << AVK_VT_SNV) | (1u << AVK_VT_INSERTION) | (1u << AVK_VT_DELETION) | (1u << AVK_VT_INDEL) |
                (1u << AVK_VT_TR_CONTRACTION) | (1u << AVK_VT_TR_EXPANSION) | (1u << AVK_VT_SV_DELETION) | (1u << AVK_VT_SV_INSERTION);
        // add_record_basepair_stats(): :455-522 (wrapping u64 like a release build).  Types without variants have
        // zero totals and zero basepair counts, so their record rows stay zero.
        __syncwarp();
        if (lane == 0) {
            u64 truth_total = 0, query_total = 0;
#pragma unroll 1
            for (int k = 0; k < n_slots; ++k) { truth_total += LD64(slot_tot + 16 * k); query_total += LD64(slot_tot + 16 * k + 8); }
            const addr bp_ = gm + 8 * AVK_M_BASEPAIR;
            const u64 tfn = LD64(bp_ + 8), qfp = LD64(bp_ + 24);
            const u64 ttp = 2 * truth_total - tfn, qtp = 2 * query_total - qfp;
            if (!(ttp >= LD64(bp_)) || !(qtp >= LD64(bp_ + 16))) status = AVK_ST_TP_UNDERFLOW;
            else {
                add4(gm + 8 * AVK_M_RECORD_BP, ttp, tfn, qtp, qfp);
#pragma unroll 1
                for (int k = 0; k < n_slots; ++k) {
                    const addr g = gm + (u32)(8 * AVK_N_METRICS * (1 + k));
                    const u64 fn_ = LD64(g + 8 * (AVK_M_BASEPAIR + 1)), fp_ = LD64(g + 8 * (AVK_M_BASEPAIR + 3));
                    add4(g + 8 * AVK_M_RECORD_BP, 2 * LD64(slot_tot + 16 * k) - fn_, fn_, 2 * LD64(slot_tot + 16 * k + 8) - fp_, fp_);
                }
            }
        }
        status = __shfl_sync(AVK_FULL, status, 0);
    }
    if (ed_overflow) return SOLVE_WORKSPACE;
    if (status != AVK_ST_OK) return status;
    __syncwarp();
    // ---- summary counters of this region straight into this CTA's partial table (only the non-zero entries)
    if (out.tot_slots) {
        unsigned long long *slot = out.tot_slots + (size_t)(blockIdx.x & (TOT_SLOTS - 1)) * TOT_STRIDE;
#pragma unroll 1
        for (int i = lane; i < AVK_N_METRICS * (1 + n_slots); i += 32) {
            const u64 v = LD64(gm + 8 * i);
            if (v) {
                const int k = i / AVK_N_METRICS, m = i - k * AVK_N_METRICS;
                const int col = (k == 0 ? 0 : (1 + slot_type[k - 1]) * AVK_N_METRICS) + m;
                atomicAdd(slot + col, (unsigned long long)v);
                if (out.strata) out.strata->add(r, col, (unsigned long long)v);
            }
        }
        if (lane == 0) { atomicOr(slot + TOT_MASK, (unsigned long long)mask); atomicAdd(slot + TOT_SOLVED, 1ull); }
    }
    // ---- write the full GroupTypeMetrics row [13][22] (coalesced), zeros for absent types
    if (out.region_metrics) {
        u64 *dst = out.region_metrics + r * (u64)(AVK_N_GROUPS * AVK_N_METRICS);
        // type -> slot lookup in a register: 4 bits per type, 15 = absent
        u64 lut = ~0ull;
#pragma unroll 1
        for (int k = 0; k < n_slots; ++k) lut = (lut & ~(15ull << (4 * slot_type[k]))) | ((u64)k << (4 * slot_type[k]));
#pragma unroll 1
        for (int i = lane; i < AVK_N_GROUPS * AVK_N_METRICS; i += 32) {
            const int g = i / AVK_N_METRICS, m = i - g * AVK_N_METRICS;
            u64 v = 0;
            if (g == 0) v = LD64(gm + 8 * m);
            else {
                const int k = (int)((lut >> (4 * (g - 1))) & 15);
                if (k != 15) v = LD64(gm + (u32)(8 * (AVK_N_METRICS * (1 + k) + m)));
            }
            dst[i] = v;
        }
    }
    if (want_seq) emit_seq(out, r, 0, -1);
    __syncwarp();
    if (lane == 0) {
        out.ed1[r] = shortcut ? 0u : (u32)LDI(rnb);
        out.ed2[r] = shortcut ? 0u : (u32)LDI(rnb + 4);
        out.type_mask[r] = (uint16_t)mask;
    }
    return AVK_ST_OK;
}

// solve_merge_region(): merge_solver.rs:110-200, split in three so that the K(K-1)/2 pair searches of a cluster -- which are
// independent -- become separate work items (a dense 5-input cluster is ten searches of ~1 ms each):
//   merge_front    per cluster: validation, variant_delta_length prefilter (:211-223), identical-lists shortcut; the pairs
//                  that need a search are appended to a task list, the others are decided here;
//   merge_pair     per task: optimize_sequences on (v_i as truth, v_j as query), is_exact_match() of the result (:135-143);
//   merge_classify per cluster: match_sets -> classification (:152-197).
// `rows[r*K + i]` is match_sets[i] as a bit mask; `pair_err[r]` keeps the error of the FIRST failing pair in the
// reference's loop order, (pair index << 8) | status, like the `?` in the sequential loop.
struct MergeWork {
    u32 *rows;        // [n][K]
    u32 *pair_err;    // [n], 0xffffffff = none
    u64 *tasks;       // (r << 16) | (i << 8) | j
    u32 *task_ctr;
};

template <bool SMEM>
__device__ int RegionSolver<SMEM>::merge_front(u64 r, const avk_merge_cfg &cfg, const MergeWork &w) {
    const DevBatch &b = *bp;
    const int lane = lane_id();
    const u32 K = b.n_inputs;
    const u32 c = b.contig[r];
    SOLVER_WRITE(start = (int)b.start[r]; end = (int)b.end[r]; mbf = (int)cfg.max_branch_factor);
    if (c >= b.n_contigs || b.start[r] > b.end[r] || (u64)b.end[r] > b.contig_len[c] || b.end[r] > 0x7fff0000u) return AVK_ST_BAD_INPUT;
    if (mbf <= 0 || K > 32) return AVK_ST_BAD_INPUT;
    {
        bool invalid = false;
        int sums[4] = {0, 0, 0, 0};
#pragma unroll 1
        for (u32 k = 0; k < K; ++k) {
            const u64 v0 = b.var_off[r * K + k];
            invalid = validate_list(v0, (int)(b.var_off[r * K + k + 1] - v0), sums) || invalid;
        }
        if (__any_sync(AVK_FULL, invalid)) return AVK_ST_BAD_INPUT;
    }
    // variant_delta_length(): :211-223, lane k holds input k
    long long delta = 0;
    bool unknown = false;
    if ((u32)lane < K) {
#pragma unroll 1
        for (u64 gv = b.var_off[r * K + lane]; gv < b.var_off[r * K + lane + 1]; ++gv) {
            const int z = b.zyg[gv];
            unknown = unknown || z == AVK_ZYG_UNKNOWN;
            const long long cnt = (z == AVK_ZYG_HOM_ALT) ? 2 : ((z == AVK_ZYG_UNPHASED_HET || z == AVK_ZYG_PHASED_HET01 || z == AVK_ZYG_PHASED_HET10) ? 1 : 0);
            delta += ((long long)b.l1[gv] - (long long)b.l0[gv]) * cnt;
        }
    }
    if (__any_sync(AVK_FULL, unknown)) return AVK_ST_BAD_ZYGOSITY;
    u32 match_row = ((u32)lane < K) ? (1u << lane) : 0;   // lane i holds match_sets[i] as a bit mask
#pragma unroll 1
    for (u32 i = 0; i < K; ++i) {
#pragma unroll 1
        for (u32 j = i + 1; j < K; ++j) {
            const long long di = __shfl_sync(AVK_FULL, delta, i), dj = __shfl_sync(AVK_FULL, delta, j);
            if (di != dj) continue;                                      // :135: different total length change, no search
            if (merge_pair_identical(r, i, j)) {
                if ((u32)lane == i) match_row |= 1u << j;
                if ((u32)lane == j) match_row |= 1u << i;
            } else if (lane == 0) {
                w.tasks[atomicAdd(w.task_ctr, 1u)] = (r << 16) | ((u64)i << 8) | j;
            }
        }
    }
    if ((u32)lane < K) w.rows[r * K + lane] = match_row;
    if (lane == 0) w.pair_err[r] = 0xffffffffu;
    return AVK_ST_OK;
}

// one pair search; *exact is meaningful when AVK_ST_OK is returned
template <bool SMEM>
__device__ int RegionSolver<SMEM>::merge_pair(u64 r, u32 i, u32 j, const avk_merge_cfg &cfg, bool *exact) {
    const DevBatch &b = *bp;
    const u32 c = b.contig[r];
    SOLVER_WRITE(start = (int)b.start[r]; end = (int)b.end[r]; mbf = (int)cfg.max_branch_factor);
    *exact = false;
    if (!begin_region(b.contig_ptr[c])) return SOLVE_WORKSPACE;
    int rc = setup_pair(r, i, j, false);
    if (rc) { drain_window(); return rc; }
    rc = optimize(true);
    if (rc) return rc;
    if (n_res > 0) {
        int s = 0;
#pragma unroll 1
        for (int k = 0; k < 6; ++k) s += LDI(res_num + 4 * k);
        *exact = s == 0;
    }
    return AVK_ST_OK;
}

// classification from the match sets (lanes = inputs); status of the cluster is returned
template <bool SMEM>
__device__ int RegionSolver<SMEM>::merge_classify(u64 r, const avk_merge_cfg &cfg, const DevMergeOut &out, const MergeWork &w) {
    const DevBatch &b = *bp;
    const int lane = lane_id();
    const u32 K = b.n_inputs;
    const u32 perr = w.pair_err[r];
    if (perr != 0xffffffffu) return (int)(perr & 0xffu);
    const u32 match_row = ((u32)lane < K) ? w.rows[r * K + lane] : 0;
    const u32 full = K >= 32 ? 0xffffffffu : ((1u << K) - 1u);
    const bool empty = (u32)lane < K && b.var_off[r * K + lane + 1] == b.var_off[r * K + lane];
    const u32 empty_mask = __ballot_sync(AVK_FULL, empty);
    const bool all_identical = __all_sync(AVK_FULL, (u32)lane >= K || match_row == full);
    // no_conflict: every pair (i, j) has empty_i || empty_j || exact (:155-157)
    const bool row_ok = (u32)lane >= K || empty || ((match_row | empty_mask) & full) == full;
    const bool no_conflict = __all_sync(AVK_FULL, row_ok);
    const u32 maj = K / 2 + 1;                                            // :167
    const unsigned has = __ballot_sync(AVK_FULL, (u32)lane < K && (u32)__popc(match_row) >= maj);
    u32 first_maj = 0;
    if (has) first_maj = __shfl_sync(AVK_FULL, match_row, __ffs(has) - 1);
    int cls;
    u32 idx_mask = 0;
    int sel = -1;
    if (all_identical) cls = AVK_MERGE_BASEPAIR_IDENTICAL;               // :174-197
    else if (cfg.no_conflict_enabled && no_conflict) { cls = AVK_MERGE_NO_CONFLICT; idx_mask = full & ~empty_mask; }
    else if (cfg.majority_voting_enabled && first_maj != 0) { cls = AVK_MERGE_MAJORITY_AGREE; idx_mask = first_maj; }
    else if (cfg.conflict_selection >= 0) { cls = AVK_MERGE_CONFLICT_SELECTION; sel = cfg.conflict_selection; }
    else cls = AVK_MERGE_DIFFERENT;
    __syncwarp();
    if (lane == 0) {
        out.cls[r] = (u8)cls;
        int n = 0;
        if (sel >= 0) { out.idx[r * K + 0] = (u8)sel; n = 1; }
        else for (u32 k = 0; k < K; ++k) if (idx_mask & (1u << k)) out.idx[r * K + (n++)] = (u8)k;
        for (u32 k = n; k < K; ++k) out.idx[r * K + k] = 0xFF;
        out.n_idx[r] = (u8)n;
    }
    return AVK_ST_OK;
}

}  // namespace avk
