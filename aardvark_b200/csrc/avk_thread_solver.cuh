// avk_thread_solver.cuh -- solve_compare_region for ONE cluster by ONE thread, written as a coroutine.
//
// The warp solvers of avk_solver.cuh put a whole warp on one cluster; for the common small cluster (a handful of
// variants, windows of a few hundred bases, edit distances of a few units) most of what such a warp executes is
// warp-uniform scalar bookkeeping replicated on 32 lanes.  Here a cluster belongs to one thread -- 32 clusters per
// warp -- and the search is restated so that a thread needs next to no memory (< 900 bytes of shared memory):
//
//   * A search node is NOT stored.  DWFALite is path independent (after every update the state equals the state of
//     one from-scratch update on the current sequences: increase_edit_distance only fires while no diagonal touches
//     an end, dynamic_wfa.rs:77), and a haplotype sequence is a pure function of the alleles assigned so far.  A queued
//     node is therefore 12 bytes: (cost, id) key, the two allele bit masks, depth and the two edit distances.  A popped
//     node rebuilds its trackers by replaying its alleles (HaplotypeTracker, haplotype_dwfa.rs:175-227) and its
//     wavefront is known in closed form when its edit distance is 0 (the single diagonal stands at the end of the
//     shorter sequence) or recomputed from scratch otherwise.
//   * A haplotype sequence is never materialised: it is a list of pieces (reference runs and ALT alleles) and the
//     longest-common-prefix walk reads the bytes in place; two reference runs at the same coordinate match without
//     being read.
//   * SIMT: 32 threads on 32 different clusters only run together where they execute the SAME instructions, and only stay
//     together if what they execute there takes about the same time.  The unit of work every alignment decomposes into is the
//     extension of ONE wavefront diagonal (a longest-common-prefix walk): task_step() does exactly one, and it is the only
//     place in the kernel where sequences are compared.  Everything else is a coroutine: advance() runs a cluster's control
//     flow (queue pops, quotas, prunes, scoring) up to the next alignment it needs and returns with a Task; task_setup()
//     builds the task's two sequences.  The kernel's main loop gives every lane one task_step() per trip and lets the lanes
//     that have finished a task advance to their next one in batches.
//
// Exactly the reference's searches are replayed -- same priority keys, node ids, quotas, prunes and tie-breaks
// (query_optimizer.rs:166-365, exact_gt_optimizer.rs:108-357, waffle_solver.rs:122-522) -- with the exactness-preserving
// shortcuts of RegionSolver::compare_score (DESIGN.md 4.1).  Whatever does not fit the fixed per-thread workspace
// (more than TS_MAXN variants, queue / result / edit-distance / piece capacity, sequence bundle or exact shortcut
// requested) is REJECTED before any output is written and solved by the warp kernels instead.
//
// The code is plain scalar C++ (AVK_HD): the same source is compiled for the host by tests/ts_host.cpp and checked
// against the CPU oracle there, cluster by cluster, before it ever runs on a GPU.
#pragma once
#include "avk_layout.h"

#if defined(__CUDACC__)
extern __shared__ __align__(128) unsigned char avk_dyn_smem[];
#endif

namespace avk_ts {

#if defined(__CUDA_ARCH__)
// unaligned 32-bit little-endian read through a generic pointer
static __device__ __forceinline__ uint32_t ld4u_any(const uint8_t *p) {
    const uint32_t *w = (const uint32_t *)((uintptr_t)p & ~(uintptr_t)3);
    return __funnelshift_r(w[0], w[1], ((uint32_t)(uintptr_t)p & 3u) * 8u);
}
#endif

typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;
using namespace avk;

enum { TS_MAXN = 12, TS_EDCAP = 16, TS_QCAP = 16, TS_RESCAP = 8, TS_MAXALT = 6, TS_MAXP = 2 * TS_MAXALT + 1, TS_MAXSLOT = 4 };
enum { TS_REJECT = -1 };   // >= 0: AVK_ST_*
// A thread gives up on a cluster after this many queue pops (search + exact-GT): 32 clusters share a warp and a launch ends with
// its slowest thread, so the rare long search is handed to the speculative solver (avk_spec_search.cuh), which pops 32 at a time.
enum { TS_POP_BUDGET = 64 };
enum { TS_WF = 2 * TS_EDCAP + 2 };
// what the thread has to do next (outside advance / exec_task)
enum { PH_FETCH = 0, PH_RUN = 1, PH_COMMIT = 2, PH_DONE = 3 };

struct VarInfo { u16 pos, aoff; u8 l0, l1, alted, pad; };                   // pos relative to the region start
struct QEnt { u32 key; u16 a1, a2; u8 depth, ed1, ed2, pad; };              // optimize_sequences: key = cost << 16 | id
struct XEnt { u32 key; u16 keep; u8 depth, pad; };                          // optimize_gt_alleles: key = errors << 27 | (31 - good) << 22 | id
struct ResEnt { u16 a1, a2; u8 ed1, ed2, tvs1, tvs2, qvs1, qvs2, p0, p1; };
// pieces of a virtual haplotype sequence, alternating reference run (even index) / ALT allele (odd index)
struct PSeq {
    u16 ls[TS_MAXP + 1];       // logical start of piece k; ls[n] == length
    u16 src[TS_MAXP];          // even k: reference position relative to the region start; odd k: offset into the allele bytes
};
enum { TS_XCAP = (TS_QCAP * sizeof(QEnt)) / sizeof(XEnt) };

// per-thread workspace (shared memory on the GPU)
struct Work {
    VarInfo var[TS_MAXN];
    u8 vtype[TS_MAXN], zyg[TS_MAXN], slot[TS_MAXN];
    u8 bucket[TS_MAXN + 2];
    u16 truth_mask;                 // bit oi: order entry oi is a truth variant
    u16 type_bits[TS_MAXSLOT];      // bit oi: order entry oi has the variant type of metric-row slot k
    union {
        QEnt q[TS_QCAP];
        XEnt x[TS_XCAP];
    };
    ResEnt res[TS_RESCAP];
    u16 wf[3][TS_WF];               // parent hap 0 / hap 1, child (also the scoring alignments)
    PSeq seq[2];
    u32 bp[1 + TS_MAXSLOT][4];      // basepair counters being accumulated by the scoring: joint row, then one per slot
};
// one workspace per thread, side by side in shared memory: an odd number of 32-bit words per workspace keeps the 32 lanes
// of a warp on 32 different banks when they touch the same field
static_assert(sizeof(Work) % 4 == 0 && (sizeof(Work) / 4) % 2 == 1, "sizeof(Work) must be an odd number of words");

// counters of the work actually executed (same meaning as avk_work_counters)
struct Counters { u64 cells, matched; u32 alignments, spops, xpops; };

// read-only view of one cluster
struct Cluster {
    const u8 *ref;     // region window: base at absolute position start + x is ref[x]
    const u8 *recs;    // N VI_* records in merged order (digest)
    const u8 *alle;    // allele bytes of the digest
    int wlen, N, nT, nQ, mbf, n_slots;   // wlen = window length (end - start)
    u32 xcap;          // optimize_gt_alleles: node expansions allowed per call (AVK_ST_TIMEOUT beyond)
    u32 slot_types;    // 4 bits per slot: variant type of metric-row slot k
    bool has_noop;     // some record's ALT equals its REF (alt_ed == 0)
};

// A sequence to build: HaplotypeTracker replay of `side` (0 truth, 1 query; 2 = the plain reference window) over the first
// `depth` order entries with ALT where `mask` has the bit, then copy_reference(region end) if to_end.
struct Spec { u8 side, depth, to_end, pad; u16 mask; };
// scalars of a built sequence: `len`; tracker ref_pos / skip distance; spliced ALTs; last_ok == 0 iff the LAST replayed
// entry was an incompatible ALT of this side; plen / prp: length and ref_pos after depth - 1 entries (the parent's)
struct SeqInfo { int len, ref_pos, skip, n_alt, last_ok, plen, prp; };

enum { TK_NONE = 0, TK_ALIGN = 1, TK_PREFIX = 2 };
enum { INIT_KEEP = 0, INIT_ZERO = 1, INIT_COPY = 2, INIT_CLOSED0 = 3 };
// One alignment job: build sequences a (baseline) and b (other), then
//   TK_ALIGN : DWFALite::update (if `update`) and finalize (if `finalize`) on wavefront buffer `buf`, initialised per `init`
//   TK_PREFIX: longest common prefix from offset d0 (DWFA with max ED 0, exact_gt_optimizer.rs:380)
struct Task {
    int kind;
    Spec a, b;
    int buf, init, src, ed_in, d0;
    bool update, finalize;
    // micro-state of the wavefront pass in flight (task_step): next diagonal, maxima of the pass, finalize pass?
    int i, mb, mo, matched;
    bool full, fin_pass;
    // results
    bool ok;            // false: capacity exceeded, reject the cluster
    int ed, m;
    SeqInfo ia, ib;
};

static AVK_HD inline u32 rec32(const Cluster &c, int oi, int field) { return *(const u32 *)(c.recs + (size_t)VI_SIZE * oi + field); }
static AVK_HD inline int min_i(int a, int b) { return a < b ? a : b; }
static AVK_HD inline int max_i(int a, int b) { return a > b ? a : b; }

// program counter of the coroutine
enum {
    PC_S_POP = 0, PC_S_PARENT, PC_S_PARENT_DONE, PC_S_FINAL, PC_S_FINAL_DONE, PC_S_CHILD, PC_S_CHILD_DONE,
    PC_SCORE_NEXT, PC_X_POP, PC_X_FINAL_DONE, PC_X_CHILD, PC_X_CHILD_DONE,
    PC_F_BEGIN, PC_F_HAP, PC_F_X_DONE, PC_F_Y_DONE, PC_F_SLOT, PC_F_EF_DONE, PC_F_ZF_DONE, PC_F_END
};

// ---------------------------------------------------------------------------------------------------------------------
// One thread's solver: scalar members live in registers, the workspace in shared memory.
struct Solver {
    Cluster c;
    Work *wp;
    Counters *ctr;
    Task task;
    int phase, pc;
    int rc;                        // status of the cluster when phase == PH_COMMIT (AVK_ST_* or TS_REJECT)
    int pops_left;                 // TS_POP_BUDGET minus the queue pops of this cluster so far
    // optimize_sequences
    int qn, nres;
    u32 best, next_id;
    u32 e_key, pm0, pm1;           // the popped entry
    int oi, ped0, ped1, h2, k, two, ced0, ccost, cm0, cm1;
    int f_ed0, f_sk0;              // finalize: first haplotype's distance and skip sum (tsk | qsk << 8)
    // scoring: iteration over the equal-best results and their two haplotypes
    int ri, hi, h, best_r, best_total, total, budget;
    bool lost;
    u32 keep0, keep1, best_keep0, best_keep1;
    // optimize_gt_alleles
    int xn, best_err, min_sync, af_index, af_counts, x_errors, x_d0;
    bool have_best, x_is_alt, x_do_alt;
    u32 x_next_id, hap_alt, x_keep, x_ekeep, x_id0, x_id1, x_expansions;
    // final scoring
    u32 f_X, f_Y, f_tp, f_Ef, f_failT, f_failQ, f_failF, f_other;
    int f_altT, f_altQ, f_side, f_alt_other;
    u32 f_mask;
    bool f_mirror;                 // truth filter == query filter (mirror_lists): one pass per slot serves both sides

#if defined(__CUDA_ARCH__)
    // on the device the workspaces sit side by side in dynamic shared memory: addressing them through the __shared__ array
    // (not through the generic pointer) lets the compiler emit LDS / STS
    __device__ __forceinline__ Work &w() const { return ((Work *)avk_dyn_smem)[threadIdx.x]; }
#else
    Work &w() const { return *wp; }
#endif
    AVK_HD int sync_pos(int i) const { return (i == c.N - 1) ? c.wlen : (int)w().var[i + 1].pos; }   // query_optimizer.rs:258-265 (relative)
    AVK_HD bool is_truth(int i) const { return (w().truth_mask >> i) & 1; }
    AVK_HD int slot_type(int s) const { return (int)((c.slot_types >> (4 * s)) & 15u); }
    AVK_HD static Spec spec(int side, u32 mask, int depth, bool to_end) { Spec s; s.side = (u8)side; s.depth = (u8)depth; s.to_end = to_end ? 1 : 0; s.pad = 0; s.mask = (u16)mask; return s; }

    // HaplotypeTracker replay (haplotype_dwfa.rs:175-227); positions relative to the region start.
    // returns false when the sequence has more than TS_MAXALT spliced ALTs.  (One out-of-line copy: it is called from a dozen
    // places of the coroutine and must not drag the solver's registers into local memory, hence static with explicit arguments.)
    static AVK_HD_NOINLINE bool replay_impl(const Work *wp_, int wlen, int N, PSeq *ps, SeqInfo *out, const Spec sp) {
#if defined(__CUDA_ARCH__)
        const Work &W = ((const Work *)avk_dyn_smem)[threadIdx.x];
        (void)wp_;
#else
        const Work &W = *wp_;
#endif
        // The tracker's ref_pos before entry i is max(end of the last spliced ALT, position of entry i): the entries are in
        // position order and every entry's sync point is the next entry's position (query_optimizer.rs:258-265).  So an ALT
        // of this side is compatible iff the last spliced ALT ends at or before it, entries that are not ALTs of this side
        // change nothing, and the walk only visits the set bits of (mask & side).
        int cur = 0, len = 0, m = 0, skip = 0, last_ok = 1, plen = 0, prp = 0, ref_pos = 0;
        const bool pieces = ps != nullptr;
        if (pieces) { ps->ls[0] = 0; ps->src[0] = 0; }
        const int depth = sp.side < 2 ? (int)sp.depth : 0;
        if (depth > 0) {
            const u32 tmask = W.truth_mask;
            const u32 side_bits = sp.side == 0 ? tmask : ~tmask;
            const u32 last_bit = 1u << (depth - 1);
            u32 bits = (u32)sp.mask & side_bits & (last_bit | (last_bit - 1u));
            bool snap = false;
            while (bits) {
                const u32 low = bits & (0u - bits);
                bits ^= low;
#if defined(__CUDA_ARCH__)
                const int i = __ffs((int)low) - 1;
#else
                const int i = __builtin_ctz(low);
#endif
                const VarInfo v = W.var[i];
                const int vpos = v.pos;
                if (low == last_bit) {                            // state before the last replayed entry (the parent's)
                    prp = depth == 1 ? 0 : (cur > vpos ? cur : vpos);
                    plen = len + (prp - cur);
                    snap = true;
                }
                if (cur <= vpos) {                                // compatible (haplotype_dwfa.rs:189)
                    if (m >= TS_MAXALT) return false;
                    len += vpos - cur;
                    if (pieces) { ps->ls[2 * m + 1] = (u16)len; ps->src[2 * m + 1] = (u16)(v.aoff + v.l0); }
                    len += v.l1;
                    cur = vpos + v.l0;
                    if (pieces) { ps->ls[2 * m + 2] = (u16)len; ps->src[2 * m + 2] = (u16)cur; }
                    m += 1;
                } else {
                    skip += v.alted;                              // edit_distance(allele0, allele1) (:199)
                    if (low == last_bit) last_ok = 0;
                }
            }
            if (!snap) {
                const int lp = W.var[depth - 1].pos;
                prp = depth == 1 ? 0 : (cur > lp ? cur : lp);
                plen = len + (prp - cur);
            }
            const int sy = (depth == N) ? wlen : (int)W.var[depth].pos;   // sync point of the last entry
            ref_pos = cur > sy ? cur : sy;
        }
        if ((sp.to_end || sp.side >= 2) && ref_pos < wlen) ref_pos = wlen;
        len += ref_pos - cur;
        if (pieces) ps->ls[2 * m + 1] = (u16)len;
        out->len = len; out->ref_pos = ref_pos; out->skip = skip; out->n_alt = m; out->last_ok = last_ok; out->plen = plen; out->prp = prp;
        return true;
    }
    template <bool PIECES>
    AVK_HD bool replay(PSeq *ps, SeqInfo &s, const Spec sp) const { return replay_impl(wp, c.wlen, c.N, PIECES ? ps : nullptr, &s, sp); }

    AVK_HD const u8 *piece_ptr(const PSeq &s, int pk, int x) const { return ((pk & 1) ? c.alle : c.ref) + s.src[pk] + (x - s.ls[pk]); }

    // equal leading bytes of A[x..] and B[y..]
    AVK_HD int lcp(const PSeq &A, int la, int x, const PSeq &B, int lb, int y) const {
        const int maxn = min_i(la - x, lb - y);
        if (maxn <= 0) return 0;
        int ka = 0, kb = 0;
        while (A.ls[ka + 1] <= x) ++ka;
        while (B.ls[kb + 1] <= y) ++kb;
        int total = 0;
        for (;;) {
            const int n = min_i(min_i(A.ls[ka + 1] - x, B.ls[kb + 1] - y), maxn - total);
            const u8 *pa = piece_ptr(A, ka, x), *pb = piece_ptr(B, kb, y);
            if (pa != pb) {                                   // same reference bytes otherwise: equal by construction
                int j = 0;
#if defined(__CUDA_ARCH__)
                while (j < n) {                                   // four bases per step (unaligned words: two aligned loads + funnel shift;
                    const u32 x = ld4u_any(pa + j) ^ ld4u_any(pb + j);   //  every buffer read here has >= 8 bytes of slack behind it)
                    if (x) { j += (__ffs((int)x) - 1) >> 3; break; }
                    j += 4;
                }
                if (j > n) j = n;
#else
                while (j < n && pa[j] == pb[j]) ++j;
#endif
                if (j < n) return total + j;
            }
            total += n; x += n; y += n;
            if (total >= maxn) return total;
            while (A.ls[ka + 1] <= x) ++ka;
            while (B.ls[kb + 1] <= y) ++kb;
        }
    }

    // ================================================================== the ONE place where sequences are built ...
    // task_setup(): builds the two sequences of the task and initialises its wavefront.  A task that cannot be set up (piece
    // capacity) ends here with ok == false.
    AVK_HD void task_setup() {
        Work &W = w();
        Task &t = task;
        {   // (out-of-line call: its outputs go through locals so that the solver itself can stay in registers)
            SeqInfo ia, ib;
            const Spec sa = t.a, sb = t.b;
            t.ok = replay<true>(&W.seq[0], ia, sa) && replay<true>(&W.seq[1], ib, sb);
            t.ia = ia; t.ib = ib;
        }
        if (!t.ok) { t.kind = TK_NONE; return; }
        if (t.kind == TK_PREFIX) return;
        u16 *wf = W.wf[t.buf];
        int ed = t.ed_in;
        if (t.init == INIT_ZERO) { wf[0] = 0; ed = 0; }
        else if (t.init == INIT_CLOSED0) { wf[0] = (u16)min_i(t.ia.plen, t.ib.plen); ed = 0; }   // parent had ED 0: its one diagonal stood at the end of its shorter sequence
        else if (t.init == INIT_COPY) { const u16 *sw = W.wf[t.src]; for (int i = 0; i < 2 * ed + 1; ++i) wf[i] = sw[i]; }
        t.ed = ed; t.i = 0; t.mb = -1; t.mo = -1; t.matched = 0; t.full = false;
        t.fin_pass = !t.update;                                // wfa_ed: finalize() only
    }
    // ================================================================== ... and where wavefronts advance: ONE diagonal per call
    // DWFALite::update (dynamic_wfa.rs:68-84) then finalize (:183-198), cut at the diagonal: extend() of diagonal t.i (:94-130);
    // at the end of a pass over the wavefront the stop rule of the current pass is tested and, if it does not hold,
    // increase_edit_distance() (:152-168) grows the wavefront in place.  finalize() starts with an extend() of its own: a pass
    // over the already extended diagonals that only evaluates reached_full_diagonal.  The task ends with kind == TK_NONE.
    AVK_HD void task_step() {
        Work &W = w();
        Task &t = task;
        const PSeq &A = W.seq[0], &B = W.seq[1];
        const int la = t.ia.len, lb = t.ib.len;
        if (t.kind == TK_PREFIX) {
            t.m = lcp(A, la, t.d0, B, lb, t.d0);
            ctr->cells += 1; ctr->matched += (u64)t.m;
            t.kind = TK_NONE;
            return;
        }
        u16 *wf = W.wf[t.buf];
        const int ed = t.ed, n = 2 * ed + 1;
        {
            const int i = t.i;
            int d = wf[i];
            int boff = d + ed - i;
            if (boff < la && d < lb) {
                const int ext = lcp(A, la, boff, B, lb, d);
                d += ext; boff += ext; t.matched += ext;
                wf[i] = (u16)d;
            }
            t.mb = max_i(t.mb, boff); t.mo = max_i(t.mo, d);
            t.full = t.full || (boff >= la && d >= lb);
            t.i = i + 1;
        }
        if (t.i < n) return;
        // ---- end of a pass over the wavefront
        ctr->cells += (u64)n; ctr->matched += (u64)t.matched;
        const bool done = t.fin_pass ? t.full : (t.mb >= la || t.mo >= lb);
        t.i = 0; t.mb = -1; t.mo = -1; t.matched = 0; t.full = false;
        if (done) {
            if (!t.fin_pass && t.finalize) { t.fin_pass = true; return; }
            if (t.fin_pass) ctr->alignments += 1;
            t.ok = true;
            t.kind = TK_NONE;
            return;
        }
        if (ed + 1 > TS_EDCAP) { t.ok = false; t.kind = TK_NONE; return; }
        for (int i = n + 1; i >= 0; --i) {                    // increase_edit_distance(): in place from the top
            int v = 0;
            if (i < n) v = wf[i];
            if (i >= 1 && i - 1 < n) v = max_i(v, wf[i - 1] + 1);
            if (i >= 2 && i - 2 < n) v = max_i(v, wf[i - 2] + 1);
            wf[i] = (u16)v;
        }
        t.ed = ed + 1;
    }
    // whole task at once (host harness)
    AVK_HD void exec_task() {
        task_setup();
        while (task.kind != TK_NONE) task_step();
    }

    // ================================================================== begin: load the cluster
    // leaves phase = PH_RUN with the workspace loaded, or PH_COMMIT with rc = an error status / TS_REJECT
    AVK_HD void begin(const u8 *digest, const u8 *contig, int start, int end, int mbf, u32 xcap, int pop_budget = TS_POP_BUDGET) {
        const int *hdr = (const int *)digest;
        task.kind = TK_NONE;
        phase = PH_COMMIT;
        pops_left = pop_budget;
        rc = hdr[PH_STATUS / 4];
        if (rc) return;
        rc = TS_REJECT;
        const int n = hdr[PH_N / 4];
        if (n > TS_MAXN || n < 1 || mbf > 255) return;
        // logical offsets are 16-bit, allele lengths 8-bit
        if ((end - start) + hdr[PH_SUM_L1 / 4] > 60000 || hdr[PH_SUM_ALLE / 4] > 60000) return;
        const int ns = hdr[PH_NSLOTS / 4];
        if (ns > TS_MAXSLOT) return;
        c.ref = contig + start; c.recs = digest + PH_SIZE; c.alle = c.recs + (size_t)VI_SIZE * n;
        c.xcap = xcap ? xcap : AVK_EXACT_GT_DEFAULT_MAX_EXPANSIONS;
        c.wlen = end - start; c.N = n; c.nT = hdr[PH_N0 / 4]; c.nQ = hdr[PH_N1 / 4]; c.mbf = mbf; c.n_slots = ns;
        c.slot_types = 0; c.has_noop = false;
        for (int s = 0; s < ns; ++s) c.slot_types |= (u32)digest[PH_SLOT_TYPE + s] << (4 * s);
        Work &W = w();
        u16 tm = 0;
        for (int s = 0; s < TS_MAXSLOT; ++s) W.type_bits[s] = 0;
        for (int i = 0; i < n; ++i) {
            const u32 *r = (const u32 *)(c.recs + (size_t)VI_SIZE * i);
            if (r[VI_L0 / 4] > 255u || r[VI_L1 / 4] > 255u) return;
            VarInfo v;
            v.pos = (u16)(r[VI_POS / 4] - (u32)start); v.aoff = (u16)r[VI_AOFF / 4];
            v.l0 = (u8)r[VI_L0 / 4]; v.l1 = (u8)r[VI_L1 / 4]; v.alted = (u8)r[VI_ALTED / 4]; v.pad = 0;   // alt_ed <= max(l0, l1)
            if (v.alted == 0) c.has_noop = true;
            W.var[i] = v;
            const u32 f = r[VI_FLAGS / 4];
            W.vtype[i] = (u8)(f & 0xff); W.zyg[i] = (u8)((f >> 8) & 0xff); W.slot[i] = (u8)(f >> 24);
            W.type_bits[f >> 24] |= (u16)(1u << i);
            if (f & 0x10000u) tm |= (u16)(1u << i);
        }
        W.truth_mask = tm;
        // optimize_sequences: root (query_optimizer.rs:184-192)
        for (int i = 0; i <= n; ++i) W.bucket[i] = 0;
        nres = 0; best = 0xffffffffu; next_id = 1; qn = 0;
        { QEnt e; e.key = 0; e.a1 = 0; e.a2 = 0; e.depth = 0; e.ed1 = 0; e.ed2 = 0; e.pad = 0; W.q[qn++] = e; }
        rc = AVK_ST_OK;
        phase = PH_RUN; pc = PC_S_POP;
    }
    AVK_HD void stop(int status) { rc = status; phase = PH_COMMIT; }

    AVK_HD void emit_align(Spec a, Spec b, int buf, int init, int src, int ed_in, bool update, bool finalize) {
        task.kind = TK_ALIGN; task.a = a; task.b = b; task.buf = buf; task.init = init; task.src = src; task.ed_in = ed_in;
        task.update = update; task.finalize = finalize; task.d0 = 0;
    }
    AVK_HD void emit_prefix(Spec a, Spec b, int d0) {
        task.kind = TK_PREFIX; task.a = a; task.b = b; task.d0 = d0; task.buf = 0; task.init = 0; task.src = 0; task.ed_in = 0;
        task.update = false; task.finalize = false;
    }
    // hap_lb: flips a result's haplotype costs at least (ED or skipped distance > 0: its zero-flip path cannot be exact).
    // hap_zero: known to cost none -- ED 0 and nothing skipped.  "Nothing skipped" is read off the skipped variants' summed edit
    // distance, which says nothing about a skipped variant whose ALT equals its REF (distance 0); an incompatible no-op ALT
    // cannot be kept (optimize_gt_alleles drops that child, exact_gt_optimizer.rs:293-305), so in a cluster that holds such a
    // record the shortcut is off and the search runs.
    AVK_HD static int hap_lb(const ResEnt &r, int hh) { return (hh ? (r.ed2 + r.tvs2 + r.qvs2) : (r.ed1 + r.tvs1 + r.qvs1)) == 0 ? 0 : 1; }
    AVK_HD bool hap_zero(const ResEnt &r, int hh) const { return hap_lb(r, hh) == 0 && !c.has_noop; }

    // ================================================================== the coroutine
    // Runs the cluster's control flow until it needs an alignment (returns with task.kind != TK_NONE) or the cluster is
    // finished (phase == PH_COMMIT: rc is the status; on AVK_ST_OK best_r / best_keep* / W.bp hold what commit needs).
    AVK_HD void advance() {
        Work &W = w();
        const int n = c.N;
        for (;;) {
            switch (pc) {
            // ---------------------------------------------------------------- optimize_sequences (query_optimizer.rs:203-328)
            case PC_S_POP: {
                if (qn == 0) {                                                  // queue drained
                    if (nres == 0) { stop(AVK_ST_NO_RESULT); return; }          // :331
                    // scoring of the equal-best results (waffle_solver.rs:169-265), see PC_SCORE_NEXT
                    best_r = 0; best_total = 0x7fffffff; best_keep0 = best_keep1 = 0;
                    ri = 0; hi = nres;
                    for (int i = 0; i < nres; ++i) if (hap_zero(W.res[i], 0) && hap_zero(W.res[i], 1)) { ri = i; hi = i + 1; break; }
                    h = 0;
                    pc = PC_SCORE_NEXT;
                    break;
                }
                int bi = 0;
                u32 bk = W.q[0].key;
                for (int i = 1; i < qn; ++i) { const u32 kk = W.q[i].key; if (kk < bk) { bk = kk; bi = i; } }
                const QEnt e = W.q[bi];
                W.q[bi] = W.q[--qn];
                ctr->spops += 1;
                if (--pops_left < 0) { stop(TS_REJECT); return; }               // a long search: not on a single thread
                if ((e.key >> 16) > best) break;                                // :204 strict
                if (W.bucket[e.depth] >= c.mbf) break;                          // :222
                W.bucket[e.depth] += 1;
                e_key = e.key; pm0 = e.a1; pm1 = e.a2; oi = e.depth; ped0 = e.ed1; ped1 = e.ed2;
                h2 = 0;
                pc = PC_S_PARENT;
                break;
            }
            case PC_S_PARENT: {                                                 // wavefront of a parent haplotype with ED > 0: recomputed from scratch
                while (h2 < 2 && (h2 ? ped1 : ped0) == 0) ++h2;
                if (h2 < 2) {
                    const u32 pm = h2 ? pm1 : pm0;
                    emit_align(spec(0, pm, oi, false), spec(1, pm, oi, false), h2, INIT_ZERO, 0, 0, true, false);
                    pc = PC_S_PARENT_DONE;
                    return;
                }
                h2 = 0;
                if (oi == n) { pc = PC_S_FINAL; break; }
                const int z = W.zyg[oi];
                const bool tr = is_truth(oi);
                const bool het = (z == AVK_ZYG_UNPHASED_HET || z == AVK_ZYG_PHASED_HET01 || z == AVK_ZYG_PHASED_HET10);
                if (!het && z != AVK_ZYG_HOM_ALT) { stop(AVK_ST_BAD_ZYGOSITY); return; }   // assert_eq! :315
                two = (het && (!tr || z == AVK_ZYG_UNPHASED_HET)) ? 1 : 0;                  // :269 both orientations, new ids
                k = two ? 0 : 1;
                pc = PC_S_CHILD;
                break;
            }
            case PC_S_PARENT_DONE: {
                if (!task.ok || task.ed != (h2 ? ped1 : ped0)) { stop(TS_REJECT); return; }   // (a differing distance cannot happen: path independence)
                h2 += 1;
                pc = PC_S_PARENT;
                break;
            }
            case PC_S_FINAL: {                                                  // :227-247 finalize_dwfa (haplotype_dwfa.rs:84-95) of haplotype h2
                const u32 pm = h2 ? pm1 : pm0;
                const int pe = h2 ? ped1 : ped0;
                // the parent's sequences at depth n and at the region end differ only by the trailing reference run, so the
                // closed-form parent diagonal (ED 0) is min of the lengths before that run: replay to_end reports them as plen
                // only for depth - 1; build the parent diagonal from a depth-n replay instead (INIT_KEEP after a closed-form write)
                if (pe == 0) {
                    SeqInfo ti, qi;
                    replay<false>(nullptr, ti, spec(0, pm, n, false)); replay<false>(nullptr, qi, spec(1, pm, n, false));
                    W.wf[h2][0] = (u16)min_i(ti.len, qi.len);
                }
                emit_align(spec(0, pm, n, true), spec(1, pm, n, true), h2, INIT_KEEP, 0, pe, true, true);
                pc = PC_S_FINAL_DONE;
                return;
            }
            case PC_S_FINAL_DONE: {
                if (!task.ok) { stop(TS_REJECT); return; }
                if (task.ia.skip > 255 || task.ib.skip > 255) { stop(TS_REJECT); return; }
                if (h2 == 0) { f_ed0 = task.ed; f_sk0 = task.ia.skip | (task.ib.skip << 8); h2 = 1; pc = PC_S_FINAL; break; }
                const int tsk0 = f_sk0 & 255, qsk0 = f_sk0 >> 8, tsk1 = task.ia.skip, qsk1 = task.ib.skip;
                const u32 cc = (u32)(f_ed0 + task.ed + tsk0 + tsk1 + qsk0 + qsk1);
                if (cc < best) { best = cc; nres = 0; }
                if (cc == best) {
                    if (nres >= TS_RESCAP) { stop(TS_REJECT); return; }
                    ResEnt r;
                    r.a1 = (u16)pm0; r.a2 = (u16)pm1; r.ed1 = (u8)f_ed0; r.ed2 = (u8)task.ed;
                    r.tvs1 = (u8)tsk0; r.tvs2 = (u8)tsk1; r.qvs1 = (u8)qsk0; r.qvs2 = (u8)qsk1; r.p0 = r.p1 = 0;
                    W.res[nres++] = r;
                }
                pc = PC_S_POP;
                break;
            }
            case PC_S_CHILD: {                                                  // child k, haplotype h2: HaplotypeDWFA::extend_variant (haplotype_dwfa.rs:46-67)
                if (h2 == 0) {
                    const int z = W.zyg[oi];
                    bool a1, a2;
                    if (two) { a1 = k == 1; a2 = k == 0; }                      // (REF, ALT) first, then (ALT, REF)
                    else if (z != AVK_ZYG_HOM_ALT) { a1 = (z == AVK_ZYG_PHASED_HET10); a2 = !a1; }   // phased truth het :294-312
                    else { a1 = true; a2 = true; }                              // hom-alt :313-327
                    cm0 = (int)(pm0 | ((a1 ? 1u : 0u) << oi)); cm1 = (int)(pm1 | ((a2 ? 1u : 0u) << oi));
                    ccost = 0;
                }
                const u32 cm = (u32)(h2 ? cm1 : cm0);
                const int pe = h2 ? ped1 : ped0;
                emit_align(spec(0, cm, oi + 1, false), spec(1, cm, oi + 1, false), 2, pe == 0 ? INIT_CLOSED0 : INIT_COPY, h2, pe, true, false);
                pc = PC_S_CHILD_DONE;
                return;
            }
            case PC_S_CHILD_DONE: {
                if (!task.ok) { stop(TS_REJECT); return; }
                ccost += task.ed + task.ia.skip + task.ib.skip;
                if (h2 == 0) { ced0 = task.ed; h2 = 1; pc = PC_S_CHILD; break; }
                u32 id;
                if (two) id = next_id++;
                else id = e_key & 0xffffu;
                if ((u32)ccost > 0xfffeu || id > 0xfffeu) { stop(TS_REJECT); return; }
                if (qn >= TS_QCAP) {                                            // garbage collection: entries the search would discard when popped (cost > best)
                    int wq = 0;
                    for (int i = 0; i < qn; ++i) if ((W.q[i].key >> 16) <= best) W.q[wq++] = W.q[i];
                    qn = wq;
                    if (qn >= TS_QCAP) { stop(TS_REJECT); return; }
                }
                QEnt ne;
                ne.key = ((u32)ccost << 16) | id; ne.a1 = (u16)cm0; ne.a2 = (u16)cm1; ne.depth = (u8)(oi + 1);
                ne.ed1 = (u8)ced0; ne.ed2 = (u8)task.ed; ne.pad = 0;
                W.q[qn++] = ne;
                k += 1; h2 = 0;
                pc = (k < 2) ? PC_S_CHILD : PC_S_POP;
                break;
            }
            // ---------------------------------------------------------------- scoring driver (waffle_solver.rs:169-265)
            // exact-GT scoring of every equal-best solution; first minimum wins, with the pruning argued in
            // RegionSolver::compare_score: a haplotype with ED 0 and nothing skipped scores 0 flips without a search; a solution
            // whose lower bound reaches the current minimum is not searched; a search stops at its budget; the first solution
            // with both haplotypes at 0 is the answer.
            case PC_SCORE_NEXT: {
                if (ri >= hi) { pc = PC_F_BEGIN; break; }
                const ResEnt r = W.res[ri];
                const bool z0 = hap_zero(r, 0), z1 = hap_zero(r, 1);
                if (h == 0) {
                    if (hap_lb(r, 0) + hap_lb(r, 1) >= best_total) { ri += 1; break; }
                    total = 0; lost = false; keep0 = keep1 = 0;
                }
                if (h < 2 && !lost) {
                    const u32 ha = h ? r.a2 : r.a1;
                    if (h ? z1 : z0) { if (h) keep1 = ha; else keep0 = ha; h += 1; break; }
                    budget = best_total - total - (h == 0 ? hap_lb(r, 1) : 0);
                    // optimize_gt_alleles (exact_gt_optimizer.rs:108-357) on this haplotype
                    hap_alt = ha; x_keep = 0;
                    x_next_id = 1; best_err = 0x7fffffff; have_best = false;
                    min_sync = 0; af_index = 0; af_counts = 0; x_expansions = 0;
                    xn = 0;
                    { XEnt e; e.key = (31u << 22); e.keep = 0; e.depth = 0; e.pad = 0; W.x[xn++] = e; }
                    pc = PC_X_POP;
                    break;
                }
                if (!lost && total < best_total) { best_total = total; best_r = ri; best_keep0 = keep0; best_keep1 = keep1; }
                ri += 1; h = 0;
                break;
            }
            // ---------------------------------------------------------------- optimize_gt_alleles: one queue pop
            case PC_X_POP: {
                int errs = -1;                                                   // >= 0: the search is over with this error count
                if (xn == 0) {
                    if (!have_best) { stop(AVK_ST_NO_RESULT); return; }          // :345-348
                    errs = best_err;
                } else {
                    int bi = 0;
                    u32 bk = W.x[0].key;
                    for (int i = 1; i < xn; ++i) { const u32 kk = W.x[i].key; if (kk < bk) { bk = kk; bi = i; } }
                    const XEnt e = W.x[bi];
                    W.x[bi] = W.x[--xn];
                    ctr->xpops += 1;
                    if (--pops_left < 0) { stop(TS_REJECT); return; }
                    x_errors = (int)(e.key >> 27);
                    if (x_errors >= budget && !have_best) errs = budget;         // nodes pop in non-decreasing error order
                    else if (x_errors >= best_err) break;                        // :169 non-strict
                    else if (++x_expansions > c.xcap) { stop(AVK_ST_TIMEOUT); return; }   // stand-in for the 300 s bail (:174-176)
                    else {
                        oi = e.depth; x_ekeep = e.keep; x_id0 = e.key & 0x3fffffu;
                        if (oi == n) {                                           // :180-192: finalize; exact <=> sequences equal
                            emit_prefix(spec(0, x_ekeep, n, true), spec(1, x_ekeep, n, true), 0);
                            pc = PC_X_FINAL_DONE;
                            return;
                        }
                        if (oi < min_sync) break;                                // :194-197
                        SeqInfo ti, qi;
                        replay<false>(nullptr, ti, spec(0, x_ekeep, oi, false)); replay<false>(nullptr, qi, spec(1, x_ekeep, oi, false));
                        if (ti.len == qi.len && ti.ref_pos == qi.ref_pos) { min_sync = oi; af_counts = 0; af_index = oi; }   // is_synchronized :206-217 (alive => ed == 0)
                        x_d0 = min_i(ti.len, qi.len);                            // the single diagonal of an alive node
                        x_is_alt = (hap_alt >> oi) & 1;
                        x_do_alt = x_is_alt && !(oi < af_index);
                        // REF allele: move, id kept (:257-273).  ALT allele: (REF, error) with id next_id, then (ALT, no error) with
                        // the following id unless auto-failed (:274-306).
                        x_id1 = 0;
                        if (x_is_alt) { x_id0 = x_next_id; if (x_do_alt) x_id1 = x_next_id + 1; x_next_id += x_do_alt ? 2 : 1; }
                        k = 0;
                        pc = PC_X_CHILD;
                        break;
                    }
                }
                // search over: back to the scoring driver
                lost = errs >= budget;
                total += errs;
                if (h) keep1 = x_keep; else keep0 = x_keep;
                h += 1;
                pc = PC_SCORE_NEXT;
                break;
            }
            case PC_X_FINAL_DONE: {
                if (!task.ok) { stop(TS_REJECT); return; }
                ctr->alignments += 1;
                const bool exact = task.ia.len == task.ib.len && task.m == task.ia.len;
                if (exact && x_errors < best_err) { best_err = x_errors; have_best = true; x_keep = x_ekeep; }
                pc = PC_X_POP;
                break;
            }
            case PC_X_CHILD: {
                const u32 kp = x_ekeep | ((k == 1 ? 1u : 0u) << oi);
                emit_prefix(spec(0, kp, oi + 1, false), spec(1, kp, oi + 1, false), x_d0);
                pc = PC_X_CHILD_DONE;
                return;
            }
            case PC_X_CHILD_DONE: {
                if (!task.ok) { stop(TS_REJECT); return; }
                const bool alt = k == 1;
                bool ok = true;
                if (alt) ok = (is_truth(oi) ? task.ia : task.ib).last_ok != 0;   // incompatible ALT: success == false -> dropped
                if (ok) ok = (x_d0 + task.m >= task.ia.len) || (x_d0 + task.m >= task.ib.len);   // DWFA with max ED 0: an end must be reached
                if (ok) {
                    const int cerr = x_errors + ((x_is_alt && !alt) ? 1 : 0);
                    const int good = (oi + 1) - cerr;
                    const u32 id = alt ? x_id1 : x_id0;
                    if (id > 0x3ffffeu || cerr > 30) { stop(TS_REJECT); return; }
                    if (xn >= TS_XCAP) {                                         // garbage collection (RegionSolver::gc_queue)
                        int wq = 0;
                        for (int i = 0; i < xn; ++i) {
                            const XEnt g = W.x[i];
                            const bool dead = (int)(g.key >> 27) >= best_err || (g.depth != n && g.depth < min_sync);
                            if (!dead) W.x[wq++] = g;
                        }
                        xn = wq;
                        if (xn >= TS_XCAP) { stop(TS_REJECT); return; }
                    }
                    XEnt ne;
                    ne.key = ((u32)cerr << 27) | ((u32)(31 - good) << 22) | id;
                    ne.keep = (u16)(x_ekeep | ((alt ? 1u : 0u) << oi)); ne.depth = (u8)(oi + 1); ne.pad = 0;
                    W.x[xn++] = ne;
                }
                k += 1;
                if (k < (x_do_alt ? 2 : 1)) { pc = PC_X_CHILD; break; }
                af_counts += 1;                                                  // :310-339
                if (af_counts >= 500) {
                    if (af_index >= n) { stop(AVK_ST_NO_RESULT); return; }
                    int wq = 0;
                    for (int i = 0; i < xn; ++i) {
                        const XEnt g = W.x[i];
                        const bool set = g.depth > af_index;
                        if (!set || !((g.keep >> af_index) & 1)) W.x[wq++] = g;
                    }
                    xn = wq;
                    af_index += 1;
                    af_counts = 0;
                }
                pc = PC_X_POP;
                break;
            }
            // ---------------------------------------------------------------- basepair metrics (waffle_solver.rs:335-449)
            // X = ED(ref, truth), Y = ED(ref, query), Z = ED(truth, query) = the optimizer's finalised distance; per supported type
            // present: the filtered sequence of one side against the full haplotype of the other.  generate_allele_sequence
            // (:726-778) == a replay over all N entries up to the region end (an ALT overlapping an applied one is skipped and
            // costs its alt_ed in both).  Counters accumulate in W.bp; nothing else is kept.
            case PC_F_BEGIN: {
                for (int s = 0; s <= c.n_slots; ++s) for (int m = 0; m < 4; ++m) W.bp[s][m] = 0;
                f_mirror = mirror_lists(W.res[best_r]);
                h2 = 0;
                pc = PC_F_HAP;
                break;
            }
            case PC_F_HAP: {
                if (h2 == 2) { pc = PC_F_END; break; }
                const ResEnt R = W.res[best_r];
                f_mask = h2 ? R.a2 : R.a1;
                SeqInfo ti, qi;
                int closed;
                if (!replay<false>(nullptr, ti, spec(0, f_mask, n, true)) || !replay<false>(nullptr, qi, spec(1, f_mask, n, true))) { stop(TS_REJECT); return; }
                f_altT = ti.n_alt; f_altQ = qi.n_alt; f_failT = (u32)ti.skip; f_failQ = (u32)qi.skip;
                f_X = 0; f_Y = 0;
                if (f_altT) {
                    closed = closed_form(0, f_mask, 0xffffu);
                    if (closed >= 0) { f_X = (u32)closed; ctr->alignments += 1; ctr->cells += 1; }
                    else { emit_align(spec(2, 0, 0, true), spec(0, f_mask, n, true), 2, INIT_ZERO, 0, 0, false, true); pc = PC_F_X_DONE; return; }
                }
                pc = PC_F_X_DONE; task.ok = true; task.ed = (int)f_X;
                break;
            }
            case PC_F_X_DONE: {
                if (!task.ok) { stop(TS_REJECT); return; }
                f_X = (u32)task.ed;
                const ResEnt R = W.res[best_r];
                const u32 Z = h2 ? R.ed2 : R.ed1;
                if (Z == 0) { task.ed = (int)f_X; pc = PC_F_Y_DONE; break; }
                if (!f_altQ) { task.ed = 0; pc = PC_F_Y_DONE; break; }
                const int closed = closed_form(1, f_mask, 0xffffu);
                if (closed >= 0) { ctr->alignments += 1; ctr->cells += 1; task.ed = closed; pc = PC_F_Y_DONE; break; }
                emit_align(spec(2, 0, 0, true), spec(1, f_mask, n, true), 2, INIT_ZERO, 0, 0, false, true);
                pc = PC_F_Y_DONE;
                return;
            }
            case PC_F_Y_DONE: {
                if (!task.ok) { stop(TS_REJECT); return; }
                f_Y = (u32)task.ed;
                const ResEnt R = W.res[best_r];
                const u32 Z = h2 ? R.ed2 : R.ed1;
                f_tp = f_X + f_Y - Z;
                W.bp[0][0] += f_tp; W.bp[0][1] += 2 * f_X - f_tp + 2 * f_failT; W.bp[0][2] += f_tp; W.bp[0][3] += 2 * f_Y - f_tp + 2 * f_failQ;
                k = 0; f_side = 1;
                pc = PC_F_SLOT;
                break;
            }
            case PC_F_SLOT: {                                                    // slot k, side f_side: query filter (:395-410) then truth filter (:422-437)
                if (k >= c.n_slots) { h2 += 1; pc = PC_F_HAP; break; }
                if (!type_supported(slot_type(k))) { k += 1; f_side = 1; break; }
                const u32 side_bits = f_side ? (u32)(u16)~W.truth_mask : (u32)W.truth_mask;
                const u32 fbits = (u32)W.type_bits[k] & side_bits;
                const int nf = popc16(fbits);
                bool next = false;
                if (nf == 0) next = true;
                else if (nf == (f_side ? c.nQ : c.nT)) {                         // filtered == full haplotype
                    W.bp[1 + k][2 * f_side] += f_tp;
                    W.bp[1 + k][2 * f_side + 1] += f_side ? (2 * f_Y - f_tp + 2 * f_failQ) : (2 * f_X - f_tp + 2 * f_failT);
                    if (f_mirror) { W.bp[1 + k][0] += f_tp; W.bp[1 + k][1] += 2 * f_Y - f_tp + 2 * f_failQ; }   // (X == Y, failT == failQ)
                    next = true;
                } else {
                    SeqInfo fi;
                    if (!replay<false>(nullptr, fi, spec(f_side, f_mask & fbits, n, true))) { stop(TS_REJECT); return; }
                    f_failF = (u32)fi.skip;
                    f_other = f_side ? f_X : f_Y;                                // ED(ref, unfiltered other haplotype)
                    f_alt_other = f_side ? f_altT : f_altQ;
                    if (!fi.n_alt) { f_Ef = 0; task.ok = true; task.ed = (int)f_other; pc = PC_F_ZF_DONE; break; }
                    const int closed = closed_form(f_side, f_mask & fbits, 0xffffu);
                    if (closed >= 0) { ctr->alignments += 1; ctr->cells += 1; task.ok = true; task.ed = closed; pc = PC_F_EF_DONE; break; }
                    emit_align(spec(2, 0, 0, true), spec(f_side, f_mask & fbits, n, true), 2, INIT_ZERO, 0, 0, false, true);
                    pc = PC_F_EF_DONE;
                    return;
                }
                if (next) { if (f_side == 1 && !f_mirror) f_side = 0; else { f_side = 1; k += 1; } }
                break;
            }
            case PC_F_EF_DONE: {
                if (!task.ok) { stop(TS_REJECT); return; }
                f_Ef = (u32)task.ed;
                if (!f_alt_other) { task.ed = (int)f_Ef; pc = PC_F_ZF_DONE; break; }
                const u32 side_bits = f_side ? (u32)(u16)~W.truth_mask : (u32)W.truth_mask;
                const u32 fm = f_mask & (u32)W.type_bits[k] & side_bits;
                // side 1 (query filtered): ED(truth, F); side 0 (truth filtered): ED(F, query)
                if (f_side) emit_align(spec(0, f_mask, n, true), spec(1, fm, n, true), 2, INIT_ZERO, 0, 0, false, true);
                else emit_align(spec(0, fm, n, true), spec(1, f_mask, n, true), 2, INIT_ZERO, 0, 0, false, true);
                pc = PC_F_ZF_DONE;
                return;
            }
            case PC_F_ZF_DONE: {
                if (!task.ok) { stop(TS_REJECT); return; }
                const u32 Zf = (u32)task.ed;
                const u32 ftp = f_other + f_Ef - Zf;
                W.bp[1 + k][2 * f_side] += ftp;
                W.bp[1 + k][2 * f_side + 1] += 2 * f_Ef - ftp + 2 * f_failF;
                if (f_mirror) { W.bp[1 + k][0] += ftp; W.bp[1 + k][1] += 2 * f_Ef - ftp + 2 * f_failF; }
                if (f_side == 1 && !f_mirror) f_side = 0; else { f_side = 1; k += 1; }
                pc = PC_F_SLOT;
                break;
            }
            case PC_F_END:
            default:
                stop(AVK_ST_OK);
                return;
            }
        }
    }

    // Basepair metrics of a result in which the truth and query lists are the same records (order t0 q0 t1 q1 ...: position,
    // REF / ALT bytes, type slot) and each query record carries its ALT on exactly the haplotypes its truth twin does -- the
    // usual true-positive cluster.  Then the two haplotypes of each side spell the same strings, and so does every per-type
    // filter of them: ED(ref, truth filter) == ED(ref, query filter), ED(truth filter, query) == ED(truth, query filter)
    // (edit distance is symmetric), X == Y and the skip sums agree, so the truth-filter pass of each slot (waffle_solver.rs
    // :422-437) adds what the query-filter pass (:395-410) adds and is not run.
    AVK_HD bool mirror_lists(const ResEnt &R) const {
        const Work &W = w();
        const int n = c.N;
        if (c.nT != c.nQ || (n & 1)) return false;
        for (int i = 0; i < n; i += 2) {
            const VarInfo a = W.var[i], b = W.var[i + 1];
            if (!is_truth(i) || is_truth(i + 1) || a.pos != b.pos || a.l0 != b.l0 || a.l1 != b.l1 || W.slot[i] != W.slot[i + 1]) return false;
            if (((R.a1 >> i) & 1u) != ((R.a1 >> (i + 1)) & 1u) || ((R.a2 >> i) & 1u) != ((R.a2 >> (i + 1)) & 1u)) return false;
            for (int x = 0; x < a.l0 + a.l1; ++x) if (c.alle[a.aoff + x] != c.alle[b.aoff + x]) return false;
        }
        return true;
    }

    AVK_HD static int popc16(u32 v) { v &= 0xffffu; int cnt = 0; while (v) { v &= v - 1; ++cnt; } return cnt; }

    // ED(reference window, haplotype of `side` with ALT mask `mask`) when it is known without aligning
    // (RegionSolver::build_hap_seq): every spliced ALT a 1->1 substitution with at most two changing a base (Hamming <= 2 ==
    // ED), or no base-changing substitution and otherwise only anchored pure insertions, or only anchored pure deletions
    // (ED == the length difference).  -1 otherwise.
    AVK_HD int closed_form(int side, u32 mask, u32 bits) const {
        const Work &W = w();
        int cur = 0, subm = 0, ins = 0, del = 0;
        bool open = false;
        u32 todo = mask & bits & (side == 0 ? (u32)W.truth_mask : ~(u32)W.truth_mask) & ((1u << c.N) - 1u);
        while (todo) {
            const u32 low = todo & (0u - todo);
            todo ^= low;
#if defined(__CUDA_ARCH__)
            const int i = __ffs((int)low) - 1;
#else
            const int i = __builtin_ctz(low);
#endif
            const VarInfo v = W.var[i];
            if ((int)v.pos < cur) continue;                                      // overlapping: skipped (:745-753)
            cur = v.pos + v.l0;
            const bool anchored = c.alle[v.aoff + v.l0] == c.ref[v.pos];
            if (v.l0 == 1 && v.l1 == 1) subm += anchored ? 0 : 1;
            else if (v.l0 == 1 && anchored) ins += v.l1 - 1;
            else if (v.l1 == 1 && anchored) del += v.l0 - 1;
            else open = true;
        }
        if (open) return -1;
        if (ins == 0 && del == 0) return subm <= 2 ? subm : -1;
        if (subm == 0 && (ins == 0 || del == 0)) return ins + del;
        return -1;
    }
};

// ---------------------------------------------------------------------------------------------------------------------
// Commit of a solved cluster (rc == AVK_ST_OK after advance()): per-variant labels and metric rows are produced on the
// fly from the chosen solution, its exact-GT result and the basepair counters, and handed to the sink:
//   sink.variant(order index, expected, observed)      (already toggled for query entries, compare_benchmark.rs:109-123)
//   sink.metric(group, metric index, value)            (non-zero entries only; group 0 = joint, 1 + type otherwise)
// returns AVK_ST_OK, or the status the region ends with (AVK_ST_TP_UNDERFLOW / AVK_ST_TRUTH_FP) -- in which case the sink has
// not been called.
template <class Sink>
AVK_HD inline int commit_solution(const Solver &S, Sink &sink, u32 *ed1, u32 *ed2, u16 *type_mask) {
    const Work &W = S.w();
    const Cluster &c = S.c;
    const int n = c.N, ns = c.n_slots;
    const ResEnt R = W.res[S.best_r];
    // RECORD_BP totals (add_record_basepair_stats :455-522, wrapping u64 like a release build) + the TP underflow ensure
    u64 tot[TS_MAXSLOT][2];
    for (int s = 0; s < TS_MAXSLOT; ++s) tot[s][0] = tot[s][1] = 0;
    u64 truth_total = 0, query_total = 0;
    for (int i = 0; i < n; ++i) {
        const int exp_ = (int)((R.a1 >> i) & 1) + (int)((R.a2 >> i) & 1);
        const int obs_ = (int)((S.best_keep0 >> i) & 1) + (int)((S.best_keep1 >> i) & 1);
        if (exp_ < obs_) return AVK_ST_TRUTH_FP;                                  // assert! :322 (cannot happen: flips only remove ALTs)
        const u64 v = (u64)(W.zyg[i] == AVK_ZYG_HOM_ALT ? 2 : 1) * rec32(c, i, VI_RAW);
        const int side = S.is_truth(i) ? 0 : 1;
        tot[W.slot[i]][side] += v;
        if (side == 0) truth_total += v; else query_total += v;
    }
    const u64 tfn = W.bp[0][1], qfp = W.bp[0][3];
    const u64 ttp = 2 * truth_total - tfn, qtp = 2 * query_total - qfp;
    if (!(ttp >= (u64)W.bp[0][0]) || !(qtp >= (u64)W.bp[0][2])) return AVK_ST_TP_UNDERFLOW;
    // per-variant expected / observed (:226-258)
    for (int i = 0; i < n; ++i) {
        const bool tr = S.is_truth(i);
        const int exp_ = (int)((R.a1 >> i) & 1) + (int)((R.a2 >> i) & 1);
        const int obs_ = (int)((S.best_keep0 >> i) & 1) + (int)((S.best_keep1 >> i) & 1);
        sink.variant(i, tr ? exp_ : obs_, tr ? obs_ : exp_);
    }
    // rows: joint (s == -1) then one per slot; GT / HAP / WEIGHTED_HAP via add_truth_zygosity (grouped_metrics.rs:183-227) with
    // the query pass in the query columns (add_swap_benchmark :268-277)
    for (int s = -1; s < ns; ++s) {
        u64 gt[6] = {0, 0, 0, 0, 0, 0}, hap[4] = {0, 0, 0, 0}, whap[4] = {0, 0, 0, 0};
        for (int i = 0; i < n; ++i) {
            if (s >= 0 && W.slot[i] != s) continue;
            const int col = S.is_truth(i) ? 0 : 2;
            const int exp_ = (int)((R.a1 >> i) & 1) + (int)((R.a2 >> i) & 1);
            const int obs_ = (int)((S.best_keep0 >> i) & 1) + (int)((S.best_keep1 >> i) & 1);
            const u64 wgt = W.var[i].alted;
            const int mn = exp_ < obs_ ? exp_ : obs_;
            hap[col] += (u64)mn; whap[col] += (u64)mn * wgt;
            if (exp_ == obs_) gt[col] += 1;
            else {
                hap[col + 1] += (u64)(exp_ - obs_); whap[col + 1] += (u64)(exp_ - obs_) * wgt; gt[col + 1] += 1;
                if (obs_ > 0) gt[col == 0 ? 4 : 5] += 1;
            }
        }
        const int g = s < 0 ? 0 : 1 + S.slot_type(s);
        for (int m = 0; m < 6; ++m) if (gt[m]) sink.metric(g, AVK_M_GT + m, gt[m]);
        for (int m = 0; m < 4; ++m) {
            if (hap[m]) sink.metric(g, AVK_M_HAP + m, hap[m]);
            if (whap[m]) sink.metric(g, AVK_M_WEIGHTED_HAP + m, whap[m]);
            if (W.bp[1 + s][m]) sink.metric(g, AVK_M_BASEPAIR + m, (u64)W.bp[1 + s][m]);
        }
        u64 rb[4];
        if (s < 0) { rb[0] = ttp; rb[1] = tfn; rb[2] = qtp; rb[3] = qfp; }
        else {
            const u64 fn_ = W.bp[1 + s][1], fp_ = W.bp[1 + s][3];
            rb[0] = 2 * tot[s][0] - fn_; rb[1] = fn_; rb[2] = 2 * tot[s][1] - fp_; rb[3] = fp_;
        }
        for (int m = 0; m < 4; ++m) if (rb[m]) sink.metric(g, AVK_M_RECORD_BP + m, rb[m]);
    }
    u32 mask = supported_type_mask();                                             // every supported type gets a (possibly all-zero) entry (:444)
    for (int s = 0; s < ns; ++s) mask |= 1u << S.slot_type(s);
    *ed1 = R.ed1; *ed2 = R.ed2; *type_mask = (u16)mask;
    return AVK_ST_OK;
}

}  // namespace avk_ts
