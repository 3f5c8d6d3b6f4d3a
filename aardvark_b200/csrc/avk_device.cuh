// avk_device.cuh -- warp-cooperative device primitives of the haplotype-comparison path.
//
// One warp owns one cluster (or one alignment).  All 32 lanes execute these functions together
// with warp-uniform scalar arguments; lanes split either
//   * the BASES of one diagonal (4 bytes per lane, 128 bytes per warp step: unaligned 32-bit
//     loads built with funnel shifts, XOR, __ffs, __ballot_sync), or
//   * the DIAGONALS of one wavefront (one diagonal per lane),
// whichever the wavefront width calls for.  No tensor cores: this is integer DP (SURVEY.md 8d).
//
// Memory spaces.  Mem<true> addresses the CTA's dynamic shared memory with 32-bit byte offsets
// (LDS/STS, no generic-address arithmetic); Mem<false> uses 64-bit global addresses.  Every kernel
// is instantiated for one of the two, so the hot shared-memory tier never touches a generic pointer.
//
// Virtual sequences.  A haplotype is "the reference with ALT alleles spliced in", and most of it
// IS reference.  A sequence is therefore kept as a materialised prefix (up to the end of its last
// spliced ALT) plus an implicit tail that reads the reference window directly:
//       byte x  =  x < mlen ? data[x] : tail[x - mlen]          for x < len
// Appending reference (HaplotypeTracker::copy_reference) costs nothing, clones copy only the
// prefix, and when both sequences of a comparison read the same reference bytes the match is
// known without touching memory.  Logical content is exactly the reference's Vec<u8>.
//
// Sequences are raw bytes (the reference compares raw bytes, dynamic_wfa.rs:118, so N / IUPAC /
// soft-masked bases stay distinct symbols).  Every buffer has >= 8 readable bytes of slack.
//
// Semantics follow DWFALite::{extend,increase_edit_distance,update,finalize}
// (src/dwfa/dynamic_wfa.rs:68-245) exactly.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define AVK_FULL 0xffffffffu

typedef uint8_t u8;
typedef uint32_t u32;
typedef uint64_t u64;

extern __shared__ __align__(128) u8 avk_dyn_smem[];

namespace avk {

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

template <bool SMEM> struct Mem;
template <> struct Mem<true> {
    typedef u32 addr;
    static __device__ __forceinline__ u8 *p(addr a) { return avk_dyn_smem + a; }
};
template <> struct Mem<false> {
    typedef u64 addr;
    static __device__ __forceinline__ u8 *p(addr a) { return (u8 *)a; }
};
#define LD8(a) (*(const u8 *)M::p(a))
#define LD32(a) (*(const u32 *)M::p(a))
#define LDI(a) (*(const int *)M::p(a))
#define LD64(a) (*(const u64 *)M::p(a))
#define ST8(a, v) (*(u8 *)M::p(a) = (u8)(v))
#define ST32(a, v) (*(u32 *)M::p(a) = (u32)(v))
#define ST64(a, v) (*(u64 *)M::p(a) = (u64)(v))

// ---- work counters (DESIGN.md "algorithmic work"); live in the arena header ---------------------
enum { WK_COOP = 8, WK_CELLS = 16, WK_MATCHED = 24, WK_ALIGN = 32, WK_SPOPS = 36, WK_XPOPS = 40, ARENA_HDR = 48 };
// WK_COOP != 0: the warp is the master warp of a k_compare_coop CTA and may hand wide wavefronts to the whole CTA

// counters that several warps of a team may bump at the same time (k_compare_team): atomic adds
template <bool SMEM>
__device__ __forceinline__ void wk_add64(typename Mem<SMEM>::addr a, u64 v) { atomicAdd((unsigned long long *)Mem<SMEM>::p(a), (unsigned long long)v); }
template <bool SMEM>
__device__ __forceinline__ void wk_add32(typename Mem<SMEM>::addr a, u32 v) { atomicAdd((u32 *)Mem<SMEM>::p(a), v); }

// ---- unaligned 32-bit load: two aligned loads + funnel shift ------------------------------------
template <bool SMEM>
__device__ __forceinline__ u32 ld4u(typename Mem<SMEM>::addr a) {
    typedef Mem<SMEM> M;
    const typename M::addr w = a & ~(typename M::addr)3;
    return __funnelshift_r(LD32(w), LD32(w + 4), ((u32)a & 3u) * 8u);   // shift 0 returns the first word
}

// ---- byte copy, any alignment ---------------------------------------------------------------------
template <bool SMEM>
__device__ __noinline__ void warp_copy(typename Mem<SMEM>::addr dst, typename Mem<SMEM>::addr src, int n) {
    typedef Mem<SMEM> M;
    const int lane = lane_id();
    if (n <= 32) {
        __syncwarp();
        if (lane < n) ST8(dst + lane, LD8(src + lane));
        return;
    }
    const int head = (int)((4u - ((u32)dst & 3u)) & 3u);
    __syncwarp();
    if (lane < head) ST8(dst + lane, LD8(src + lane));
    const int nw = (n - head) >> 2;
#pragma unroll 1
    for (int i = lane; i < nw; i += 32) ST32(dst + head + 4 * i, ld4u<SMEM>(src + head + 4 * i));
    const int done = head + (nw << 2);
    if (done + lane < n) ST8(dst + done + lane, LD8(src + done + lane));
}

// ---- longest common prefix of two physical byte ranges (128 bytes per step) -----------------------
template <bool SMEM>
__device__ __forceinline__ int raw_lcp(typename Mem<SMEM>::addr a, typename Mem<SMEM>::addr b, int maxn) {
    const int lane = lane_id();
    int total = 0;
#pragma unroll 1
    while (total < maxn) {
        const int k = total + 4 * lane;
        int good = 0;   // equal bytes in this lane's word, capped by the bytes that exist
        const int valid = min(4, maxn - k);
        if (valid > 0) {
            const u32 x = ld4u<SMEM>(a + k) ^ ld4u<SMEM>(b + k);
            good = x ? ((__ffs(x) - 1) >> 3) : 4;
            good = min(good, valid);
        }
        const unsigned m = __ballot_sync(AVK_FULL, good == 4);
        if (m == AVK_FULL) { total += 128; continue; }
        const int f = __ffs(~m) - 1;
        total += 4 * f + __shfl_sync(AVK_FULL, good, f);
        break;
    }
    return min(total, maxn);
}

// ---- virtual sequence ---------------------------------------------------------------------------------
template <bool SMEM>
struct VSeq {
    typename Mem<SMEM>::addr data;   // materialised prefix
    typename Mem<SMEM>::addr tail;   // address of the byte at logical offset mlen (a reference position)
    int mlen;                        // materialised bytes
    int len;                         // logical length
    __device__ __forceinline__ typename Mem<SMEM>::addr at(int x) const { return x < mlen ? data + x : tail + (x - mlen); }
    __device__ __forceinline__ int run(int x, int cap) const { return x < mlen ? mlen - x : cap; }   // bytes left in this piece
};

// number of equal leading bytes of A[ia..] and B[ib..]; warp-uniform.  At most three pieces.
template <bool SMEM>
__device__ __noinline__ int vs_lcp(const VSeq<SMEM> A, int ia, const VSeq<SMEM> B, int ib) {
    const int maxn = min(A.len - ia, B.len - ib);
    int total = 0;
#pragma unroll 1
    while (total < maxn) {
        const int xa = ia + total, xb = ib + total;
        const int n = min(min(A.run(xa, maxn), B.run(xb, maxn)), maxn - total);
        const typename Mem<SMEM>::addr pa = A.at(xa), pb = B.at(xb);
        if (pa == pb) { total += n; continue; }   // both read the same reference bytes: equal by construction
        const int m = raw_lcp<SMEM>(pa, pb, n);
        total += m;
        if (m < n) break;
    }
    return total;
}

// ---- DWFA -------------------------------------------------------------------------------------------
// State: ed, wavefront wf[0 .. 2*ed] (int32, bases consumed in `other` == B), kept by the caller.
// baseline (A) offset of entry i is wf[i] + ed - i (dynamic_wfa.rs:114).
struct Reach {
    int max_base;   // max_i (wf[i] + ed - i)     (maximum_baseline_distance :201-208)
    int max_other;  // max_i wf[i]                (maximum_other_distance    :212-215)
    bool full;      // any i: base >= la && other >= lb (reached_full_diagonal :237-245)
};

// extend(): dynamic_wfa.rs:94-130.  Narrow wavefronts: one warp-wide LCP per diagonal.  Wide
// wavefronts: one diagonal per lane, one word compare each; lanes whose word matched completely are
// finished with a warp-wide LCP so that one long run does not serialise the warp.
template <bool SMEM>
__device__ __noinline__ Reach dwfa_extend(typename Mem<SMEM>::addr wf, int ed, const VSeq<SMEM> A, const VSeq<SMEM> B,
                                          typename Mem<SMEM>::addr wk) {
    typedef Mem<SMEM> M;
    const int lane = lane_id();
    const int n = 2 * ed + 1;
    const int la = A.len, lb = B.len;
    int mb = -1, mo = -1;
    bool full = false;
    int matched = 0;
    if (n <= 3) {
#pragma unroll 1
        for (int i = 0; i < n; ++i) {
            int d = LDI(wf + 4 * i);
            int boff = d + ed - i;
            int ext = 0;
            if (boff < la && d < lb) ext = vs_lcp<SMEM>(A, boff, B, d);
            d += ext; boff += ext; matched += ext;
            __syncwarp();
            if (ext && lane == 0) ST32(wf + 4 * i, d);
            mb = max(mb, boff); mo = max(mo, d);
            full = full || (boff >= la && d >= lb);
        }
    } else {
#pragma unroll 1
        for (int base = 0; base < n; base += 32) {
            const int i = base + lane;
            const bool act = i < n;
            int d = act ? LDI(wf + 4 * i) : 0;
            int boff = d + ed - i;
            const int d0 = d;
            bool more = false;
            if (act && boff < la && d < lb) {
                const int lim = min(la - boff, lb - d);
                const int valid = min(min(4, lim), min(A.run(boff, 4), B.run(d, 4)));
                const typename M::addr pa = A.at(boff), pb = B.at(d);
                int good = valid;
                if (pa != pb) {
                    const u32 x = ld4u<SMEM>(pa) ^ ld4u<SMEM>(pb);
                    good = min(x ? ((__ffs(x) - 1) >> 3) : 4, valid);
                }
                d += good; boff += good;
                more = (good == valid) && good < lim;
            }
            unsigned m = __ballot_sync(AVK_FULL, more);
#pragma unroll 1
            while (m) {
                const int src = __ffs(m) - 1;
                m &= m - 1;
                const int dd = __shfl_sync(AVK_FULL, d, src);
                const int bb = __shfl_sync(AVK_FULL, boff, src);
                const int ext = vs_lcp<SMEM>(A, bb, B, dd);
                if (lane == src) { d += ext; boff += ext; }
            }
            if (act) {
                if (d != d0) ST32(wf + 4 * i, d);
                matched += d - d0;
                mb = max(mb, boff); mo = max(mo, d);
                full = full || (boff >= la && d >= lb);
            }
        }
        mb = __reduce_max_sync(AVK_FULL, mb);
        mo = __reduce_max_sync(AVK_FULL, mo);
        full = __any_sync(AVK_FULL, full);
        matched = __reduce_add_sync(AVK_FULL, matched);
    }
    __syncwarp();
    if (lane == 0) { wk_add64<SMEM>(wk + WK_CELLS, (u64)n); wk_add64<SMEM>(wk + WK_MATCHED, (u64)matched); }
    Reach r;
    r.max_base = mb; r.max_other = mo; r.full = full;
    return r;
}

// increase_edit_distance() without the re-extend: dynamic_wfa.rs:152-168, in place.
// new[i] = max(old[i], old[i-1]+1, old[i-2]+1) over the entries that exist; chunks are processed from
// the top so that every read of old[] precedes the write that replaces it.
template <bool SMEM>
__device__ __noinline__ void dwfa_grow(typename Mem<SMEM>::addr wf, int old_ed) {
    typedef Mem<SMEM> M;
    const int lane = lane_id();
    const int n_old = 2 * old_ed + 1;
    const int n_new = n_old + 2;
#pragma unroll 1
    for (int base = ((n_new - 1) >> 5) << 5; base >= 0; base -= 32) {
        const int i = base + lane;
        int v = 0;
        if (i < n_new) {
            if (i < n_old) v = LDI(wf + 4 * i);
            if (i >= 1 && i - 1 < n_old) v = max(v, LDI(wf + 4 * (i - 1)) + 1);
            if (i >= 2 && i - 2 < n_old) v = max(v, LDI(wf + 4 * (i - 2)) + 1);
        }
        __syncwarp();
        if (i < n_new) ST32(wf + 4 * i, v);
    }
    __syncwarp();
}


enum { DWFA_OK = 0, DWFA_MAX_ED = 1 };

// ---- CTA-cooperative DWFA for wide wavefronts (SV / long-indel clusters) -------------------------------------
// A 10 kbp event means an edit distance of ~10^4: 10^8 wavefront cells in ONE alignment, far too much for one warp.
// In k_compare_coop one master warp runs the solver; when a wavefront reaches COOP_MIN_ED it posts the alignment as
// a job and all COOP_THREADS threads of the CTA advance it together: wavefront ping-ponged in shared memory, one
// diagonal per thread (thread-serial word compares), grow + extend fused so that a step costs one barrier
// (__syncthreads_or doubles as the termination vote).  Same recurrence and stop rules as dwfa_grow/dwfa_extend.
enum { COOP_THREADS = 512, COOP_MIN_ED = 48, COOP_JOB_BYTES = 128, DWFA_COOP_SPILL = 2 };
struct CoopJob {
    u64 wf;                                  // the node's wavefront ints (global memory)
    u64 a_data, a_tail, b_data, b_tail;
    int a_mlen, a_len, b_mlen, b_len;
    int ed, max_ed, to_full, status, exit_, cap_ints;
    unsigned long long matched, cells;
};
static_assert(sizeof(CoopJob) <= COOP_JOB_BYTES, "CoopJob must fit its slot");

__device__ __forceinline__ int lcp_thread(const VSeq<false> &A, int ia, const VSeq<false> &B, int ib) {
    typedef Mem<false> M;
    const int maxn = min(A.len - ia, B.len - ib);
    int total = 0;
#pragma unroll 1
    while (total < maxn) {
        const int xa = ia + total, xb = ib + total;
        const int n = min(min(A.run(xa, maxn), B.run(xb, maxn)), maxn - total);
        const u64 pa = A.at(xa), pb = B.at(xb);
        if (pa == pb) { total += n; continue; }
        int k = 0;
#pragma unroll 1
        while (k < n) {
            const u32 x = ld4u<false>(pa + k) ^ ld4u<false>(pb + k);
            const int good = min(x ? ((__ffs(x) - 1) >> 3) : 4, n - k);
            k += good;
            if (x && good < 4) break;
        }
        total += k;
        if (k < n) break;
    }
    return total;
}

// ---- fast path of the CTA-wide DWFA: both sequences staged in shared memory, 16-bit wavefront --------------------------------
// Shared-memory layout behind the job slot (area = 8 * cap_ints bytes, the same allocation the 32-bit path ping-pongs in):
//   [sequence A bytes, 8 bytes slack][sequence B bytes, 8 bytes slack][cur: cap16 u16][nxt: cap16 u16]
// The sequences take what they need and the two wavefront buffers share the rest (208 KB in all at the default capacity:
// two 45 kbp haplotypes still leave room for edit distances up to ~14,000).  Per wavefront entry a thread then
// executes: three 16-bit shared loads for the recurrence (dynamic_wfa.rs:152-168), one byte compare that ends the extension
// of 3 diagonals in 4 on unrelated sequence, and only for the others an aligned-word XOR + ffs loop (4 bases per step) --
// ~20 instructions instead of ~57 with virtual sequences read through 64-bit global addresses.
__device__ __forceinline__ u32 lds4u(const u8 *p) {          // unaligned 32-bit read from shared memory: two aligned words + funnel shift
    const u32 *w = (const u32 *)((uintptr_t)p & ~(uintptr_t)3);
    return __funnelshift_r(w[0], w[1], ((u32)(uintptr_t)p & 3u) * 8u);
}
__device__ __forceinline__ int lcp_staged(const u8 *sa, int ia, int la, const u8 *sb, int ib, int lb) {   // ia < la && ib < lb
    if (sa[ia] != sb[ib]) return 0;
    const int maxn = min(la - ia, lb - ib);
    int k = 1;
#pragma unroll 1
    while (k < maxn) {
        const u32 x = lds4u(sa + ia + k) ^ lds4u(sb + ib + k);
        if (x) { k += (__ffs(x) - 1) >> 3; break; }
        k += 4;
    }
    return min(k, maxn);
}
// stage the logical bytes [0, len) of a virtual sequence into shared memory (4 bytes per thread and trip)
__device__ __forceinline__ void coop_stage(u8 *dst, const VSeq<false> &S) {
    typedef Mem<false> M;
    const int tid = threadIdx.x, T = blockDim.x;
    const int words = (S.len + 3) >> 2;
#pragma unroll 1
    for (int wi = tid; wi < words; wi += T) {
        const int x = 4 * wi;
        u32 v;
        if (x + 4 <= S.mlen) v = ld4u<false>(S.data + x);
        else if (x >= S.mlen) v = ld4u<false>(S.tail + (x - S.mlen));
        else { v = 0; for (int k = 0; k < 4; ++k) v |= (u32)LD8(S.at(min(x + k, S.len - 1))) << (8 * k); }   // the word that straddles the two pieces
        *(u32 *)(dst + x) = v;
    }
}
// entries of each of the two 16-bit wavefront buffers once both sequences are staged (<= 0: they do not fit); offsets must
// stay below 65535 even with the +1 per step of an untrimmed wavefront
__device__ __forceinline__ int coop_staged_cap16(int la, int lb, int cap_ints) {
    const long long seq = (long long)((la + 8 + 3) & ~3) + ((lb + 8 + 3) & ~3);
    long long cap = (8LL * cap_ints - seq) / 4;
    cap = min(cap, 2LL * (64000 - lb));
    return (int)max(cap, 0LL);
}
// unaligned 32-bit read at a shared-window byte address (two aligned ld.shared + funnel shift); the address is the 32-bit
// shared-space one so the reads stay LDS -- through a generic u8 pointer the compiler falls back to 64-bit generic loads
__device__ __forceinline__ u32 lds4u_s(u32 saddr) {
    u32 w0, w1;
    const u32 a = saddr & ~3u;
    asm("ld.shared.u32 %0, [%1];" : "=r"(w0) : "r"(a));
    asm("ld.shared.u32 %0, [%1+4];" : "=r"(w1) : "r"(a));
    return __funnelshift_r(w0, w1, (saddr & 3u) * 8u);
}
// equal leading bytes of a[ia..la) and b[ib..lb), ia < la && ib < lb, a/b shared-space addresses: four bases per step for every
// lane alike (on unrelated sequence three diagonals in four end at the first base: a byte test first and a word loop for the
// rest would leave the loop to a quarter of the lanes at the full issue cost)
__device__ __forceinline__ int lcp_staged_w(u32 sa, int ia, int la, u32 sb, int ib, int lb) {
    const int maxn = min(la - ia, lb - ib);
    u32 pa = sa + (u32)ia, pb = sb + (u32)ib;
    int k = 0;
#pragma unroll 1
    for (;;) {
        const u32 x = lds4u_s(pa + k) ^ lds4u_s(pb + k);
        if (x) { k += (__ffs(x) - 1) >> 3; break; }
        k += 4;
        if (k >= maxn) break;
    }
    return min(k, maxn);
}
// Wavefront entries are stored as offset + 1 with 0 = "no diagonal": two zero entries in front of each buffer and the zeroes
// behind the old wavefront stand for the missing neighbours, so increase_edit_distance() (dynamic_wfa.rs:152-168) is three loads
// and two max operations without a single bounds test.
template <bool TO_FULL>
__device__ __noinline__ void coop_dwfa_body_staged_t() {
    CoopJob &J = *(CoopJob *)avk_dyn_smem;
    const int tid = threadIdx.x, T = blockDim.x;
    VSeq<false> A, B;
    A.data = J.a_data; A.tail = J.a_tail; A.mlen = J.a_mlen; A.len = J.a_len;
    B.data = J.b_data; B.tail = J.b_tail; B.mlen = J.b_mlen; B.len = J.b_len;
    const int la = A.len, lb = B.len, max_ed = J.max_ed;
    u8 *sa = avk_dyn_smem + COOP_JOB_BYTES;
    u8 *sb = sa + ((la + 8 + 3) & ~3);
    const int cap = (coop_staged_cap16(la, lb, J.cap_ints) - 4) & ~1;      // (two pad entries per buffer; even: both buffers 4-byte aligned)
    unsigned short *cur = (unsigned short *)(sb + ((lb + 8 + 3) & ~3)) + 2, *nxt = cur + cap + 2;
    const int e_cap = (cap - 3) / 2;
    int *gw = (int *)(uintptr_t)J.wf;
    int e = J.ed, status = DWFA_OK;
    const u32 sa_s = (u32)__cvta_generic_to_shared(sa), sb_s = (u32)__cvta_generic_to_shared(sb);
    coop_stage(sa, A);
    coop_stage(sb, B);
#pragma unroll 1
    for (int i = tid; i < 2 * cap + 4; i += T) cur[i - 2] = 0;       // both buffers and their pads (they are adjacent)
    __syncthreads();
#pragma unroll 1
    for (int i = tid; i < 2 * e + 1; i += T) cur[i] = (unsigned short)(gw[i] + 1);
    __syncthreads();
    unsigned long long matched = 0, cells = 0;
    u32 reached = 0;
#pragma unroll 1
    for (int i = tid; i < 2 * e + 1; i += T) {           // extend() of the wavefront as it stands
        int d = (int)cur[i] - 1;
        int boff = d + e - i;
        if (boff < la && d < lb) { const int ext = lcp_staged_w(sa_s, boff, la, sb_s, d, lb); d += ext; boff += ext; matched += ext; cur[i] = (unsigned short)(d + 1); }
        const u32 ra = boff >= la, rb = d >= lb;
        reached |= TO_FULL ? (ra & rb) : (ra | rb);
    }
    cells += 2 * e + 1;
    int stop = __syncthreads_or(reached != 0u);
#pragma unroll 1
    while (!stop) {
        e += 1;
        if (e > max_ed) { status = DWFA_MAX_ED; break; }                 // *ed stays incremented, wavefront not grown
        if (e > e_cap) { status = DWFA_COOP_SPILL; e -= 1; break; }      // does not fit shared memory: back to the warp path
        const int n = 2 * e + 1;
        reached = 0;
        // two adjacent diagonals per thread: their five neighbours are two aligned 32-bit loads, increase_edit_distance() for
        // both is one byte permute and three 16-bit-pair operations, and the two extensions are independent work for one thread
#pragma unroll 1
        for (int i = 2 * tid; i < n; i += 2 * T) {
            const u32 w0 = *(const u32 *)(cur + i - 2), w1 = *(const u32 *)(cur + i);      // (cur[i-2], cur[i-1]), (cur[i], cur[i+1])
            const u32 mid = __byte_perm(w0, w1, 0x5432);                                   // (cur[i-1], cur[i])
            const u32 nv = __vmaxu2(w1, __vadd2(__vmaxu2(w0, mid), 0x00010001u));
            const bool two = i + 1 < n;
            int d0 = (int)(nv & 0xffffu) - 1, d1 = (int)(nv >> 16) - 1;
            int b0 = d0 + e - i, b1 = d1 + e - i - 1;
            if (b0 < la && d0 < lb) { const int ext = lcp_staged_w(sa_s, b0, la, sb_s, d0, lb); d0 += ext; b0 += ext; matched += ext; }
            if (two && b1 < la && d1 < lb) { const int ext = lcp_staged_w(sa_s, b1, la, sb_s, d1, lb); d1 += ext; b1 += ext; matched += ext; }
            if (two) *(u32 *)(nxt + i) = (u32)(d0 + 1) | ((u32)(d1 + 1) << 16);
            else nxt[i] = (unsigned short)(d0 + 1);                                        // (entries behind the wavefront stay 0)
            const u32 ra0 = b0 >= la, rb0 = d0 >= lb, ra1 = two && b1 >= la, rb1 = two && d1 >= lb;
            reached |= TO_FULL ? ((ra0 & rb0) | (ra1 & rb1)) : (ra0 | rb0 | ra1 | rb1);
        }
        cells += n;
        stop = __syncthreads_or(reached != 0u);
        unsigned short *t = cur; cur = nxt; nxt = t;
    }
    const int n_out = 2 * (status == DWFA_MAX_ED ? e - 1 : e) + 1;
#pragma unroll 1
    for (int i = tid; i < n_out; i += T) gw[i] = (int)cur[i] - 1;
    if (matched) atomicAdd(&J.matched, matched);
    if (tid == 0) { J.ed = e; J.status = status; J.cells = cells; }
    __threadfence_block();
    __syncthreads();
}
__device__ __forceinline__ void coop_dwfa_body_staged() {
    if (((CoopJob *)avk_dyn_smem)->to_full) coop_dwfa_body_staged_t<true>(); else coop_dwfa_body_staged_t<false>();
}

// ---- fastest path of the CTA-wide DWFA: 2-bit packed sequences, four diagonals per thread and trip ---------------------------------
// When both sequences are plain upper-case ACGT (the reference compares raw bytes, dynamic_wfa.rs:118, so anything else --
// N, IUPAC, soft-masked bases -- takes the byte path above) they are staged as 2 bits per base, 16 bases per word.  Layout
// behind the job slot:  [A words + 2][B words + 2][2 pad][cur: cap16 u16][2 pad][nxt: cap16 u16]
// A wavefront entry is stored as offset + 1 with 0 meaning "no diagonal", which turns the recurrence (dynamic_wfa.rs:152-168)
// into three unconditional max operations: the two pad entries before and the zeroed entries behind a wavefront stand for
// its missing neighbours.  A thread takes one contiguous run of diagonals, FOUR per trip: one 64-bit and one 32-bit shared load
// bring the six old entries they depend on, one 64-bit store writes the four new ones; the extension of a diagonal compares 16
// bases per step (two words per sequence, funnel shift to the base offset, XOR, find-first-set), and the four extensions are
// independent, so their shared-memory latencies overlap.
enum { PK_DIAGS = 4 };
__device__ int g_avk_packed_dwfa = 0;   // AVK_PACKED_DWFA=1: take this path when the sequences allow it (off by default: measured slower
                                        // than the byte-staged path on the wide-wavefront microbenchmark, DESIGN.md section 5)
__device__ __forceinline__ u32 pk_code4(u32 v, bool &bad) {      // four ASCII bases -> 8 bits; anything but ACGT sets bad
    u32 out = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const u32 c = (v >> (8 * k)) & 0xffu;
        bad = bad || (c & 0xe0u) != 0x40u || !((0x0010008au >> (c & 31u)) & 1u);   // 'A' 0x41, 'C' 0x43, 'G' 0x47, 'T' 0x54
        out |= ((c >> 1) & 3u) << (2 * k);
    }
    return out;
}
// stage the logical bases [0, len) of a virtual sequence, 16 per word (the tail of the last word and two slack words are zero)
__device__ __forceinline__ bool coop_stage_packed(u32 *dst, const VSeq<false> &S) {
    typedef Mem<false> M;
    const int tid = threadIdx.x, T = blockDim.x;
    const int words = (S.len + 15) >> 4;
    bool bad = false;
#pragma unroll 1
    for (int wi = tid; wi < words + 2; wi += T) {
        u32 w = 0;
        if (wi < words) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int x = 16 * wi + 4 * q;
                if (x >= S.len) break;
                u32 v;
                if (x + 4 <= S.mlen) v = ld4u<false>(S.data + x);
                else if (x >= S.mlen && x + 4 <= S.len) v = ld4u<false>(S.tail + (x - S.mlen));
                else { v = 0; for (int k = 0; k < 4; ++k) v |= (u32)(x + k < S.len ? LD8(S.at(x + k)) : (u8)'A') << (8 * k); }   // straddles the two pieces or the end
                w |= pk_code4(v, bad) << (8 * q);
            }
        }
        dst[wi] = w;
    }
    return bad;
}
// equal leading bases of A[ia..la) and B[ib..lb), ia < la && ib < lb
__device__ __forceinline__ int lcp_packed(const u32 *pa, int ia, int la, const u32 *pb, int ib, int lb) {
    const int maxn = min(la - ia, lb - ib);
    int k = 0;
#pragma unroll 1
    for (;;) {
        const int xa = ia + k, xb = ib + k;
        const u32 a = __funnelshift_r(pa[xa >> 4], pa[(xa >> 4) + 1], 2 * (xa & 15));
        const u32 b = __funnelshift_r(pb[xb >> 4], pb[(xb >> 4) + 1], 2 * (xb & 15));
        const u32 x = a ^ b;
        if (x) { k += (__ffs((int)x) - 1) >> 1; break; }
        k += 16;
        if (k >= maxn) break;
    }
    return min(k, maxn);
}
// shared-memory words the packed layout needs for wavefronts of `cap` entries each
__device__ __forceinline__ long long coop_packed_bytes(int la, int lb, long long cap) {
    return 4LL * (((la + 15) >> 4) + 2 + ((lb + 15) >> 4) + 2) + 2LL * (2 * (cap + 16) + 8);
}
__device__ __forceinline__ int coop_packed_cap16(int la, int lb, int cap_ints) {
    long long cap = (8LL * cap_ints - 4LL * (((la + 15) >> 4) + ((lb + 15) >> 4) + 4) - 64) / 4 - 16;
    cap = min(cap, 2LL * (64000 - lb));
    cap &= ~7LL;
    return (int)max(cap, 0LL);
}
// returns false (nothing done, every thread agrees) when a sequence holds anything but ACGT
template <bool TO_FULL>
__device__ __noinline__ bool coop_dwfa_body_packed() {
    CoopJob &J = *(CoopJob *)avk_dyn_smem;
    const int tid = threadIdx.x, T = blockDim.x;
    VSeq<false> A, B;
    A.data = J.a_data; A.tail = J.a_tail; A.mlen = J.a_mlen; A.len = J.a_len;
    B.data = J.b_data; B.tail = J.b_tail; B.mlen = J.b_mlen; B.len = J.b_len;
    const int la = A.len, lb = B.len, max_ed = J.max_ed;
    u32 *pa = (u32 *)(avk_dyn_smem + COOP_JOB_BYTES);
    u32 *pb = pa + ((la + 15) >> 4) + 2;
    const int cap = coop_packed_cap16(la, lb, J.cap_ints);
    // wavefront buffers: 16-byte aligned at entry 0, with 8 entries (only 2 are read) of zero padding in front
    unsigned short *w0 = (unsigned short *)((((uintptr_t)(pb + ((lb + 15) >> 4) + 2)) + 15) & ~(uintptr_t)15) + 8;
    unsigned short *w1 = w0 + cap + 16;
    const int e_cap = (cap - 3) / 2;
    int *gw = (int *)(uintptr_t)J.wf;
    int e = J.ed, status = DWFA_OK;
    bool bad = coop_stage_packed(pa, A);
    bad = coop_stage_packed(pb, B) || bad;
    if (__syncthreads_or(bad)) return false;
    unsigned short *cur = w0, *nxt = w1;
#pragma unroll 1
    for (int i = tid; i < cap + 16; i += T) { w0[i - 8] = 0; w1[i - 8] = 0; }
    __syncthreads();
#pragma unroll 1
    for (int i = tid; i < 2 * e + 1; i += T) cur[i] = (unsigned short)(gw[i] + 1);
    __syncthreads();
    unsigned long long matched = 0, cells = 0;
    bool flag = false;
#pragma unroll 1
    for (int i = tid; i < 2 * e + 1; i += T) {           // extend() of the wavefront as it stands
        int d = (int)cur[i] - 1;
        int boff = d + e - i;
        if (boff < la && d < lb) { const int ext = lcp_packed(pa, boff, la, pb, d, lb); d += ext; boff += ext; matched += ext; cur[i] = (unsigned short)(d + 1); }
        flag = flag || (TO_FULL ? (boff >= la && d >= lb) : (boff >= la || d >= lb));
    }
    cells += 2 * e + 1;
    int stop = __syncthreads_or(flag);
#pragma unroll 1
    while (!stop) {
        e += 1;
        if (e > max_ed) { status = DWFA_MAX_ED; break; }                 // *ed stays incremented, wavefront not grown
        if (e > e_cap) { status = DWFA_COOP_SPILL; e -= 1; break; }      // does not fit shared memory: back to the warp path
        const int n = 2 * e + 1;
        // every thread takes one contiguous run of diagonals, a multiple of PK_DIAGS long: the step ends with a barrier, so the
        // runs must be as equal as they can be
        const int per = (((n + T - 1) / T) + PK_DIAGS - 1) & ~(PK_DIAGS - 1);
        const int i_end = min(n, (tid + 1) * per);
        u32 reached = 0;
#pragma unroll 1
        for (int i0 = tid * per; i0 < i_end; i0 += PK_DIAGS) {
            // old entries i0 - 2 .. i0 + 3 (stored + 1; 0 = absent: the pads in front, the zeroes behind the old wavefront)
            const uint2 v = *(const uint2 *)(cur + i0);
            const u32 p = *(const u32 *)(cur + i0 - 2);
            u32 o[PK_DIAGS + 2];
            o[0] = p & 0xffffu; o[1] = p >> 16;
            o[2] = v.x & 0xffffu; o[3] = v.x >> 16; o[4] = v.y & 0xffffu; o[5] = v.y >> 16;
            u32 r[PK_DIAGS];
#pragma unroll
            for (int j = 0; j < PK_DIAGS; ++j) {
                // increase_edit_distance(): max(old[i], old[i - 1] + 1, old[i - 2] + 1) on the + 1 representation; an absent
                // neighbour contributes 0 or 1, below every real entry
                int d = (int)max(o[j + 2], max(o[j + 1], o[j]) + 1u) - 1;
                int boff = d + e - (i0 + j);
                const bool live = i0 + j < n;
                if (live && boff < la && d < lb) { const int ext = lcp_packed(pa, boff, la, pb, d, lb); d += ext; boff += ext; matched += ext; }
                const u32 ra = boff >= la, rb = d >= lb;
                reached |= live ? (TO_FULL ? (ra & rb) : (ra | rb)) : 0u;
                r[j] = live ? (u32)(d + 1) : 0u;
            }
            uint2 w;
            w.x = r[0] | (r[1] << 16); w.y = r[2] | (r[3] << 16);
            *(uint2 *)(nxt + i0) = w;
        }
        cells += n;
        stop = __syncthreads_or(reached != 0u);
        unsigned short *t = cur; cur = nxt; nxt = t;
    }
    const int n_out = 2 * (status == DWFA_MAX_ED ? e - 1 : e) + 1;
#pragma unroll 1
    for (int i = tid; i < n_out; i += T) gw[i] = (int)cur[i] - 1;
    if (matched) atomicAdd(&J.matched, matched);
    if (tid == 0) { J.ed = e; J.status = status; J.cells = cells; }
    __threadfence_block();
    __syncthreads();
    return true;
}

// executed by every thread of the CTA; the job is in CoopJob at the start of dynamic shared memory
__device__ __noinline__ void coop_dwfa_body() {
    CoopJob &J = *(CoopJob *)avk_dyn_smem;
    // plain ACGT on both sides and room for the wavefront to grow: 2-bit packed path (declines when it meets another byte)
    if (g_avk_packed_dwfa && J.a_len < 64000 && J.b_len < 64000 && J.a_len > 0 && J.b_len > 0 && coop_packed_cap16(J.a_len, J.b_len, J.cap_ints) >= 2 * J.ed + 256) {
        if (J.to_full ? coop_dwfa_body_packed<true>() : coop_dwfa_body_packed<false>()) return;
    }
    // both sequences fit beside a 16-bit wavefront with room to grow: byte-staged path
    if (J.a_len < 64000 && J.b_len < 64000 && coop_staged_cap16(J.a_len, J.b_len, J.cap_ints) >= 2 * J.ed + 256) { coop_dwfa_body_staged(); return; }
    int *cur = (int *)(avk_dyn_smem + COOP_JOB_BYTES), *nxt = cur + J.cap_ints;
    const int tid = threadIdx.x, T = blockDim.x;
    VSeq<false> A, B;
    A.data = J.a_data; A.tail = J.a_tail; A.mlen = J.a_mlen; A.len = J.a_len;
    B.data = J.b_data; B.tail = J.b_tail; B.mlen = J.b_mlen; B.len = J.b_len;
    const int la = A.len, lb = B.len, max_ed = J.max_ed, e_cap = (J.cap_ints - 3) / 2;
    const bool to_full = J.to_full != 0;
    int *gw = (int *)(uintptr_t)J.wf;
    int e = J.ed, status = DWFA_OK;
    if (e > e_cap) {      // resumed past what cur / nxt hold (an earlier update of this alignment spilled): straight back to the warp path
        if (tid == 0) { J.status = DWFA_COOP_SPILL; J.cells = 0; }
        __syncthreads();
        return;
    }
    unsigned long long matched = 0, cells = 0;
    bool flag = false;
#pragma unroll 1
    for (int i = tid; i < 2 * e + 1; i += T) {           // extend() of the wavefront as it stands
        int d = gw[i];
        int boff = d + e - i;
        if (boff < la && d < lb) { const int ext = lcp_thread(A, boff, B, d); d += ext; boff += ext; matched += ext; }
        cur[i] = d;
        flag = flag || (to_full ? (boff >= la && d >= lb) : (boff >= la || d >= lb));
    }
    cells += 2 * e + 1;
    int stop = __syncthreads_or(flag);
#pragma unroll 1
    while (!stop) {
        e += 1;
        if (e > max_ed) { status = DWFA_MAX_ED; break; }                 // *ed stays incremented, wavefront not grown
        if (e > e_cap) { status = DWFA_COOP_SPILL; e -= 1; break; }      // does not fit shared memory: back to the warp path
        const int n = 2 * e + 1, n_old = n - 2;
        flag = false;
#pragma unroll 1
        for (int i = tid; i < n; i += T) {
            int d = 0;                                                   // increase_edit_distance(): dynamic_wfa.rs:152-168
            if (i < n_old) d = cur[i];
            if (i >= 1 && i - 1 < n_old) d = max(d, cur[i - 1] + 1);
            if (i >= 2 && i - 2 < n_old) d = max(d, cur[i - 2] + 1);
            int boff = d + e - i;
            if (boff < la && d < lb) { const int ext = lcp_thread(A, boff, B, d); d += ext; boff += ext; matched += ext; }
            nxt[i] = d;
            flag = flag || (to_full ? (boff >= la && d >= lb) : (boff >= la || d >= lb));
        }
        cells += n;
        stop = __syncthreads_or(flag);
        int *t = cur; cur = nxt; nxt = t;
    }
    const int n_out = 2 * (status == DWFA_MAX_ED ? e - 1 : e) + 1;
#pragma unroll 1
    for (int i = tid; i < n_out; i += T) gw[i] = cur[i];
    if (matched) atomicAdd(&J.matched, matched);
    if (tid == 0) { J.ed = e; J.status = status; J.cells = cells; }
    __threadfence_block();
    __syncthreads();
}

// master warp: post the job, work on it with everybody else, collect the result
__device__ __noinline__ int dwfa_run_coop(u64 wf, int *ed, int max_ed, const VSeq<false> A, const VSeq<false> B, bool to_full, u64 wk) {
    typedef Mem<false> M;
    CoopJob &J = *(CoopJob *)avk_dyn_smem;
    __syncwarp();
    if (lane_id() == 0) {
        J.wf = wf; J.a_data = A.data; J.a_tail = A.tail; J.b_data = B.data; J.b_tail = B.tail;
        J.a_mlen = A.mlen; J.a_len = A.len; J.b_mlen = B.mlen; J.b_len = B.len;
        J.ed = *ed; J.max_ed = max_ed; J.to_full = to_full ? 1 : 0; J.status = 0; J.exit_ = 0; J.matched = 0; J.cells = 0;
    }
    __threadfence();                                   // the wavefront ints were written by this warp through global memory
    __syncwarp();
    asm volatile("bar.sync 1, %0;" ::"r"((int)COOP_THREADS) : "memory");
    coop_dwfa_body();
    const int st = J.status;
    *ed = J.ed;
    if (lane_id() == 0) { ST64(wk + WK_CELLS, LD64(wk + WK_CELLS) + J.cells); ST64(wk + WK_MATCHED, LD64(wk + WK_MATCHED) + J.matched); }
    __syncwarp();
    return st;
}
// helper warps of k_compare_coop
__device__ __forceinline__ void coop_helper_loop() {
    CoopJob &J = *(CoopJob *)avk_dyn_smem;
    for (;;) {
        asm volatile("bar.sync 1, %0;" ::"r"((int)COOP_THREADS) : "memory");
        if (J.exit_) return;
        coop_dwfa_body();
    }
}
__device__ __forceinline__ void coop_release_helpers() {   // master warp, all lanes
    CoopJob &J = *(CoopJob *)avk_dyn_smem;
    __syncwarp();
    if (lane_id() == 0) J.exit_ = 1;
    __syncwarp();
    asm volatile("bar.sync 1, %0;" ::"r"((int)COOP_THREADS) : "memory");
}

// update() (dynamic_wfa.rs:68-84) when !to_full, finalize() (:183-198) when to_full.
// *ed is left incremented when the cap is hit (:146-149).
template <bool SMEM>
__device__ __noinline__ int dwfa_run(typename Mem<SMEM>::addr wf, int *ed, int max_ed, const VSeq<SMEM> A, const VSeq<SMEM> B,
                                     bool to_full, typename Mem<SMEM>::addr wk) {
    typedef Mem<SMEM> M;
    int e = *ed;
    bool coop = !SMEM && LD32(wk + WK_COOP) != 0;
    Reach r = dwfa_extend<SMEM>(wf, e, A, B, wk);
#pragma unroll 1
    while (to_full ? !r.full : (!(r.max_base >= A.len) && !(r.max_other >= B.len))) {
        if constexpr (!SMEM) {
            if (coop && e >= COOP_MIN_ED) {            // wide wavefront: the whole CTA takes over from here
                const int rc = dwfa_run_coop(wf, &e, max_ed, A, B, to_full, wk);
                *ed = e;
                if (rc != DWFA_COOP_SPILL) return rc;
                coop = false;                          // wavefront outgrew shared memory: finish on the warp path
                r = dwfa_extend<SMEM>(wf, e, A, B, wk);
                continue;
            }
        }
        e += 1;
        *ed = e;
        if (e > max_ed) return DWFA_MAX_ED;
        dwfa_grow<SMEM>(wf, e - 1);
        r = dwfa_extend<SMEM>(wf, e, A, B, wk);
    }
    return DWFA_OK;
}

// wfa_ed(): src/util/sequence_alignment.rs:9-13.  wf holds 2*max_ed+3 ints; returns -1 if the distance
// would exceed max_ed (callers size the buffer from a proven bound, so -1 is a bug trap).
template <bool SMEM>
__device__ __noinline__ int wfa_ed_warp(const VSeq<SMEM> A, const VSeq<SMEM> B, typename Mem<SMEM>::addr wf, int max_ed,
                                        typename Mem<SMEM>::addr wk) {
    typedef Mem<SMEM> M;
    __syncwarp();
    if (lane_id() == 0) { ST32(wf, 0); ST32(wk + WK_ALIGN, LD32(wk + WK_ALIGN) + 1); }
    __syncwarp();
    int ed = 0;
    if (dwfa_run<SMEM>(wf, &ed, max_ed, A, B, true, wk) != DWFA_OK) return -1;
    return ed;
}

// ---- TMA bulk copy of a reference window into shared memory -------------------------------------------
// cp.async.bulk (1-D bulk TMA, SASS UBLKCP) + mbarrier completion.  src/dst 16-byte aligned, bytes a
// multiple of 16.  One mbarrier per warp (arena bytes [0,8)); `phase` toggles per use.
__device__ __forceinline__ u32 smem_u32(const void *p) { return (u32)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(u32 mbar_off) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(avk_dyn_smem + mbar_off)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void tma_window_issue(u32 dst_off, const u8 *gsrc, u32 bytes, u32 mbar_off) {
    // order this warp's earlier generic-proxy accesses to the window before the async-proxy write
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (lane_id() == 0) {
        const u32 mbar = smem_u32(avk_dyn_smem + mbar_off);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(avk_dyn_smem + dst_off)), "l"(gsrc), "r"(bytes), "r"(mbar) : "memory");
    }
}
// two bulk copies (reference window + cluster digest) completing on one mbarrier
__device__ __forceinline__ void tma_issue2(u32 dst0, const u8 *src0, u32 bytes0, u32 dst1, const u8 *src1, u32 bytes1, u32 mbar_off) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (lane_id() == 0) {
        const u32 mbar = smem_u32(avk_dyn_smem + mbar_off);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes0 + bytes1) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(avk_dyn_smem + dst0)), "l"(src0), "r"(bytes0), "r"(mbar) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(avk_dyn_smem + dst1)), "l"(src1), "r"(bytes1), "r"(mbar) : "memory");
    }
}
__device__ __forceinline__ void tma_window_wait(u32 mbar_off, u32 phase) {
    const u32 mbar = smem_u32(avk_dyn_smem + mbar_off);
    u32 done = 0;
#pragma unroll 1
    while (!done) {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(done) : "r"(mbar), "r"(phase) : "memory");
    }
    __syncwarp();
}

}  // namespace avk
