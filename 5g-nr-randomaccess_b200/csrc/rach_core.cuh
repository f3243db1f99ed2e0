/*
 * rach_core.cuh -- the per-replication RACH engine (variant W/B dynamics), written once as
 * "phase" functions that a CUDA thread block executes with __syncthreads() between them
 * (rach_engine.cu).  tests/emu/ compiles the same phases for the host and runs them thread
 * by thread (test infrastructure only; the product library has no CPU path).
 *
 * WHAT IT COMPUTES: exactly the per-ms state machine of RandomAccessWithNOMA.c:267-335
 * (selectPreamble :475-562, preambleCollision :607-665, requestResourceAllocation :667-710,
 * timerIncrease :712-718, successUEs :720-728) -- bit-identical per-UE outcomes under the
 * Philox draw tape (include/rach_tape.h) -- but NOT by touching every UE every ms.
 *
 * HOW (event-driven restatement, DESIGN.md section 3):
 *  * A UE in the Msg1 phase lives in exactly one 16-byte RECORD that sits in the calendar
 *    bucket of the ms in which its RAR window will expire ("move time" m).  Between two moves
 *    nothing about the UE changes that cannot be derived from (txTime, m): once it has
 *    transmitted at txTime=X it is postponed every ms (W:647 or W:658) until it is granted
 *    or rarWindow reaches maxRarWindow at m = X + Wn - 1 (W:493-496).
 *  * Per preamble p and move time m a COHORT entry in shared memory holds the number of
 *    such UEs and the lowest UE index among them.  The UEs visible to a collision scan at
 *    ms T (active==1 && txTime==T, W:615) are the cohorts m in [T, T+Wn-1].
 *  * Index order (the reference walks UEs 0..n-1 sequentially, W:302) is reproduced through
 *    the index of the FIRST scan of each preamble class in the ms,
 *        s[p] = min( lowest visible non-mover of p,  lowest UE that re-transmits in this very
 *                    ms into p ("lander": backoff draw 0, W:540-549) ),
 *    members of p above s[p] are postponed before their turn (which changes the base of the
 *    limit-branch backoff, W:516), movers below s[p] have left before the scan (group size),
 *    later landers scan alone, and UL grants go to singleton scans in index order (W:639-641).
 *  * Msg3 (W:667-710) is a second small calendar.
 *
 * Every function cites the reference lines it restates.
 */
#ifndef RACH_CORE_CUH
#define RACH_CORE_CUH

#include <stddef.h>
#include <stdint.h>
#include "rach_tape.h"
#include "rach_warp.cuh"

#ifdef __CUDACC__
#define RA_HD __host__ __device__ __forceinline__
#define RA_HDM __host__ __device__ __forceinline__      /* member functions */
#else
#define RA_HD static inline
#define RA_HDM inline
struct uint4 { unsigned x, y, z, w; };
static inline uint4 make_uint4(unsigned a, unsigned b, unsigned c, unsigned d) { uint4 r = {a, b, c, d}; return r; }
#endif

typedef unsigned long long ra_u64;

#define RA_INF32 0xFFFFFFFFu
#define RA_INF64 0xFFFFFFFFFFFFFFFFull
#define RA_DEAD  0xFFFFFFFFu
#define RA_M3RING 64
#define RA_DUMP_W 16
#ifndef RA_HBINS
#define RA_HBINS 512        /* histogram bins of the grant selection            */
#endif
#ifndef RA_SCAP
#define RA_SCAP  512        /* singleton scans of one ms kept in shared memory (rest: global).  Shared memory is
                               kept small on purpose: at 5 resident blocks x 48 registers the spills live in L1 */
#endif

/* ---- atomics: CUDA on the device, plain read-modify-write in the host emulator ---------- */
#ifdef __CUDA_ARCH__
#define RA_AADD(p, v)   atomicAdd((p), (v))
#define RA_AMIN(p, v)   atomicMin((p), (v))
/* 64-bit sum in shared memory fed with 32-bit addends: one native 32-bit atomic on the low word and a carry (a 64-bit
 * shared-memory atomicAdd is a compare-and-swap loop) */
__device__ __forceinline__ void ra_aadd64(unsigned long long* p, unsigned v) {
    unsigned* w = reinterpret_cast<unsigned*>(p);
    const unsigned old = atomicAdd(w, v);
    if (old + v < old) atomicAdd(w + 1, 1u);
}
#define RA_AADD64(p, v) ra_aadd64((p), (v))
#else
template <class T> static inline T ra_emu_add(T* p, T v) { T o = *p; *p = o + v; return o; }
template <class T> static inline T ra_emu_min(T* p, T v) { T o = *p; if (v < o) *p = v; return o; }
#define RA_AADD(p, v)   ra_emu_add((p), (v))
#define RA_AMIN(p, v)   ra_emu_min((p), (v))
#define RA_AADD64(p, v) (*(p) += (unsigned long long)(v))
#endif

/* x % d for x < 2^31 and 1 <= d <= 2^16 without a division.  With l = ceil(log2 d), magic = floor(2^(31+l) / d) + 1 fits
 * in 32 bits and floor(x * magic / 2^(31+l)) is exactly x / d: magic = 2^(31+l)/d + e with 0 < e <= 1, so the product
 * overshoots x/d by x*e / 2^(31+l) < 2^-l <= 1/d, which cannot carry x/d = q + r/d (r <= d-1) past q + 1.  The quotient is
 * (x * magic >> 32) >> (l - 1).  d == 1 (l = 0) takes magic = 0xFFFFFFFF, shift 0: the quotient comes out as x - 1 and the
 * one conditional subtraction below makes the remainder 0. */
RA_HD unsigned ra_mod_shift(unsigned d) { unsigned l = 0; while ((1u << l) < d) ++l; return l ? l - 1 : 0; }
RA_HD unsigned ra_magic(unsigned d) {
    if (d <= 1) return 0xFFFFFFFFu;
    unsigned l = 0; while ((1u << l) < d) ++l;
    return (unsigned)((1ull << (31 + l)) / d) + 1u;
}
RA_HD unsigned ra_mod(unsigned x, unsigned d, unsigned magic, unsigned shift) {
    const unsigned q = rach_mulhi32(x, magic) >> shift;
    unsigned r = x - q * d;
    if (r >= d) r -= d;
    return r;
}

/* A calendar record is written once and read once, several ms later, by which time a thousand other replications have been
 * through the caches: streaming (evict-first) stores and loads keep the 16-byte records from displacing what IS re-used
 * (work lists, position hints).  Measured on the bench workload: 965 -> 945 ms. */
#ifdef __CUDA_ARCH__
__device__ __forceinline__ ::uint4 ra_ldrec(const ::uint4* p) { return __ldcs(p); }
__device__ __forceinline__ void ra_strec(::uint4* p, const ::uint4& v) { __stcs(p, v); }
#define RA_STREC(p, v) ra_strec((p), (v))
#define RA_LDREC(p)    ra_ldrec(p)
#else
#define RA_STREC(p, v) (*(p) = (v))
#define RA_LDREC(p)    (*(p))
#endif

/* ---- one parameter point, device view ---------------------------------------------------- */
struct RaPointDev {
    int nUE, P, BI, G, Wn, M, A, maxTime;
    int geometry, R, nOcc, hshift;  /* hshift: idx >> hshift < RA_HBINS */
    unsigned magicBI, magicP, magicA;      /* ra_magic() of the three runtime divisors (shifts: modSh) */
    float cellRadius;                      /* variant N: per point (N:56, used by activeUE N:168) */
    ra_u64 seed;
    const int* arrCum;        /* [nOcc] activeCheck after the arrival step of ms occ*A (W:280-292) */
    /* byte offsets of the block's tables in dynamic shared memory (ra_layout): a function of (R, P) only, kept
     * here so that a launch whose replications share one point reads them as kernel constants */
    unsigned oMinI, oCnt, oBcount, oM3count, oN, oL1, oNlList, oL1m, oL2, oBefore, oExtraFirst, oClsSize;
    unsigned oHist, oSIdx, smemBytes, oDead;
    unsigned modSh;                        /* ra_mod_shift() of BI | P << 8 | A << 16 */
    /* rand() % backoffIndicator (W:514,540,685), rand() % nPreamble (W:478,502,701), subTime % accessTime (W:518) */
    RA_HDM unsigned modBI(unsigned x) const { return ra_mod(x, (unsigned)BI, magicBI, modSh & 0xFFu); }
    RA_HDM unsigned modP(unsigned x) const { return ra_mod(x, (unsigned)P, magicP, (modSh >> 8) & 0xFFu); }
    RA_HDM unsigned modA(unsigned x) const { return ra_mod(x, (unsigned)A, magicA, modSh >> 16); }
};

/* table layout for (R, P).  One definition for the runtime point (ra_layout) and for the compile-time view below. */
struct RaLayout {
    unsigned oMinI, oCnt, oBcount, oDead, oM3count, oN, oL1, oNlList, oL1m, oL2, oBefore, oExtraFirst, oClsSize, oHist,
             oSIdx, smemBytes;
};
#define RA_LAYOUT_BODY(R_, P_) \
    RaLayout l = {}; unsigned o = 0; const unsigned RP = (unsigned)(R_) * (unsigned)(P_), P4 = 4u * (unsigned)(P_); \
    l.oMinI = o;       o += 4u * RP; \
    l.oCnt = o;        o += 4u * RP; \
    l.oBcount = o;     o += 4u * (unsigned)(R_); \
    l.oDead = o;       o += 4u * (unsigned)(R_); \
    l.oM3count = o;    o += 4u * RA_M3RING; \
    l.oN = o;          o += P4; \
    l.oL1 = o;         o += P4; \
    l.oNlList = o;     o += P4; \
    l.oL1m = o;        o += P4; \
    l.oL2 = o;         o += P4; \
    l.oBefore = o;     o += P4; \
    l.oExtraFirst = o; o += P4; \
    l.oClsSize = o;    o += P4; \
    l.oHist = o;       o += 4u * RA_HBINS; \
    l.oSIdx = o;       o += 4u * RA_SCAP; \
    l.smemBytes = o; \
    return l;
#ifdef __CUDACC__
__host__ __device__
#endif
constexpr RaLayout ra_layout_of(int R, int P) { RA_LAYOUT_BODY(R, P) }

/* Compile-time view of a point of the family (P, BI, A, Wn): every reference default that the step's inner loops
 * divide by or index with (W:71-72,76,78: 54 preambles, BI 20, maxRarWindow 6, accessTime 5) becomes an immediate --
 * `% BI`, `% P`, `% A` turn into multiply-shift sequences without corrections, table offsets into immediates, and the
 * dozen shared-memory loads of these values per event disappear.  Same layout as RaPointDev (no data members
 * added): the kernel casts its shared-memory copy of the point.  nUE, G, M, horizon, seed ... stay runtime values. */
template <int P_, int BI_, int A_, int Wn_, int R_>
struct RaPointFixed : RaPointDev {
    static constexpr int P = P_, BI = BI_, A = A_, Wn = Wn_, R = R_;
    static constexpr RaLayout L = ra_layout_of(R_, P_);
    static constexpr unsigned oMinI = L.oMinI, oCnt = L.oCnt, oBcount = L.oBcount, oDead = L.oDead, oM3count = L.oM3count, oN = L.oN, oL1 = L.oL1, oNlList = L.oNlList, oL1m = L.oL1m, oL2 = L.oL2,
        oBefore = L.oBefore, oExtraFirst = L.oExtraFirst, oClsSize = L.oClsSize, oHist = L.oHist, oSIdx = L.oSIdx,
        smemBytes = L.smemBytes;
    RA_HDM unsigned modBI(unsigned x) const { return x % (unsigned)BI_; }
    RA_HDM unsigned modP(unsigned x) const { return x % (unsigned)P_; }
    RA_HDM unsigned modA(unsigned x) const { return x % (unsigned)A_; }
};
/* the reference's defaults (RandomAccessWithNOMA.c:71-78); ring = next_pow2(BI + max(A,5) + Wn) = 32 */
typedef RaPointFixed<54, 20, 5, 6, 32> RaPointDef;
RA_HD bool ra_point_is_default_family(const RaPointDev& pt) {
    return pt.P == RaPointDef::P && pt.BI == RaPointDef::BI && pt.A == RaPointDef::A && pt.Wn == RaPointDef::Wn && pt.R == RaPointDef::R;
}

/* ---- per-CTA global workspace ------------------------------------------------------------ */
struct RaWork {
    uint4*    bucket;         /* [R][cap]   move calendar                                  */
    uint4*    msg3;           /* [RA_M3RING][cap3]  Msg3 calendar                           */
    uint4*    landerRec;      /* [cap]  UEs re-transmitting in the current ms               */
    unsigned* landerMeta;     /* [cap]  bit0: member of its class at start of ms; bits 8..: late joins */
    uint4*    uncertain;      /* [cap]  movers below the natural leader: pos, idx, p0|limit<<31 */
    uint4*    c3;             /* [cap]  limit movers that land iff not postponed: idx,p0,pnew,landed */
    unsigned* singles;        /* [cap]  UE index of every singleton scan of the ms          */
    unsigned* minPos;         /* [R*P]  bucket position of each cohort's lowest UE -- a HINT (no atomic pair; verified on
                                 use).  Global on purpose: 7 KB more shared memory per block shrinks L1 below the
                                 register-spill working set of 5 resident blocks (measured: 10 % slower) */
    uint4*    e1Rec;          /* [cap3] Msg3 restarts that land on the current ms (W:693)   */
    unsigned* e1Meta;         /* [cap3] 1 = absorbed by a later scan                        */
    unsigned* hist;           /* [histLen] the replication's histograms (ra_hist_add), or NULL */
    int cap, cap3;
};

/* the next 256-byte aligned table of `bytes` in a workspace at `base` (NULL: sizing only, no pointer) */
static inline void* ra_carve_next(unsigned char* base, size_t& off, size_t bytes) {
    void* p = base ? base + off : NULL;
    off = (off + bytes + 255) / 256 * 256;
    return p;
}

/* lays out one block's workspace at `base` for a ring of R move buckets and P preambles, with a histogram region of
 * histLen counters (0 = none); returns its size in bytes */
static inline size_t ra_work_carve(unsigned char* base, int cap, int cap3, int R, int P, RaWork* w, int histLen = 0) {
    const size_t c = (size_t)cap, c3 = (size_t)cap3;
    size_t off = 0;
    w->bucket = (uint4*)ra_carve_next(base, off, sizeof(uint4) * c * (size_t)R);
    w->msg3 = (uint4*)ra_carve_next(base, off, sizeof(uint4) * c3 * RA_M3RING);
    w->landerRec = (uint4*)ra_carve_next(base, off, sizeof(uint4) * c);
    w->landerMeta = (unsigned*)ra_carve_next(base, off, sizeof(unsigned) * c);
    w->uncertain = (uint4*)ra_carve_next(base, off, sizeof(uint4) * c);
    w->c3 = (uint4*)ra_carve_next(base, off, sizeof(uint4) * c);
    w->singles = (unsigned*)ra_carve_next(base, off, sizeof(unsigned) * c);
    w->e1Rec = (uint4*)ra_carve_next(base, off, sizeof(uint4) * c3);
    w->e1Meta = (unsigned*)ra_carve_next(base, off, sizeof(unsigned) * c3);
    w->minPos = (unsigned*)ra_carve_next(base, off, sizeof(unsigned) * (size_t)R * (size_t)P);
    w->hist = histLen ? (unsigned*)ra_carve_next(base, off, sizeof(unsigned) * (size_t)histLen) : NULL;
    w->cap = cap; w->cap3 = cap3;
    return off;
}

/* ---- per-CTA shared state ---------------------------------------------------------------- */
struct RaShared {
    int grantCheck, activeCheck, acOld, nArr, overflow, nextAc;   /* nextAc: activeCheck after the next arrival step */
    int nextArrMs, occ;       /* next ms with T % A == 0 and its occasion number (no division in the ms loop) */
    int gcAdd;                /* singleton scans of the ms just finished that phase 5 did not have to rank (all answered):
                                 added to grantCheck by the thread that opens the next ms (ra_gc_apply) */
    unsigned nLanders, nUnc, nC3, nSingles, nE1, nMov, nM3, tau;
    unsigned nSuccess, noGrant, nNl, nNlLight;      /* nNlLight: stale position hints met by ra_light_ms (its own counter:
                                                      the block may still be reading nNl of the ms it has just finished) */
    ra_u64 txSum, delaySum, failSum, contFailed, collP, txop, collScans, totScans;
    ra_u64 recMoves;          /* records read from the calendars (move buckets, Msg3 ring, same-ms work list)     */
};

/* per-thread counters, folded into RaShared at the end of the replication */
struct RaAcc { unsigned contFailed, collP, txop, collScans, totScans; };

/* the histogram region a job starts with: none on the device (the kernels set it); in the host emulation the caller's
 * (NULL: none), as with ra_emu_smem_base */
#ifdef __CUDA_ARCH__
#define RA_JOB_HIST0 nullptr
#else
static thread_local unsigned* ra_emu_hist_base;
#define RA_JOB_HIST0 ra_emu_hist_base
#endif

template <class PT>
struct RaJobT {
    const PT* pt;             /* RaPointDev, or a compile-time view of it (RaPointDef)      */
    unsigned rep;             /* tape replication id                                        */
    int* dump;                /* [nUE][16] or NULL                                          */
    unsigned* hist = RA_JOB_HIST0;   /* the block's (U0: the warp's) histogram region, or NULL */
};
typedef RaJobT<RaPointDev> RaJob;

/* ---- histograms of the successful UEs (ra_options.histograms) ----------------------------
 * A point's region holds three histograms back to back, 32-bit counters (a replication has fewer than 2^24 successes):
 *   [0, maxTime + 7)   delay: timer at success in ms.  W and N record T - timerStart + 6 with T < maxTime (W:674,
 *                      N:504-508), U0's timer is at most maxTime: so 0 .. maxTime + 6
 *   [+0, +256)         preambleTxCounter (N: nTxPreamble), the last bin counts 255 and above
 *   [+256, +512)       failCount (W/B only; N and U0 pass 0 and that part is never reported) */
#define RA_HIST_TOP 256
RA_HD int ra_hist_delay_bins(int maxTime) { return maxTime + 7; }
RA_HD int ra_hist_len(int maxTime) { return maxTime + 7 + 2 * RA_HIST_TOP; }

/* the success event of one UE (W:720-728 / N:504-508 / U0:113-115) */
template <class PT>
RA_HD void ra_hist_add(const RaJobT<PT>& job, unsigned delay, unsigned tx, unsigned fail) {
    unsigned* h = job.hist;
    if (!h) return;
    const unsigned nD = (unsigned)ra_hist_delay_bins(job.pt->maxTime);
    /* the clamps keep the adds in the region; the delay bound above makes its clamp unreachable */
    RA_AADD(&h[delay < nD ? delay : nD - 1u], 1u);
    RA_AADD(&h[nD + (tx < RA_HIST_TOP - 1u ? tx : RA_HIST_TOP - 1u)], 1u);
    RA_AADD(&h[nD + RA_HIST_TOP + (fail < RA_HIST_TOP - 1u ? fail : RA_HIST_TOP - 1u)], 1u);
}

/* ---- record packing ---------------------------------------------------------------------- */
/* x: idx   y: txTime   z: timerStart | failCount<<16   w: preamble | mrc<<8 | ptc<<16 | flag<<31
 * flag: move bucket: 1 = stale (invisible);  Msg3 calendar: 1 = second visit (connectionRequest 48) */
RA_HD unsigned ra_w3(unsigned p, unsigned mrc, unsigned ptc, unsigned flag) {
    return (p & 0xFFu) | ((mrc & 0xFFu) << 8) | ((ptc & 0x7FFFu) << 16) | (flag << 31);
}
RA_HD unsigned ra_rec_p(const uint4& r)    { return r.w & 0xFFu; }
RA_HD unsigned ra_rec_mrc(const uint4& r)  { return (r.w >> 8) & 0xFFu; }
RA_HD unsigned ra_rec_ptc(const uint4& r)  { return (r.w >> 16) & 0x7FFFu; }
RA_HD unsigned ra_rec_flag(const uint4& r) { return r.w >> 31; }
RA_HD unsigned ra_rec_ts(const uint4& r)   { return r.z & 0xFFFFu; }
RA_HD unsigned ra_rec_fail(const uint4& r) { return r.z >> 16; }
RA_HD unsigned ra_z(unsigned ts, unsigned fail) { return (ts & 0xFFFFu) | (fail << 16); }

/* slot alignment, W:518-527 (= W:544-553, W:688-697) */
RA_HD int ra_align5(int subTime) {                       /* the literal 5 of the Msg3 restart, W:687-697 */
    const int r = (int)((unsigned)subTime % 5u);
    if (r == 0) return subTime + 1;
    if (r == 1) return subTime;
    return subTime + (5 - r + 1);
}

template <class PT>
RA_HD int ra_align_pt(const PT& pt, int subTime) {
    const int r = (int)pt.modA((unsigned)subTime);
    if (r == 0) return subTime + 1;
    if (r == 1) return subTime;
    return subTime + (pt.A - r + 1);
}

/* the same with a compile-time subframe A >= 2: the first ms congruent to 1 (mod A) at or after subTime -- one
 * multiply-shift division, no branch (r == 0 -> +1, r == 1 -> +0, else +(A - r + 1), all of them A * floor((subTime + A - 2) / A) + 1) */
template <int P_, int BI_, int A_, int Wn_, int R_>
RA_HD int ra_align_pt(const RaPointFixed<P_, BI_, A_, Wn_, R_>&, int subTime) {
    if (A_ >= 2) return (int)(((unsigned)subTime + (unsigned)(A_ - 2)) / (unsigned)A_ * (unsigned)A_) + 1;
    return subTime + 1;
}

template <class PT>
RA_HD rach_u32x4 ra_draws(const RaJobT<PT>& job, unsigned ue, int ms) {
    return rach_tape_block(job.pt->seed, job.rep, ue, (unsigned)ms, 0u, RACH_TAPE_TAG_UE);
}

/* ---- the block's tables in dynamic shared memory ------------------------------------------ */
/* Tables are addressed as base + pt.o<Table> (32-bit shared addresses: LDS / ATOMS).  Keeping 64-bit table
 * pointers in shared memory instead made every access a generic LD / ATOM behind a pointer load: 9 % slower at two
 * replications per block, equal in the long steady state (measured on B200). */
#ifdef __CUDA_ARCH__
__device__ __forceinline__ unsigned char* ra_smem() {
    extern __shared__ __align__(16) unsigned char ra_dyn_smem[];
    return ra_dyn_smem;
}
#else
static thread_local unsigned char* ra_emu_smem_base;      /* host emulation of the phases: set by the caller */
static inline unsigned char* ra_smem() { return ra_emu_smem_base; }
#endif
#define RA_TAB_U(off)  (reinterpret_cast<unsigned*>(ra_smem() + (off)))
#define RA_TAB_Q(off)  (reinterpret_cast<uint4*>(ra_smem() + (off)))
struct RaTabsT { unsigned *minI, *cnt, *bcount, *dead, *m3count, *N, *l1, *nlList, *l1m, *l2, *before, *extraFirst, *clsSize, *hist, *sIdx; };
#define RA_T(name, O) (reinterpret_cast<decltype(RaTabsT::name)>(ra_smem() + pt.O))
#define S_minI       RA_T(minI, oMinI)             /* [R*P] lowest UE index of the cohort                        */
#define S_cnt        RA_T(cnt, oCnt)               /* [R*P] cohort size                                          */
#define S_bcount     RA_T(bcount, oBcount)         /* [R]   records in each move bucket                          */
#define S_dead       RA_T(dead, oDead)             /* [R]   ... of which granted away since (left as RA_DEAD records) */
#define S_m3count    RA_T(m3count, oM3count)       /* [RA_M3RING]                                                */
#define S_N          RA_T(N, oN)                   /* [P] each, N .. clsSize                                     */
#define S_l1         RA_T(l1, oL1)
#define S_nlList     RA_T(nlList, oNlList)
#define S_l1m        RA_T(l1m, oL1m)
#define S_l2         RA_T(l2, oL2)
#define S_before     RA_T(before, oBefore)
#define S_extraFirst RA_T(extraFirst, oExtraFirst)
#define S_clsSize    RA_T(clsSize, oClsSize)
#define S_hist       RA_T(hist, oHist)             /* [RA_HBINS] singleton scans per index bin (grant selection) */
#define S_sIdx       RA_T(sIdx, oSIdx)             /* [RA_SCAP]  first singleton indices of the ms                */

RA_HD void ra_layout(RaPointDev& pt) {
    const RaLayout l = ra_layout_of(pt.R, pt.P);
    pt.oMinI = l.oMinI; pt.oCnt = l.oCnt;
    pt.oBcount = l.oBcount; pt.oDead = l.oDead; pt.oM3count = l.oM3count; pt.oN = l.oN; pt.oL1 = l.oL1; pt.oNlList = l.oNlList;
    pt.oL1m = l.oL1m; pt.oL2 = l.oL2; pt.oBefore = l.oBefore; pt.oExtraFirst = l.oExtraFirst; pt.oClsSize = l.oClsSize;
    pt.oHist = l.oHist; pt.oSIdx = l.oSIdx; pt.smemBytes = l.smemBytes;
}

template <class PT>
RA_HD unsigned ra_first_scan(const PT& pt, unsigned p) {     /* s[p] of the header comment */
    unsigned a = S_l1[p], b = S_l2[p];
    return a < b ? a : b;
}

/* append a record to move bucket `m`; returns its position */
template <class PT>
RA_HD unsigned ra_bucket_push(const PT& pt, const RaWork& w, RaShared& s, int m, const uint4& rec) {
    unsigned slot = (unsigned)m & (unsigned)(pt.R - 1);
    /* one shared-memory atomic per record: measured 8 % faster on B200 than aggregating the lanes of a warp
     * per bucket with __match_any_sync (the variable-mask shuffle that follows costs more than the contention) */
    unsigned pos = RA_AADD(&S_bcount[slot], 1u);
    if (pos >= (unsigned)w.cap) { s.overflow = 1; return 0; }
    RA_STREC(&w.bucket[slot * (unsigned)w.cap + pos], rec);      /* ring x capacity < 2^32 records (checked at create) */
    return pos;
}

/* a UE (re)enters the Msg1 phase with transmission time X = rec.y > now: visible from X on,
 * its RAR window expires at X + Wn - 1 (rarWindow is 1 at X, W:493) */
template <class PT>
RA_HD void ra_schedule(const PT& pt, const RaWork& w, RaShared& s, const uint4& rec) {
    int m = (int)rec.y + pt.Wn - 1;
    const unsigned pos = ra_bucket_push(pt, w, s, m, rec);
    unsigned c = ((unsigned)m & (unsigned)(pt.R - 1)) * (unsigned)pt.P + ra_rec_p(rec);
    RA_AADD(&S_cnt[c], 1u);
    /* a bare atomic: 0.6 % faster than reading the minimum first */
    if (RA_AMIN(&S_minI[c], rec.x) > rec.x) w.minPos[c] = pos;
}

/* a UE whose txTime is not in the future and that nobody postpones (W:516 applied to an old
 * txTime, or a Msg3 restart landing on `now`, W:693): invisible to scans, rarWindow counts
 * from 0 at `now`, so it expires at now + Wn */
template <class PT>
RA_HD void ra_park_stale(const PT& pt, const RaWork& w, RaShared& s, int now, uint4 rec) {
    rec.w |= 0x80000000u;
    ra_bucket_push(pt, w, s, now + pt.Wn, rec);
}

template <class PT>
RA_HD void ra_msg3_push(const PT& pt, const RaWork& w, RaShared& s, int due, const uint4& rec) {
    unsigned slot = (unsigned)due & (RA_M3RING - 1);
    unsigned pos = RA_AADD(&S_m3count[slot], 1u);
    if (pos >= (unsigned)w.cap3) { s.overflow = 1; return; }
    w.msg3[(size_t)slot * w.cap3 + pos] = rec;
}

RA_HD void ra_lander_push(const RaWork& w, RaShared& s, const uint4& rec, unsigned member) {
    unsigned l = RA_AADD(&s.nLanders, 1u);
    if (l >= (unsigned)w.cap) { s.overflow = 1; return; }
    w.landerRec[l] = rec; w.landerMeta[l] = member;
}

/* ---- dump helpers (DUMP builds only) ------------------------------------------------------ */
RA_HD void ra_dump_init_row(int* d) {           /* calloc + initialUE, W:229,374-381 */
    for (int k = 0; k < RA_DUMP_W; ++k) d[k] = 0;
    d[0] = -1; d[1] = -1; d[2] = -1; d[6] = -1; d[15] = -1;
}

/* sector of activateUEs, W:392-410, from the first activation draw */
RA_HD int ra_sector(int r31) {
    float pi = 3.14;
    float theta = (float)r31 / (float)(2147483647) * 2 * pi;
    if (theta >= 0 && theta < ((1. / 3.) * pi)) return 0;
    else if (theta >= ((1. / 3.) * pi) && theta < ((2. / 3.) * pi)) return 1;
    else if (theta >= ((2. / 3.) * pi) && theta < 3.14) return 2;
    else if (theta >= pi && theta < ((4. / 3.) * pi)) return 3;
    else if (theta >= ((4. / 3.) * pi) && theta < ((5. / 3.) * pi)) return 4;
    return 5;
}

/* =========================================================================================
 * Job start: empty calendars and cohort tables (calloc + initialUE, W:229-234).
 * ========================================================================================= */
template <bool DUMP, class PT>
RA_HD void ra_job_init(const RaJobT<PT>& job, RaShared& s, int tid, int nt) {
    const PT& pt = *job.pt;
    for (int i = tid; i < pt.R * pt.P; i += nt) { S_cnt[i] = 0; S_minI[i] = RA_INF32; }
    for (int i = tid; i < pt.R; i += nt) { S_bcount[i] = 0; S_dead[i] = 0; }
    for (int i = tid; i < RA_M3RING; i += nt) S_m3count[i] = 0;
    for (int i = tid; i < RA_HBINS; i += nt) S_hist[i] = 0;
    if (DUMP) for (int i = tid; i < pt.nUE; i += nt) ra_dump_init_row(job.dump + (size_t)i * RA_DUMP_W);
    if (tid == 0) {
        s.grantCheck = 0; s.activeCheck = 0; s.overflow = 0; s.gcAdd = 0;
        s.nextAc = pt.arrCum[0]; s.nextArrMs = 0; s.occ = 0;
        s.nSuccess = 0; s.noGrant = 0;
        s.txSum = s.delaySum = s.failSum = s.contFailed = s.collP = s.txop = s.collScans = s.totScans = 0;
        s.recMoves = 0;
    }
}

/* =========================================================================================
 * Phase 0 -- start of ms T: grant reset (W:268-269), arrival gate (W:276-292), per-class
 * view of the visible cohorts.
 * ========================================================================================= */
template <class PT>
RA_HD void ra_phase0_classes(const RaJobT<PT>& job, RaShared& s, int T, int tid, int nt) {
    const PT& pt = *job.pt;
    const int P = pt.P, Wn = pt.Wn;
    const unsigned Rm = (unsigned)(pt.R - 1);
    /* (straight-line on purpose: the loads of the Wn rows pipeline; skipping rows known to be empty through a mask was
     * measured slower at every load -- 5 % on Uniform traffic, 8 % at 20k UEs Beta) */
    for (int p = tid; p < P; p += nt) {
        unsigned n = 0, best = RA_INF32, bestm = 0;
        for (int d = 0; d < Wn; ++d) {
            unsigned m = ((unsigned)(T + d) & Rm);
            n += S_cnt[m * P + p];
            if (d > 0) { unsigned v = S_minI[m * P + p]; if (v < best) { best = v; bestm = m; } }
        }
        S_N[p] = n;
        S_l1[p] = best; S_l1m[p] = bestm;
        S_l2[p] = RA_INF32; S_before[p] = 0; S_extraFirst[p] = 0; S_clsSize[p] = 0;
    }
}

/* the control block of ms T (one thread) */
template <class PT>
RA_HD void ra_phase0_ctl(const RaJobT<PT>& job, RaShared& s, int T) {
    const PT& pt = *job.pt;
    const unsigned Rm = (unsigned)(pt.R - 1);
    if ((unsigned)T % 5u == 0) s.grantCheck = 0;          /* literal 5, W:268 */
    s.nLanders = 0; s.nUnc = 0; s.nC3 = 0; s.nSingles = 0; s.nE1 = 0; s.tau = RA_INF32; s.noGrant = 0; s.nNl = 0;
    s.acOld = s.activeCheck;
    if (T == s.nextArrMs) {                                                 /* T % accessTime == 0, W:280 */
        if (s.activeCheck != pt.nUE) s.activeCheck = s.nextAc;
        s.nextArrMs = T + pt.A; s.occ++;
        if (s.occ < pt.nOcc) s.nextAc = pt.arrCum[s.occ];                   /* needed A ms from now: latency hidden */
    }
    s.nArr = s.activeCheck - s.acOld;
    s.nMov = S_bcount[(unsigned)T & Rm];
    /* every record of the bucket was granted before its window expired (the normal case under light load: the
     * first scan of a lone UE is answered): nothing to read, nothing to move */
    if (S_dead[(unsigned)T & Rm] == s.nMov) s.nMov = 0;
    s.nM3 = S_m3count[(unsigned)T & (RA_M3RING - 1)];
    s.recMoves += (ra_u64)s.nMov + s.nM3;
}

template <class PT>
RA_HD void ra_phase0(const RaJobT<PT>& job, RaShared& s, int T, int tid, int nt) {
    ra_phase0_classes(job, s, T, tid, nt);
    if (tid == 0) ra_phase0_ctl(job, s, T);
}

/* =========================================================================================
 * Phase 1 -- one pass over the UEs that have an event in ms T (item = work index):
 *   [0, nMov)            movers (bucket T): rarWindow reaches maxRarWindow, W:496-558
 *   [nMov, +nArr)        arrivals: activateUEs + first selectPreamble, W:294-298,383-394,477-487
 *   [.., +nM3)           Msg3 due: requestResourceAllocation, W:667-710
 * ========================================================================================= */
/* A mover that re-transmits in this very ms (backoff draw 0 on a tx slot, W:540-549: one mover in twenty) joins the
 * ms' work list of re-transmitters.  Done on the spot that is a 40-instruction branch which three of four warp
 * iterations enter for a single lane (measured: 14 % of the step kernel's warp instructions at 1 of 32 lanes).  So the
 * mover only parks the record in its thread's registers (RaPend) and the thread puts it on the list later -- the
 * kernel when two of them meet in one lane of the warp (then every lane of the warp flushes) and at the end of the
 * bucket.  The list has no order (entries are appended by atomics), so when an entry gets there is immaterial as long
 * as it is before the barrier that ends phase 1. */
struct RaPend { unsigned x, z, w; };      /* x = idx | member << 31 (idx < 2^24), RA_INF32 = empty; z, w as in the record */

template <class PT>
RA_HD void ra_pend_flush(const PT& pt, const RaWork& w, RaShared& s, int T, RaPend& pd) {
    if (pd.x == RA_INF32) return;
    const unsigned idx = pd.x & 0x7FFFFFFFu;
    RA_AMIN(&S_l2[pd.w & 0xFFu], idx);
    ra_lander_push(w, s, make_uint4(idx, (unsigned)T, pd.z, pd.w), pd.x >> 31);
    pd.x = RA_INF32;
}

template <bool DUMP, class PT>
RA_HD bool ra_phase1_mover_d(const RaJobT<PT>& job, const RaWork& w, RaShared& s, RaAcc& acc, int T, unsigned item, const uint4& rec, const rach_u32x4& d, RaPend& land);

/* one mover, its re-transmission (if any) parked in `pd` (the caller flushes it before the phase ends): the mover loop of
 * the kernel one record at a time (used by the host emulation) */
template <bool DUMP, class PT>
RA_HD void ra_phase1_mover(const RaJobT<PT>& job, const RaWork& w, RaShared& s, RaAcc& acc, int T, unsigned item, const uint4& rec, RaPend& pd) {
    if (rec.x == RA_DEAD) return;
    RaPend land;
    if (ra_phase1_mover_d<DUMP>(job, w, s, acc, T, item, rec, ra_draws(job, rec.x, T), land)) {
        ra_pend_flush(*job.pt, w, s, T, pd);
        pd = land;
    }
}

/* one mover (work item `item` < nMov); the draws of (UE, T) are passed in so that the kernel can run two Philox chains
 * side by side.  Returns true if the UE re-transmits in this ms: its new record is then in `land` and has NOT been put
 * on the work list. */
template <bool DUMP, class PT>
RA_HD bool ra_phase1_mover_d(const RaJobT<PT>& job, const RaWork& w, RaShared& s, RaAcc& acc, int T, unsigned item, const uint4& rec, const rach_u32x4& d, RaPend& land) {
    const PT& pt = *job.pt;
    land.x = RA_INF32; land.z = 0; land.w = 0;
    if (rec.x == RA_DEAD) return false;
    const unsigned idx = rec.x, p0 = ra_rec_p(rec), stale = ra_rec_flag(rec);
    /* below the lowest visible non-mover of my class: nobody is sure to have postponed me */
    const bool uncertain = !stale && idx < S_l1[p0];
    const bool limit = (int)ra_rec_mrc(rec) >= pt.M;
    /* both branches draw the backoff: retry W:540 (1st draw), limit W:514 (2nd draw) */
    const int tmp = (int)pt.modBI((limit ? d.v[1] : d.v[0]) >> 1);
    /* Both branches written as selects: one mover in ten takes the limit branch, so almost every warp would
     * otherwise execute both sides of an if/else.
     *   retry branch, W:532-558: subTime = time + tmp (W:542); maxRarCounter++, preambleTxCounter++
     *   limit branch, W:498-531: new preamble, counters reset, timer = 0, failCount++, subTime = CURRENT
     *     txTime + tmp (W:516): an old txTime if stale, T+1 if a lower index postponed me (certain above the
     *     leader), T under the not-postponed hypothesis if uncertain (settled in phase 3)
     * The counters are updated inside the packed words (no unpack / repack): retry adds 1 to maxRarCounter (bits 8..15;
     * it is below M <= 255 here, so no carry) and to preambleTxCounter (bits 16..30; a carry into bit 31 is the overflow
     * check), limit writes preamble | 0 << 8 | 1 << 16 and adds 1 to failCount (bits 16..31 of z; carry = overflow). */
    const unsigned pl = pt.modP(d.v[0] >> 1);
    const unsigned pnew = limit ? pl : p0;
    const unsigned wRetry = (rec.w & 0x7FFFFFFFu) + 0x00010100u;
    const unsigned nw = limit ? (pl | 0x00010000u) : wRetry;
    const unsigned z = limit ? (((rec.z & 0xFFFF0000u) + 0x00010000u) | (unsigned)T) : rec.z;
    acc.contFailed += limit ? 1u : 0u;
    const int base = limit ? (stale ? (int)rec.y : (uncertain ? T : T + 1)) : T;
    if (limit ? rec.z >= 0xFFFF0000u : (wRetry >> 31) != 0u) s.overflow = 2;
    const int X = ra_align_pt(pt, base + tmp);
    const uint4 nr = make_uint4(idx, (unsigned)X, z, nw);
    land.z = z; land.w = nw;                               /* (assigned on every path: the values stay in registers) */
    if (uncertain) {
        unsigned u = RA_AADD(&s.nUnc, 1u);
        w.uncertain[u] = make_uint4(item, idx, p0 | (limit ? 0x80000000u : 0u), 0);
        if (limit) {
            if (X == T) { unsigned c = RA_AADD(&s.nC3, 1u); w.c3[c] = make_uint4(idx, p0, pnew, 0); }
            return false;
        }
    }
    if (DUMP) job.dump[(size_t)idx * RA_DUMP_W + (limit ? 3 : 4)] = limit ? T + 1 : X;   /* W:510 / W:557 */
    if (X > T) {
        ra_schedule(pt, w, s, nr);                          /* the common case, one call site */
    } else if (X == T) {                                    /* backoff 0 on a tx slot: transmits now (class pnew = nw & 0xFF) */
        land.x = idx | ((!stale && !limit) ? 0x80000000u : 0u);
        return true;
    } else {
        ra_park_stale(pt, w, s, T, nr);                     /* only from an old txTime */
    }
    return false;
}

/* arrival of UE idx, W:383-394 + first draw W:477-487 */
template <bool DUMP, class PT>
RA_HD void ra_arrival_item(const RaJobT<PT>& job, const RaWork& w, RaShared& s, int T, unsigned idx) {
    const PT& pt = *job.pt;
    rach_u32x4 d = ra_draws(job, idx, T);
    unsigned p = pt.modP(d.v[pt.geometry ? 2 : 0] >> 1);
    uint4 nr = make_uint4(idx, (unsigned)(T + 1), ra_z((unsigned)T, 0), ra_w3(p, 0, 1, 0));
    if (DUMP) {
        int* row = job.dump + (size_t)idx * RA_DUMP_W;
        row[3] = T + 1; row[7] = 1;
        row[15] = pt.geometry ? ra_sector((int)(d.v[0] >> 1)) : -1;
    }
    ra_schedule(pt, w, s, nr);
}

/* Msg3 / Msg4 of entry `item` of the Msg3 calendar of ms T, W:667-710; returns 1 if the UE finished */
template <bool DUMP, class PT>
RA_HD int ra_msg3_item(const RaJobT<PT>& job, const RaWork& w, RaShared& s, RaAcc& acc, int T, unsigned item) {
    const PT& pt = *job.pt;
    uint4 rec = w.msg3[(size_t)((unsigned)T & (RA_M3RING - 1)) * w.cap3 + item];
    const unsigned idx = rec.x;
    rach_u32x4 d = ra_draws(job, idx, T);
    if (ra_rec_flag(rec) == 0) {                        /* connectionRequest 0 -> 1 < 48 */
        if (rach_msg3_success((int)(d.v[0] >> 1))) {
            unsigned timer = (unsigned)T - ra_rec_ts(rec) + 6;         /* W:674 */
            RA_AADD(&s.nSuccess, 1u);
            RA_AADD64(&s.txSum, ra_rec_ptc(rec));
            RA_AADD64(&s.delaySum, timer);
            RA_AADD64(&s.failSum, ra_rec_fail(rec));
            ra_hist_add(job, timer, ra_rec_ptc(rec), ra_rec_fail(rec));
            if (DUMP) {
                int* row = job.dump + (size_t)idx * RA_DUMP_W;
                row[0] = (int)timer; row[1] = 0; row[2] = T; row[5] = 0;
                row[6] = (int)ra_rec_p(rec); row[10] = (int)ra_rec_ptc(rec); row[11] = 1;
                row[12] = 1; row[13] = 1; row[14] = (int)ra_rec_fail(rec);
            }
            return 1;
        }
        rec.y = (unsigned)(T + 48); rec.w |= 0x80000000u;   /* W:678-679 */
        ra_msg3_push(pt, w, s, T + 48, rec);
        return 0;
    }
    /* 48 ms later: full restart, W:682-708 (accessTime is the literal 5, W:687) */
    acc.contFailed++;
    int tmp = (int)pt.modBI(d.v[0] >> 1);
    int X = ra_align5(T + tmp);
    unsigned pnew = pt.modP(d.v[1] >> 1);
    unsigned fail = ra_rec_fail(rec) + 1;
    if (fail > 0xFFFFu) s.overflow = 2;
    uint4 nr = make_uint4(idx, (unsigned)X, ra_z((unsigned)T, fail), ra_w3(pnew, 0, ra_rec_ptc(rec), 0));
    if (X == T) {                                       /* visible to later scanners, never scans */
        unsigned e = RA_AADD(&s.nE1, 1u);
        w.e1Rec[e] = nr; w.e1Meta[e] = 0;
    } else {
        ra_schedule(pt, w, s, nr);
    }
    return 0;
}

/* the events after the movers: item >= nMov */
template <bool DUMP, class PT>
RA_HD void ra_phase1_item(const RaJobT<PT>& job, const RaWork& w, RaShared& s, RaAcc& acc, int T, unsigned item) {
    item -= s.nMov;
    if (item < (unsigned)s.nArr) { ra_arrival_item<DUMP>(job, w, s, T, (unsigned)s.acOld + item); return; }
    item -= (unsigned)s.nArr;
    if (item < s.nM3) ra_msg3_item<DUMP>(job, w, s, acc, T, item);
}

/* =========================================================================================
 * Phase 2 (one thread, only if nC3 > 0) -- limit-branch movers that would re-transmit now if
 * nobody has postponed them: decide in index order (a landing is itself a scan of its new
 * class and postpones the members above it).
 * ========================================================================================= */
template <class PT>
RA_HD void ra_phase2_serial(const PT& pt, const RaWork& w, RaShared& s) {
    const unsigned n = s.nC3;
    for (unsigned i = 0; i < n; ++i) {                      /* selection by ascending idx */
        unsigned best = i;
        for (unsigned j = i + 1; j < n; ++j) if (w.c3[j].x < w.c3[best].x) best = j;
        uint4 c = w.c3[best]; w.c3[best] = w.c3[i];
        if (c.x < ra_first_scan(pt, c.y)) {                  /* not postponed: lands on pnew */
            c.w = 1;
            if (c.x < S_l2[c.z]) S_l2[c.z] = c.x;
        }
        w.c3[i] = c;
    }
}

/* =========================================================================================
 * Phase 3 -- movers below the natural leader of their class, now that s[] is final.
 * ========================================================================================= */
template <bool DUMP, class PT>
RA_HD void ra_phase3_item(const RaJobT<PT>& job, const RaWork& w, RaShared& s, int T, unsigned u) {
    const PT& pt = *job.pt;
    const uint4 e = w.uncertain[u];
    const unsigned idx = e.y, p0 = e.z & 0xFFu;
    const unsigned sp = ra_first_scan(pt, p0);
    if (idx < sp) RA_AADD(&S_before[p0], 1u);              /* left the class before its first scan */
    if (!(e.z >> 31)) return;
    /* limit branch, W:498-531 */
    uint4 rec = w.bucket[(size_t)((unsigned)T & (unsigned)(pt.R - 1)) * w.cap + e.x];
    rach_u32x4 d = ra_draws(job, idx, T);
    unsigned pnew = pt.modP(d.v[0] >> 1);
    int tmp = (int)pt.modBI(d.v[1] >> 1);
    int base = T + (idx > sp ? 1 : 0);                      /* postponed by the first scan, W:658 */
    int X = ra_align_pt(pt, base + tmp);
    uint4 nr = make_uint4(idx, (unsigned)X, ra_z((unsigned)T, ra_rec_fail(rec) + 1), ra_w3(pnew, 0, 1, 0));
    if (DUMP) job.dump[(size_t)idx * RA_DUMP_W + 3] = T + 1;
    if (X == T) ra_lander_push(w, s, nr, pnew == p0 ? 1u : 0u);   /* S_l2 already holds it (phase 2) */
    else ra_schedule(pt, w, s, nr);                         /* X > T always: base >= T */
}

/* =========================================================================================
 * Phase 3b (only if nE1 > 0) -- a Msg3 restart that landed on T at index k is counted by the
 * first scan of its class at an index above k (W:613-621), which postpones it.
 * ========================================================================================= */
template <class PT>
RA_HD void ra_phase3b_item(const PT& pt, const RaWork& w, RaShared& s, unsigned e) {
    const uint4 r = w.e1Rec[e];
    const unsigned k = r.x, q = ra_rec_p(r);
    unsigned bestIdx = RA_INF32, bestRef = RA_INF32;
    unsigned sq = ra_first_scan(pt, q);
    if (sq != RA_INF32 && sq > k && sq == S_l1[q]) { bestIdx = sq; bestRef = 0x80000000u | q; }
    for (unsigned l = 0; l < s.nLanders; ++l) {
        const uint4 lr = w.landerRec[l];
        if (ra_rec_p(lr) == q && lr.x > k && lr.x < bestIdx) { bestIdx = lr.x; bestRef = l; }
    }
    if (bestIdx == RA_INF32) return;
    w.e1Meta[e] = 1;
    if (bestRef & 0x80000000u) RA_AADD(&S_extraFirst[q], 1u);
    else RA_AADD(&w.landerMeta[bestRef], 256u);
}

/* =========================================================================================
 * Phase 4 -- the collision scans of ms T, W:607-665.
 *   class items  [0, P):        first scan by the natural leader (a visible non-mover)
 *   lander items [P, P+nLanders): scan by a UE that re-transmits in this ms
 * ========================================================================================= */
/* singleton j of the ms: the first RA_SCAP in shared memory, all of them in the workspace */
template <class PT>
RA_HD unsigned ra_single(const PT& pt, const RaWork& w, unsigned j) { return j < RA_SCAP ? S_sIdx[j] : w.singles[j]; }

template <class PT>
RA_HD void ra_single_push(const PT& pt, const RaWork& w, RaShared& s, unsigned idx) {
    unsigned k = RA_AADD(&s.nSingles, 1u);
    if (k < RA_SCAP) S_sIdx[k] = idx;
    w.singles[k] = idx;
    RA_AADD(&S_hist[idx >> pt.hshift], 1u);
}

RA_HD void ra_count_scan(RaAcc& acc, unsigned size) {
    acc.totScans++;                                         /* B:334,351 */
    if (size == 1) { acc.txop++; }                          /* W:625 */
    else { acc.collP += size; acc.txop += size; acc.collScans++; }   /* W:650-652, B:349 */
}

template <class PT>
RA_HD void ra_phase4_item(const PT& pt, const RaWork& w, RaShared& s, RaAcc& acc, unsigned item) {
    if (item < (unsigned)pt.P) {
        const unsigned q = item;
        const unsigned sq = ra_first_scan(pt, q);
        if (sq == RA_INF32 || sq != S_l1[q]) return;        /* no scan, or a lander scans first */
        unsigned size = S_N[q] - S_before[q] + S_extraFirst[q];
        S_clsSize[q] = size;
        ra_count_scan(acc, size);
        if (size == 1) {
            ra_single_push(pt, w, s, sq);
        }
        return;
    }
    const unsigned l = item - (unsigned)pt.P;
    if (l >= s.nLanders) return;
    const uint4 r = w.landerRec[l];
    const unsigned q = ra_rec_p(r), meta = w.landerMeta[l];
    unsigned size;
    if (r.x == ra_first_scan(pt, q)) size = S_N[q] - S_before[q] + ((meta & 1u) ? 0u : 1u) + (meta >> 8);
    else size = 1u + (meta >> 8);
    ra_count_scan(acc, size);
    if (size == 1) {
        ra_single_push(pt, w, s, r.x);
    } else {
        w.landerMeta[l] = meta | 2u;                        /* collided */
    }
}

/* =========================================================================================
 * Phase 5 (one warp, vector form of rach_warp.cuh) -- UL grants: the first G-1-grantCheck
 * singleton scans in UE index order are granted (strict '<' after the increment, W:639-641).
 * tau = highest granted index (RA_INF32: all, 0 with nobody granted handled by flag).
 * Histogram over index bins (filled by phase 4) -> the bin holding the K-th smallest -> exact
 * rank inside that bin.
 * ========================================================================================= */
/* the same threshold by one thread, straight from the definition: the reference formulation the host emulation checks
 * ra_phase5_warp against */
template <class PT>
RA_HD void ra_phase5_serial(const PT& pt, const RaWork& w, RaShared& s) {
    const unsigned n = s.nSingles;
    long long K = (long long)pt.G - 1 - s.grantCheck;
    if (K < 0) K = 0;
    if ((long long)n <= K) { s.tau = RA_INF32; }
    else if (K == 0) { s.tau = 0; s.noGrant = 1; }
    else {
        unsigned prev = 0; bool first = true;
        for (long long r = 0; r < K; ++r) {
            unsigned best = RA_INF32;
            for (unsigned j = 0; j < n; ++j) {
                unsigned v = w.singles[j];
                if ((first || v > prev) && v < best) best = v;
            }
            prev = best; first = false;
        }
        s.tau = prev;
    }
    s.grantCheck += (int)n;
}

template <class PT>
RW_FN void ra_phase5_warp(const PT& pt, const RaWork& w, RaShared& s) {
    const unsigned n = s.nSingles;
    long long K = (long long)pt.G - 1 - s.grantCheck;
    if (K < 0) K = 0;
    unsigned tau = RA_INF32, noGrant = 0;
    if ((long long)n > K) {
        if (K == 0) { noGrant = 1; tau = 0; }
        else if (n <= 32u) {
            /* at most one singleton per lane (the normal case away from the overload peak, where the singletons of a ms are
             * the UEs of one arrival step -- consecutive indices, all in ONE histogram bin, so the bin walk below would
             * take K full passes): rank by counting, the K-th smallest is the lane whose rank is K - 1 (indices are distinct) */
            unsigned v[RW_LANES];
            int hit[RW_LANES];
            RW_EACH(l) v[l] = (unsigned)lane < n ? ra_single(pt, w, (unsigned)lane) : RA_INF32;
            RW_EACH(l) {
                unsigned rank = 0;
                for (unsigned i = 0; i < n; ++i) rank += RW_SHFL(v, (int)i) < v[l] ? 1u : 0u;
                hit[l] = (unsigned)lane < n && rank == (unsigned)K - 1u;
            }
            tau = RW_SHFL(v, RW_FFS(RW_BALLOT(hit)) - 1);
        }
        else {
            const unsigned k = (unsigned)K;
            const int per = RA_HBINS / 32;
            unsigned sum[RW_LANES], incl[RW_LANES], bstar[RW_LANES], before[RW_LANES];
            int ge[RW_LANES];
            RW_EACH(l) { sum[l] = 0; for (int b = 0; b < per; ++b) sum[l] += S_hist[lane * per + b]; }
            rw_scan_u32(sum, incl);
            RW_EACH(l) ge[l] = incl[l] >= k;
            const int L = RW_FFS(RW_BALLOT(ge)) - 1;
            RW_EACH(l) {
                bstar[l] = 0; before[l] = 0;
                if (lane == L) {
                    unsigned c = incl[l] - sum[l];
                    for (int b = 0; b < per; ++b) {
                        const unsigned h = S_hist[lane * per + b];
                        if (c + h >= k) { bstar[l] = (unsigned)(lane * per + b); before[l] = c; break; }
                        c += h;
                    }
                }
            }
            const unsigned bin = RW_SHFL(bstar, L);
            const unsigned kk = k - RW_SHFL(before, L);     /* 1-based rank inside bin `bin` */
            unsigned prev = 0; bool first = true;
            for (unsigned r = 0; r < kk; ++r) {
                unsigned best[RW_LANES];
                RW_EACH(l) {
                    best[l] = RA_INF32;
                    for (unsigned j = lane; j < n; j += 32) {
                        const unsigned x = ra_single(pt, w, j);
                        if ((x >> pt.hshift) == bin && (first || x > prev) && x < best[l]) best[l] = x;
                    }
                }
                prev = rw_min_u32(best); first = false;
            }
            tau = prev;
        }
    }
    RW_EACH(l) if (lane == 0) { s.tau = tau; s.noGrant = noGrant; s.grantCheck += (int)n; }
}

RA_HD bool ra_granted(const RaShared& s, unsigned idx) { return !s.noGrant && idx <= s.tau; }

/* Phase 5 is not needed when every singleton scan of the ms is answered (grantCheck + n < G, W:639-641): the flags the
 * ms started with (tau = everybody, noGrant = 0) already say so.  Every thread evaluates this after phase 4 (same
 * answer); one thread notes the count, and grantCheck itself is only touched once nobody reads it any more: by the
 * thread that opens the next ms (ra_gc_apply).  Saves a block barrier in most ms of a lightly or moderately loaded cell. */
template <class PT>
RA_HD bool ra_phase5_trivial(const PT& pt, const RaShared& s) {
    return (long long)s.nSingles <= (long long)pt.G - 1 - (long long)s.grantCheck;
}
RA_HD void ra_gc_apply(RaShared& s) {                            /* one thread, before the next ms reads grantCheck */
    if (s.gcAdd) { s.grantCheck += s.gcAdd; s.gcAdd = 0; }
}

/* a granted visible non-mover leaves its bucket and cohort and queues Msg3 (W:642-645) */
template <bool DUMP, class PT>
RA_HD void ra_grant_nonmover(const RaJobT<PT>& job, const RaWork& w, RaShared& s, int T, unsigned q, unsigned slot, size_t at) {
    const PT& pt = *job.pt;
    uint4 rec = w.bucket[at];
    w.bucket[at].x = RA_DEAD;
    RA_AADD(&S_dead[slot], 1u);
    S_cnt[slot * pt.P + q] -= 1; S_minI[slot * pt.P + q] = RA_INF32;   /* it was alone in its class */
    if (DUMP) {
        int* row = job.dump + (size_t)rec.x * RA_DUMP_W;
        row[8] = T - (int)rec.y + 1; row[9] = (int)ra_rec_mrc(rec);
    }
    rec.y = (unsigned)(T + 11); rec.w &= 0x7FFFFFFFu;
    ra_msg3_push(pt, w, s, T + 11, rec);
}

/* =========================================================================================
 * Phase 6 -- apply the outcomes of the scans (W:641-648, W:653-661), retire ms T.
 * items: [0,P) classes, [P, P+nLanders) landers, [.., +nE1) late restarts
 * ========================================================================================= */
template <bool DUMP, class PT>
RA_HD void ra_phase6_item(const RaJobT<PT>& job, const RaWork& w, RaShared& s, int T, unsigned item) {
    const PT& pt = *job.pt;
    const unsigned Rm = (unsigned)(pt.R - 1);
    if (item < (unsigned)pt.P) {
        const unsigned q = item;
        const unsigned sq = ra_first_scan(pt, q);
        if (sq != RA_INF32 && sq == S_l1[q] && S_clsSize[q] == 1 && ra_granted(s, sq)) {
            /* a visible non-mover scanned alone and was granted: active=2, txTime=T+11, W:642-645.  Its record
             * sits in the bucket of its move time, normally at the hinted position */
            const unsigned slot = S_l1m[q], hint = w.minPos[slot * pt.P + q];
            const size_t at = (size_t)slot * w.cap + hint;
#ifndef RA_NO_POS_HINT
            if (hint < S_bcount[slot] && w.bucket[at].x == sq) ra_grant_nonmover<DUMP>(job, w, s, T, q, slot, at);
            else
#endif
            { unsigned k = RA_AADD(&s.nNl, 1u); S_nlList[k] = q; }      /* rare: found by ra_phase6b */
        }
        if (q == 0) { S_bcount[(unsigned)T & Rm] = 0; S_dead[(unsigned)T & Rm] = 0; S_m3count[(unsigned)T & (RA_M3RING - 1)] = 0; }
        /* the cohort that moved in this ms is gone */
        S_cnt[((unsigned)T & Rm) * pt.P + q] = 0; S_minI[((unsigned)T & Rm) * pt.P + q] = RA_INF32;
        return;
    }
    item -= (unsigned)pt.P;
    if (item < s.nLanders) {
        uint4 r = w.landerRec[item];
        const unsigned meta = w.landerMeta[item];
        if (!(meta & 2u) && ra_granted(s, r.x)) {
            if (DUMP) { int* row = job.dump + (size_t)r.x * RA_DUMP_W; row[8] = 0; row[9] = (int)ra_rec_mrc(r); }
            r.y = (unsigned)(T + 11);
            ra_msg3_push(pt, w, s, T + 11, r);
        } else {
            r.y = (unsigned)(T + 1);                        /* txTime++, W:647 / W:658 */
            ra_schedule(pt, w, s, r);                       /* rarWindow 0 now -> expires at T+Wn */
        }
        return;
    }
    item -= s.nLanders;
    if (item < s.nE1) {
        uint4 r = w.e1Rec[item];
        if (w.e1Meta[item]) { r.y = (unsigned)(T + 1); ra_schedule(pt, w, s, r); }
        else ra_park_stale(pt, w, s, T, r);
    }
}

/* Phase 6b (every thread, only if nNl > 0) -- fallback for a granted visible non-mover whose position hint
 * was stale (two UEs lowered the cohort minimum at the same time): find the record in the bucket of its move
 * time by index. */
template <bool DUMP, class PT>
RA_HD void ra_phase6b(const RaJobT<PT>& job, const RaWork& w, RaShared& s, int T, int tid, int nt, unsigned nNl) {
    const PT& pt = *job.pt;
    for (unsigned e = 0; e < nNl; ++e) {
        const unsigned q = S_nlList[e], slot = S_l1m[q], want = S_l1[q];
        const unsigned n = S_bcount[slot];
        for (unsigned j = tid; j < n; j += nt) {
            const size_t at = (size_t)slot * w.cap + j;
            if (w.bucket[at].x != want) continue;
            ra_grant_nonmover<DUMP>(job, w, s, T, q, slot, at);
        }
    }
}

/* with phase 6 (every thread), only if the ms had singleton scans */
template <class PT>
RA_HD void ra_hist_clear(const PT& pt, const RaWork& w, RaShared& s, int tid, int nt) {
    const unsigned n = s.nSingles;
    if (n > RA_HBINS / 2) { for (int i = tid; i < RA_HBINS; i += nt) S_hist[i] = 0; }
    else for (unsigned j = tid; j < n; j += nt) S_hist[ra_single(pt, w, j) >> pt.hshift] = 0;
}

/* =========================================================================================
 * A LIGHT ms, start to end, by ONE WARP without a block barrier (vector form of rach_warp.cuh).
 *
 * Most simulated ms have no mover at all: under Uniform traffic a lone UE is answered at its first scan and leaves
 * only a dead record behind; under overload the movers sit in one ms of five.  What such a ms still does is small:
 * a few arrivals and Msg3 answers (at most one per lane here), the re-scan of the visible classes -- every member is
 * a non-mover, so a class of size n is one scan by its lowest index (W:613-662: n == 1 -> singleton, UL grant in index
 * order while grantCheck < G, W:639-641; n > 1 -> collision counters) -- and the retirement of an empty bucket.
 * The general path spends five block-wide barriers and seven passes on it; this routine fuses phases 0, 1, 4, 5 and 6
 * into one warp-synchronous pass, and the kernel runs such ms back to back while the other warps wait at one barrier.
 *
 * returns 0  not a light ms (real movers, or more than 32 events): nothing was touched, run the general path
 *         1  ms T is complete
 *         2  the events (phase 1) are done but a Msg3 restart landed on this ms (W:693): continue with the general
 *            path from the class view (ra_phase0_classes) and phase 2
 *         3  complete except for a granted UE whose position hint was stale: run ra_phase6b
 * ========================================================================================= */
/* the control block of the replication as warp-uniform registers: warp 0 keeps it there while it runs light ms back to
 * back (every lane computes the same updates) and writes it back to shared memory when the block takes over */
struct RaCtl { int grantCheck, activeCheck, nextAc, nextArrMs, occ; unsigned nM3sum; };
RA_HD RaCtl ra_ctl_load(const RaShared& s) {
    RaCtl c; c.grantCheck = s.grantCheck; c.activeCheck = s.activeCheck; c.nextAc = s.nextAc; c.nextArrMs = s.nextArrMs;
    c.occ = s.occ; c.nM3sum = 0;
    return c;
}
RA_HD void ra_ctl_store(RaShared& s, const RaCtl& c) {           /* one thread */
    s.grantCheck = c.grantCheck; s.activeCheck = c.activeCheck; s.nextAc = c.nextAc; s.nextArrMs = c.nextArrMs;
    s.occ = c.occ; s.recMoves += c.nM3sum;
}

RA_HD void ra_lists_reset(RaShared& s) {                         /* one thread; what ra_phase0_ctl does per ms */
    s.nLanders = 0; s.nUnc = 0; s.nC3 = 0; s.nSingles = 0; s.nE1 = 0; s.tau = RA_INF32; s.noGrant = 0; s.nNl = 0;
    s.nNlLight = 0;
}

/* done = 1 if the replication ended with this ms (everybody succeeded, or the horizon); on entry s.nE1 == s.nNlLight == 0 */
template <bool DUMP, class PT>
RW_FN int ra_light_ms(const RaJobT<PT>& job, const RaWork& w, RaShared& s, RaCtl& c, RaAcc* acc, int T, int* done, int* simTime) {
    const PT& pt = *job.pt;
    const int P = pt.P, Wn = pt.Wn;
    const unsigned Rm = (unsigned)(pt.R - 1), slotT = (unsigned)T & Rm;
    /* eligibility: no state is touched before the ms is known to be light.  One ballot answers it together with the
     * question the class view asks below -- which cohorts of the window [T, T+Wn-1] have a live record at all (lane d
     * looks at the bucket of T+d; bit 0 = bucket T itself).  The events of this ms cannot change the answer: an arrival
     * or a Msg3 restart transmits at T+1 or later and so joins the cohort of T+Wn or later. */
    const bool canSkip = Wn <= 32;                          /* one bit per cohort of the window */
    unsigned liveWin = 0;
    if (canSkip) {
        int lv[RW_LANES];
        RW_EACH(l) { const unsigned m = ((unsigned)(T + lane) & Rm); lv[l] = lane < Wn && S_bcount[m] != S_dead[m]; }
        liveWin = RW_BALLOT(lv);
        if (liveWin & 1u) return 0;
    } else if (S_bcount[slotT] != S_dead[slotT]) return 0;
    const bool arrivalMs = T == c.nextArrMs;
    const int newAc = (arrivalMs && c.activeCheck != pt.nUE) ? c.nextAc : c.activeCheck;
    const unsigned nArr = (unsigned)(newAc - c.activeCheck), nM3 = S_m3count[(unsigned)T & (RA_M3RING - 1)];
    if (nArr + nM3 > 32u) return 0;
    /* control block of ms T (ra_phase0_ctl on registers) */
    if ((unsigned)T % 5u == 0) c.grantCheck = 0;          /* literal 5, W:268 */
    const unsigned acOld = (unsigned)c.activeCheck;
    c.activeCheck = newAc;
    if (arrivalMs) {
        c.nextArrMs = T + pt.A; c.occ++;
        if (c.occ < pt.nOcc) c.nextAc = pt.arrCum[c.occ];
    }
    c.nM3sum += nM3;
    /* phase 1: arrivals (W:294-298), then Msg3 answers (W:318-321), one per lane */
    int fin[RW_LANES];
    RW_EACH(l) {
        fin[l] = 0;
        if ((unsigned)lane < nArr) ra_arrival_item<DUMP>(job, w, s, T, acOld + (unsigned)lane);
        else if ((unsigned)lane < nArr + nM3) fin[l] = ra_msg3_item<DUMP>(job, w, s, acc[l], T, (unsigned)lane - nArr);
    }
    const unsigned anyFin = nM3 ? RW_BALLOT(fin) : 0u;
    RW_SYNC();
    if (nM3 && s.nE1) return 2;
    /* phases 0 + 4 fused: the class view, and the one scan per visible class (no mover, no re-transmitter, nobody left
     * early: size = N, first scan by the lowest visible index).  A cohort whose bucket holds no live record (empty, or
     * every record granted away) has an all-zero row: skipped for all classes at once. */
    const unsigned liveSlots = canSkip ? liveWin : 1u;
    unsigned nSing = 0;
    if (liveSlots) {
        int f[RW_LANES];
        for (int base = 0; base < P; base += 32) {
            RW_EACH(l) {
                const int q = base + lane;
                f[l] = 0;
                if (q < P) {
                    unsigned n = 0, best = RA_INF32, bestm = 0;
                    for (int d = 1; d < Wn; ++d) {      /* all rows: skipping the dead ones measured 1-2 % slower */
                        const unsigned m = ((unsigned)(T + d) & Rm);
                        n += S_cnt[m * P + q];
                        const unsigned v = S_minI[m * P + q]; if (v < best) { best = v; bestm = m; }
                    }
                    S_N[q] = n; S_l1[q] = best; S_l1m[q] = bestm;
                    if (n) ra_count_scan(acc[l], n);
                    f[l] = n == 1u;
                }
            }
            nSing += (unsigned)RW_POPC(RW_BALLOT(f));
        }
    }
    if (nSing) {
        /* phase 5: the first G-1-grantCheck singleton scans in UE index order are granted (W:639-641) */
        RW_SYNC();
        long long K = (long long)pt.G - 1 - c.grantCheck;
        if (K < 0) K = 0;
        unsigned tau = RA_INF32, noGrant = 0;
        if ((long long)nSing > K) {
            if (K == 0) noGrant = 1;
            else {
                unsigned prev = 0; bool first = true;
                for (long long r = 0; r < K; ++r) {
                    unsigned bv[RW_LANES];
                    RW_EACH(l) {
                        bv[l] = RA_INF32;
                        for (int q = lane; q < P; q += 32)
                            if (S_N[q] == 1u) { const unsigned v = S_l1[q]; if ((first || v > prev) && v < bv[l]) bv[l] = v; }
                    }
                    prev = rw_min_u32(bv); first = false;
                }
                tau = prev;
            }
        }
        /* phase 6: granted -> Msg3 calendar (W:642-645); the others stay where they are (txTime++ is implicit) */
        if (!noGrant) {
            RW_EACH(l) for (int q = lane; q < P; q += 32) {
                if (S_N[q] != 1u || S_l1[q] > tau) continue;
                const unsigned slot = S_l1m[q], hint = w.minPos[slot * P + q];
                const size_t at = (size_t)slot * w.cap + hint;
#ifndef RA_NO_POS_HINT
                if (hint < S_bcount[slot] && w.bucket[at].x == S_l1[q]) ra_grant_nonmover<DUMP>(job, w, s, T, (unsigned)q, slot, at);
                else
#endif
                { const unsigned k = RA_AADD(&s.nNlLight, 1u); S_nlList[k] = (unsigned)q; }      /* rare: found by ra_phase6b */
            }
        }
        c.grantCheck += (int)nSing;
    }
    /* retire ms T: its bucket held dead records only, so its cohorts are already empty */
    if (S_bcount[slotT] | nM3) {
        RW_EACH(l) if (lane == 0) { S_bcount[slotT] = 0; S_dead[slotT] = 0; S_m3count[(unsigned)T & (RA_M3RING - 1)] = 0; }
    }
    RW_SYNC();
    if (nSing && s.nNlLight) return 3;
    /* W:330-334 and the loop bound W:267 */
    *done = 0;
    if (anyFin && s.nSuccess == (unsigned)pt.nUE) { *simTime = T; *done = 1; }
    else if (T + 1 >= pt.maxTime) { *simTime = pt.maxTime; *done = 1; }
    return 1;
}

/* after phase 6 (every thread, same answer): W:330-334 and the loop bound W:267 */
template <class PT>
RA_HD bool ra_ms_done(const PT& pt, const RaShared& s, int T, int* simTime) {
    if (s.nSuccess == (unsigned)pt.nUE) { *simTime = T; return true; }
    if (T + 1 >= pt.maxTime) { *simTime = pt.maxTime; return true; }
    return false;
}

/* =========================================================================================
 * End of the replication (DUMP only): state of the UEs still in flight after the last
 * executed ms `last`, as the reference's per-ms bookkeeping would have left it.
 * ========================================================================================= */
template <class PT>
RA_HD void ra_dump_inflight(const RaJobT<PT>& job, const RaWork& w, RaShared& s, int last, int tid, int nt) {
    const PT& pt = *job.pt;
    for (int slot = 0; slot < pt.R; ++slot) {
        /* absolute move time of this slot: the value in (last, last+R] congruent to slot */
        int m = last + 1 + (int)(((unsigned)slot - (unsigned)(last + 1)) & (unsigned)(pt.R - 1));
        for (unsigned j = tid; j < S_bcount[slot]; j += nt) {
            uint4 r = w.bucket[(size_t)slot * w.cap + j];
            if (r.x == RA_DEAD) continue;
            int* row = job.dump + (size_t)r.x * RA_DUMP_W;
            int X = (int)r.y;
            row[0] = last + 1 - (int)ra_rec_ts(r);                         /* timer, W:713 */
            row[1] = 1;
            if (ra_rec_flag(r)) {                                          /* stale */
                int t0 = m - pt.Wn;
                row[2] = X; row[8] = last - t0; row[5] = X - t0 < 0 ? X - t0 : 0;
            } else if (X > last) {                                         /* in backoff */
                row[2] = X; row[8] = 0; row[5] = X - last - 1;
            } else {                                                       /* transmitted, postponed */
                row[2] = last + 1; row[8] = last - X + 1; row[5] = 0;
            }
            row[6] = (int)ra_rec_p(r); row[7] = 1; row[9] = (int)ra_rec_mrc(r);
            row[10] = (int)ra_rec_ptc(r); row[11] = 0; row[12] = 0; row[13] = 0;
            row[14] = (int)ra_rec_fail(r);
        }
    }
    for (int slot = 0; slot < RA_M3RING; ++slot) {
        for (unsigned j = tid; j < S_m3count[slot]; j += nt) {
            uint4 r = w.msg3[(size_t)slot * w.cap3 + j];
            int* row = job.dump + (size_t)r.x * RA_DUMP_W;
            row[0] = last + 1 - (int)ra_rec_ts(r);
            row[1] = 2; row[2] = (int)r.y; row[5] = 0; row[6] = (int)ra_rec_p(r); row[7] = 1;
            row[10] = (int)ra_rec_ptc(r); row[11] = 1; row[12] = ra_rec_flag(r) ? 48 : 0;
            row[13] = 0; row[14] = (int)ra_rec_fail(r);
        }
    }
}

#endif /* RACH_CORE_CUH */
