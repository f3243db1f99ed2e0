/*
 * rach_core_n.cuh -- per-replication engine of variant N: the sector / gain-pairing simulator
 * NOMA.c (main loop N:665-711, activeUE N:131-192, preambleSectorCollisionDetection N:194-324,
 * msg2Results N:449-498, resourceRequestAllocation N:499-546, timers N:702-706).
 *
 * NOMA.c is already phase-structured per RACH occasion (every accessTime ms): all UEs whose
 * txTime is occasion+1 transmit, the base station decides per sector, every transmitter then
 * learns its fate.  Event-driven form used here:
 *   * a UE waiting to transmit is one 16-byte record in the calendar bucket of its occasion
 *     (txTime - 1); arrivals are appended to the bucket of the current occasion;
 *   * per occasion: histogram over (sector, preamble) in shared memory -> singletons in preamble
 *     order per sector -> grants (<= G per sector: in preamble order, N:252-260; more singletons
 *     than grants: stable sort by channel gain N:90-103, pairing 10*log(h)-10*log(l) > 15.
 *     N:268-298 with the base-station draws N:284,286, leftovers N:299-307) -> every record is
 *     re-read and moved: granted -> Msg3 calendar (txTime += 10, N:494), else backoff
 *     (N:453-479) or dropped after maxMsg1ReTx (RaFailed, N:481-488);
 *   * Msg3 (N:499-546) is a per-ms calendar: 90 % success, else +49 ms, then restart with a new
 *     preamble and an aligned backoff; a restart whose txTime is not after the current ms can
 *     never transmit again in the reference (txTime == time+1 is tested only at occasions):
 *     such a UE becomes a "zombie" (kept only for the per-UE dump).
 * pt.geometry == 0 selects NOMA.c's alternative, non-sector collision function (N:325-447; its call is commented
 * out at N:688): one grant counter for the whole cell, no sector buckets, a lone singleton is always answered
 * (N:377-384), one base-station draw per granted pair and p < 0.3 answers only the weaker UE (N:411-415).
 * timer / nowBackoff are derived from (timerStart, txTime) as in variant W.
 * fp64 follows the C semantics of the reference (float locals, double libm); products and sums
 * that C would not fuse are written with explicit round-to-nearest intrinsics on the device.
 */
#ifndef RACH_CORE_N_CUH
#define RACH_CORE_N_CUH

#include <math.h>
#include "rach_core.cuh"
#include "rach_warp.cuh"

#ifdef __CUDA_ARCH__
#define RA_FMUL(a, b) __fmul_rn((a), (b))
#define RA_FADD(a, b) __fadd_rn((a), (b))
#define RA_DMUL(a, b) __dmul_rn((a), (b))
#define RA_DADD(a, b) __dadd_rn((a), (b))
#define RA_DSUB(a, b) __dsub_rn((a), (b))
#else
#define RA_FMUL(a, b) ((a) * (b))
#define RA_FADD(a, b) ((a) + (b))
#define RA_DMUL(a, b) ((a) * (b))
#define RA_DADD(a, b) ((a) + (b))
#define RA_DSUB(a, b) ((a) - (b))
#endif

#define RA_NSECT 6

/* record: x idx | y txTime (Msg3: due ms) | z timerStart:16 nTxPreamble:8 msg1ReTx:8 |
 * w preamble:8 sector:3 msg3Faile:8 fromRestart:1 ... flag:1 (Msg3 calendar: second visit) */
RA_HD unsigned rn_z(unsigned ts, unsigned nTx, unsigned reTx) { return (ts & 0xFFFFu) | ((nTx & 0xFFu) << 16) | ((reTx & 0xFFu) << 24); }
RA_HD unsigned rn_ts(const uint4& r)   { return r.z & 0xFFFFu; }
RA_HD unsigned rn_ntx(const uint4& r)  { return (r.z >> 16) & 0xFFu; }
RA_HD unsigned rn_retx(const uint4& r) { return r.z >> 24; }
RA_HD unsigned rn_w(unsigned p, unsigned sector, unsigned m3f, unsigned fromRestart, unsigned flag) {
    return (p & 0xFFu) | ((sector & 7u) << 8) | ((m3f & 0xFFu) << 11) | ((fromRestart & 1u) << 19) | (flag << 31);
}
RA_HD unsigned rn_p(const uint4& r)       { return r.w & 0xFFu; }
RA_HD unsigned rn_sector(const uint4& r)  { return (r.w >> 8) & 7u; }
RA_HD unsigned rn_m3f(const uint4& r)     { return (r.w >> 11) & 0xFFu; }
RA_HD unsigned rn_restart(const uint4& r) { return (r.w >> 19) & 1u; }

struct RaWorkN {
    uint4*  bucket;      /* [R][cap] tx calendar, keyed by occasion ms                       */
    uint4*  msg3;        /* [RA_M3RING][cap3]                                                */
    uint4*  zombie;      /* [cap]  restarts that can never transmit again (dump only)        */
    double* gain;        /* [cap]  channelGain of every arrived UE (N:191)                   */
    unsigned* hist;      /* [histLen] the replication's histograms (ra_hist_add), or NULL    */
    int cap, cap3;
};

/* lays out one block's workspace at `base` for a ring of R buckets and histLen histogram counters (0 = none); returns its
 * size in bytes (ra_work_carve) */
static inline size_t rn_work_carve(unsigned char* base, int cap, int cap3, int R, RaWorkN* w, int histLen = 0) {
    const size_t c = (size_t)cap, c3 = (size_t)cap3;
    size_t off = 0;
    w->bucket = (uint4*)ra_carve_next(base, off, sizeof(uint4) * c * (size_t)R);
    w->msg3 = (uint4*)ra_carve_next(base, off, sizeof(uint4) * c3 * RA_M3RING);
    w->zombie = (uint4*)ra_carve_next(base, off, sizeof(uint4) * c);
    w->gain = (double*)ra_carve_next(base, off, sizeof(double) * c);
    w->hist = histLen ? (unsigned*)ra_carve_next(base, off, sizeof(unsigned) * (size_t)histLen) : NULL;
    w->cap = cap; w->cap3 = cap3;
    return off;
}

struct RaSharedN {
    unsigned* cnt;       /* [6*P] transmitters per (sector, preamble)                         */
    unsigned* who;       /* [6*P] bucket position of the first one                            */
    unsigned* grant;     /* [6*P] 1 = the singleton of this cell got msg2                     */
    unsigned* bcount;    /* [R]                                                               */
    unsigned* m3count;   /* [RA_M3RING]                                                       */
    unsigned* sPos;      /* [6*P] singles of a sector: bucket position                        */
    int*      sIdx;      /* [6*P] ... UE index (-1 = paired away, N:280-281)                  */
    double*   sLg;       /* [6*P] ... 10*log(channelGain)                                     */
    double*   sGain;     /* [6*P] ... channelGain                                             */
    unsigned* ord;       /* [6*P] ... the singles in ascending gain order (positions into sPos/sIdx/sGain) */
    int activeCheck, acOld, nArr, overflow;
    unsigned nSuccess, nZombie, nDropped, pad;
    ra_u64 txSum, delaySum;
};

/* the block's tables in dynamic shared memory (the kernel's; the host emulation carves a host buffer the same way) */
RA_HD void rn_carve(RaSharedN& s, unsigned char* base, int R, int P) {
    const size_t c = (size_t)RA_NSECT * P;
    s.sLg = reinterpret_cast<double*>(base);     base += sizeof(double) * c;
    s.sGain = reinterpret_cast<double*>(base);   base += sizeof(double) * c;
    s.cnt = reinterpret_cast<unsigned*>(base);   base += sizeof(unsigned) * c;
    s.who = reinterpret_cast<unsigned*>(base);   base += sizeof(unsigned) * c;
    s.grant = reinterpret_cast<unsigned*>(base); base += sizeof(unsigned) * c;
    s.sPos = reinterpret_cast<unsigned*>(base);  base += sizeof(unsigned) * c;
    s.sIdx = reinterpret_cast<int*>(base);       base += sizeof(int) * c;
    s.ord = reinterpret_cast<unsigned*>(base);   base += sizeof(unsigned) * c;
    s.bcount = reinterpret_cast<unsigned*>(base); base += sizeof(unsigned) * (size_t)R;
    s.m3count = reinterpret_cast<unsigned*>(base);
}
RA_HD size_t rn_smem_bytes(int R, int P) {
    return (size_t)RA_NSECT * P * (2 * sizeof(double) + 6 * sizeof(unsigned)) + sizeof(unsigned) * ((size_t)R + RA_M3RING);
}

/* UE draw stream of one (ue, ms): draw k is word k&3 of block k>>2 */
struct RaStream {
    ra_u64 seed; unsigned rep, ue, ms, k; rach_u32x4 blk;
};
RA_HD RaStream ra_stream(const RaJob& job, unsigned ue, int ms) {
    RaStream s; s.seed = job.pt->seed; s.rep = job.rep; s.ue = ue; s.ms = (unsigned)ms; s.k = 0;
    s.blk.v[0] = s.blk.v[1] = s.blk.v[2] = s.blk.v[3] = 0;
    return s;
}
RA_HD int ra_stream_next(RaStream& s) {
    if ((s.k & 3u) == 0) s.blk = rach_tape_block(s.seed, s.rep, s.ue, s.ms, s.k >> 2, RACH_TAPE_TAG_UE);
    int r = (int)(s.blk.v[s.k & 3u] >> 1);
    s.k++;
    return r;
}

RA_HD unsigned rn_bucket_push(const RaPointDev& pt, const RaWorkN& w, RaSharedN& s, int occasionMs, const uint4& rec) {
    unsigned slot = (unsigned)occasionMs & (unsigned)(pt.R - 1);
    unsigned pos = RA_AADD(&s.bcount[slot], 1u);
    if (pos >= (unsigned)w.cap) { s.overflow = 1; return 0; }
    w.bucket[(size_t)slot * w.cap + pos] = rec;
    return pos;
}
RA_HD void rn_msg3_push(const RaWorkN& w, RaSharedN& s, int due, const uint4& rec) {
    unsigned slot = (unsigned)due & (RA_M3RING - 1);
    unsigned pos = RA_AADD(&s.m3count[slot], 1u);
    if (pos >= (unsigned)w.cap3) { s.overflow = 1; return; }
    w.msg3[(size_t)slot * w.cap3 + pos] = rec;
}

/* dump row order (saveResultLogs fields, N:577-592, + nTxPreamble): 0 timer 1 active 2 txTime 3 firstTxTime 4 secondTxTime
 * 5 nowBackoff 6 preamble 7 sector 8 rarWindow 9 msg1ReTx 10 nTxPreamble 11 msg2 12 msg3Wait
 * 13 RA 14 msg3Faile 15 RaFailed */
RA_HD void rn_dump_init_row(int* d) { for (int k = 0; k < RA_DUMP_W; ++k) d[k] = 0; d[7] = -1; }   /* N:104-130 */

template <bool DUMP>
RA_HD void rn_job_init(const RaJob& job, RaSharedN& s, int tid, int nt) {
    const RaPointDev& pt = *job.pt;
    for (int i = tid; i < pt.R; i += nt) s.bcount[i] = 0;
    for (int i = tid; i < RA_M3RING; i += nt) s.m3count[i] = 0;
    if (DUMP) for (int i = tid; i < pt.nUE; i += nt) rn_dump_init_row(job.dump + (size_t)i * RA_DUMP_W);
    if (tid == 0) {
        s.activeCheck = 0; s.overflow = 0; s.nSuccess = 0; s.nZombie = 0; s.nDropped = 0;
        s.txSum = 0; s.delaySum = 0;
    }
}

/* ---- occasion phase A0: arrival gate N:675-681, clear the (sector, preamble) tables ---- */
RA_HD void rn_phaseA0(const RaJob& job, RaSharedN& s, int T, int tid, int nt) {
    const RaPointDev& pt = *job.pt;
    for (int i = tid; i < RA_NSECT * pt.P; i += nt) { s.cnt[i] = 0; s.grant[i] = 0; }
    if (tid == 0) {
        s.acOld = s.activeCheck;
        s.activeCheck = pt.arrCum[T / pt.A];
        s.nArr = s.activeCheck - s.acOld;
    }
}

/* ---- occasion phase A1: activeUE N:131-192 for the new arrivals; they transmit in this occasion ---- */
template <bool DUMP>
#define RN_MAX_REJECT 65536   /* draws one rejection loop of activeUE may take before the engine gives up (RA_E_INTERNAL) */
RA_HD void rn_phaseA1_item(const RaJob& job, const RaWorkN& w, RaSharedN& s, int T, unsigned idx) {
    const RaPointDev& pt = *job.pt;
    const float cellRadius = pt.cellRadius;
    RaStream st = ra_stream(job, idx, T);
    const float pi = 3.14;
    const unsigned p = pt.modP((unsigned)ra_stream_next(st));            /* N:133 */
    const int ra = ra_stream_next(st);                                                             /* N:142 */
    const float angle = (float)ra / (float)(2147483647) * 2 * pi;
    const int sector = ra_sector(ra);                                                              /* N:146-163 */
    float r;
    /* the reference's loops have no bound; validation keeps the radius where they end quickly, the cap only turns a
     * hang on absurd parameters into an error */
    for (int it = 0;; ++it) {                                                                      /* N:167-172 */
        r = (float)((double)cellRadius * sqrt((double)((float)ra_stream_next(st) / (float)2147483647)));
        if ((double)r > 35.0) break;
        if (it >= RN_MAX_REJECT) { s.overflow = 3; break; }
    }
    const float x = (float)((double)r * cos((double)angle)), y = (float)((double)r * sin((double)angle));   /* N:176,178 */
    const double env = sqrt((double)RA_FADD(RA_FMUL(x, x), RA_FMUL(y, y)));                         /* N:183 */
    double ch_g = 0;
    for (int it = 0; ch_g < 1e-7; ++it) {                                                          /* N:185-189 */
        if (it >= RN_MAX_REJECT) { s.overflow = 3; break; }
        const float pathloss = (float)sqrt(RA_DADD(1.0, RA_DMUL(env, env)));
        const double rayleigh = sqrt(RA_DMUL(-2.0, log((double)ra_stream_next(st) / (double)2147483647)));
        const double q = rayleigh / (double)pathloss;
        ch_g = RA_DMUL(q, q);
    }
    w.gain[idx] = ch_g;
    const uint4 rec = make_uint4(idx, (unsigned)(T + 1), rn_z((unsigned)T, 1, 0), rn_w(p, (unsigned)sector, 0, 0, 0));
    if (DUMP) { int* row = job.dump + (size_t)idx * RA_DUMP_W; row[3] = T + 1; row[7] = sector; }
    rn_bucket_push(pt, w, s, T, rec);
}

/* ---- occasion phase A2: histogram of the transmitters, N:206-226 ---- */
RA_HD void rn_phaseA2_item(const RaPointDev& pt, const RaWorkN& w, RaSharedN& s, int T, unsigned j) {
    const uint4 r = w.bucket[(size_t)((unsigned)T & (unsigned)(pt.R - 1)) * w.cap + j];
    const unsigned k = (pt.geometry ? rn_sector(r) : 0u) * (unsigned)pt.P + rn_p(r);
    if (RA_AADD(&s.cnt[k], 1u) == 0) s.who[k] = j;
}

/* ---- occasion phase B: the base station's decision for one sector, N:243-309 (one thread) ---- */
RA_HD void rn_phaseB_sector(const RaJob& job, const RaWorkN& w, RaSharedN& s, int T, int sec) {
    const RaPointDev& pt = *job.pt;
    const int P = pt.P, G = pt.G;
    unsigned* sPos = s.sPos + sec * P; int* sIdx = s.sIdx + sec * P;
    double* sLg = s.sLg + sec * P; double* sGain = s.sGain + sec * P;
    const uint4* bT = w.bucket + (size_t)((unsigned)T & (unsigned)(pt.R - 1)) * w.cap;
    int count = 0;
    for (int p = 0; p < P; ++p)                             /* singles in preamble order, N:244-249 */
        if (s.cnt[sec * P + p] == 1) {
            const unsigned pos = s.who[sec * P + p];
            const int idx = (int)bT[pos].x;
            sPos[count] = (unsigned)p; sIdx[count] = idx; sGain[count] = w.gain[idx]; count++;
        }
    if (count == 0) return;
    int grants = 0;
    const bool nonSector = pt.geometry == 0;
    if (count <= G) {                                       /* N:252-260; N:377-384 answers every lone singleton */
        for (int i = 0; i < count; ++i) if (grants < G || nonSector) { grants++; s.grant[sec * P + sPos[i]] = 1; }
        return;
    }
    for (int i = 1; i < count; ++i) {                       /* sortUE N:90-103 == stable ascending sort */
        const unsigned tp = sPos[i]; const int ti = sIdx[i]; const double tg = sGain[i];
        int j = i - 1;
        while (j >= 0 && tg < sGain[j]) { sPos[j + 1] = sPos[j]; sIdx[j + 1] = sIdx[j]; sGain[j + 1] = sGain[j]; --j; }
        sPos[j + 1] = tp; sIdx[j + 1] = ti; sGain[j + 1] = tg;
    }
    for (int i = 0; i < count; ++i) sLg[i] = RA_DMUL(10.0, log(sGain[i]));
    unsigned bsK = 0;
    int pair = 0;
    /* once the sector has no grant left nothing below can change any UE (no msg2, no draw) */
    for (int i = 0; i < count - 1 && grants < G; ++i) {     /* N:268-298 */
        for (int j = 1; j < count; ++j) {
            if (sIdx[i] != -1 && sIdx[j] != -1 && RA_DSUB(sLg[j], sLg[i]) > 15.) {
                pair += 2;
                const unsigned pi_ = sPos[i], pj_ = sPos[j];
                sIdx[i] = -1; sIdx[j] = -1;
                if (grants < G) {
                    grants++;
                    const int r0 = rach_tape_rand31(pt.seed, job.rep, (unsigned)sec, (unsigned)T, bsK++, RACH_TAPE_TAG_BS);
                    const double pr = (double)r0 / (double)2147483647;                         /* N:284 */
                    if (pr < 0.3) {
                        if (nonSector) s.grant[sec * P + pi_] = 1;                             /* N:413-415 */
                        else {
                            const int r1 = rach_tape_rand31(pt.seed, job.rep, (unsigned)sec, (unsigned)T, bsK++, RACH_TAPE_TAG_BS);
                            s.grant[sec * P + ((r1 % 2) ? pj_ : pi_)] = 1;                     /* N:286-287 */
                        }
                    } else { s.grant[sec * P + pi_] = 1; s.grant[sec * P + pj_] = 1; }         /* N:290-291 */
                }
                break;
            }
        }
    }
    (void)pair;                                             /* count - pair > 0 whenever an unpaired single is left */
    for (int i = 0; i < count && grants < G; ++i)           /* N:299-307 */
        if (sIdx[i] != -1) { grants++; s.grant[sec * P + sPos[i]] = 1; }
}

/* ---- occasion phase B, warp form: ONE WARP decides one sector (same decisions as rn_phaseB_sector above, which stays
 * as the one-thread statement of N:243-309 for cross-checks).  Written in the vector form of rach_warp.cuh.
 *   gather   singles in preamble order: ballot + prefix count per 32 preambles (N:244-249)
 *   sort     sortUE (N:90-103) is a stable ascending sort by channelGain: every single counts the singles that sort
 *            before it (gain, then position) and takes that rank -- O(count) per lane instead of O(count^2) on one
 *   pairing  N:268-298 walks the sorted singles i = 0.. and pairs i with the FIRST j >= 1 still unpaired whose
 *            10*log(gain_j) - 10*log(gain_i) > 15.: one ballot per 32 candidates; the base-station draws (N:284,286) are
 *            keyed (sector, ms, k) and computed redundantly by every lane
 *   rest     N:299-307: unpaired singles in gain order while the sector has grants left: ballot + prefix count */
RW_FN void rn_phaseB_warp(const RaJob& job, const RaWorkN& w, RaSharedN& s, int T, int sec) {
    const RaPointDev& pt = *job.pt;
    const int P = pt.P, G = pt.G;
    unsigned* sPos = s.sPos + sec * P; int* sIdx = s.sIdx + sec * P; unsigned* ord = s.ord + sec * P;
    double* sLg = s.sLg + sec * P; double* sGain = s.sGain + sec * P;
    const uint4* bT = w.bucket + (size_t)((unsigned)T & (unsigned)(pt.R - 1)) * w.cap;
    const bool nonSector = pt.geometry == 0;
    int f[RW_LANES];
    int count = 0;
    for (int base = 0; base < P; base += 32) {
        RW_EACH(l) { const int p = base + lane; f[l] = p < P && s.cnt[sec * P + p] == 1; }
        const unsigned mask = RW_BALLOT(f);
        RW_EACH(l) if (f[l]) {
            const int p = base + lane, k = count + RW_POPC(mask & ((1u << lane) - 1u));
            const int idx = (int)bT[s.who[sec * P + p]].x;
            sPos[k] = (unsigned)p; sIdx[k] = idx; sGain[k] = w.gain[idx];
        }
        count += RW_POPC(mask);
    }
    RW_SYNC();
    if (count == 0) return;
    if (count <= G) {                                       /* N:252-260 / N:377-384: every single is answered */
        RW_EACH(l) for (int i = lane; i < count; i += 32) s.grant[sec * P + sPos[i]] = 1;
        return;
    }
    RW_EACH(l) for (int i = lane; i < count; i += 32) {
        const double g = sGain[i];
        int rank = 0;
        for (int j = 0; j < count; ++j) { const double h = sGain[j]; rank += (h < g || (h == g && j < i)) ? 1 : 0; }
        ord[rank] = (unsigned)i;
        sLg[i] = RA_DMUL(10.0, log(g));
    }
    RW_SYNC();
    int grants = 0;
    unsigned bsK = 0;
    for (int ri = 0; ri < count - 1 && grants < G; ++ri) {  /* N:268-298; nothing changes any UE once the grants are gone */
        const unsigned ei = ord[ri];
        if (sIdx[ei] == -1) continue;
        const double lgi = sLg[ei];
        int rj = -1;
        for (int base = 0; base < count && rj < 0; base += 32) {
            RW_EACH(l) {
                const int r = base + lane;
                f[l] = 0;
                if (r >= 1 && r < count) { const unsigned e = ord[r]; f[l] = sIdx[e] != -1 && RA_DSUB(sLg[e], lgi) > 15.; }
            }
            const unsigned mask = RW_BALLOT(f);
            if (mask) rj = base + RW_FFS(mask) - 1;
        }
        if (rj < 0) continue;
        const unsigned ej = ord[rj], pi_ = sPos[ei], pj_ = sPos[ej];
        RW_SYNC();                                          /* every lane has read the marks of this round */
        grants++;
        const int r0 = rach_tape_rand31(pt.seed, job.rep, (unsigned)sec, (unsigned)T, bsK++, RACH_TAPE_TAG_BS);
        const double pr = (double)r0 / (double)2147483647;                                     /* N:284 */
        unsigned g0 = pi_, g1 = pj_;                        /* N:290-291: both */
        if (pr < 0.3) {
            if (nonSector) g1 = pi_;                                                          /* N:413-415 */
            else {
                const int r1 = rach_tape_rand31(pt.seed, job.rep, (unsigned)sec, (unsigned)T, bsK++, RACH_TAPE_TAG_BS);
                g0 = g1 = (r1 % 2) ? pj_ : pi_;                                               /* N:286-287 */
            }
        }
        RW_EACH(l) if (lane == 0) {
            sIdx[ei] = -1; sIdx[ej] = -1;
            s.grant[sec * P + g0] = 1; s.grant[sec * P + g1] = 1;
        }
        RW_SYNC();
    }
    for (int base = 0; base < count && grants < G; base += 32) {                              /* N:299-307 */
        RW_EACH(l) { const int r = base + lane; f[l] = r < count && sIdx[ord[r]] != -1; }
        const unsigned mask = RW_BALLOT(f);
        RW_EACH(l) if (f[l] && grants + RW_POPC(mask & ((1u << lane) - 1u)) < G) s.grant[sec * P + sPos[ord[base + lane]]] = 1;
        grants += RW_POPC(mask);
    }
}

/* ---- occasion phase C: msg2Results(UE, T+1) for every transmitter, N:449-498 ---- */
template <bool DUMP>
RA_HD void rn_phaseC_item(const RaJob& job, const RaWorkN& w, RaSharedN& s, int T, unsigned j) {
    const RaPointDev& pt = *job.pt;
    uint4 r = w.bucket[(size_t)((unsigned)T & (unsigned)(pt.R - 1)) * w.cap + j];
    const unsigned idx = r.x, k = (pt.geometry ? rn_sector(r) : 0u) * (unsigned)pt.P + rn_p(r);
    if (s.cnt[k] == 1 && s.grant[k]) {                      /* msg2 == 1: N:491-497 */
        r.y = (unsigned)(T + 1 + 10);
        if (DUMP) { int* row = job.dump + (size_t)idx * RA_DUMP_W; row[4] = T + 11; }
        rn_msg3_push(w, s, T + 11, r);
        return;
    }
    /* msg2 == 0: rarWindow = 5 >= maxRarWindow -> retransmission, N:452-479 */
    unsigned nTx = rn_ntx(r) + 1, reTx = rn_retx(r) + 1;
    const rach_u32x4 d = ra_draws(job, idx, T + 1);
    const int tmp = (int)pt.modBI(d.v[0] >> 1);
    const int X = ra_align_pt(pt, T + 1 + 3 + tmp);
    if ((int)reTx >= pt.M) {                                /* N:481-488: dropped for good */
        const unsigned pnew = pt.modP(d.v[1] >> 1);
        RA_AADD(&s.nDropped, 1u);
        if (DUMP) {
            int* row = job.dump + (size_t)idx * RA_DUMP_W;
            row[0] = 0; row[1] = 1; row[2] = X; row[4] = X; row[5] = X - (T + 1) - 1; row[6] = (int)pnew;
            row[8] = 0; row[9] = 0; row[10] = 0; row[11] = 0; row[12] = rn_m3f(r) ? 49 : 0; row[13] = 0;
            row[14] = (int)rn_m3f(r); row[15] = 1;
        }
        return;
    }
    if (nTx > 0xFFu) s.overflow = 2;
    const uint4 nr = make_uint4(idx, (unsigned)X, rn_z(rn_ts(r), nTx, reTx), rn_w(rn_p(r), rn_sector(r), rn_m3f(r), 0, 0));
    if (DUMP) job.dump[(size_t)idx * RA_DUMP_W + 4] = X;   /* secondTxTime, N:479 */
    rn_bucket_push(pt, w, s, X - 1, nr);
}

/* ---- every ms: resourceRequestAllocation for the UEs whose Msg3 is due, N:499-546 ---- */
template <bool DUMP>
RA_HD void rn_msg3_item(const RaJob& job, const RaWorkN& w, RaSharedN& s, int T, unsigned j) {
    const RaPointDev& pt = *job.pt;
    uint4 r = w.msg3[(size_t)((unsigned)T & (RA_M3RING - 1)) * w.cap3 + j];
    const unsigned idx = r.x;
    const rach_u32x4 d = ra_draws(job, idx, T);
    if (ra_rec_flag(r) == 0) {                              /* msg3Wait <= 48 */
        if (rach_msg3_success((int)(d.v[0] >> 1))) {        /* N:504-508 */
            const unsigned timer = (unsigned)T - rn_ts(r) + 6;
            RA_AADD(&s.nSuccess, 1u);
            RA_AADD64(&s.txSum, rn_ntx(r));
            RA_AADD64(&s.delaySum, timer);
            ra_hist_add(job, timer, rn_ntx(r), 0u);                /* N has no failCount */
            if (DUMP) {
                int* row = job.dump + (size_t)idx * RA_DUMP_W;
                row[0] = (int)timer; row[1] = 0; row[2] = T; row[5] = 0; row[6] = (int)rn_p(r); row[8] = 0;
                row[9] = (int)rn_retx(r); row[10] = (int)rn_ntx(r); row[11] = 1; row[12] = 0; row[13] = 1;
                row[14] = (int)rn_m3f(r); row[15] = 0;
            }
        } else {                                            /* N:509-512 */
            r.y = (unsigned)(T + 49); r.w |= 0x80000000u;
            rn_msg3_push(w, s, T + 49, r);
        }
        return;
    }
    /* restart, N:514-543: new preamble first (N:519), then the backoff draw (N:520) */
    const unsigned pnew = pt.modP(d.v[0] >> 1);
    const int tmp = (int)pt.modBI(d.v[1] >> 1);
    const int X = ra_align_pt(pt, T + tmp);
    unsigned m3f = rn_m3f(r) + 1;
    if (m3f > 0xFFu) s.overflow = 2;
    const uint4 nr = make_uint4(idx, (unsigned)X, rn_z((unsigned)T, 0, 0), rn_w(pnew, rn_sector(r), m3f, 1, 0));
    if (DUMP) job.dump[(size_t)idx * RA_DUMP_W + 4] = X;
    if (X - 1 > T) rn_bucket_push(pt, w, s, X - 1, nr);     /* next tested at occasion X-1 (N:692) */
    else if (DUMP) {                                        /* txTime == time+1 can never hold again */
        unsigned z = RA_AADD(&s.nZombie, 1u);
        if (z < (unsigned)w.cap) w.zombie[z] = nr; else s.overflow = 1;
    }
}

/* ---- end (DUMP): UEs still in flight after the last executed ms `last` ---- */
RA_HD void rn_dump_row_active1(int* row, const uint4& r, int last, int nowBackoff) {
    row[0] = last + 1 - (int)rn_ts(r); row[1] = 1; row[2] = (int)r.y; row[5] = nowBackoff;
    row[6] = (int)rn_p(r); row[8] = 0; row[9] = (int)rn_retx(r); row[10] = (int)rn_ntx(r); row[11] = 0;
    row[12] = rn_m3f(r) ? 49 : 0; row[13] = 0; row[14] = (int)rn_m3f(r); row[15] = 0;
}
RA_HD void rn_dump_inflight(const RaJob& job, const RaWorkN& w, RaSharedN& s, int last, int tid, int nt) {
    const RaPointDev& pt = *job.pt;
    for (int slot = 0; slot < pt.R; ++slot)
        for (unsigned j = tid; j < s.bcount[slot]; j += nt) {
            const uint4 r = w.bucket[(size_t)slot * w.cap + j];
            const int X = (int)r.y;
            /* backoff set at occasion T (msg2Results: X-T-2, N:478) or at restart ms S (X-S-1, N:538),
             * decremented once per ms since, never below 0 (N:550-552) */
            int nb = X - last - (rn_restart(r) ? 2 : 3);
            if (nb < 0) nb = 0;
            rn_dump_row_active1(job.dump + (size_t)r.x * RA_DUMP_W, r, last, nb);
        }
    for (unsigned j = tid; j < s.nZombie; j += nt) {
        const uint4 r = w.zombie[j];
        const int S = (int)rn_ts(r);
        rn_dump_row_active1(job.dump + (size_t)r.x * RA_DUMP_W, r, last, (int)r.y - S - 1);   /* never > 0 */
    }
    for (int slot = 0; slot < RA_M3RING; ++slot)
        for (unsigned j = tid; j < s.m3count[slot]; j += nt) {
            const uint4 r = w.msg3[(size_t)slot * w.cap3 + j];
            int* row = job.dump + (size_t)r.x * RA_DUMP_W;
            row[0] = last + 1 - (int)rn_ts(r); row[1] = 2; row[2] = (int)r.y; row[5] = 0; row[6] = (int)rn_p(r);
            row[8] = 0; row[9] = (int)rn_retx(r); row[10] = (int)rn_ntx(r); row[11] = 1;
            row[12] = ra_rec_flag(r) ? 49 : 0; row[13] = 0; row[14] = (int)rn_m3f(r); row[15] = 0;
        }
}

#endif /* RACH_CORE_N_CUH */
