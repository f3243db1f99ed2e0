/*
 * rach_core_u0.cuh -- variant U0: the oldest simulator, RandomAccessSimulator.c (main loop
 * U0:75-126, selectPreamble U0:157-197, preambleCollision U0:200-233,
 * requestResourceAllocation U0:235-257, timerIncrease U0:259-266).
 *
 * U0 has index-order effects that differ from W (the group update of U0:228-229 makes the
 * members above the scanner back off in the same ms and the scanner one ms later; UEs in the
 * Msg3 phase scan too, U0:107; dropped UEs keep colliding, U0:207 has no raFailed test), a
 * 60 s Uniform horizon and a live set of a few dozen UEs (arrived, not finished; dropped UEs
 * leave it and stay as "phantoms").  The O(nUE) loops of the reference shrink to O(live).
 *
 * Two exact formulations over the same compact, index-ordered live list:
 *   ru_serial_ms  one thread performs the reference's own steps, UE after UE;
 *   ru_warp_ms    ONE WARP PER REPLICATION, one lane per live UE (up to 32; a ms with more falls back to
 *                 the serial step on lane 0).  The only coupling between UEs inside a ms is the collision
 *                 scan (reads active / txTime / preamble of the others, group-updates rarWindow / txTime),
 *                 and it is resolved with ballots in index order -- see ru_warp_ms.
 * The warp step is written in "vector form" (per-lane variables are arrays indexed by l, RW_EACH runs a
 * statement for every lane): on the device the arrays have one element and the lanes are the threads of the
 * warp, in the host emulation of tests/emu they have 32 elements and a loop plays the lanes -- the same source.
 */
#ifndef RACH_CORE_U0_CUH
#define RACH_CORE_U0_CUH

#include "rach_core.cuh"
#include "rach_warp.cuh"

#ifdef __CUDACC__
#define RU_ALIGN __align__(16)
#else
#define RU_ALIGN alignas(16)
#endif
struct RU_ALIGN RuUE {   /* 64 bytes; the first 16 are all a collision scan reads (U0:207-209) */
    int idx, active, txTime, preamble;      /* live-list copy: active == -2 = gone (finished / moved to ph[]) */
    int timer, rarWindow, maxRarCounter, preambleTxCounter;
    int msg2Flag, connectionRequest, msg4Flag, preambleChange;
    int raFailed, nowBackoff, pad0, pad1;   /* pad0: next node of a phantom chain */
};

/* RuUE entries of one replication's global workspace: live-list overflow [cap], phantom store [cap], phantom calendar
 * heads [maxR ints] */
RA_HD size_t ru_work_elems(int cap, int maxR) {
    return 2 * (size_t)cap + ((size_t)maxR * sizeof(int) + sizeof(RuUE) - 1) / sizeof(RuUE);
}

struct RuStats { int simTime, nSuccess; long long txSum, delaySum, collisionPreambles, totalPreambleTxop, dropped; int overflow; };

/* dump row: timer active txTime preamble preambleChange rarWindow maxRarCounter preambleTxCounter
 * msg2Flag connectionRequest msg4Flag raFailed nowBackoff 0 0 0 (saveResult order, U0:339-341) */
RA_HD void ru_dump_row(int* o, const RuUE& u) {
    o[0] = u.timer; o[1] = u.active; o[2] = u.txTime; o[3] = u.preamble; o[4] = u.preambleChange;
    o[5] = u.rarWindow; o[6] = u.maxRarCounter; o[7] = u.preambleTxCounter; o[8] = u.msg2Flag;
    o[9] = u.connectionRequest; o[10] = u.msg4Flag; o[11] = u.raFailed; o[12] = u.nowBackoff;
    o[13] = 0; o[14] = 0; o[15] = 0;
}

RA_HD int ru_rand(const RaJob& job, const RuUE& u, int time, unsigned& k) {
    return rach_tape_rand31(job.pt->seed, job.rep, (unsigned)u.idx, (unsigned)time, k++, RACH_TAPE_TAG_UE);
}

/* selectPreamble, U0:157-197.  Returns 1 if the UE was dropped (raFailed = -1) in this step. */
RA_HD int ru_select(const RaJob& job, RuUE& u, int time, unsigned& k) {
    const RaPointDev& pt = *job.pt;
    int dropped = 0;
    if (u.active == 1 && u.msg2Flag == 0) {
        if (u.preamble == -1) {
            u.preamble = (int)pt.modP((unsigned)ru_rand(job, u, time, k));
            u.rarWindow = 0; u.maxRarCounter = 0; u.preambleTxCounter = 0; u.preambleChange = 1;
        } else if (u.nowBackoff == 0) {
            u.rarWindow++;
            if (u.rarWindow >= 5) {
                int tmp = (int)pt.modBI((unsigned)ru_rand(job, u, time, k)) + 2;
                u.txTime = time + tmp; u.nowBackoff = tmp; u.rarWindow = 0; u.maxRarCounter++;
                if (u.maxRarCounter >= 10) {
                    u.raFailed = -1; dropped = 1;
                    u.preamble = (int)pt.modP((unsigned)ru_rand(job, u, time, k));
                    u.maxRarCounter = 0; u.preambleChange++;
                }
            }
        }
    }
    return dropped;
}

/* the single transmitter of a preamble, U0:213-219 */
RA_HD void ru_scan_success(RuUE& u, int time) {
    u.preambleTxCounter++; u.active = 2; u.txTime = time + 2; u.connectionRequest = 0; u.msg2Flag = 1;
}

/* requestResourceAllocation U0:113-115, 235-257 and timerIncrease U0:118-119, 259-266.  Returns 1 on success. */
RA_HD int ru_msg3_timer(const RaJob& job, RuUE& u, int time, unsigned& k) {
    const RaPointDev& pt = *job.pt;
    int success = 0;
    if (u.active == 2 && u.txTime + 2 == time) {
        u.connectionRequest++;
        if (u.connectionRequest < 48) {
            int r = ru_rand(job, u, time, k);
            if (rach_msg3_success(r)) { u.msg4Flag = 1; u.active = 0; success = 1; }
            else u.txTime = time + 1;
        } else {
            u.active = 1;
            u.txTime = time + (int)pt.modBI((unsigned)ru_rand(job, u, time, k)) + 2;
            u.preamble = (int)pt.modP((unsigned)ru_rand(job, u, time, k));
            u.msg2Flag = 0; u.rarWindow = 0; u.maxRarCounter = 0; u.preambleTxCounter++;
        }
    }
    if (u.active > 0 && u.msg4Flag == 0) {
        u.timer++;
        if (u.nowBackoff != 0) u.nowBackoff--;
    }
    return success;
}

/* Dropped UEs ("phantoms", raFailed == -1) are never processed again (U0:99) but still match the scan
 * predicate of U0:207 in the one ms where txTime+2 == time; a group update then moves them to time+3
 * (U0:228-229) so they can match again 5 ms later.  They are kept out of the live list in `ph[]`,
 * chained per ms of their next possible match (pad0 = next node, -1 ends the chain). */
RA_HD int ru_phantom_count(const RuUE* ph, const int* phHead, int slot, int time, int preamble) {
    int c = 0;
    for (int n = phHead[slot]; n >= 0; n = ph[n].pad0)
        if (ph[n].txTime + 2 == time && ph[n].preamble == preamble) c++;
    return c;
}
RA_HD void ru_phantom_group_update(RuUE* ph, int* phHead, int slot, int ringMask, int time, int preamble) {
    int prev = -1;
    for (int n = phHead[slot]; n >= 0;) {
        const int next = ph[n].pad0;
        if (ph[n].txTime + 2 == time && ph[n].preamble == preamble) {
            ph[n].rarWindow = 5; ph[n].txTime = time + 3;
            if (prev < 0) phHead[slot] = next; else ph[prev].pad0 = next;
            ph[n].pad0 = phHead[(time + 5) & ringMask]; phHead[(time + 5) & ringMask] = n;
        } else prev = n;
        n = next;
    }
}
RA_HD void ru_phantom_add(RuUE* ph, int* phHead, int ringMask, int pos, const RuUE& u) {
    RuUE n = u; const int s2 = (u.txTime + 2) & ringMask;
    n.pad0 = phHead[s2]; ph[pos] = n; phHead[s2] = pos;
}

/* the per-replication control state both formulations share */
struct RuRun { int nLive, nPh, activeCheck, arrived, nSuccess, overflow; };

/* The first `winCap` entries of the live list live in `win` (shared memory on the device: the live set is a few dozen
 * UEs, and a walk that fetches it every ms out of L2 spends its time waiting), the rest in `live` (global). */
#define RU_L(x) (*((x) < winCap ? win + (x) : live + (x)))

/* One ms, one thread, the reference's own order (U0:96-121).  The list is dense on entry and on exit. */
template <bool DUMP>
RA_HD void ru_serial_ms(const RaJob& job, RuUE* live, RuUE* win, int winCap, RuUE* ph, int* phHead, int cap, int time,
                        RuRun& r, RuStats& st) {
    const int ringMask = job.pt->R - 1, slot = time & ringMask;
    const int nLive = r.nLive;
    int nGone = 0;
    for (int a = 0; a < nLive; ++a) {
        RuUE u = RU_L(a);
        unsigned k = 0;
        st.dropped += ru_select(job, u, time, k);
        if (u.txTime + 2 == time && u.txTime != -1) {                     /* preambleCollision U0:107-110, 200-233 */
            RU_L(a) = u;                                                  /* the scan below reads the list */
            int check = 0;
            for (int b = 0; b < nLive; ++b)
                { const RuUE& o = RU_L(b); if (o.active == 1 && o.txTime + 2 == time && o.preamble == u.preamble) check++; }
            check += ru_phantom_count(ph, phHead, slot, time, u.preamble);
            if (check == 1) {
                st.totalPreambleTxop++;
                ru_scan_success(u, time);
            } else {
                st.collisionPreambles += check;
                for (int b = 0; b < nLive; ++b) {
                    RuUE& o = RU_L(b);
                    if (o.active == 1 && o.txTime + 2 == time && o.preamble == u.preamble) { o.rarWindow = 5; o.txTime = time + 3; }
                }
                ru_phantom_group_update(ph, phHead, slot, ringMask, time, u.preamble);   /* they can match again at time+5 */
                u = RU_L(a);                                              /* the scanner may be a member */
            }
        }
        r.nSuccess += ru_msg3_timer(job, u, time, k);
        if (u.msg4Flag == 1) {
            st.txSum += u.preambleTxCounter; st.delaySum += u.timer; nGone++;
            if (DUMP) ru_dump_row(job.dump + (size_t)u.idx * RA_DUMP_W, u);
            u.active = -2;
        } else if (u.raFailed == -1) {                                    /* frozen from now on: to the phantom calendar */
            if (r.nPh >= cap) r.overflow = 1;
            else { ru_phantom_add(ph, phHead, ringMask, r.nPh, u); r.nPh++; }
            nGone++; u.active = -2;
        }
        RU_L(a) = u;
    }
    if (nGone) {                                                          /* compact, keeping index order */
        int w = 0;
        for (int a = 0; a < nLive; ++a) if (RU_L(a).active != -2) { if (w != a) RU_L(w) = RU_L(a); ++w; }
        r.nLive = w;
    }
}

/* ---- vector form (rach_warp.cuh) ---------------------------------------------------------------------------- */
/* per-lane partial sums, folded at the end of the replication */
struct RuLaneSums { long long txSum[RW_LANES], delaySum[RW_LANES], coll[RW_LANES], txop[RW_LANES], dropped[RW_LANES]; };

/* One ms, one warp, one lane per live UE (r.nLive <= 32 <= winCap; the list is dense on entry and on exit).
 *
 * Sequentially, UE a (index order) runs selectPreamble on itself, then -- if txTime+2 == time -- scans the list:
 * check = UEs with active==1, txTime+2 == time and its preamble, as the list stands at that moment: lower indices
 * after their whole turn, higher indices BEFORE theirs.  After its own turn a UE never matches (it was the only one
 * and succeeded, or the group update moved it to time+3, or it did not match to begin with), so the members a
 * scanner sees are: itself (after its selectPreamble) and the higher indices in their start-of-ms state, minus
 * those a previous group update of this ms has hit.  A hit UE above the scanner then runs selectPreamble on the
 * updated state (rarWindow 5 -> backs off in this very ms) and is no scanner any more.
 * So: every lane runs selectPreamble tentatively; the scanners are resolved one after the other in index order
 * with ballots (a handful per ms); lanes hit by a group update redo selectPreamble from their start state;
 * Msg3 / timers / leaving the list are per-lane again. */
template <bool DUMP>
RW_FN void ru_warp_ms(const RaJob& job, RuUE* win, RuUE* ph, int* phHead, int cap, int time, RuRun& r, RuLaneSums& sm) {
    const int ringMask = job.pt->R - 1, slot = time & ringMask;
    const int nLive = r.nLive;
    RuUE u0[RW_LANES], u[RW_LANES];
    unsigned k[RW_LANES];
    int alive[RW_LANES], preM[RW_LANES], sc[RW_LANES], selfM[RW_LANES], hit[RW_LANES], drop1[RW_LANES], pre1[RW_LANES], m[RW_LANES];
    RW_EACH(l) {
        alive[l] = lane < nLive; hit[l] = 0; drop1[l] = 0; k[l] = 0; preM[l] = sc[l] = selfM[l] = 0; pre1[l] = -2;
        if (alive[l]) {
            u0[l] = win[lane]; u[l] = u0[l];
            drop1[l] = ru_select(job, u[l], time, k[l]);
            preM[l] = u0[l].active == 1 && u0[l].txTime + 2 == time;
            sc[l] = u[l].txTime + 2 == time && u[l].txTime != -1;
            selfM[l] = u[l].active == 1 && u[l].txTime + 2 == time;
            pre1[l] = u[l].preamble;
        }
    }
    unsigned pending = RW_BALLOT(sc);
    while (pending) {
        const int a = RW_FFS(pending) - 1;
        const int pa = RW_SHFL(pre1, a);
        RW_EACH(l) m[l] = lane > a ? (preM[l] && !hit[l] && u0[l].preamble == pa) : (lane == a ? selfM[l] : 0);
        const unsigned mask = RW_BALLOT(m);
        const int check = RW_POPC(mask) + ru_phantom_count(ph, phHead, slot, time, pa);
        if (check == 1) {
            RW_EACH(l) if (lane == a) { sm.txop[l]++; ru_scan_success(u[l], time); selfM[l] = 0; }
        } else {
            RW_EACH(l) {
                if (lane == a) sm.coll[l] += check;
                if (m[l]) {
                    if (lane == a) { u[l].rarWindow = 5; u[l].txTime = time + 3; selfM[l] = 0; }
                    else {                                    /* hit before my turn: selectPreamble sees the update */
                        hit[l] = 1; sc[l] = 0;
                        u[l] = u0[l]; u[l].rarWindow = 5; u[l].txTime = time + 3;
                        k[l] = 0; drop1[l] = ru_select(job, u[l], time, k[l]);
                    }
                }
            }
            RW_SYNC();
            RW_EACH(l) if (lane == 0) ru_phantom_group_update(ph, phHead, slot, ringMask, time, pa);
            RW_SYNC();
            pending &= ~mask;                                 /* the hit lanes are no scanners any more */
        }
        pending &= ~(1u << a);
    }
    int fin[RW_LANES], drp[RW_LANES], keep[RW_LANES];
    RW_EACH(l) {
        fin[l] = drp[l] = keep[l] = 0;
        if (alive[l]) {
            sm.dropped[l] += drop1[l];
            ru_msg3_timer(job, u[l], time, k[l]);
            fin[l] = u[l].msg4Flag == 1;
            drp[l] = !fin[l] && u[l].raFailed == -1;
            keep[l] = !fin[l] && !drp[l];
            if (fin[l]) {
                sm.txSum[l] += u[l].preambleTxCounter; sm.delaySum[l] += u[l].timer;
                if (DUMP) ru_dump_row(job.dump + (size_t)u[l].idx * RA_DUMP_W, u[l]);
            }
        }
    }
    r.nSuccess += RW_POPC(RW_BALLOT(fin));
    unsigned dmask = RW_BALLOT(drp);
    while (dmask) {                                          /* rare: one chain insertion after the other */
        const int j = RW_FFS(dmask) - 1;
        if (r.nPh >= cap) r.overflow = 1;
        else {
            RW_EACH(l) if (lane == j) ru_phantom_add(ph, phHead, ringMask, r.nPh, u[l]);
            r.nPh++;
        }
        RW_SYNC();
        dmask &= dmask - 1;
    }
    const unsigned kmask = RW_BALLOT(keep);
    RW_SYNC();                                               /* every lane holds its entry in registers by now */
    RW_EACH(l) if (keep[l]) win[RW_POPC(kmask & ((1u << lane) - 1u))] = u[l];
    r.nLive = RW_POPC(kmask);
    RW_SYNC();
}

/* arrivals of the ms, U0:77-94 (bound fixed: i < nUE); lanes stride over the new entries */
RW_FN void ru_arrivals(const RaPointDev& pt, RuUE* live, RuUE* win, int winCap, int cap, int time, RuRun& r) {
    const int nAccessUE = pt.G;                       /* host: ceil(n*5/60000), at least 1 (U0:60-64) */
    if (r.activeCheck >= pt.nUE) r.activeCheck = pt.nUE; else r.activeCheck += nAccessUE;
    const int upto = r.activeCheck + 1 < pt.nUE ? r.activeCheck + 1 : pt.nUE;
    int n = upto - r.arrived;
    if (n < 0) n = 0;
    if (r.nLive + n > cap) { r.overflow = 1; n = cap - r.nLive; }
    RW_EACH(l) for (int j = lane; j < n; j += 32) {
        RuUE u; u.idx = r.arrived + j; u.timer = 0; u.active = 1; u.txTime = time + 1; u.preamble = -1;
        u.rarWindow = 0; u.maxRarCounter = 0; u.preambleTxCounter = 0; u.msg2Flag = 0;
        u.connectionRequest = 0; u.msg4Flag = 0; u.preambleChange = 0; u.raFailed = 0; u.nowBackoff = 0;
        u.pad0 = u.pad1 = 0;
        RU_L(r.nLive + j) = u;
    }
    r.nLive += n; r.arrived += n;
    RW_SYNC();
}

/* One replication, one warp (device) / one host thread playing the 32 lanes (emulation).  `lanesOn` = 0 forces the
 * serial step in every ms (the one-thread formulation, kept as the cross-check of the warp step). */
template <bool DUMP>
RW_FN void ru_run_replication(const RaJob& job, RuUE* live, RuUE* win, int winCap, RuUE* ph, int* phHead, int cap,
                              int lanesOn, RuStats* out) {
    const RaPointDev& pt = *job.pt;
    const int nUE = pt.nUE, maxTime = pt.maxTime, accessTime = 5;   /* U0:57,59 */
    const int ringMask = pt.R - 1;
    RuStats st; st.simTime = maxTime; st.nSuccess = 0; st.txSum = st.delaySum = 0;
    st.collisionPreambles = st.totalPreambleTxop = st.dropped = 0; st.overflow = 0;
    RuLaneSums sm;
    RW_EACH(l) { sm.txSum[l] = sm.delaySum[l] = sm.coll[l] = sm.txop[l] = sm.dropped[l] = 0; }
    if (DUMP) RW_EACH(l) for (int i = lane; i < nUE; i += 32) {      /* calloc + initialUE, U0:46,149-155 */
        int* o = job.dump + (size_t)i * RA_DUMP_W;
        for (int q = 0; q < RA_DUMP_W; ++q) o[q] = 0;
        o[0] = -1; o[1] = -1; o[2] = -1; o[3] = -1;
    }
    RW_EACH(l) for (int i = lane; i <= ringMask; i += 32) phHead[i] = -1;
    RW_SYNC();
    RuRun r; r.nLive = r.nPh = r.activeCheck = r.arrived = r.nSuccess = r.overflow = 0;
    int time;
    for (time = 0; time < maxTime; time++) {
        if (time % accessTime == 1) ru_arrivals(pt, live, win, winCap, cap, time, r);
        if (lanesOn && r.nLive <= 32 && winCap >= 32) {
            ru_warp_ms<DUMP>(job, win, ph, phHead, cap, time, r, sm);
        } else {
            /* a crowded ms: lane 0 walks the list the reference's way; the control state is broadcast afterwards */
            int c0[RW_LANES], c1[RW_LANES], c2[RW_LANES], c3[RW_LANES];
            RW_EACH(l) {
                c0[l] = c1[l] = c2[l] = c3[l] = 0;
                if (lane == 0) {
                    RuRun r1 = r;
                    ru_serial_ms<DUMP>(job, live, win, winCap, ph, phHead, cap, time, r1, st);
                    c0[l] = r1.nLive; c1[l] = r1.nPh; c2[l] = r1.nSuccess; c3[l] = r1.overflow;
                }
            }
            RW_SYNC();
            r.nLive = RW_SHFL(c0, 0); r.nPh = RW_SHFL(c1, 0); r.nSuccess = RW_SHFL(c2, 0); r.overflow = RW_SHFL(c3, 0);
        }
        RW_EACH(l) if (lane == 0) phHead[time & ringMask] = -1;               /* whoever was not hit never matches again */
        RW_SYNC();
        if (r.nSuccess == nUE) break;                                         /* U0:122-125 */
    }
    if (DUMP) {
        const int nLive = r.nLive, nPh = r.nPh;
        RW_EACH(l) {
            for (int a = lane; a < nLive; a += 32) ru_dump_row(job.dump + (size_t)RU_L(a).idx * RA_DUMP_W, RU_L(a));
            for (int n = lane; n < nPh; n += 32) ru_dump_row(job.dump + (size_t)ph[n].idx * RA_DUMP_W, ph[n]);
        }
    }
    /* `st` holds what the serial steps added (on lane 0 only); the lane sums hold the warp steps' share */
    long long tot[5];
    for (int q = 0; q < 5; ++q) {
        long long v[RW_LANES];
        RW_EACH(l) {
            const bool z = lane == 0;
            v[l] = q == 0 ? sm.txSum[l] + (z ? st.txSum : 0) : q == 1 ? sm.delaySum[l] + (z ? st.delaySum : 0)
                 : q == 2 ? sm.coll[l] + (z ? st.collisionPreambles : 0) : q == 3 ? sm.txop[l] + (z ? st.totalPreambleTxop : 0)
                 : sm.dropped[l] + (z ? st.dropped : 0);
        }
        tot[q] = rw_sum(v);
    }
    st.txSum = tot[0]; st.delaySum = tot[1]; st.collisionPreambles = tot[2]; st.totalPreambleTxop = tot[3]; st.dropped = tot[4];
    st.simTime = time; st.nSuccess = r.nSuccess; st.overflow = r.overflow;
    *out = st;
}

#undef RU_L

#endif /* RACH_CORE_U0_CUH */
