/*
 * rach_emu.cpp -- TEST INFRASTRUCTURE.  Runs the phase functions of the CUDA engine
 * (5g-nr-randomaccess_b200/csrc/rach_core.cuh) on the host, one emulated thread after the
 * other with the phase boundaries where the kernel has __syncthreads(), so that the
 * event-driven algorithm can be fuzzed against the oracle without a GPU.  It is NOT a CPU
 * fallback: nothing in the product loads it, and librach_gpu fails without a device.
 *
 * Same ABI as oracle_run()/ref_run() (oracle/ref_api.h).
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <vector>

#include "rach_core.cuh"
#include "rach_gpu.h"
#include "rach_host.h"
extern "C" {
#include "ref_api.h"
}

extern "C" { int emu_use_fixed = 1; int emu_light = 1; long long emu_light_ms = 0, emu_light_code2 = 0, emu_light_code3 = 0, emu_total_ms = 0; }

template <bool DUMP, class PT>
static int emu_body(const PT& pt, const RaWork& w, RaShared& s, const ref_config* cfg, ref_result* res, int* perUE, int NT) {
    RaJobT<PT> job; job.pt = &pt; job.rep = (unsigned)cfg->rep; job.dump = DUMP ? perUE : NULL;
    std::vector<RaAcc> acc(NT); memset(acc.data(), 0, sizeof(RaAcc) * NT);

    for (int t = 0; t < NT; ++t) ra_job_init<DUMP>(job, s, t, NT);
    int simTime = pt.maxTime;
    RaAcc lacc[32]; memset(lacc, 0, sizeof lacc);              /* the 32 lanes of warp 0 in the light path */
    bool done = false;
    for (int T = 0;; ++T) {
        /* the kernel's control flow: warp 0 runs light ms back to back (ra_light_ms, vector form: the 32 lanes are played
         * by a loop), then prepares the first ms that needs the whole block */
        int code = 0;
        ra_gc_apply(s);
        if (emu_light) {
            ra_lists_reset(s);
            RaCtl c = ra_ctl_load(s);
            int fin = 0;
            for (;;) {
                code = ra_light_ms<DUMP>(job, w, s, c, lacc, T, &fin, &simTime);
                if (code == 2) emu_light_code2++;
                if (code == 3) emu_light_code3++;
                if (code != 1) break;
                emu_light_ms++; emu_total_ms++;
                if (fin) { code = 4; break; }
                ++T;
            }
            ra_ctl_store(s, c);
        }
        if (code == 4) { done = true; break; }
        emu_total_ms++;
        if (code == 0) {
            for (int t = 0; t < 32; ++t) ra_phase0(job, s, T, t, 32);
            unsigned n1 = s.nMov + (unsigned)s.nArr + s.nM3;
            /* as in the kernel: a thread walks its movers first, a re-transmitter among them waits in the thread's RaPend until
             * the next one arrives or the bucket ends; then the arrivals and Msg3 answers */
            const uint4* bT = w.bucket + (size_t)((unsigned)T & (unsigned)(pt.R - 1)) * w.cap;
            for (int t = 0; t < NT; ++t) {
                RaPend pd; pd.x = RA_INF32; pd.z = pd.w = 0;
                unsigned i = t;
                for (; i < s.nMov; i += NT) ra_phase1_mover<DUMP>(job, w, s, acc[t], T, i, bT[i], pd);
                ra_pend_flush(pt, w, s, T, pd);
                for (; i < n1; i += NT) ra_phase1_item<DUMP>(job, w, s, acc[t], T, i);
            }
        } else if (code == 2) {
            for (int t = 0; t < 32; ++t) ra_phase0_classes(job, s, T, t, 32);
        }
        if (code != 3) {
        if (s.nC3) ra_phase2_serial(pt, w, s);
        if (s.nUnc) { unsigned n = s.nUnc; for (int t = 0; t < NT; ++t) for (unsigned i = t; i < n; i += NT) ra_phase3_item<DUMP>(job, w, s, T, i); }
        if (s.nE1) { unsigned n = s.nE1; for (int t = 0; t < NT; ++t) for (unsigned i = t; i < n; i += NT) ra_phase3b_item(pt, w, s, i); }
        unsigned n4 = (unsigned)pt.P + s.nLanders;
        for (int t = 0; t < NT; ++t) for (unsigned i = t; i < n4; i += NT) ra_phase4_item(pt, w, s, acc[t], i);
        if (s.nSingles) {
            if (ra_phase5_trivial(pt, s)) s.gcAdd = (int)s.nSingles;
            else {                                  /* the kernel's phase 5, checked against the one-thread statement */
                RaShared ref = s;
                ra_phase5_serial(pt, w, ref);
                ra_phase5_warp(pt, w, s);
                if (s.tau != ref.tau || s.noGrant != ref.noGrant) {
                    fprintf(stderr, "emu: phase 5 tau %u/%u noGrant %u/%u at ms %d\n", s.tau, ref.tau, s.noGrant, ref.noGrant, T);
                    return -4;
                }
            }
        }
        unsigned n6 = (unsigned)pt.P + s.nLanders + s.nE1;
        for (int t = 0; t < NT; ++t) for (unsigned i = t; i < n6; i += NT) ra_phase6_item<DUMP>(job, w, s, T, i);
        if (s.nSingles) for (int t = 0; t < NT; ++t) ra_hist_clear(pt, w, s, t, NT);
        }
        { const unsigned nNl = code == 3 ? s.nNlLight : s.nNl;
          if (nNl) for (int t = 0; t < NT; ++t) ra_phase6b<DUMP>(job, w, s, T, t, NT, nNl); }
        if (s.overflow) { fprintf(stderr, "emu: overflow flag %d at ms %d\n", s.overflow, T); return -3; }
        if (ra_ms_done(pt, s, T, &simTime)) break;
    }
    (void)done;
    const int last = simTime < pt.maxTime ? simTime : pt.maxTime - 1;
    if (DUMP) for (int t = 0; t < NT; ++t) ra_dump_inflight(job, w, s, last, t, NT);
    for (int t = 0; t < 32; ++t) {
        s.contFailed += lacc[t].contFailed; s.collP += lacc[t].collP; s.txop += lacc[t].txop;
        s.collScans += lacc[t].collScans; s.totScans += lacc[t].totScans;
    }
    for (int t = 0; t < NT; ++t) {
        s.contFailed += acc[t].contFailed; s.collP += acc[t].collP; s.txop += acc[t].txop;
        s.collScans += acc[t].collScans; s.totScans += acc[t].totScans;
    }
    memset(res, 0, sizeof *res);
    res->simTimeMs = simTime; res->nSuccess = (int)s.nSuccess; res->preambleTxSum = (long long)s.txSum;
    res->delaySum = (long long)s.delaySum; res->failCountSum = (long long)s.failSum;
    res->continueFailed = (long long)s.contFailed; res->collisionPreambles = (long long)s.collP;
    res->totalPreambleTxop = (long long)s.txop; res->collisionScans = (long long)s.collScans;
    res->totalScans = (long long)s.totScans; res->captured = 1; res->lastMs = last;
    return 0;
}

template <bool DUMP>
static int emu_run_t(const ref_config* cfg, ref_result* res, int* perUE, int NT) {
    ra_params p; ra_params_default(&p, RA_VARIANT_W);
    p.nUE = cfg->nUE; p.distribution = cfg->distribution; p.nPreamble = cfg->nPreamble;
    p.backoffIndicator = cfg->backoffIndicator; p.nGrantUL = cfg->nGrantUL;
    p.maxRarWindow = cfg->maxRarWindow; p.maxMsg2TxCount = cfg->maxMsg2TxCount;
    p.accessTime = cfg->accessTime; p.cellRadius = cfg->cellRadius; p.geometry = cfg->geometry;
    p.seed = cfg->seed; p.maxTimeMs = cfg->stopMs > 0 ? cfg->stopMs : 0;
    char err[256];
    if (ra_host_validate(&p, err, sizeof err) != RA_OK) { fprintf(stderr, "emu: %s\n", err); return -1; }

    RaPointDev pt;
    ra_host_point(&p, &pt);
    std::vector<int> arrCum(pt.nOcc);
    ra_host_arrcum(&p, arrCum.data(), pt.nOcc);
    pt.arrCum = arrCum.data();

    /* the block's global workspace and dynamic shared memory, laid out as the engine lays them out */
    RaWork w;
    const int cap3 = ra_host_cap3(RA_VARIANT_W, &pt);
    std::vector<uint4> work((ra_work_carve(NULL, pt.nUE, cap3, pt.R, pt.P, &w) + 15) / 16);
    ra_work_carve(reinterpret_cast<unsigned char*>(work.data()), pt.nUE, cap3, pt.R, pt.P, &w);
    RaShared s; memset(&s, 0, sizeof s);
    std::vector<uint4> smem((pt.smemBytes + 15) / 16 + 1);
    ra_emu_smem_base = reinterpret_cast<unsigned char*>(smem.data());

    /* the kernel's two views of a point: runtime values, or the compile-time family of the reference defaults */
    int rc;
    if (emu_use_fixed && ra_point_is_default_family(pt)) rc = emu_body<DUMP>(static_cast<const RaPointDef&>(pt), w, s, cfg, res, perUE, NT);
    else rc = emu_body<DUMP>(pt, w, s, cfg, res, perUE, NT);
    return rc;
}

extern "C" { int emu_threads = 64; }

extern "C" int emu_run(const ref_config* cfg, ref_result* res, int* perUE, float* geom) {
    (void)geom;
    struct timespec t0, t1; clock_gettime(CLOCK_MONOTONIC, &t0);
    int rc = perUE ? emu_run_t<true>(cfg, res, perUE, emu_threads) : emu_run_t<false>(cfg, res, NULL, emu_threads);
    clock_gettime(CLOCK_MONOTONIC, &t1);
    res->seconds = (double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec);
    return rc;
}

/* ------------------------------------------------------------------------------------------
 * Variant N: the phases of rach_core_n.cuh, same emulation scheme.
 * perUE: nUE*16 ints in N dump order; geom: nUE doubles (channelGain).
 * ------------------------------------------------------------------------------------------ */
#include "rach_core_n.cuh"

extern "C" { int emu_n_serialB = 0; }

template <bool DUMP>
static int emu_run_n_t(const ref_config* cfg, ref_result* res, int* perUE, double* gains, int NT) {
    ra_params p; ra_params_default(&p, RA_VARIANT_N);
    p.nUE = cfg->nUE; p.distribution = 2; p.nPreamble = cfg->nPreamble;
    p.backoffIndicator = cfg->backoffIndicator; p.nGrantUL = cfg->nGrantUL;
    p.maxRarWindow = cfg->maxRarWindow; p.maxMsg2TxCount = cfg->maxMsg2TxCount;
    p.accessTime = cfg->accessTime; p.cellRadius = cfg->cellRadius; p.geometry = cfg->geometry; p.seed = cfg->seed;
    char err[256];
    if (ra_host_validate(&p, err, sizeof err) != RA_OK) { fprintf(stderr, "emu: %s\n", err); return -1; }
    RaPointDev pt;
    ra_host_point(&p, &pt);
    std::vector<int> arrCum(pt.nOcc);
    ra_host_arrcum(&p, arrCum.data(), pt.nOcc);
    pt.arrCum = arrCum.data();

    /* the block's global workspace and its tables in dynamic shared memory, laid out as the engine lays them out */
    RaWorkN w;
    const int cap3 = ra_host_cap3(RA_VARIANT_N, &pt);
    std::vector<uint4> work((rn_work_carve(NULL, pt.nUE, cap3, pt.R, &w) + 15) / 16);
    rn_work_carve(reinterpret_cast<unsigned char*>(work.data()), pt.nUE, cap3, pt.R, &w);
    RaSharedN s; memset(&s, 0, sizeof s);
    std::vector<uint4> smem((rn_smem_bytes(pt.R, pt.P) + 15) / 16);
    rn_carve(s, reinterpret_cast<unsigned char*>(smem.data()), pt.R, pt.P);
    RaJob job; job.pt = &pt; job.rep = (unsigned)cfg->rep; job.dump = DUMP ? perUE : NULL;

    for (int t = 0; t < NT; ++t) rn_job_init<DUMP>(job, s, t, NT);
    int simTime = pt.maxTime;
    const unsigned Rm = (unsigned)(pt.R - 1);
    for (int T = 0; T < pt.maxTime; ++T) {
        if (T % pt.A == 0) {
            for (int t = 0; t < NT; ++t) rn_phaseA0(job, s, T, t, NT);
            for (int t = 0; t < NT; ++t) for (unsigned i = t; i < (unsigned)s.nArr; i += NT) rn_phaseA1_item<DUMP>(job, w, s, T, (unsigned)s.acOld + i);
            const unsigned nTx = s.bcount[(unsigned)T & Rm];
            for (int t = 0; t < NT; ++t) for (unsigned j = t; j < nTx; j += NT) rn_phaseA2_item(pt, w, s, T, j);
            for (int sec = 0; sec < (pt.geometry ? RA_NSECT : 1); ++sec) {       /* warp form (the kernel's) or the one-thread statement */
                if (emu_n_serialB) rn_phaseB_sector(job, w, s, T, sec); else rn_phaseB_warp(job, w, s, T, sec);
            }
            for (int t = 0; t < NT; ++t) for (unsigned j = t; j < nTx; j += NT) rn_phaseC_item<DUMP>(job, w, s, T, j);
            s.bcount[(unsigned)T & Rm] = 0;
        }
        const unsigned nM3 = s.m3count[(unsigned)T & (RA_M3RING - 1)];
        if (nM3) {
            for (int t = 0; t < NT; ++t) for (unsigned j = t; j < nM3; j += NT) rn_msg3_item<DUMP>(job, w, s, T, j);
            s.m3count[(unsigned)T & (RA_M3RING - 1)] = 0;
            if (s.nSuccess == (unsigned)pt.nUE) { simTime = T; break; }
        }
        if (s.overflow) { fprintf(stderr, "emu N: overflow flag %d at ms %d\n", s.overflow, T); return -3; }
    }
    const int last = simTime < pt.maxTime ? simTime : pt.maxTime - 1;
    if (DUMP) {
        for (int t = 0; t < NT; ++t) rn_dump_inflight(job, w, s, last, t, NT);
        if (gains) for (int i = 0; i < pt.nUE; ++i) gains[i] = i < s.activeCheck ? w.gain[i] : 0.0;
    }
    memset(res, 0, sizeof *res);
    res->simTimeMs = simTime; res->nSuccess = (int)s.nSuccess; res->preambleTxSum = (long long)s.txSum;
    res->delaySum = (long long)s.delaySum; res->continueFailed = (long long)s.nDropped; res->captured = 1;
    return 0;
}

extern "C" int emu_run_n(const ref_config* cfg, ref_result* res, int* perUE, float* geom) {
    return perUE ? emu_run_n_t<true>(cfg, res, perUE, (double*)geom, emu_threads)
                 : emu_run_n_t<false>(cfg, res, NULL, NULL, emu_threads);
}

/* ------------------------------------------------------------------------------------------
 * Variant U0: rach_core_u0.cuh runs one replication per thread; here: called once.
 * ------------------------------------------------------------------------------------------ */
#include "rach_core_u0.cuh"

extern "C" { int emu_u0_mode = 1; }

extern "C" int emu_run_u0(const ref_config* cfg, ref_result* res, int* perUE, float* geom) {
    (void)geom;
    ra_params p; ra_params_default(&p, RA_VARIANT_U0);
    p.nUE = cfg->nUE; p.nPreamble = cfg->nPreamble; p.backoffIndicator = cfg->backoffIndicator; p.seed = cfg->seed;
    p.maxTimeMs = cfg->stopMs > 0 ? cfg->stopMs : 0;
    char err[256];
    if (ra_host_validate(&p, err, sizeof err) != RA_OK) { fprintf(stderr, "emu: %s\n", err); return -1; }
    RaPointDev pt;
    ra_host_point(&p, &pt);
    std::vector<RuUE> live((size_t)pt.nUE), ph((size_t)pt.nUE);
    std::vector<int> phHead((size_t)pt.R);
    RaJob job; job.pt = &pt; job.rep = (unsigned)cfg->rep; job.dump = perUE;
    RuStats st;
    /* emu_u0_mode 1: the warp step (32 lanes played by a loop), 40-entry window so that crowded ms spill to the
     * global list; 0: the serial step in every ms, 5-entry window */
    std::vector<RuUE> win(emu_u0_mode ? 40 : 5);
    if (perUE) ru_run_replication<true>(job, live.data(), win.data(), (int)win.size(), ph.data(), phHead.data(), pt.nUE, emu_u0_mode, &st);
    else ru_run_replication<false>(job, live.data(), win.data(), (int)win.size(), ph.data(), phHead.data(), pt.nUE, emu_u0_mode, &st);
    memset(res, 0, sizeof *res);
    res->simTimeMs = st.simTime; res->nSuccess = st.nSuccess; res->preambleTxSum = st.txSum; res->delaySum = st.delaySum;
    res->collisionPreambles = st.collisionPreambles; res->totalPreambleTxop = st.totalPreambleTxop;
    res->continueFailed = st.dropped; res->captured = 1;
    return st.overflow ? -3 : 0;
}

/* the engine's division-free modulo (rach_core.cuh: ra_magic / ra_mod_shift / ra_mod), for the exactness test */
extern "C" unsigned emu_mod(unsigned x, unsigned d) { return ra_mod(x, d, ra_magic(d), ra_mod_shift(d)); }
