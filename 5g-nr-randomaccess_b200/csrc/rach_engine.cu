/*
 * rach_engine.cu -- librach_gpu: the CUDA (sm_100a) step kernel and the C ABI of
 * include/rach_gpu.h.
 *
 * One thread block simulates one replication from ms 0 to the horizon: it owns the move /
 * Msg3 calendars of that replication in HBM (16-byte records, 128-bit loads and stores) and
 * the per-preamble cohort tables in shared memory, and runs the phases of rach_core.cuh with
 * __syncthreads() in between -- except the ms without movers, which warp 0 runs alone, back to
 * back, without a block barrier (ra_light_ms).  Blocks are persistent: grid = min(jobs, SMs *
 * CTAs/SM) and each block pulls replications from an atomic job counter.  Replications never
 * exchange data, so multi-GPU is a partition of the job list (no collective in the data path).
 *
 * Replaces the body of the reference's (seed, nUE) loop, RandomAccessWithNOMA.c:229-368.
 * There is no CPU path in this library.
 */
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <type_traits>
#include <string>
#include <vector>

#include "rach_core.cuh"
#include "rach_core_n.cuh"
#include "rach_core_u0.cuh"
#include "rach_gpu.h"
#include "rach_host.h"

/* Block shapes of the W step kernel (threads, resident blocks per SM the register budget is sized for).
 * Measured on B200, 4096 replications x 100k UEs, round 1 (runtime parameters): 128 x 8 (64 registers, no spills) 1215 ms,
 * 256 x 5 (48 registers) 1259 ms, 192 x 6 1241 ms, 96 x 10 1286 ms, 64 x 11 1337 ms, 512 x 2 1515 ms -- the block-wide
 * barriers between the phases cost less with 4 warps than with 8.  Round 2, default-family instantiation (compile-time
 * P / BI / subframe / window): 128 x 8 1061 ms, 128 x 9 (56 registers) 1030 ms, 128 x 10 1050 ms, 96 x 10 1102 ms.
 * The small shape needs its blocks' tables in one SM's shared memory; points with a large ring x preamble product fall
 * back to 256 x 5 (fewer, larger blocks). */
#ifndef RA_NT
#define RA_NT 128          /* small shape */
#endif
#ifndef RA_MINB
#define RA_MINB 9
#endif
#ifndef RA_NT_BIG
#define RA_NT_BIG 256
#define RA_MINB_BIG 5
#endif
/* few replications per device (strong scaling, small sweeps): one replication cannot be split over blocks, so the block
 * grows instead -- 512 threads x 2 per SM (64 registers) when there are at most two replications per SM */
#define RA_NT_HUGE 512
#define RA_MINB_HUGE 2
#ifndef RA_NT_N
#define RA_NT_N 128        /* variant N, one warp per sector in the base-station phase.  Measured (50k UEs x 2048 replications,  */
#define RA_MINB_N 8        /* round 2): 128 x 8 57.0 ms, 96 x 10 57.5 ms, 192 x 5 63.6 ms, 256 x 4 76.2 ms (round 1, one lane per
                              sector: 192 x 5 169 ms) */
#endif
#define RA_NPHASE 10
#ifndef RA_ILP
#define RA_ILP 2             /* movers per thread and loop iteration (interleaved Philox chains) */
#endif
#define RA_TICK(k) do { if (timers && tid == 0) { long long now_ = clock64(); sCyc[k] += (ra_u64)(now_ - tick); tick = now_; } } while (0)

struct RaKernelArgs {
    const RaPointDev* points;
    const int*        jobPoint;     /* [nJobs] point index                       */
    const unsigned*   jobRep;       /* [nJobs] tape replication id               */
    const RaWork*     works;        /* [gridDim.x]  (variant W)                  */
    const RaWorkN*    worksN;       /* [gridDim.x]  (variant N)                  */
    double*           gainDump;     /* [nJobs][cap] channelGain per UE (variant N, DUMP) or NULL */
    RuUE*             liveBase;     /* [threads][cap] live lists (variant U0)    */
    size_t            gainStride;
    unsigned*         jobCounter;
    ra_stats*         stats;        /* [nJobs]                                   */
    int*              dump;         /* [nJobs][dumpStride] or NULL               */
    int*              errFlag;
    volatile int*     doneFlags;    /* [nJobs] host-mapped: 1 = the replication's stats and dump rows are complete (streaming), or NULL */
    ra_u64*           phaseCycles;  /* [RA_NPHASE] cycles of thread 0 per phase, summed over blocks */
    size_t            dumpStride;
    int               nJobs, maxP, maxR;
};

template <bool DUMP, int NT, int MINB, bool FIXED, bool TIMERS = false>
__global__ void __launch_bounds__(NT, MINB) ra_step_kernel(RaKernelArgs a) {
    /* FIXED: every point of the launch belongs to the reference's default family (54 preambles, BI 20, subframe 5, RAR
     * window 5): those values are immediates in this instantiation (RaPointDef); otherwise they are read from the point */
    typedef typename std::conditional<FIXED, RaPointDef, RaPointDev>::type PT;
    __shared__ RaShared s;
    __shared__ RaPointDev sPt;
    __shared__ int sJob;
    __shared__ int sLight[4];                           /* warp 0 -> block: ms to resume at, how (ra_light_ms code), simTime */
    __shared__ ra_u64 sCyc[RA_NPHASE];
    long long tick = 0;
    /* profiling aid (ra_options.phaseTimers): its own instantiation, so that the product kernel carries none of the
     * per-phase tests (a dozen per ms and warp: 9 % of the instructions of a lightly loaded ms) */
    const bool timers = TIMERS && a.phaseCycles != nullptr;
    if (threadIdx.x < RA_NPHASE) sCyc[threadIdx.x] = 0;
    const int tid = threadIdx.x, nt = blockDim.x;
    const RaWork w = a.works[blockIdx.x];

    for (;;) {
        __syncthreads();
        if (tid == 0) sJob = (int)atomicAdd(a.jobCounter, 1u);
        __syncthreads();
        const int jobId = sJob;
        if (jobId >= a.nJobs) break;
        if (tid == 0) sPt = a.points[a.jobPoint[jobId]];
        __syncthreads();
        /* (a thread-local copy of the point was measured: spills, 3 % slower; the point as a kernel constant, for
         * launches with one point: constant-bank loads in divergent code, 4-7 % slower than these shared loads) */
        const PT& pt = static_cast<const PT&>(sPt);
        RaJobT<PT> job; job.pt = &pt; job.rep = a.jobRep[jobId];
        job.dump = DUMP ? a.dump + (size_t)jobId * a.dumpStride : nullptr;
        ra_job_init<DUMP>(job, s, tid, nt);
        RaAcc acc; acc.contFailed = acc.collP = acc.txop = acc.collScans = acc.totScans = 0;
        __syncthreads();

        int simTime = pt.maxTime;
        if (timers && tid == 0) tick = clock64();
        /* The loop over the ms.  Warp 0 owns the control flow: it decides whether the replication has ended (W:330-334 and
         * the loop bound W:267; no other warp reads nSuccess, which warp 0 may already be changing in a later light ms),
         * runs light ms (no movers, at most 32 events) back to back without any block barrier (ra_light_ms), and at the
         * first ms that needs the block prepares that ms' class view and control block.  It publishes (ms to run, how,
         * simTime) through sLight. */
        for (int T = 0, first = 1;; first = 0) {
            if (tid < 32) {
                int code = 0;
                if (!first && ra_ms_done(pt, s, T, &simTime)) code = 4;           /* the ms the block has just finished */
                else {
                    if (!first) ++T;
                    if (tid == 0) ra_gc_apply(s);
                    if (tid == 0) ra_lists_reset(s);
                    __syncwarp();
                    RaCtl c = ra_ctl_load(s);
                    int done = 0;
                    for (;;) {
                        code = ra_light_ms<DUMP>(job, w, s, c, &acc, T, &done, &simTime);
                        if (code != 1) break;
                        if (done) { code = 4; break; }
                        ++T;
                    }
                    __syncwarp();
                    if (tid == 0) ra_ctl_store(s, c);
                    __syncwarp();
                    if (code == 0) ra_phase0(job, s, T, tid, 32);
                    else if (code == 2) ra_phase0_classes(job, s, T, tid, 32);
                }
                if (tid == 0) { sLight[0] = T; sLight[1] = code; sLight[2] = simTime; sLight[3] = (int)s.nNlLight; }
            }
            __syncthreads();
            T = sLight[0];
            const int lightCode = sLight[1];
            RA_TICK(0);
            if (lightCode == 4) { simTime = sLight[2]; break; }
            if (lightCode == 0) {
                /* movers: 128-bit coalesced loads of bucket T; two records per thread and iteration so that
                 * their two Philox chains interleave (the chain is 10 dependent rounds), next pair prefetched */
                const unsigned nMov = s.nMov;
                const uint4* bT = w.bucket + (size_t)((unsigned)T & (unsigned)(pt.R - 1)) * w.cap;
                const uint4 dead = make_uint4(RA_DEAD, 0, 0, 0);
                unsigned i = tid;
                /* the thread walks records tid, tid + NT, ...: one pointer stepped by a compile-time stride (loads at
                 * immediate offsets), `left` = records from the thread's current one to the end of the bucket */
                const uint4* pr = bT + tid;
                int left = (int)nMov - tid;
                /* the trip count is the warp's (that of its first lane; lanes past the end of the bucket carry dead
                 * records): the warp votes inside the loop */
                int leftW = (int)nMov - (tid & ~31);
                RaPend pd; pd.x = RA_INF32; pd.z = pd.w = 0;      /* this thread's parked re-transmitter (ra_pend_flush) */
                uint4 c[RA_ILP];
#pragma unroll
                for (int k = 0; k < RA_ILP; ++k) c[k] = left > k * NT ? RA_LDREC(&pr[k * NT]) : dead;
                while (leftW > 0) {
                    uint4 n[RA_ILP];
                    rach_u32x4 d[RA_ILP];
#pragma unroll
                    for (int k = 0; k < RA_ILP; ++k) n[k] = left > (RA_ILP + k) * NT ? RA_LDREC(&pr[(RA_ILP + k) * NT]) : dead;
#pragma unroll
                    for (int k = 0; k < RA_ILP; ++k) d[k] = ra_draws(job, c[k].x, T);
#pragma unroll
                    for (int k = 0; k < RA_ILP; ++k) {
                        RaPend land;
                        const bool lands = ra_phase1_mover_d<DUMP>(job, w, s, acc, T, i + k * NT, c[k], d[k], land);
                        if (FIXED) {
                            /* a second re-transmitter in a lane that still holds one: the whole warp empties its registers
                             * (one pass of the list code for a dozen lanes instead of one pass per lane).  Only with the
                             * compile-time point view: with runtime parameters the three extra live registers cost more
                             * than the branch (measured on the configs[4] grid: 1062 vs 1014 ms) */
                            if (__any_sync(0xFFFFFFFFu, lands && pd.x != RA_INF32)) ra_pend_flush(pt, w, s, T, pd);
                            if (lands) pd = land;
                        } else if (lands) { pd = land; ra_pend_flush(pt, w, s, T, pd); }
                    }
#pragma unroll
                    for (int k = 0; k < RA_ILP; ++k) c[k] = n[k];
                    i += RA_ILP * NT; pr += RA_ILP * NT; left -= RA_ILP * NT; leftW -= RA_ILP * NT;
                }
                ra_pend_flush(pt, w, s, T, pd);
                const unsigned n1 = nMov + (unsigned)s.nArr + s.nM3;
                for (i = nMov + tid; i < n1; i += nt) ra_phase1_item<DUMP>(job, w, s, acc, T, i);
                __syncthreads();
                RA_TICK(1);
            }
            if (lightCode != 3) {
            if (s.nC3) {
                if (tid == 0) ra_phase2_serial(pt, w, s);
                __syncthreads();
                RA_TICK(2);
            }
            if (s.nUnc) {
                const unsigned n = s.nUnc;
                for (unsigned i = tid; i < n; i += nt) ra_phase3_item<DUMP>(job, w, s, T, i);
                __syncthreads();
                RA_TICK(3);
            }
            if (s.nE1) {
                const unsigned n = s.nE1;
                for (unsigned i = tid; i < n; i += nt) ra_phase3b_item(pt, w, s, i);
                __syncthreads();
                RA_TICK(4);
            }
            {
                const unsigned n4 = (unsigned)pt.P + s.nLanders;
                for (unsigned i = tid; i < n4; i += nt) ra_phase4_item(pt, w, s, acc, i);
            }
            __syncthreads();
            RA_TICK(5);
            if (s.nSingles) {
                if (ra_phase5_trivial(pt, s)) {                    /* every scan answered: no threshold, no barrier */
                    if (tid == 0) s.gcAdd = (int)s.nSingles;
                } else {
                    if (tid < 32) ra_phase5_warp(pt, w, s);
                    __syncthreads();
                    RA_TICK(6);
                }
            }
            {
                const unsigned n6 = (unsigned)pt.P + s.nLanders + s.nE1;
                for (unsigned i = tid; i < n6; i += nt) ra_phase6_item<DUMP>(job, w, s, T, i);
                if (s.nSingles) ra_hist_clear(pt, w, s, tid, nt);
            }
            __syncthreads();
            RA_TICK(7);
            }
            {
                /* stale position hints: of this ms' general phase 6, or handed over by ra_light_ms (code 3, count in sLight) */
                const unsigned nNl = lightCode == 3 ? (unsigned)sLight[3] : s.nNl;
                if (nNl) {
                    ra_phase6b<DUMP>(job, w, s, T, tid, nt, nNl);
                    __syncthreads();
                    RA_TICK(8);
                }
            }
        }
        const int last = simTime < pt.maxTime ? simTime : pt.maxTime - 1;
        if (DUMP) ra_dump_inflight(job, w, s, last, tid, nt);
        if (acc.contFailed) atomicAdd(&s.contFailed, (ra_u64)acc.contFailed);
        if (acc.collP) atomicAdd(&s.collP, (ra_u64)acc.collP);
        if (acc.txop) atomicAdd(&s.txop, (ra_u64)acc.txop);
        if (acc.collScans) atomicAdd(&s.collScans, (ra_u64)acc.collScans);
        if (acc.totScans) atomicAdd(&s.totScans, (ra_u64)acc.totScans);
        __syncthreads();
        if (tid == 0) {
            ra_stats st; memset(&st, 0, sizeof st);
            st.simTimeMs = simTime; st.nSuccess = (int)s.nSuccess;
            st.preambleTxSum = (long long)s.txSum; st.delaySum = (long long)s.delaySum;
            st.failCountSum = (long long)s.failSum; st.continueFailed = (long long)s.contFailed;
            st.finalSuccess = (long long)s.nSuccess;                 /* W:676: one per success */
            st.collisionPreambles = (long long)s.collP; st.totalPreambleTxop = (long long)s.txop;
            st.collisionScans = (long long)s.collScans; st.totalScans = (long long)s.totScans;
            st.updates = (long long)pt.nUE * (long long)((simTime + pt.A - 1) / pt.A);
            st.recordMoves = (long long)s.recMoves;
            a.stats[jobId] = st;
            if (s.overflow) atomicExch(a.errFlag, s.overflow);
            /* every thread's dump rows were written before the barrier above; publish them system-wide, then the flag */
            if (a.doneFlags) { __threadfence_system(); a.doneFlags[jobId] = 1; }
        }
    }
    __syncthreads();
    if (timers && tid < RA_NPHASE && sCyc[tid]) atomicAdd(&a.phaseCycles[tid], sCyc[tid]);
}

/* ------------------------------------------------------------------------------------------
 * Variant N (NOMA.c): one block per replication, phases of rach_core_n.cuh.
 * ------------------------------------------------------------------------------------------ */
template <bool DUMP>
__global__ void __launch_bounds__(RA_NT_N, RA_MINB_N) ra_step_kernel_n(RaKernelArgs a) {     /* fp64 activation math: 64 registers, no spills */
    extern __shared__ __align__(16) unsigned char ra_dyn_smem[];
    __shared__ RaSharedN s;
    __shared__ RaPointDev sPt;
    __shared__ int sJob;
    const int tid = threadIdx.x, nt = blockDim.x;
    const RaWorkN w = a.worksN[blockIdx.x];
    for (;;) {
        __syncthreads();
        if (tid == 0) sJob = (int)atomicAdd(a.jobCounter, 1u);
        __syncthreads();
        const int jobId = sJob;
        if (jobId >= a.nJobs) break;
        if (tid == 0) { sPt = a.points[a.jobPoint[jobId]]; rn_carve(s, ra_dyn_smem, sPt.R, sPt.P); }
        __syncthreads();
        const RaPointDev& pt = sPt;
        RaJob job; job.pt = &pt; job.rep = a.jobRep[jobId];
        job.dump = DUMP ? a.dump + (size_t)jobId * a.dumpStride : nullptr;
        rn_job_init<DUMP>(job, s, tid, nt);
        __syncthreads();
        int simTime = pt.maxTime;
        const unsigned Rm = (unsigned)(pt.R - 1);
        int nextOcc = 0, occ = 0;                                      /* next ms with T % accessTime == 0 (no division per ms) */
        for (int T = 0; T < pt.maxTime; ++T) {
            if (T == nextOcc) {                                         /* a RACH occasion, N:668 */
                nextOcc += pt.A;
                /* the arrival gate (N:675-681) is read by every thread from the schedule, so the table clearing / control
                 * block (A0) and the arrivals (A1: calendar appends only) share one phase */
                const unsigned acOld = occ ? (unsigned)pt.arrCum[occ - 1] : 0u, acNew = (unsigned)pt.arrCum[occ];
                ++occ;
                rn_phaseA0(job, s, T, tid, nt);
                for (unsigned i = acOld + tid; i < acNew; i += nt) rn_phaseA1_item<DUMP>(job, w, s, T, i);
                __syncthreads();
                const unsigned nTx = s.bcount[(unsigned)T & Rm];
                for (unsigned j = tid; j < nTx; j += nt) rn_phaseA2_item(pt, w, s, T, j);
                __syncthreads();
                for (int sec = tid >> 5; sec < (pt.geometry ? RA_NSECT : 1); sec += nt >> 5) rn_phaseB_warp(job, w, s, T, sec);   /* one warp per sector */
                __syncthreads();
                for (unsigned j = tid; j < nTx; j += nt) rn_phaseC_item<DUMP>(job, w, s, T, j);
                __syncthreads();
                if (tid == 0) s.bcount[(unsigned)T & Rm] = 0;           /* the slot is next used a ring later */
            }
            const unsigned nM3 = s.m3count[(unsigned)T & (RA_M3RING - 1)];
            if (nM3) {                                                  /* N:699 */
                for (unsigned j = tid; j < nM3; j += nt) rn_msg3_item<DUMP>(job, w, s, T, j);
                __syncthreads();
                if (tid == 0) s.m3count[(unsigned)T & (RA_M3RING - 1)] = 0;
                const bool allDone = s.nSuccess == (unsigned)pt.nUE;          /* N:707-710 */
                /* nobody may start the Msg3 answers of a later ms (they change nSuccess) before every thread has taken
                 * this decision */
                __syncthreads();
                if (allDone) { simTime = T; break; }
            }
        }
        __syncthreads();
        const int last = simTime < pt.maxTime ? simTime : pt.maxTime - 1;
        if (DUMP) {
            rn_dump_inflight(job, w, s, last, tid, nt);
            double* g = a.gainDump + (size_t)jobId * a.gainStride;
            for (int i = tid; i < pt.nUE; i += nt) g[i] = i < s.activeCheck ? w.gain[i] : 0.0;
        }
        if (tid == 0) {
            ra_stats st; memset(&st, 0, sizeof st);
            st.simTimeMs = simTime; st.nSuccess = (int)s.nSuccess;
            st.preambleTxSum = (long long)s.txSum; st.delaySum = (long long)s.delaySum;
            st.continueFailed = (long long)s.nDropped;                  /* RaFailed UEs, N:483 */
            st.finalSuccess = (long long)s.nSuccess;
            st.updates = (long long)pt.nUE * (long long)((simTime + pt.A - 1) / pt.A);
            a.stats[jobId] = st;
            if (s.overflow) atomicExch(a.errFlag, s.overflow);
        }
        if (a.doneFlags) {                                  /* the dump rows of every thread, then the flag */
            __syncthreads();
            if (tid == 0) { __threadfence_system(); a.doneFlags[jobId] = 1; }
        }
    }
}

/* ------------------------------------------------------------------------------------------
 * Variant U0 (RandomAccessSimulator.c): one warp per replication, one lane per live UE (rach_core_u0.cuh).
 * Measured on the way here (100k UEs x 1024 replications): one thread per replication, 8 replications per warp 2680 ms
 * (the walks serialise each other's branches), one per warp 848 ms.
 * ------------------------------------------------------------------------------------------ */
#define RU_WIN 64            /* live-list entries per replication kept in shared memory (the warp step needs >= 32) */
static size_t ru_smem_bytes(int maxR, bool headsInSmem) {
    return RU_WIN * sizeof(RuUE) + (headsInSmem ? (size_t)maxR * sizeof(int) : 0);
}

/* one warp (= one block) per replication; lanesOn = 0 runs the serial step on lane 0 in every ms */
template <bool DUMP>
__global__ void __launch_bounds__(32) ra_u0_kernel(RaKernelArgs a, int cap, int headsInSmem, int lanesOn) {
    extern __shared__ __align__(16) unsigned char ru_dyn_smem[];
    const int lane = threadIdx.x;
    RuUE* live = a.liveBase + (size_t)blockIdx.x * ru_work_elems(cap, a.maxR);
    RuUE* ph = live + cap;
    int* phHead = reinterpret_cast<int*>(ph + cap);
    RuUE* win = reinterpret_cast<RuUE*>(ru_dyn_smem);
    if (headsInSmem) phHead = reinterpret_cast<int*>(ru_dyn_smem + RU_WIN * sizeof(RuUE));
    for (;;) {
        int jobId = 0;
        if (lane == 0) jobId = (int)atomicAdd(a.jobCounter, 1u);
        jobId = __shfl_sync(0xFFFFFFFFu, jobId, 0);
        if (jobId >= a.nJobs) break;
        const RaPointDev* pt = &a.points[a.jobPoint[jobId]];
        RaJob job; job.pt = pt; job.rep = a.jobRep[jobId];
        job.dump = DUMP ? a.dump + (size_t)jobId * a.dumpStride : nullptr;
        RuStats st;
        ru_run_replication<DUMP>(job, live, win, RU_WIN, ph, phHead, cap, lanesOn, &st);
        __syncwarp();
        if (lane != 0) continue;
        ra_stats o; memset(&o, 0, sizeof o);
        o.simTimeMs = st.simTime; o.nSuccess = st.nSuccess; o.preambleTxSum = st.txSum; o.delaySum = st.delaySum;
        o.continueFailed = st.dropped; o.finalSuccess = st.nSuccess;
        o.collisionPreambles = st.collisionPreambles; o.totalPreambleTxop = st.totalPreambleTxop;
        o.updates = (long long)pt->nUE * (long long)((st.simTime + 4) / 5);
        a.stats[jobId] = o;
        if (st.overflow) atomicExch(a.errFlag, st.overflow);
        if (a.doneFlags) { __threadfence_system(); a.doneFlags[jobId] = 1; }      /* after the __syncwarp() above */
    }
}

/* ------------------------------------------------------------------------------------------
 * activateUEs side outputs, RandomAccessWithNOMA.c:392-415, recomputed from the draw tape.
 * Types follow the C semantics of the reference: float locals, double libm calls.
 * ------------------------------------------------------------------------------------------ */
__global__ void ra_geometry_kernel(RaPointDev pt, unsigned rep, int lastArrivalMs, float cellRadius, float* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= pt.nUE) return;
    float* o = out + (size_t)i * 6;
    /* arrival ms: first occasion whose cumulative count exceeds i */
    int lo = 0, hi = pt.nOcc;
    while (lo < hi) { int mid = (lo + hi) >> 1; if (pt.arrCum[mid] > i) hi = mid; else lo = mid + 1; }
    const int time = lo * pt.A;
    if (lo >= pt.nOcc || time > lastArrivalMs) { for (int k = 0; k < 6; ++k) o[k] = 0.f; return; }
    rach_u32x4 d = rach_tape_block(pt.seed, rep, (unsigned)i, (unsigned)time, 0u, RACH_TAPE_TAG_UE);
    const float bandwidth = 5;                                                    /* W:64 */
    float pi = 3.14;
    float theta = (float)(int)(d.v[0] >> 1) / (float)(2147483647) * 2 * pi;      /* W:393 */
    float r = (float)((double)cellRadius * sqrt((double)((float)(int)(d.v[1] >> 1) / (float)2147483647)));   /* W:394 */
    int sector = ra_sector((int)(d.v[0] >> 1));
    o[0] = theta;
    o[1] = (float)((double)r * cos((double)theta));                              /* W:412 */
    o[2] = (float)((double)r * sin((double)theta));                              /* W:413 */
    o[3] = r;                                                                    /* W:414 */
    o[4] = (float)(20 * log10(4. * (double)pi * (double)r / (double)(bandwidth / 1000)));   /* W:415 */
    o[5] = (float)sector;
}

/* ========================================================================================== */
/*                                        host side                                           */
/* ========================================================================================== */
struct RaDev {
    int id = 0;
    std::vector<int> jobs;            /* global job ids run on this device */
    RaPointDev* dPoints = nullptr;
    std::vector<int*> dArrCum;
    int* dJobPoint = nullptr; unsigned* dJobRep = nullptr; unsigned* dCounter = nullptr;
    ra_stats* dStats = nullptr; RaWork* dWorks = nullptr; RaWorkN* dWorksN = nullptr; unsigned char* dWorkspace = nullptr;
    double* dGainDump = nullptr;
    int* dDump = nullptr; int* dErr = nullptr; float* dGeom = nullptr; ra_u64* dCyc = nullptr;
    int grid = 0, nt = 0; size_t smem = 0; const void* kern = nullptr;
    cudaStream_t stream = nullptr; cudaEvent_t e0 = nullptr, e1 = nullptr;
    std::vector<ra_stats> hStats;
    int hErr = 0;
    /* streaming of per-UE dumps while the kernel runs (ra_sim_run_stream) */
    int* hDone = nullptr;             /* [nJobs] pinned, mapped: written by the kernel                   */
    cudaStream_t copyStream = nullptr;
};

/* shape: 0 = 128 x 8, 1 = 256 x 5, 2 = 512 x 2 (threads x resident blocks per SM) */
static const int kShapeNT[3] = {RA_NT, RA_NT_BIG, RA_NT_HUGE};
static const int kShapeMinB[3] = {RA_MINB, RA_MINB_BIG, RA_MINB_HUGE};
template <bool DUMP, bool FIXED, bool TIMERS>
static const void* ra_step_entry2(int shape) {
    if (shape == 2) return (const void*)ra_step_kernel<DUMP, RA_NT_HUGE, RA_MINB_HUGE, FIXED, TIMERS>;
    return shape == 1 ? (const void*)ra_step_kernel<DUMP, RA_NT_BIG, RA_MINB_BIG, FIXED, TIMERS>
                      : (const void*)ra_step_kernel<DUMP, RA_NT, RA_MINB, FIXED, TIMERS>;
}
/* (the phase timers exist without the per-UE dump only: ra_sim_create refuses the combination) */
static const void* ra_step_entry(bool dump, int shape, bool fixed, bool timers) {
    if (dump) return fixed ? ra_step_entry2<true, true, false>(shape) : ra_step_entry2<true, false, false>(shape);
    if (timers) return fixed ? ra_step_entry2<false, true, true>(shape) : ra_step_entry2<false, false, true>(shape);
    return fixed ? ra_step_entry2<false, true, false>(shape) : ra_step_entry2<false, false, false>(shape);
}

struct ra_sim {
    std::vector<ra_params> points;
    std::vector<RaPointDev> hostPoints;       /* arrCum unset; per-device copies carry the pointers */
    std::vector<std::vector<int>> arrCum;
    int nPoints = 0, reps = 0;
    ra_options opt;
    std::vector<RaDev> devs;
    std::vector<ra_stats> stats;              /* [nPoints*reps] */
    std::vector<int> jobDev, jobLocal;        /* where each global job ran */
    bool ran = false;
    double kernelMs = 0; long long launches = 0;
    size_t dumpStride = 0;
    int maxP = 0, maxR = 0, cap = 0, cap3 = 0, variant = RA_VARIANT_W;
    std::string err;
};


static thread_local std::string g_createErr;
static thread_local int g_createCode = RA_OK;

#define RA_CUDA(sim, call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
    char b_[512]; snprintf(b_, sizeof b_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    (sim)->err = b_; return RA_E_CUDA; } } while (0)

static void ra_free_dev(RaDev& d) {
    cudaSetDevice(d.id);
    for (int* p : d.dArrCum) cudaFree(p);
    cudaFree(d.dPoints); cudaFree(d.dJobPoint); cudaFree(d.dJobRep); cudaFree(d.dCounter);
    cudaFree(d.dStats); cudaFree(d.dWorks); cudaFree(d.dWorkspace); cudaFree(d.dDump); cudaFree(d.dErr);
    cudaFree(d.dGeom); cudaFree(d.dCyc); cudaFree(d.dWorksN); cudaFree(d.dGainDump);
    if (d.e0) cudaEventDestroy(d.e0);
    if (d.e1) cudaEventDestroy(d.e1);
    if (d.stream) cudaStreamDestroy(d.stream);
    if (d.copyStream) cudaStreamDestroy(d.copyStream);
    if (d.hDone) cudaFreeHost(d.hDone);
}

static int ra_setup_device(ra_sim* sim, RaDev& d) {
    RA_CUDA(sim, cudaSetDevice(d.id));
    cudaDeviceProp prop;
    RA_CUDA(sim, cudaGetDeviceProperties(&prop, d.id));
    RA_CUDA(sim, cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking));
    RA_CUDA(sim, cudaEventCreate(&d.e0));
    RA_CUDA(sim, cudaEventCreate(&d.e1));
    const int nJobs = (int)d.jobs.size();

    /* points + arrival tables */
    std::vector<RaPointDev> pts = sim->hostPoints;
    d.dArrCum.resize(sim->nPoints, nullptr);
    for (int i = 0; i < sim->nPoints; ++i) {
        RA_CUDA(sim, cudaMalloc(&d.dArrCum[i], sizeof(int) * sim->arrCum[i].size()));
        RA_CUDA(sim, cudaMemcpy(d.dArrCum[i], sim->arrCum[i].data(), sizeof(int) * sim->arrCum[i].size(), cudaMemcpyHostToDevice));
        pts[i].arrCum = d.dArrCum[i];
    }
    RA_CUDA(sim, cudaMalloc(&d.dPoints, sizeof(RaPointDev) * pts.size()));
    RA_CUDA(sim, cudaMemcpy(d.dPoints, pts.data(), sizeof(RaPointDev) * pts.size(), cudaMemcpyHostToDevice));

    /* job list */
    std::vector<int> jp(nJobs); std::vector<unsigned> jr(nJobs);
    for (int j = 0; j < nJobs; ++j) {
        jp[j] = d.jobs[j] / sim->reps;
        jr[j] = (unsigned)(sim->opt.repOffset + d.jobs[j] % sim->reps);
    }
    RA_CUDA(sim, cudaMalloc(&d.dJobPoint, sizeof(int) * std::max(nJobs, 1)));
    RA_CUDA(sim, cudaMalloc(&d.dJobRep, sizeof(unsigned) * std::max(nJobs, 1)));
    RA_CUDA(sim, cudaMemcpy(d.dJobPoint, jp.data(), sizeof(int) * nJobs, cudaMemcpyHostToDevice));
    RA_CUDA(sim, cudaMemcpy(d.dJobRep, jr.data(), sizeof(unsigned) * nJobs, cudaMemcpyHostToDevice));
    RA_CUDA(sim, cudaMalloc(&d.dCounter, sizeof(unsigned)));
    RA_CUDA(sim, cudaMalloc(&d.dErr, sizeof(int)));
    RA_CUDA(sim, cudaMalloc(&d.dCyc, sizeof(ra_u64) * RA_NPHASE));
    RA_CUDA(sim, cudaMalloc(&d.dStats, sizeof(ra_stats) * std::max(nJobs, 1)));
    d.hStats.resize(nJobs);
    if (sim->opt.dumpUEs) {
        size_t bytes = sizeof(int) * sim->dumpStride * (size_t)std::max(nJobs, 1);
        cudaError_t e = cudaMalloc(&d.dDump, bytes);
        if (e != cudaSuccess) { sim->err = "dump buffer does not fit on the device (dumpUEs keeps nUE*16 ints per replication)"; return RA_E_NOMEM; }
    }

    if (sim->variant == RA_VARIANT_U0) {
        /* one warp (block) per replication; global live-list overflow + phantom store of cap UEs (64 B each) per block */
        size_t freeB = 0, totalB = 0;
        RA_CUDA(sim, cudaMemGetInfo(&freeB, &totalB));
        const size_t perThread = sizeof(RuUE) * ru_work_elems(sim->cap, sim->maxR);
        long long threads = std::min<long long>(nJobs, (long long)((double)freeB * 0.85 / (double)perThread));
        threads = std::min<long long>(threads, (long long)prop.multiProcessorCount * 32);   /* resident blocks */
        if (threads < 1) { sim->err = "not enough device memory for one U0 live list"; return RA_E_NOMEM; }
        d.grid = (int)threads;
        d.smem = 0;
        cudaError_t e = cudaMalloc(&d.dWorkspace, perThread * (size_t)d.grid);
        if (e != cudaSuccess) { sim->err = std::string("U0 workspace cudaMalloc failed: ") + cudaGetErrorString(e); return RA_E_NOMEM; }
        return RA_OK;
    }
    /* grid and per-block workspace */
    const bool isN = sim->variant == RA_VARIANT_N;
    const bool dump = sim->opt.dumpUEs != 0;
    d.smem = 0;
    if (isN) d.smem = rn_smem_bytes(sim->maxR, sim->maxP);
    else for (const RaPointDev& hp : sim->hostPoints) d.smem = std::max(d.smem, (size_t)hp.smemBytes);
    if (d.smem > (size_t)prop.sharedMemPerBlockOptin) {
        sim->err = "per-replication tables (ring x preambles) exceed the shared memory of one block"; return RA_E_INVAL;
    }
    /* W block shape.  Enough replications to fill the device: 128 x 8 if eight blocks' tables (+1 KB reserved per block)
     * fit in one SM's shared memory, else 256 x 5.  Fewer replications than block slots (strong scaling over GPUs, small
     * sweeps): a replication cannot be split over blocks, so the blocks grow with the free room -- at most 5 per SM:
     * 256 threads, at most 2 per SM: 512 threads.  RACH_BLOCK=small|big|huge overrides, for tuning. */
    int shape = (d.smem + 1024) * RA_MINB > (size_t)prop.sharedMemPerMultiprocessor ? 1 : 0;
    {
        /* larger blocks only pay where a ms has hundreds of events to share out; a lightly loaded point (Uniform traffic:
         * 9 arrivals per occasion at 100k UEs) is barrier latency, which grows with the block (measured, Uniform 100k x 256:
         * 128 threads 129 ms, 256 137 ms, 512 143 ms) */
        int peak = 0;
        for (const std::vector<int>& ac : sim->arrCum)
            for (size_t o = 0; o < ac.size(); ++o) peak = std::max(peak, ac[o] - (o ? ac[o - 1] : 0));
        const int perSMjobs = (nJobs + prop.multiProcessorCount - 1) / prop.multiProcessorCount;
        if (peak >= 24) {
            if (perSMjobs <= RA_MINB_HUGE) shape = 2;
            else if (perSMjobs <= RA_MINB_BIG) shape = 1;
        }
    }
    if (const char* bs = getenv("RACH_BLOCK")) shape = bs[0] == 'h' ? 2 : (bs[0] == 'b' ? 1 : 0);
    /* all points in the reference's default family (P 54, BI 20, subframe 5, RAR window 5): the instantiation with those
     * values as immediates (RACH_FIXED=0 forces the general one, for cross-checks) */
    bool fixed = !isN;
    for (const RaPointDev& hp : sim->hostPoints) fixed = fixed && ra_point_is_default_family(hp);
    if (const char* fx = getenv("RACH_FIXED")) fixed = fixed && fx[0] != '0';
    d.nt = isN ? RA_NT_N : kShapeNT[shape];
    const int minb = isN ? RA_MINB_N : kShapeMinB[shape];
    const void* kern = isN ? (dump ? (const void*)ra_step_kernel_n<true> : (const void*)ra_step_kernel_n<false>)
                           : ra_step_entry(dump, shape, fixed, sim->opt.phaseTimers != 0);
    d.kern = kern;
    RA_CUDA(sim, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)d.smem));
    /* shared-memory carveout: the driver's default was the best of {default, 50, 60, 75, 100 %} (within 0.6 %) */
    int occ = 0;
    RA_CUDA(sim, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, d.nt, d.smem));
    if (occ < 1) { sim->err = "step kernel does not fit on an SM"; return RA_E_INVAL; }
    int perSM = sim->opt.ctasPerSM > 0 ? std::min(sim->opt.ctasPerSM, occ) : std::min(occ, minb);
    if (isN && dump) {
        cudaError_t e = cudaMalloc(&d.dGainDump, sizeof(double) * (size_t)sim->cap * (size_t)std::max(nJobs, 1));
        if (e != cudaSuccess) { sim->err = "gain dump buffer does not fit on the device"; return RA_E_NOMEM; }
    }

    RaWork sizeW; RaWorkN sizeN;
    const size_t perBlock = isN ? rn_work_carve(nullptr, sim->cap, sim->cap3, sim->maxR, &sizeN)
                                : ra_work_carve(nullptr, sim->cap, sim->cap3, sim->maxR, sim->maxP, &sizeW);

    size_t freeB = 0, totalB = 0;
    RA_CUDA(sim, cudaMemGetInfo(&freeB, &totalB));
    size_t budget = (size_t)((double)freeB * 0.85);
    int grid = std::min(nJobs, prop.multiProcessorCount * perSM);
    if ((size_t)grid * perBlock > budget) grid = (int)(budget / perBlock);
    if (grid < 1) { sim->err = "not enough device memory for one replication workspace"; return RA_E_NOMEM; }
    d.grid = grid;
    {
        cudaError_t e = cudaMalloc(&d.dWorkspace, perBlock * (size_t)grid);
        if (e != cudaSuccess) { sim->err = std::string("workspace cudaMalloc failed: ") + cudaGetErrorString(e); return RA_E_NOMEM; }
    }
    if (isN) {
        std::vector<RaWorkN> worksN(grid);
        for (int b = 0; b < grid; ++b) rn_work_carve(d.dWorkspace + perBlock * (size_t)b, sim->cap, sim->cap3, sim->maxR, &worksN[b]);
        RA_CUDA(sim, cudaMalloc(&d.dWorksN, sizeof(RaWorkN) * grid));
        RA_CUDA(sim, cudaMemcpy(d.dWorksN, worksN.data(), sizeof(RaWorkN) * grid, cudaMemcpyHostToDevice));
        return RA_OK;
    }
    std::vector<RaWork> works(grid);
    for (int b = 0; b < grid; ++b) ra_work_carve(d.dWorkspace + perBlock * (size_t)b, sim->cap, sim->cap3, sim->maxR, sim->maxP, &works[b]);
    RA_CUDA(sim, cudaMalloc(&d.dWorks, sizeof(RaWork) * grid));
    RA_CUDA(sim, cudaMemcpy(d.dWorks, works.data(), sizeof(RaWork) * grid, cudaMemcpyHostToDevice));
    return RA_OK;
}

extern "C" const char* ra_last_create_error(void) { return g_createErr.c_str(); }
extern "C" int ra_last_create_code(void) { return g_createCode; }

extern "C" ra_sim* ra_sim_create_ex(const ra_params* points, int nPoints, int repsPerPoint,
                                    const int* devices, int nDevices, const ra_options* opt) {
    g_createErr.clear(); g_createCode = RA_E_INVAL;      /* every early return below is a parameter error unless it says otherwise */
    if (!points || nPoints < 1 || repsPerPoint < 1) { g_createErr = "points/nPoints/repsPerPoint invalid"; return nullptr; }
    int devCount = 0;
    if (cudaGetDeviceCount(&devCount) != cudaSuccess || devCount < 1) {
        g_createErr = "no CUDA device: librach_gpu has no CPU path"; g_createCode = RA_E_NODEVICE; return nullptr;
    }
    ra_sim* sim = new ra_sim();
    memset(&sim->opt, 0, sizeof sim->opt);
    if (opt) sim->opt = *opt;
    if (sim->opt.phaseTimers && sim->opt.dumpUEs) {
        g_createErr = "phaseTimers and dumpUEs cannot be combined (the timed kernel is the one without the per-UE dump)"; delete sim; return nullptr;
    }
    sim->nPoints = nPoints; sim->reps = repsPerPoint;
    sim->points.assign(points, points + nPoints);
    char err[256];
    for (int i = 0; i < nPoints; ++i) {
        if (ra_host_validate(&points[i], err, sizeof err) != RA_OK) {
            g_createErr = std::string("point ") + std::to_string(i) + ": " + err; delete sim; return nullptr;
        }
        const ra_params& p = points[i];
        if (i == 0) sim->variant = p.variant;
        else if (p.variant != sim->variant) { g_createErr = "all points of one ra_sim must share the variant"; delete sim; return nullptr; }
        RaPointDev pt;
        ra_host_point(&p, &pt);
        sim->hostPoints.push_back(pt);
        sim->arrCum.emplace_back(pt.nOcc);
        ra_host_arrcum(&p, sim->arrCum.back().data(), pt.nOcc);
        {   /* the device reads arrivals as differences of this schedule: it must never decrease nor pass nUE */
            const std::vector<int>& ac = sim->arrCum.back();
            for (size_t o = 0; o < ac.size(); ++o)
                if (ac[o] < (o ? ac[o - 1] : 0) || ac[o] > pt.nUE) {
                    g_createErr = std::string("point ") + std::to_string(i) + ": arrival schedule is not monotone"; g_createCode = RA_E_INTERNAL;
                    delete sim; return nullptr;
                }
        }
        sim->maxP = std::max(sim->maxP, pt.P); sim->maxR = std::max(sim->maxR, pt.R);
        sim->cap = std::max(sim->cap, pt.nUE);
        sim->cap3 = std::max(sim->cap3, ra_host_cap3(p.variant, &pt));
        sim->dumpStride = std::max(sim->dumpStride, (size_t)pt.nUE * RA_DUMP_W);
    }
    /* the engines index a block's move calendar with 32 bits (ring x capacity records of 16 bytes: 64 GB) */
    if ((unsigned long long)sim->maxR * (unsigned long long)sim->cap >= (1ull << 32)) {
        g_createErr = "ring x nUE exceeds 2^32 calendar records per replication"; g_createCode = RA_E_INVAL; delete sim; return nullptr;
    }
    std::vector<int> devs;
    if (!devices || nDevices < 1) devs.push_back(0);
    else devs.assign(devices, devices + nDevices);
    for (int dv : devs) if (dv < 0 || dv >= devCount) { g_createErr = "device index out of range"; delete sim; return nullptr; }

    /* longest replications first, dealt round-robin to the devices */
    const int nJobs = nPoints * repsPerPoint;
    std::vector<int> order(nJobs);
    for (int j = 0; j < nJobs; ++j) order[j] = j;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
        const RaPointDev& pa = sim->hostPoints[a / repsPerPoint]; const RaPointDev& pb = sim->hostPoints[b / repsPerPoint];
        return (long long)pa.nUE * pa.maxTime > (long long)pb.nUE * pb.maxTime; });
    sim->devs.resize(devs.size());
    sim->jobDev.resize(nJobs); sim->jobLocal.resize(nJobs);
    for (size_t k = 0; k < devs.size(); ++k) sim->devs[k].id = devs[k];
    for (int k = 0; k < nJobs; ++k) {
        RaDev& d = sim->devs[k % devs.size()];
        sim->jobDev[order[k]] = (int)(k % devs.size()); sim->jobLocal[order[k]] = (int)d.jobs.size();
        d.jobs.push_back(order[k]);
    }
    sim->stats.resize(nJobs);
    for (RaDev& d : sim->devs) {
        if (d.jobs.empty()) continue;                     /* more devices than replications: nothing to set up there */
        int rc = ra_setup_device(sim, d);
        if (rc != RA_OK) { g_createErr = sim->err; g_createCode = rc; ra_sim_destroy(sim); return nullptr; }
    }
    g_createCode = RA_OK;
    return sim;
}

extern "C" ra_sim* ra_sim_create(const ra_params* points, int nPoints, int repsPerPoint,
                                 const int* devices, int nDevices) {
    return ra_sim_create_ex(points, nPoints, repsPerPoint, devices, nDevices, nullptr);
}

/* launch on one device (asynchronous); the caller synchronises */
static int ra_launch_device(ra_sim* sim, RaDev& d, bool stream = false) {
    const int nJobs = (int)d.jobs.size();
    RA_CUDA(sim, cudaSetDevice(d.id));
    RA_CUDA(sim, cudaMemsetAsync(d.dCounter, 0, sizeof(unsigned), d.stream));
    RA_CUDA(sim, cudaMemsetAsync(d.dErr, 0, sizeof(int), d.stream));
    RA_CUDA(sim, cudaMemsetAsync(d.dCyc, 0, sizeof(ra_u64) * RA_NPHASE, d.stream));
    RaKernelArgs a; memset(&a, 0, sizeof a);
    a.points = d.dPoints; a.jobPoint = d.dJobPoint; a.jobRep = d.dJobRep; a.works = d.dWorks;
    a.jobCounter = d.dCounter; a.stats = d.dStats; a.dump = d.dDump; a.errFlag = d.dErr; a.phaseCycles = sim->opt.phaseTimers ? d.dCyc : nullptr;
    a.dumpStride = sim->dumpStride; a.nJobs = nJobs; a.maxP = sim->maxP; a.maxR = sim->maxR;
    if (stream) {
        if (!d.hDone) {
            RA_CUDA(sim, cudaHostAlloc(&d.hDone, sizeof(int) * (size_t)nJobs, cudaHostAllocMapped | cudaHostAllocPortable));
            RA_CUDA(sim, cudaStreamCreateWithFlags(&d.copyStream, cudaStreamNonBlocking));
        }
        memset(d.hDone, 0, sizeof(int) * (size_t)nJobs);
        int* dv = nullptr;
        RA_CUDA(sim, cudaHostGetDevicePointer(&dv, d.hDone, 0));
        a.doneFlags = dv;
    }
    RA_CUDA(sim, cudaEventRecord(d.e0, d.stream));
    a.worksN = d.dWorksN;
    a.gainDump = d.dGainDump; a.gainStride = (size_t)sim->cap;
    a.liveBase = (RuUE*)d.dWorkspace;
    if (sim->variant == RA_VARIANT_U0) {
        const int heads = sim->maxR <= 1024;    /* phantom calendar heads in shared memory unless BI is huge */
        const size_t sm = ru_smem_bytes(sim->maxR, heads != 0);
        const char* mode = getenv("RACH_U0");   /* RACH_U0=serial: the one-thread formulation, for cross-checks */
        const int lanesOn = !(mode && mode[0] == 's');
        if (sim->opt.dumpUEs) ra_u0_kernel<true><<<d.grid, 32, sm, d.stream>>>(a, sim->cap, heads, lanesOn);
        else ra_u0_kernel<false><<<d.grid, 32, sm, d.stream>>>(a, sim->cap, heads, lanesOn);
    } else {
        void* kargs[] = {&a};
        RA_CUDA(sim, cudaLaunchKernel(d.kern, dim3(d.grid), dim3(d.nt), kargs, d.smem, d.stream));
    }
    RA_CUDA(sim, cudaGetLastError());
    RA_CUDA(sim, cudaEventRecord(d.e1, d.stream));
    RA_CUDA(sim, cudaMemcpyAsync(d.hStats.data(), d.dStats, sizeof(ra_stats) * nJobs, cudaMemcpyDeviceToHost, d.stream));
    RA_CUDA(sim, cudaMemcpyAsync(&d.hErr, d.dErr, sizeof(int), cudaMemcpyDeviceToHost, d.stream));
    return RA_OK;
}

/* wait for one device and collect its results */
static int ra_collect_device(ra_sim* sim, RaDev& d, double* ms) {
    RA_CUDA(sim, cudaSetDevice(d.id));
    RA_CUDA(sim, cudaStreamSynchronize(d.stream));
    float t = 0; RA_CUDA(sim, cudaEventElapsedTime(&t, d.e0, d.e1));
    *ms = std::max(*ms, (double)t);
    if (d.hErr) {
        sim->err = d.hErr == 1 ? "engine self-check: a calendar bucket overflowed"
                 : d.hErr == 3 ? "engine self-check: a rejection loop of activeUE (NOMA.c:167-172, 185-189) did not end within 65536 draws"
                 : "engine self-check: a packed per-UE counter overflowed (preambleTxCounter > 32767, failCount > 65535)";
        return RA_E_INTERNAL;
    }
    for (size_t j = 0; j < d.jobs.size(); ++j) sim->stats[d.jobs[j]] = d.hStats[j];
    return RA_OK;
}

extern "C" int ra_sim_run(ra_sim* sim) {
    if (!sim) return RA_E_INVAL;
    sim->launches = 0; sim->ran = false;
    /* every device is launched, then every launched device is drained -- also after an error, so that no stream is
     * still writing into this handle's buffers when the caller sees the error code (and may destroy the handle) */
    int rc = RA_OK;
    std::string firstErr;
    std::vector<char> launched(sim->devs.size(), 0);
    for (size_t k = 0; k < sim->devs.size() && rc == RA_OK; ++k) {
        RaDev& d = sim->devs[k];
        if (d.jobs.empty()) continue;
        d.hErr = 0;
        launched[k] = 1;                      /* part of the sequence may be in flight even if a later call failed */
        rc = ra_launch_device(sim, d);
        if (rc == RA_OK) sim->launches++; else firstErr = sim->err;
    }
    double ms = 0;
    for (size_t k = 0; k < sim->devs.size(); ++k) {
        if (!launched[k]) continue;
        RaDev& d = sim->devs[k];
        if (rc == RA_OK) {
            rc = ra_collect_device(sim, d, &ms);
            if (rc != RA_OK) firstErr = sim->err;
        } else {                              /* already failing: just drain */
            cudaSetDevice(d.id); cudaStreamSynchronize(d.stream);
        }
    }
    if (rc != RA_OK) { sim->err = firstErr; return rc; }
    sim->kernelMs = ms; sim->ran = true;
    return RA_OK;
}

/* ------------------------------------------------------------------------------------------
 * Per-UE logs at scale (the role of saveResult, RandomAccessWithNOMA.c:797-825, for thousands of replications): the step
 * kernel never waits for the host.  Each replication raises a flag in host-mapped memory when its counters and its
 * nUE x 16 dump rows are complete; this thread polls the flags while the kernel keeps running, copies finished
 * replications out with one cudaMemcpyAsync each on a second stream into a ring of pinned staging buffers, and hands
 * them to the callback in completion order.
 * ------------------------------------------------------------------------------------------ */
#include <unistd.h>
extern "C" int ra_sim_run_stream(ra_sim* sim, ra_dump_cb cb, void* user) {
    if (!sim || !cb) return RA_E_INVAL;
    if (!sim->opt.dumpUEs) { sim->err = "ra_sim_run_stream needs ra_options.dumpUEs = 1 at create time"; return RA_E_STATE; }
    sim->launches = 0; sim->ran = false;
    const int kSlots = 4;                                  /* staging buffers in flight per device */
    struct Slot { int* rows = nullptr; ra_stats* st = nullptr; cudaEvent_t ev = nullptr; int job = -1; };
    struct Ring { std::vector<Slot> slots; int head = 0, inflight = 0; std::vector<char> issued; };
    const size_t nDev = sim->devs.size();
    std::vector<Ring> rings(nDev);
    int rc = RA_OK;
    std::string firstErr;
    auto fail = [&](int code, const std::string& msg) { if (rc == RA_OK) { rc = code; firstErr = msg; } };
    std::vector<char> launched(nDev, 0);
    for (size_t k = 0; k < nDev && rc == RA_OK; ++k) {
        RaDev& d = sim->devs[k];
        if (d.jobs.empty()) continue;
        cudaSetDevice(d.id);                               /* events belong to the device that is current when they are made */
        rings[k].slots.resize(kSlots);
        rings[k].issued.assign(d.jobs.size(), 0);
        for (Slot& sl : rings[k].slots) {
            if (cudaHostAlloc(&sl.rows, sizeof(int) * sim->dumpStride, cudaHostAllocPortable) != cudaSuccess ||
                cudaHostAlloc(&sl.st, sizeof(ra_stats), cudaHostAllocPortable) != cudaSuccess ||
                cudaEventCreateWithFlags(&sl.ev, cudaEventDisableTiming) != cudaSuccess) { fail(RA_E_NOMEM, "pinned staging buffers for the dump stream"); break; }
        }
        if (rc != RA_OK) break;
        d.hErr = 0;
        launched[k] = 1;
        const int lrc = ra_launch_device(sim, d, true);
        if (lrc == RA_OK) sim->launches++; else fail(lrc, sim->err);
    }
    if (rc == RA_OK) {
        size_t total = 0, delivered = 0;
        for (size_t k = 0; k < nDev; ++k) total += sim->devs[k].jobs.size();
        while (delivered < total && rc == RA_OK) {
            bool progress = false;
            for (size_t k = 0; k < nDev && rc == RA_OK; ++k) {
                if (!launched[k]) continue;
                RaDev& d = sim->devs[k];
                Ring& r = rings[k];
                cudaSetDevice(d.id);
                /* finished replications -> one asynchronous copy each, into the next free staging buffer */
                for (size_t j = 0; j < d.jobs.size() && r.inflight < kSlots; ++j) {
                    if (r.issued[j] || !((volatile int*)d.hDone)[j]) continue;
                    Slot& sl = r.slots[(r.head + r.inflight) % kSlots];
                    const int point = d.jobs[j] / sim->reps;
                    cudaError_t e1 = cudaMemcpyAsync(sl.rows, d.dDump + j * sim->dumpStride,
                                                     sizeof(int) * (size_t)sim->points[point].nUE * RA_DUMP_W, cudaMemcpyDeviceToHost, d.copyStream);
                    cudaError_t e2 = cudaMemcpyAsync(sl.st, d.dStats + j, sizeof(ra_stats), cudaMemcpyDeviceToHost, d.copyStream);
                    cudaError_t e3 = cudaEventRecord(sl.ev, d.copyStream);
                    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) {
                        const cudaError_t e = e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3);
                        fail(RA_E_CUDA, std::string("dump stream copy failed: ") + cudaGetErrorString(e)); break;
                    }
                    sl.job = (int)j; r.issued[j] = 1; ++r.inflight; progress = true;
                }
                /* copies that have arrived -> the callback, in issue order */
                while (r.inflight > 0 && rc == RA_OK) {
                    Slot& sl = r.slots[r.head];
                    const cudaError_t q = cudaEventQuery(sl.ev);
                    if (q == cudaErrorNotReady) break;
                    if (q != cudaSuccess) { fail(RA_E_CUDA, std::string("dump stream: ") + cudaGetErrorString(q)); break; }
                    const int gj = d.jobs[sl.job];
                    cb(user, gj / sim->reps, gj % sim->reps, sl.st, sl.rows);
                    r.head = (r.head + 1) % kSlots; --r.inflight; ++delivered; progress = true;
                }
            }
            if (!progress && rc == RA_OK) {
                /* nothing finished since the last look: make sure the kernels are still healthy, then wait a little */
                for (size_t k = 0; k < nDev; ++k) {
                    if (!launched[k]) continue;
                    cudaSetDevice(sim->devs[k].id);
                    const cudaError_t q = cudaStreamQuery(sim->devs[k].stream);
                    if (q != cudaSuccess && q != cudaErrorNotReady) fail(RA_E_CUDA, std::string("step kernel: ") + cudaGetErrorString(q));
                }
                usleep(200);
            }
        }
    }
    double ms = 0;
    for (size_t k = 0; k < nDev; ++k) {                     /* drain every launched device, also after an error */
        RaDev& d = sim->devs[k];
        cudaSetDevice(d.id);
        if (launched[k]) {
            if (d.copyStream) cudaStreamSynchronize(d.copyStream);
            if (rc == RA_OK) { const int crc = ra_collect_device(sim, d, &ms); if (crc != RA_OK) fail(crc, sim->err); }
            else cudaStreamSynchronize(d.stream);
        }
        for (Slot& sl : rings[k].slots) { if (sl.rows) cudaFreeHost(sl.rows); if (sl.st) cudaFreeHost(sl.st); if (sl.ev) cudaEventDestroy(sl.ev); }
    }
    if (rc != RA_OK) { sim->err = firstErr; return rc; }
    sim->kernelMs = ms; sim->ran = true;
    return RA_OK;
}

extern "C" int ra_sim_stats(ra_sim* sim, int point, int rep, ra_stats* out) {
    if (!sim || !out) return RA_E_INVAL;
    if (!sim->ran) { sim->err = "ra_sim_stats before ra_sim_run"; return RA_E_STATE; }
    if (point < 0 || point >= sim->nPoints || rep < 0 || rep >= sim->reps) { sim->err = "point/rep out of range"; return RA_E_INVAL; }
    *out = sim->stats[(size_t)point * sim->reps + rep];
    return RA_OK;
}

extern "C" int ra_sim_stats_all(ra_sim* sim, ra_stats* out) {
    if (!sim || !out) return RA_E_INVAL;
    if (!sim->ran) { sim->err = "ra_sim_stats_all before ra_sim_run"; return RA_E_STATE; }
    memcpy(out, sim->stats.data(), sizeof(ra_stats) * sim->stats.size());
    return RA_OK;
}

extern "C" int ra_sim_dump_ues(ra_sim* sim, int point, int rep, int* out) {
    if (!sim || !out) return RA_E_INVAL;
    if (!sim->ran) { sim->err = "ra_sim_dump_ues before ra_sim_run"; return RA_E_STATE; }
    if (!sim->opt.dumpUEs) { sim->err = "ra_sim_dump_ues needs ra_options.dumpUEs = 1 at create time"; return RA_E_STATE; }
    if (point < 0 || point >= sim->nPoints || rep < 0 || rep >= sim->reps) { sim->err = "point/rep out of range"; return RA_E_INVAL; }
    const int job = point * sim->reps + rep;
    RaDev& d = sim->devs[sim->jobDev[job]];
    RA_CUDA(sim, cudaSetDevice(d.id));
    RA_CUDA(sim, cudaMemcpy(out, d.dDump + (size_t)sim->jobLocal[job] * sim->dumpStride,
                            sizeof(int) * (size_t)sim->points[point].nUE * RA_DUMP_W, cudaMemcpyDeviceToHost));
    return RA_OK;
}

extern "C" int ra_sim_geometry(ra_sim* sim, int point, int rep, float* out) {
    if (!sim || !out) return RA_E_INVAL;
    if (!sim->ran) { sim->err = "ra_sim_geometry before ra_sim_run"; return RA_E_STATE; }
    if (point < 0 || point >= sim->nPoints || rep < 0 || rep >= sim->reps) { sim->err = "point/rep out of range"; return RA_E_INVAL; }
    if (sim->variant != RA_VARIANT_W) { sim->err = "ra_sim_geometry is for variant W; variant N reports ra_sim_gains"; return RA_E_STATE; }
    if (!sim->points[point].geometry) { sim->err = "ra_sim_geometry needs geometry = 1 (variant B draws no positions)"; return RA_E_STATE; }
    RaDev& d = sim->devs[0];
    RA_CUDA(sim, cudaSetDevice(d.id));
    const int n = sim->points[point].nUE;
    if (!d.dGeom) RA_CUDA(sim, cudaMalloc(&d.dGeom, sizeof(float) * 6 * (size_t)sim->cap));
    RaPointDev pt = sim->hostPoints[point]; pt.arrCum = d.dArrCum[point];
    /* UEs arrive only in ms the loop executed: up to simTime (break ms) or horizon-1 */
    const ra_stats& st = sim->stats[(size_t)point * sim->reps + rep];
    const int lastMs = st.simTimeMs < pt.maxTime ? st.simTimeMs : pt.maxTime - 1;
    ra_geometry_kernel<<<(n + 255) / 256, 256, 0, d.stream>>>(pt, (unsigned)(sim->opt.repOffset + rep), lastMs,
                                                               sim->points[point].cellRadius, d.dGeom);
    RA_CUDA(sim, cudaGetLastError());
    RA_CUDA(sim, cudaMemcpyAsync(out, d.dGeom, sizeof(float) * 6 * (size_t)n, cudaMemcpyDeviceToHost, d.stream));
    RA_CUDA(sim, cudaStreamSynchronize(d.stream));
    return RA_OK;
}

/* debug/profiling: cycles thread 0 of every block spent up to the barrier that ends each phase
 * (0 setup, 1 events, 2 C3 resolve, 3 uncertain, 4 late restarts, 5 scans, 6 grants, 7 apply) */
extern "C" int ra_sim_phase_cycles(ra_sim* sim, unsigned long long* out10) {
    if (!sim || !out10) return RA_E_INVAL;
    for (int k = 0; k < RA_NPHASE; ++k) out10[k] = 0;
    for (RaDev& d : sim->devs) {
        if (d.jobs.empty()) continue;
        ra_u64 h[RA_NPHASE];
        RA_CUDA(sim, cudaSetDevice(d.id));
        RA_CUDA(sim, cudaMemcpy(h, d.dCyc, sizeof h, cudaMemcpyDeviceToHost));
        for (int k = 0; k < RA_NPHASE; ++k) out10[k] += h[k];
    }
    return RA_OK;
}

extern "C" int ra_sim_gains(ra_sim* sim, int point, int rep, double* out) {
    if (!sim || !out) return RA_E_INVAL;
    if (!sim->ran) { sim->err = "ra_sim_gains before ra_sim_run"; return RA_E_STATE; }
    if (sim->variant != RA_VARIANT_N || !sim->opt.dumpUEs) { sim->err = "ra_sim_gains needs variant N and ra_options.dumpUEs = 1"; return RA_E_STATE; }
    if (point < 0 || point >= sim->nPoints || rep < 0 || rep >= sim->reps) { sim->err = "point/rep out of range"; return RA_E_INVAL; }
    const int job = point * sim->reps + rep;
    RaDev& d = sim->devs[sim->jobDev[job]];
    RA_CUDA(sim, cudaSetDevice(d.id));
    RA_CUDA(sim, cudaMemcpy(out, d.dGainDump + (size_t)sim->jobLocal[job] * (size_t)sim->cap,
                            sizeof(double) * (size_t)sim->points[point].nUE, cudaMemcpyDeviceToHost));
    return RA_OK;
}

extern "C" double ra_sim_kernel_ms(const ra_sim* sim) { return sim ? sim->kernelMs : 0.0; }
extern "C" long long ra_sim_gpu_launches(const ra_sim* sim) { return sim ? sim->launches : 0; }
extern "C" const char* ra_sim_last_error(const ra_sim* sim) { return sim ? sim->err.c_str() : "null handle"; }

extern "C" void ra_sim_destroy(ra_sim* sim) {
    if (!sim) return;
    for (RaDev& d : sim->devs) ra_free_dev(d);
    delete sim;
}
