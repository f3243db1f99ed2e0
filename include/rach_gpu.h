/*
 * rach_gpu.h -- C ABI of librach_gpu, the B200 (sm_100a) engine for the per-RACH-occasion
 * UE state machine of yaki-toki/5G-NR-RandomAccess.
 *
 * The reference has no plugin / FFI interface: every simulator is one `main`.  This ABI is
 * cut at the body of the reference's (seed, nUE) iteration -- everything between
 * `calloc(nUE, sizeof(struct UEinfo))` and `free(UE)` minus printing:
 *
 *   RandomAccessWithNOMA.c:229-368      (variant W, the only file with a CLI)
 *   RandomAccessSimulatorBeta.c:78-210  (variant B = W dynamics, no geometry draws)
 *
 * What each entry point replaces:
 *
 *   ra_sim_create      the per-point setup: parameter locals W:69-88 (+ argv overrides
 *                      W:90-206), calloc + initialUE W:229-234,374-381, maxTime/nAccessUE
 *                      W:241-255, srand W:219 (-> the Philox draw tape, rach_tape.h)
 *   ra_sim_run         the time loop W:267-335 (B:111-183): grant reset, arrivals,
 *                      activateUEs W:383-415, selectPreamble W:475-562, preambleCollision
 *                      W:607-665, requestResourceAllocation W:667-710, timerIncrease
 *                      W:712-718, successUEs + early break W:330-334,720-728
 *   ra_sim_stats       the aggregation loop W:337-351 and the globals W:62-63; the derived
 *                      floats of saveSimulationLog W:735-739 stay in the host
 *   ra_sim_dump_ues    the per-UE fields saveResult prints, W:809-822 (15 ints per UE)
 *   ra_sim_geometry    the activateUEs side outputs W:392-415 (never read back by W)
 *   ra_sim_histogram   the distributions behind the means of W:346-348: per-UE timer, preambleTxCounter and
 *                      failCount of the UEs with msg4Flag == 1, as histograms summed over replications
 *   ra_arrival_schedule  W:246-251 / W:285-287 (B:95-100 / B:127-129): UEs arriving per ms
 *
 * Conventions: plain pointers and sizes, caller-owned outputs, no exit() inside the
 * library (the reference's printf+exit(-1) convention, W:94-97, stays in the host main).
 * Every function that can fail returns 0 on success and a negative RA_E_* code on error;
 * ra_sim_last_error() gives the message.  ra_sim_create returns NULL on failure;
 * ra_last_create_code() / ra_last_create_error() then give the RA_E_* code and the message
 * (per calling thread).  There is no CPU fallback: without a CUDA device ra_sim_create
 * fails with RA_E_NODEVICE.
 */
#ifndef RACH_GPU_H
#define RACH_GPU_H

#ifdef __cplusplus
extern "C" {
#endif

#define RA_VARIANT_W  0   /* RandomAccessWithNOMA.c / RandomAccessSimulatorBeta.c dynamics */
#define RA_VARIANT_U0 1   /* RandomAccessSimulator.c legacy dynamics (U0:75-126, 157-266): Uniform 60 s,
                             subframe 5, 64 preambles by default, no grant limit, hard drop after 10
                             backoffs; ra_sim_dump_ues rows: timer active txTime preamble preambleChange
                             rarWindow maxRarCounter preambleTxCounter msg2Flag connectionRequest msg4Flag
                             raFailed nowBackoff 0 0 0 */
#define RA_VARIANT_N  2   /* NOMA.c sector / gain-pairing dynamics (N:131-324, 449-566, 665-711):
                             nGrantUL = grants per sector (N:43), maxRarWindow <= 5 (N:45),
                             maxMsg2TxCount carries maxMsg1ReTx (N:46), cellRadius (N:56), Beta only;
                             geometry = 0 selects NOMA.c's alternative non-sector collision function
                             (N:325-447, call commented out at N:688) */

#define RA_OK            0
#define RA_E_INVAL      -1   /* bad argument / unsupported parameter value */
#define RA_E_NODEVICE   -2   /* no usable CUDA device                      */
#define RA_E_CUDA       -3   /* a CUDA runtime call failed                 */
#define RA_E_NOMEM      -4   /* host or device allocation failed           */
#define RA_E_STATE      -5   /* call out of order (e.g. stats before run)  */
#define RA_E_INTERNAL   -6   /* engine self-check tripped (overflow flag)  */

#define RA_DUMP_FIELDS 16    /* ints per UE written by ra_sim_dump_ues     */

/* histogram kinds of ra_sim_histogram, over the UEs with msg4Flag == 1 (W:337-348, N:504-508, U0:127-139) */
#define RA_HIST_DELAY   0    /* timer at success in ms (the quantity delaySum sums, W:346): bins 0 .. horizon + 6, exact */
#define RA_HIST_TX      1    /* preambleTxCounter (preambleTxSum, W:347; N: nTxPreamble): 256 bins, the last counts >= 255 */
#define RA_HIST_FAIL    2    /* failCount (failCountSum, W:348), variant W/B only: 256 bins, the last counts >= 255 */

/* One parameter point == one iteration of the reference's nUE sweep (W:221). */
typedef struct ra_params {
    int variant;            /* RA_VARIANT_*                                                  */
    int nUE;                /* W:226                                                         */
    int distribution;       /* 1 = Uniform over 60 s, anything else = Beta(3,4) over 10 s    */
                            /*   (W:88,208,241; note B encodes 0/1, B:57,90)                 */
    int nPreamble;          /* W:71  -p                                                      */
    int backoffIndicator;   /* W:72  -b                                                      */
    int nGrantUL;           /* W:73  -g   (strict '<' after increment, W:639-641)            */
    int maxRarWindow;       /* W:76  = RAR window + 1   (-rc N stores N+1, W:128)            */
    int maxMsg2TxCount;     /* W:77  = max retx - 1     (-mrc N stores N-1, W:134)           */
    int accessTime;         /* W:78  -s                                                      */
    int maxTimeMs;          /* 0 = reference horizon (60000 Uniform / 10000 Beta, W:243,254) */
    float cellRadius;       /* W:80  -c   (geometry side outputs only)                       */
    float hBS;              /* W:81  -bs  (parsed, passed, unused by the reference)          */
    float hUT;              /* W:82  -ut  (idem)                                             */
    int geometry;           /* 1 = W: two draws per arriving UE before the first preamble    */
                            /*     draw (W:393-394); 0 = B: none (B:137-145)                 */
    unsigned long long seed;/* Philox key of the draw tape (replaces srand(seed), W:219)     */
} ra_params;

/* Per-replication counters (integers only; the host derives the reference's floats). */
typedef struct ra_stats {
    int simTimeMs;               /* `time` after the loop: break value or maxTime (W:267,332) */
    int nSuccess;                /* successUEs, W:330,720-728                                 */
    long long preambleTxSum;     /* sum of preambleTxCounter over msg4Flag==1, W:347           */
    long long delaySum;          /* sum of timer over msg4Flag==1, W:346 (float in the ref.)   */
    long long failCountSum;      /* sum of failCount over msg4Flag==1, W:348                   */
    long long continueFailed;    /* continueFaliedUEs, W:499,682 (U0: drops, raFailed = -1, U0:181-184)  */
    long long finalSuccess;      /* finalSuccessUEs, W:676                                     */
    long long collisionPreambles;/* W:62,650  (+= group size per collided scan)                */
    long long totalPreambleTxop; /* W:63,625,652                                               */
    long long collisionScans;    /* B:41,349  (B counts one per collided scan)                 */
    long long totalScans;        /* B:42,334,351 (one per scan)                                */
    long long updates;           /* nUE * ceil(simTimeMs / accessTime): the throughput unit    */
    long long recordMoves;       /* engine bookkeeping (variant W): 16-byte calendar records read at their event time =
                                    records written earlier; x 32 B = the state bytes the replication really moved  */
} ra_stats;

/* Engine options (all zero = defaults).
 * Cross-check switches read from the environment at create / run time, never needed in normal use:
 *   RACH_BLOCK=small|big|huge  force one of the three block shapes of the W/B step kernel (128 x 9 / 256 x 5 / 512 x 2 per SM)
 *   RACH_FIXED=0               W/B: the runtime point view even when every point is in the reference's default family
 *   RACH_U0=serial             variant U0: the one-lane serial step in every ms instead of the warp step */
typedef struct ra_options {
    int repOffset;      /* tape replication id of local rep 0 (multi-process sharding)        */
    int dumpUEs;        /* 1 = keep the 16-int per-UE final record of every replication       */
    int ctasPerSM;      /* 0 = engine default; resident CTAs per SM of the step kernel        */
    int phaseTimers;    /* 1 = collect per-phase cycle counters (ra_sim_phase_cycles): a separate kernel instantiation
                           (costs ~2 %), W/B dynamics only, not together with dumpUEs (RA_E_INVAL) */
    int histograms;     /* 1 = accumulate the RA_HIST_* histograms of every point on the device (ra_sim_histogram);
                           combines with dumpUEs and phaseTimers */
    int reserved[3];
} ra_options;

typedef struct ra_sim ra_sim;

/* points[nPoints] x repsPerPoint replications, sharded over devices[nDevices]
 * (devices == NULL: device 0).  Returns NULL on failure; ra_last_create_error() says why. */
ra_sim*     ra_sim_create(const ra_params* points, int nPoints, int repsPerPoint,
                          const int* devices, int nDevices);
ra_sim*     ra_sim_create_ex(const ra_params* points, int nPoints, int repsPerPoint,
                             const int* devices, int nDevices, const ra_options* opt);
const char* ra_last_create_error(void);
int         ra_last_create_code(void);               /* RA_E_* of the last failed create on this thread, RA_OK otherwise */

int         ra_sim_run(ra_sim* sim);                 /* blocking; may be called repeatedly */
/* Per-UE logs at scale (saveResult W:797-825 for many replications): like ra_sim_run, and while the kernel is still
 * running every finished replication is copied out (one asynchronous copy per replication on a second stream, pinned
 * staging) and handed to `cb` -- in completion order, from the calling thread; `rows` (nUE x RA_DUMP_FIELDS ints, layout
 * of ra_sim_dump_ues) and `st` are valid during the call only.  The step kernel never waits for the host.
 * Needs ra_options.dumpUEs = 1.  ra_sim_stats / ra_sim_dump_ues work afterwards as after ra_sim_run. */
typedef void (*ra_dump_cb)(void* user, int point, int rep, const ra_stats* st, const int* rows);
int         ra_sim_run_stream(ra_sim* sim, ra_dump_cb cb, void* user);
int         ra_sim_stats(ra_sim* sim, int point, int rep, ra_stats* out);
int         ra_sim_stats_all(ra_sim* sim, ra_stats* out /* [nPoints*repsPerPoint] */);
/* out[nUE * RA_DUMP_FIELDS]: idx-major, fields in saveResult order (W:812-819) after idx:
 *  0 timer 1 active 2 txTime 3 firstTxTime 4 secondTxTime 5 nowBackoff 6 preamble
 *  7 preambleChange 8 rarWindow 9 maxRarCounter 10 preambleTxCounter 11 msg2Flag
 *  12 connectionRequest 13 msg4Flag 14 failCount 15 sector (W:398-410, -1 if geometry off) */
int         ra_sim_dump_ues(ra_sim* sim, int point, int rep, int* out);
/* out[nUE * 6] floats: angle, xCoordinate, yCoordinate, distance, channelGain, (float)sector
 * (W:396-415).  Requires geometry=1. */
int         ra_sim_geometry(ra_sim* sim, int point, int rep, float* out);
/* out[ra_hist_bins(point, kind)]: the RA_HIST_* histogram of one point over the UEs that finished (msg4Flag == 1,
 * W:337-348), summed over the point's replications and over all devices of the handle.  Filled by ra_sim_run and
 * ra_sim_run_stream on the GPU; the sums of a bin times its value give delaySum / preambleTxSum / failCountSum of
 * ra_sim_stats (for TX and FAIL while the last bin is empty).  Needs ra_options.histograms = 1 and a run (RA_E_STATE);
 * RA_E_INVAL for a bad point or kind, and for RA_HIST_FAIL on variant N or U0 (no failCount there). */
int         ra_sim_histogram(ra_sim* sim, int point, int kind, unsigned long long* out);
/* variant N with dumpUEs: out[nUE] doubles = channelGain (N:183-191), 0 for UEs that never arrived;
 * ra_sim_dump_ues then writes: timer active txTime firstTxTime secondTxTime nowBackoff preamble sector
 * rarWindow msg1ReTx nTxPreamble msg2 msg3Wait RA msg3Faile RaFailed (saveResultLogs order, N:577-592) */
int         ra_sim_gains(ra_sim* sim, int point, int rep, double* out);
double      ra_sim_kernel_ms(const ra_sim* sim);     /* device time of the last run (max over devices) */
long long   ra_sim_gpu_launches(const ra_sim* sim);  /* kernels launched by the last run */
/* profiling aid: cycles spent per engine phase by thread 0 of every block, summed (out[10]) */
int         ra_sim_phase_cycles(ra_sim* sim, unsigned long long* out10);
void        ra_sim_destroy(ra_sim* sim);
const char* ra_sim_last_error(const ra_sim* sim);

/* Host-side helpers (no device needed). */
int         ra_params_default(ra_params* p, int variant);   /* W:69-88 defaults */
int         ra_horizon_ms(const ra_params* p);              /* W:243,254 */
/* bins of the RA_HIST_* histogram `kind` of point p: horizon + 7 for RA_HIST_DELAY, 256 for RA_HIST_TX and (variant W
 * only) RA_HIST_FAIL; RA_E_INVAL otherwise */
int         ra_hist_bins(const ra_params* p, int kind);
/* the parameter checks of ra_sim_create without a device: RA_OK, or RA_E_INVAL with the reason in err[errLen]
 * (the reference checks only "> 0" style ranges in main, W:94-158; the engine adds its packing limits: nUE <= 2^24,
 * nPreamble <= 256, backoffIndicator <= 4096, RAR window <= 255, max retx <= 256, horizon <= 65535 ms, and
 * ring x nUE < 2^32 calendar records per replication, ring = next power of two >= backoffIndicator + max(accessTime, 5)
 * + maxRarWindow) */
int         ra_params_validate(const ra_params* p, char* err, int errLen);
/* arrivals[ms] for ms in [0, horizon): UEs that become active in that ms (after the clamp of
 * W:290-292), 0 for ms % accessTime != 0.  Returns the ms at which all nUE have arrived, or -1. */
int         ra_arrival_schedule(const ra_params* p, int* arrivals, int horizon);
const char* ra_version(void);

#ifdef __cplusplus
}
#endif
#endif /* RACH_GPU_H */
