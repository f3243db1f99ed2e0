/*
 * rach_sim.c -- host program: the command line and report formats of the reference's only CLI
 * (RandomAccessWithNOMA.c), with the (seed, nUE) loop body replaced by librach_gpu.
 *
 *   flags accepted by the reference parser (W:93-158):  -t -d -p -b -g -rc -mrc -s -c -bs -ut
 *     (and their long forms); same validation messages, same exit status (255), same help text
 *     on an unknown flag (W:159-204).  The README spells some of them -r -m -u; those are
 *     accepted here as aliases (a superset; the reference itself rejects them).
 *   added:  --format w|b|n  report layout: w (default) RandomAccessWithNOMA.c:354-366,731-825;
 *                           b = RandomAccessSimulatorBeta.c:200-209,432-514 (54 grants by default, no
 *                               activation draws, its own counters and file names, a "Latency" line / 6th
 *                               file line that carries the kernel time of the whole launch);
 *                           n = NOMA.c:598-635,712-716 (variant N: "nUE nSuccess ratio meanTx meanDelay",
 *                               appended to TestResults/Sector_<nUE>_Result.txt, "Done" after each seed)
 *                           u = RandomAccessSimulator.c:69-70,141-143,277-345 (variant U0: 64 preambles, no seed loop,
 *                               the two "Result" banners, 2_SimulationResults/2_Exclude_msg2_failures_UE<nUE>_*;
 *                               its collision / tx-opportunity counters are globals that the file never resets,
 *                               so they accumulate over the sweep -- reproduced; U0:321 does not compile as
 *                               shipped: read as a plain assignment to the parameter)
 *           --nue a,b,c  (points; default the reference sweep 10000..100000 step 10000, W:221)
 *           --no-logs    (skip the per-UE *_Logs.txt, W:797-825)
 *           --outdir DIR (default "."), --device N, --seed64 S (tape key, default 0)
 *           --devices a,b,c  shard the (point, seed) list over several GPUs of the box (ra_sim_create devices[])
 *           --binlog     per-UE logs as compact binary instead of text: <seed>_<P>_UE<nUE>_Logs.bin = 32-byte header
 *                        ("RAUELOG1", int32 nUE, nFields = 14, seed, nPreamble, 0, 0) + nUE x 14 int32, the fields
 *                        saveResult prints after Idx (W:812-819), 56 B per UE instead of ~240 B of text
 *           --hist       per point, <P>_<nUE>_Distributions.csv in the result directory: "metric,value,count", one row per
 *                        non-zero bin of the histograms of the successful UEs, summed over the -t seeds (built on the GPU,
 *                        ra_sim_histogram): delay_ms (timer, W:346), preamble_tx (preambleTxCounter, W:347; 255 = 255 and
 *                        above) and, for --format w only, fail_count (failCount, W:348; 255 = 255 and above)
 *   The per-UE logs are written WHILE the kernel runs (ra_sim_run_stream): each finished replication is copied out
 *   asynchronously and written by the host thread; the report itself is printed afterwards in the reference's order.
 *
 * Differences that cannot be hidden: randomness is the Philox draw tape keyed by
 * (seed64, replication = the reference's randomSeed, UE, ms), not libc rand(); the whole sweep
 * is ONE library call (all points x seeds in one launch), results are printed afterwards in the
 * reference's order.
 */
#include <errno.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>

#include "rach_gpu.h"

static void die(const char* msg) { printf("%s", msg); exit(-1); }

static void usage_and_exit(void) {
    static const char* rows[][4] = {
        {"--times         -t", "Simulation times (int)", "Simulation count must be greater than zero.", "Default 1"},
        {"--distribution  -d", "Traffic model (1 or 2)", NULL, NULL},
        {"--preambles     -p", "Number of preambles (int)", "Number of preamble must be greater than zero.", "Default 54"},
        {"--backoff       -b", "Backoff indicator (int)", "Backoff indicator must be greater than zero.", "Default 20"},
        {"--grant         -g", "The number of Up Link Grant per RAR (int)", "The number of Up Link Grant per RAR must be greater than zero.", "Default 12"},
        {"--rarCount      -r", "RAR window size (int)", "The maximum RAR window size must be greater than zero.", "Default 5"},
        {"--maxRar        -m", "Maximum retransmission (int)", "Maximum retransmissions must be greater than zero.", "Default 10"},
        {"--subframe      -s", "Subframe units (int)", "The size of the subframe must be at least 5. (float)", "Default 5"},
        {"--cell          -c", "Cell radius Size", "The radius of the cell is entered in diameter units and must be greater than 400m.", "Default 400.0"},
        {"--hbs           -b", "Height of BS from ground (float)", "The height of the BS must be between 10m and 20m.", "Default 10.0"},
        {"--hut           -u", "Height of UE from ground (float)", "The height of the UE must be between 1.5m and 22.5m.", "Default 1.8"},
    };
    const char* pad = "                     ";
    for (size_t i = 0; i < sizeof rows / sizeof rows[0]; ++i) {
        printf("%s : %s\n", rows[i][0], rows[i][1]);
        if (i == 1) {           /* W:164-166 */
            printf("%s1: traffic model 1 (Uniform distribution)\n", pad);
            printf("%s2: traffic model 2 (Beta distribution)\n\n", pad);
            continue;
        }
        printf("%s%s\n", pad, rows[i][2]);
        printf("%s%s\n\n", pad, rows[i][3]);
    }
    exit(-1);
}

/* --hist: <dir>/<P>_<nUE>_Distributions.csv for every point of the handle */
static int write_distributions(ra_sim* sim, const ra_params* pts, int nNue, const char* dir, int withFail) {
    static const char* metric[3] = {"delay_ms", "preamble_tx", "fail_count"};
    const int kinds[3] = {RA_HIST_DELAY, RA_HIST_TX, RA_HIST_FAIL};
    for (int k = 0; k < nNue; ++k) {
        char path[800];
        snprintf(path, sizeof path, "%s/%d_%d_Distributions.csv", dir, pts[k].nPreamble, pts[k].nUE);
        FILE* fp = fopen(path, "w");
        if (!fp) { fprintf(stderr, "rach_sim: cannot write %s: %s\n", path, strerror(errno)); return 2; }
        fprintf(fp, "metric,value,count\n");
        for (int m = 0; m < (withFail ? 3 : 2); ++m) {
            const int n = ra_hist_bins(&pts[k], kinds[m]);
            unsigned long long* h = (unsigned long long*)malloc(sizeof *h * (size_t)n);
            if (ra_sim_histogram(sim, k, kinds[m], h) != RA_OK) {
                fprintf(stderr, "rach_sim: %s\n", ra_sim_last_error(sim)); free(h); fclose(fp); return 2;
            }
            for (int v = 0; v < n; ++v) if (h[v]) fprintf(fp, "%s,%d,%llu\n", metric[m], v, h[v]);
            free(h);
        }
        fclose(fp);
    }
    return 0;
}

/* --format u: the report of RandomAccessSimulator.c (U0:42-143 main, U0:277-345 writers), one replication per point */
static int report_u0(const ra_params* base, const int* nueList, int nNue, const char* outdir, int writeLogs, int device,
                     int preambleSet, int backoffSet, int hist) {
    ra_params* pts = (ra_params*)calloc((size_t)nNue, sizeof *pts);
    for (int k = 0; k < nNue; ++k) {
        ra_params_default(&pts[k], RA_VARIANT_U0);                    /* U0:48-59: 64 preambles, BI 20, 60 s */
        if (preambleSet) pts[k].nPreamble = base->nPreamble;
        if (backoffSet) pts[k].backoffIndicator = base->backoffIndicator;
        pts[k].seed = base->seed; pts[k].nUE = nueList[k];
    }
    char dir[600];
    snprintf(dir, sizeof dir, "%s/2_SimulationResults", outdir);
    mkdir(outdir, 0755);
    mkdir(dir, 0755);
    ra_options opt; memset(&opt, 0, sizeof opt);
    opt.dumpUEs = 1;                                                  /* the delay sum is a float accumulation in UE order */
    opt.histograms = hist;
    ra_sim* sim = ra_sim_create_ex(pts, nNue, 1, &device, 1, &opt);
    if (!sim) { fprintf(stderr, "rach_sim: %s\n", ra_last_create_error()); return 2; }
    if (ra_sim_run(sim) != RA_OK) { fprintf(stderr, "rach_sim: %s\n", ra_sim_last_error(sim)); return 2; }
    int collisionPreambles = 0, totalPreambleTxop = 0;                /* U0:36-37: globals, never reset */
    for (int k = 0; k < nNue; ++k) {
        const int nUE = pts[k].nUE, maxTime = 60000, accessTime = 5;
        int nAccessUE = ceil((float)nUE * (float)accessTime * 1.0 / (float)maxTime);   /* U0:60 */
        if (nAccessUE == 0) nAccessUE = 1;
        printf("-------- %05d Result ---------\n", nUE);                               /* U0:69-70 */
        printf("%d\n", nAccessUE);
        ra_stats st;
        if (ra_sim_stats(sim, k, 0, &st) != RA_OK) { fprintf(stderr, "rach_sim: %s\n", ra_sim_last_error(sim)); return 2; }
        int* ue = (int*)malloc(sizeof(int) * (size_t)nUE * RA_DUMP_FIELDS);
        if (ra_sim_dump_ues(sim, k, 0, ue) != RA_OK) { fprintf(stderr, "rach_sim: %s\n", ra_sim_last_error(sim)); return 2; }
        const int time = st.simTimeMs;
        const int lastMs = time < maxTime ? time : maxTime - 1;
        int activeCheck = 0;
        for (int t = 1; t <= lastMs; t += accessTime) {                                /* U0:77-81 */
            if (activeCheck >= nUE) activeCheck = nUE; else activeCheck += nAccessUE;
        }
        float averageDelay = 0; int failedUEs = 0, preambleTxCount = 0;                /* U0:127-139 */
        for (int i = 0; i < nUE; ++i) {
            const int* r = ue + (size_t)i * RA_DUMP_FIELDS;
            if (r[10] == 0) failedUEs++;
            else { averageDelay += (float)r[0]; preambleTxCount += r[7]; }
        }
        const int nSuccessUE = st.nSuccess;
        collisionPreambles += (int)st.collisionPreambles; totalPreambleTxop += (int)st.totalPreambleTxop;
        printf("-------- %05d Result ---------\n", activeCheck);                       /* U0:141 */
        char path[800], buf[1000];
        snprintf(path, sizeof path, "%s/2_Exclude_msg2_failures_UE%05d_Results.txt", dir, nUE);   /* U0:282 */
        FILE* fp = fopen(path, "w+");
        if (!fp) { fprintf(stderr, "rach_sim: cannot write %s: %s\n", path, strerror(errno)); return 2; }
#define U0_LINE(...) do { snprintf(buf, sizeof buf, __VA_ARGS__); fputs(buf, stdout); fputs(buf, fp); } while (0)
        U0_LINE("Number of UEs: %d\n", nUE);
        U0_LINE("Total simulation time: %dms\n", time);
        U0_LINE("Number of succeed UEs: %d\n", nSuccessUE);
        float ratioSuccess = (float)nSuccessUE / (float)nUE;
        U0_LINE("Success ratio: %lf\n", ratioSuccess);
        U0_LINE("Number of failed UEs: %d\n", failedUEs);
        float ratioFailed = (float)failedUEs / (float)nUE;
        U0_LINE("Fail probability: %lf\n", ratioFailed);
        float nCollisionPreambles = (float)collisionPreambles / (float)preambleTxCount;
        U0_LINE("Number of collision preambles: %lf\n", nCollisionPreambles);
        float averagePreambleTx = (float)totalPreambleTxop / (float)nSuccessUE;
        U0_LINE("Average preamble tx count: %lf\n", averagePreambleTx);
        averageDelay = averageDelay / (float)nSuccessUE;                               /* U0:321, see the header */
        U0_LINE("Average delay: %lfms\n", averageDelay);
#undef U0_LINE
        fclose(fp);
        if (writeLogs) {                                                               /* U0:328-345 */
            snprintf(path, sizeof path, "%s/2_Exclude_msg2_failures_UE%05d_Logs.txt", dir, nUE);
            fp = fopen(path, "w+");
            if (!fp) { fprintf(stderr, "rach_sim: cannot write %s: %s\n", path, strerror(errno)); return 2; }
            for (int i = 0; i < nUE; ++i) {
                const int* r = ue + (size_t)i * RA_DUMP_FIELDS;
                fprintf(fp, "Idx: %d | Timer: %d | Active: %d | txTime: %d | Preamble: %d | Preamble change: %d | RAR window: %d | "
                            "Max RAR: %d | Preamble reTx: %d | MSG 2 Flag: %d | ConnectRequest: %d | MSG 4 Flag: %d\n",
                        i, r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[7], r[8], r[9], r[10]);
            }
            fclose(fp);
        }
        free(ue);
    }
    if (hist && write_distributions(sim, pts, nNue, dir, 0) != 0) return 2;
    fprintf(stderr, "rach_sim: %d points, kernel %.1f ms (%s)\n", nNue, ra_sim_kernel_ms(sim), ra_version());
    ra_sim_destroy(sim);
    free(pts);
    return 0;
}

/* ---- per-UE logs, written from the streaming callback (completion order) ------------------------------------- */
typedef struct {
    const ra_params* pts; int times; const char* dir; char format; int uniform, binlog;
    float* totalDelay;          /* [point * times + seed]: float accumulation in UE order, W:338,346 */
    int failed;
} log_ctx;

static void log_cb(void* user, int point, int seed, const ra_stats* st, const int* ue) {
    log_ctx* c = (log_ctx*)user;
    (void)st;
    const int nUE = c->pts[point].nUE, nPreamble = c->pts[point].nPreamble;
    float totalDelay = 0;
    for (int i = 0; i < nUE; ++i) if (ue[i * RA_DUMP_FIELDS + 13] == 1) totalDelay += (float)ue[i * RA_DUMP_FIELDS + 0];
    c->totalDelay[(size_t)point * c->times + seed] = totalDelay;
    if (c->format == 'n') return;
    char path[800];
    if (c->binlog) {
        snprintf(path, sizeof path, "%s/%d_%d_UE%05d_Logs.bin", c->dir, seed, nPreamble, nUE);
        FILE* fp = fopen(path, "wb");
        if (!fp) { fprintf(stderr, "rach_sim: cannot write %s: %s\n", path, strerror(errno)); c->failed = 1; return; }
        int hdr[8] = {0, 0, nUE, 14, seed, nPreamble, 0, 0};
        memcpy(hdr, "RAUELOG1", 8);
        fwrite(hdr, sizeof hdr, 1, fp);
        int* row = (int*)malloc(sizeof(int) * 14 * 4096);
        for (int i0 = 0; i0 < nUE; i0 += 4096) {
            const int n = nUE - i0 < 4096 ? nUE - i0 : 4096;
            for (int i = 0; i < n; ++i) memcpy(row + i * 14, ue + (size_t)(i0 + i) * RA_DUMP_FIELDS, sizeof(int) * 14);
            fwrite(row, sizeof(int) * 14, (size_t)n, fp);
        }
        free(row);
        fclose(fp);
        return;
    }
    if (c->format == 'b' && c->uniform) snprintf(path, sizeof path, "%s/%d_Exclude_msg2_failures_UE%05d_Logs.txt", c->dir, nPreamble, nUE);   /* B:488 */
    else snprintf(path, sizeof path, "%s/%d_%d_UE%05d_Logs.txt", c->dir, seed, nPreamble, nUE);      /* W:797-825 */
    FILE* fp = fopen(path, "w+");
    if (!fp) { fprintf(stderr, "rach_sim: cannot write %s: %s\n", path, strerror(errno)); c->failed = 1; return; }
    static const char* names[15] = {"Idx", "Timer", "Active", "txTime", "FirstTxTime", "SecondTxTime", "NowBackoff",
        "Preamble", "Preamble change", "RAR window", "Max RAR", "Preamble reTx", "MSG 2 Flag", "ConnectRequest", "MSG 4 Flag"};
    for (int i = 0; i < nUE; ++i) {
        const int* r = ue + (size_t)i * RA_DUMP_FIELDS;
        fprintf(fp, "%s: %d", names[0], i);
        for (int f = 0; f < 14; ++f) fprintf(fp, " | %s: %d", names[f + 1], r[f]);
        fputc('\n', fp);
    }
    fclose(fp);
}

static int is_flag(const char* a, const char* l, const char* s, const char* alias) {
    return strcmp(a, l) == 0 || strcmp(a, s) == 0 || (alias && strcmp(a, alias) == 0);
}

int main(int argc, char* argv[]) {
    ra_params base;
    ra_params_default(&base, RA_VARIANT_W);
    int times = 1, writeLogs = 1, device = 0, grantSet = 0, preambleSet = 0, backoffSet = 0, binlog = 0, hist = 0;
    int devList[64], nDev = 0;
    char format = 'w';
    const char* outdir = ".";
    int nueList[64], nNue = 0;
    unsigned long long seed64 = 0;

    for (int i = 1; i < argc; i += 2) {
        const char* a = argv[i];
        if (strcmp(a, "--no-logs") == 0) { writeLogs = 0; i -= 1; continue; }
        if (strcmp(a, "--binlog") == 0) { binlog = 1; i -= 1; continue; }
        if (strcmp(a, "--hist") == 0) { hist = 1; i -= 1; continue; }
        const char* v = (i + 1 < argc) ? argv[i + 1] : "";      /* the reference dereferences argv[i+1] blindly (W:94) */
        if (is_flag(a, "--times", "-t", NULL)) {
            if (atoi(v) < 1) die("Simulation count must be greater than zero.");
            times = atoi(v);
        } else if (is_flag(a, "--distribution", "-d", NULL)) {
            if (atoi(v) != 1 && atoi(v) != 0) die("Traffic model just choose 1 or 2");       /* W:100-102 */
            base.distribution = atoi(v);
        } else if (is_flag(a, "--preambles", "-p", NULL)) {
            if (atoi(v) < 1) die("Number of preamble must be greater than zero.");
            base.nPreamble = atoi(v); preambleSet = 1;
        } else if (is_flag(a, "--backoff", "-b", NULL)) {
            if (atoi(v) < 1) die("Backoff indicator must be greater than zero.");
            base.backoffIndicator = atoi(v); backoffSet = 1;
        } else if (is_flag(a, "--grant", "-g", NULL)) {
            if (atoi(v) < 1) die("The number of Up Link Grant per RAR must be greater than zero.");
            base.nGrantUL = atoi(v); grantSet = 1;
        } else if (is_flag(a, "--rarCount", "-rc", "-r")) {
            if (atoi(v) < 1) die("The maximum RAR window size must be greater than zero.");
            base.maxRarWindow = atoi(v) + 1;                                                  /* W:128 */
        } else if (is_flag(a, "--maxRar", "-mrc", "-m")) {
            if (atoi(v) < 1) die("Maximum retransmissions must be greater than zero.");
            base.maxMsg2TxCount = atoi(v) - 1;                                                /* W:134 */
        } else if (is_flag(a, "--subframe", "-s", NULL)) {
            if (atoi(v) < 5) die("The size of the subframe must be at least 5.");
            base.accessTime = atoi(v);
        } else if (is_flag(a, "--cell", "-c", NULL)) {
            if (atof(v) < 400.0) die("The radius of the cell is entered in diameter units and must be greater than 400m.");
            base.cellRadius = atof(v);
        } else if (is_flag(a, "--hbs", "-bs", NULL)) {
            if (atof(v) < 10.0 || atof(v) > 20.0) die("The height of the BS must be between 10m and 20m.");
            base.hBS = atof(v);
        } else if (is_flag(a, "--hut", "-ut", "-u")) {
            if (atof(v) < 1.5 || atof(v) > 22.5) die("The height of the UE must be between 1.5m and 22.5m.");
            base.hUT = atof(v);
        } else if (strcmp(a, "--nue") == 0) {
            char* dup = strdup(v);
            for (char* tok = strtok(dup, ","); tok && nNue < 64; tok = strtok(NULL, ",")) nueList[nNue++] = atoi(tok);
            free(dup);
        } else if (strcmp(a, "--format") == 0) { format = v[0];
        } else if (strcmp(a, "--outdir") == 0) { outdir = v;
        } else if (strcmp(a, "--device") == 0) { device = atoi(v);
        } else if (strcmp(a, "--devices") == 0) {
            char* dup = strdup(v);
            for (char* tok = strtok(dup, ","); tok && nDev < 64; tok = strtok(NULL, ",")) devList[nDev++] = atoi(tok);
            free(dup);
        } else if (strcmp(a, "--seed64") == 0) { seed64 = strtoull(v, NULL, 0);
        } else usage_and_exit();
    }
    if (nNue == 0) for (int n = 10000; n <= 100000; n += 10000) nueList[nNue++] = n;   /* W:221 */
    if (nDev == 0) devList[nDev++] = device; else device = devList[0];
    base.seed = seed64;
    if (format != 'w' && format != 'b' && format != 'n' && format != 'u') usage_and_exit();
    if (format == 'u') return report_u0(&base, nueList, nNue, outdir, writeLogs, device, preambleSet, backoffSet, hist);
    if (format == 'b') { base.geometry = 0; if (!grantSet) base.nGrantUL = 54; }         /* B:49, B:137-145 */
    if (format == 'n') {                                                                 /* NOMA.c:41-57 */
        ra_params n; ra_params_default(&n, RA_VARIANT_N);
        n.nPreamble = base.nPreamble; n.backoffIndicator = base.backoffIndicator; n.accessTime = base.accessTime;
        if (grantSet) n.nGrantUL = base.nGrantUL;
        n.seed = seed64; base = n; writeLogs = 0;
    }

    const int uniform = base.distribution == 1;
    if (format != 'n') printf(uniform ? "Traffic model: Uniform\n\n" : "Traffic model: Beta\n\n");   /* W:208-213, B:59-64 */

    char dir[600];
    snprintf(dir, sizeof dir, "%s/%s", outdir, format == 'n' ? "TestResults" :
             format == 'b' ? (uniform ? "BasicUniformSimulationResults" : "BasicBetaSimulationResults")
                           : (uniform ? "NomaUniformResults" : "NomaBetaResults"));
    mkdir(outdir, 0755);
    mkdir(dir, 0755);                                                                    /* W:67-68; README.md:6-10 for B */

    ra_params* pts = (ra_params*)calloc((size_t)nNue, sizeof *pts);
    for (int k = 0; k < nNue; ++k) { pts[k] = base; pts[k].nUE = nueList[k]; }
    ra_options opt; memset(&opt, 0, sizeof opt);
    opt.dumpUEs = writeLogs;
    opt.histograms = hist;
    ra_sim* sim = ra_sim_create_ex(pts, nNue, times, devList, nDev, &opt);
    if (!sim) { fprintf(stderr, "rach_sim: %s\n", ra_last_create_error()); return 2; }
    log_ctx lc; memset(&lc, 0, sizeof lc);
    lc.pts = pts; lc.times = times; lc.dir = dir; lc.format = format; lc.uniform = uniform; lc.binlog = binlog;
    lc.totalDelay = (float*)calloc((size_t)nNue * (size_t)times, sizeof(float));
    /* with logs: every replication is copied out and written while the kernel is still running */
    const int rrc = writeLogs ? ra_sim_run_stream(sim, log_cb, &lc) : ra_sim_run(sim);
    if (rrc != RA_OK) { fprintf(stderr, "rach_sim: %s\n", ra_sim_last_error(sim)); return 2; }
    if (lc.failed) return 2;

    for (int seed = 0; seed < times; ++seed) {                   /* W:216 */
        for (int k = 0; k < nNue; ++k) {                         /* W:221 */
            const ra_params* p = &pts[k];
            const int nUE = p->nUE, nPreamble = p->nPreamble;
            ra_stats st;
            if (ra_sim_stats(sim, k, seed, &st) != RA_OK) { fprintf(stderr, "rach_sim: %s\n", ra_sim_last_error(sim)); return 2; }
            const int horizon = ra_horizon_ms(p);
            int* arr = (int*)malloc(sizeof(int) * (size_t)horizon);
            ra_arrival_schedule(p, arr, horizon);
            const int lastMs = st.simTimeMs < horizon ? st.simTimeMs : horizon - 1;
            int activeCheck = 0;
            for (int t = 0; t <= lastMs; ++t) activeCheck += arr[t];
            const int nAccessUE = arr[0];
            free(arr);

            /* float accumulation in UE order, W:338,346 (from the streamed rows); without logs the integer sum, which is
             * identical while it stays below 2^24 */
            const float totalDelay = writeLogs ? lc.totalDelay[(size_t)k * times + seed] : (float)st.delaySum;
            if (format == 'n') {                                 /* NOMA.c:598-635 */
                char path[800];
                snprintf(path, sizeof path, "%s/Sector_%d_Result.txt", dir, nUE);
                FILE* fp = fopen(path, "a");
                if (!fp) { fprintf(stderr, "rach_sim: cannot write %s: %s\n", path, strerror(errno)); return 2; }
                char line[256];
                snprintf(line, sizeof line, "%d %d %lf %lf %lf\n", nUE, st.nSuccess, ((float)st.nSuccess / (float)nUE) * 100.0,
                         ((float)(int)st.preambleTxSum / (float)st.nSuccess), ((float)(int)st.delaySum / (float)st.nSuccess));
                fputs(line, stdout); fputs(line, fp);
                fclose(fp);
                if (k == nNue - 1) printf("Done\n");             /* NOMA.c:716 */
                continue;
            }
            const int nSuccessUE = st.nSuccess, failedUEs = nUE - nSuccessUE;
            const int preambleTxCount = (int)st.preambleTxSum;
            const int continueFailed = (int)st.continueFailed, finalSuccess = (int)st.finalSuccess;
            (void)failedUEs;

            printf("-------- %05d Result ---------\n", activeCheck);                     /* W:354 */
            if (uniform) printf("Number of RA try UEs per Subframe: %d\n", nAccessUE);   /* W:355-357 */
            const double latency = ra_sim_kernel_ms(sim) / 1e3;   /* B:205-206: cumulative clock(); here the whole launch */
            if (format == 'b') printf("Latency: %lf\n", latency);
            else printf("Fail Counts: %d\n", (int)st.failCountSum);                      /* W:361 */

            /* W:735-739 */
            float ratioSuccess = (float)nSuccessUE / (float)nUE * 100.0;
            float nCollisionPreambles = (float)(format == 'b' ? st.collisionScans : st.collisionPreambles) / ((float)nUE * (float)nPreamble);   /* B:349 vs W:650 */
            float averagePreambleTx = (float)preambleTxCount / (float)nSuccessUE;
            float averageDelay = totalDelay / (float)nSuccessUE;
            printf("Number of UEs: %d\n", nUE);
            printf("Total simulation time: %dms\n", st.simTimeMs);
            printf("Success ratio: %.2lf\n", ratioSuccess);
            printf("Number of succeed UEs: %d\n", nSuccessUE);
            if (format == 'w') printf("Number of falied UEs: %d\n", continueFailed);
            printf("Number of collision preambles: %.6lf\n", nCollisionPreambles);
            printf("Average preamble tx count: %.2lf\n", averagePreambleTx);
            printf("Average delay: %.2lf\n", averageDelay);

            char path[800];
            snprintf(path, sizeof path, "%s/%d_%d_%d_Results.txt", dir, seed, nPreamble, nUE);   /* W:754-758 */
            FILE* fp = fopen(path, "w+");
            if (!fp) { fprintf(stderr, "rach_sim: cannot write %s: %s\n", path, strerror(errno)); return 2; }
            fprintf(fp, "%d\n%.2lf\n%d\n%.2lf\n%.2lf\n", nUE, ratioSuccess, nSuccessUE, averagePreambleTx, averageDelay);
            if (format == 'b') fprintf(fp, "%lf", latency);                              /* B:481 */
            else {
                fprintf(fp, "Number of total preamble tx: %d\n", preambleTxCount);
                fprintf(fp, "Finally Falied: %d\n", continueFailed);
                fprintf(fp, "Finally Success: %lf\n", (float)finalSuccess / (float)(continueFailed + finalSuccess));
            }
            fclose(fp);

        }
    }
    if (hist && write_distributions(sim, pts, nNue, dir, format == 'w') != 0) return 2;   /* B has no failCount */
    fprintf(stderr, "rach_sim: %d points x %d seeds on %d device(s), kernel %.1f ms (%s)\n", nNue, times, nDev, ra_sim_kernel_ms(sim), ra_version());
    free(lc.totalDelay);
    ra_sim_destroy(sim);
    free(pts);
    return 0;
}
