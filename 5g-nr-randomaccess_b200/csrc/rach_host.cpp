/*
 * rach_host.cpp -- host-side logic of librach_gpu that needs no device: parameter defaults
 * and validation, the horizon, and the deterministic arrival schedule.
 *
 * Reference: RandomAccessWithNOMA.c:69-88 (defaults), :241-255 (horizon, nAccessUE),
 * :276-292 (arrival gate), :844-847 (beta_dist).  The float/double mix of the reference's
 * expressions is kept verbatim because ceil() of a float quotient decides integer counts.
 */
#include <math.h>
#include <stdio.h>
#include <string.h>

#include "rach_gpu.h"
#include "rach_host.h"
#include "rach_core.cuh"

#define betaF 0.0165

/* W:844-847.  The reference is C: pow() takes doubles whatever the argument types.  This file is C++,
 * where pow(float, float) would select the float overload and change ceil() of the quotient below for
 * some nUE (caught at nUE = 300000) -- hence the explicit promotions. */
static float ra_beta_dist(float a, float b, float x) {
    float betaValue = (1 / betaF) * (pow((double)x, (double)(a - 1))) * (pow((double)(1 - x), (double)(b - 1)));
    return betaValue;
}

extern "C" int ra_params_default(ra_params* p, int variant) {
    if (!p) return RA_E_INVAL;
    memset(p, 0, sizeof(*p));
    p->variant = variant;
    p->nUE = 10000;
    p->distribution = 2;            /* W:88 */
    p->nPreamble = 54;              /* W:71 */
    p->backoffIndicator = 20;       /* W:72 */
    p->nGrantUL = 12;               /* W:73 */
    p->maxRarWindow = 6;            /* W:76 */
    p->maxMsg2TxCount = 9;          /* W:77 */
    p->accessTime = 5;              /* W:78 */
    p->maxTimeMs = 0;
    p->cellRadius = 400;            /* W:80 */
    p->hBS = 10.0;                  /* W:81 */
    p->hUT = 1.8;                   /* W:82 */
    p->geometry = 1;
    p->seed = 0;
    if (variant == RA_VARIANT_U0) {    /* RandomAccessSimulator.c:48-59 */
        p->nPreamble = 64; p->distribution = 1; p->geometry = 0;
    }
    if (variant == RA_VARIANT_N) {     /* NOMA.c:41-57 */
        p->nGrantUL = 2; p->maxRarWindow = 5; p->maxMsg2TxCount = 10; p->cellRadius = 500;
    }
    return RA_OK;
}

extern "C" int ra_horizon_ms(const ra_params* p) {
    if (!p) return RA_E_INVAL;
    if (p->maxTimeMs > 0) return p->maxTimeMs;
    return p->distribution == 1 ? 60000 : 10000;     /* W:243, W:254 */
}

extern "C" int ra_hist_bins(const ra_params* p, int kind) {
    if (!p) return RA_E_INVAL;
    const int h = ra_horizon_ms(p);
    if (h < 1) return RA_E_INVAL;
    if (kind == RA_HIST_DELAY) return ra_hist_delay_bins(h);
    if (kind == RA_HIST_TX) return RA_HIST_TOP;
    if (kind == RA_HIST_FAIL && p->variant == RA_VARIANT_W) return RA_HIST_TOP;
    return RA_E_INVAL;
}

extern "C" int ra_arrival_schedule(const ra_params* p, int* arrivals, int horizon) {
    if (!p || !arrivals || horizon < 0 || p->accessTime < 1 || p->nUE < 0) return RA_E_INVAL;
    const int n = p->nUE, accessTime = p->accessTime;
    /* the reference's maxTime also scales the Beta shape (time/maxTime, W:285) */
    const int maxTime = p->distribution == 1 ? 60000 : 10000;
    int nAccessUE = 0;
    if (p->distribution == 1) {
        nAccessUE = ceil((float)n * (float)accessTime * 1.0 / (float)maxTime);   /* W:246 */
        if (nAccessUE <= 0) nAccessUE = 1;                                         /* W:249-251 */
    }
    int activeCheck = 0, allAt = -1;
    const int nUE = n;
    for (int time = 0; time < horizon; ++time) {
        arrivals[time] = 0;
        if (activeCheck >= nUE) activeCheck = nUE;                                /* W:276-278 */
        if (time % accessTime == 0 && activeCheck != nUE) {                       /* W:280 */
            const int before = activeCheck;
            if (p->distribution == 1) {
                activeCheck += nAccessUE;
            } else {
                float betaDist = ra_beta_dist(3, 4, (float)time / (float)maxTime);
                int accessUEs = (int)ceil((float)nUE * betaDist / ((float)maxTime / (float)accessTime));
                /* a horizon beyond the reference's 10 s (maxTimeMs) puts x above 1 where (1-x)^3 < 0: nobody arrives
                 * there (the reference never evaluates it) -- keeps the cumulative schedule monotone */
                if (accessUEs < 0) accessUEs = 0;
                activeCheck += accessUEs;
            }
            if (activeCheck >= nUE) activeCheck = nUE;                            /* W:290-292 */
            arrivals[time] = activeCheck - before;
            if (activeCheck == nUE && allAt < 0) allAt = time;
        }
    }
    return allAt;
}

extern "C" int ra_params_validate(const ra_params* p, char* err, int errLen) {
    char local[256];
    if (!p) return RA_E_INVAL;
    const int rc = ra_host_validate(p, local, sizeof local);
    if (rc != RA_OK && err && errLen > 0) snprintf(err, (size_t)errLen, "%s", local);
    else if (err && errLen > 0) err[0] = 0;
    return rc;
}

static int next_pow2(int v) { int r = 1; while (r < v) r <<= 1; return r; }

int ra_host_validate(const ra_params* p, char* err, size_t errLen) {
#define RA_BAD(...) do { snprintf(err, errLen, __VA_ARGS__); return RA_E_INVAL; } while (0)
    if (p->variant != RA_VARIANT_W && p->variant != RA_VARIANT_N && p->variant != RA_VARIANT_U0)
        RA_BAD("unknown variant %d (RA_VARIANT_W = 0, RA_VARIANT_U0 = 1, RA_VARIANT_N = 2)", p->variant);
    if (p->variant == RA_VARIANT_U0) {
        /* RandomAccessSimulator.c: Uniform traffic over 60 s with subframe 5 only (U0:57-60,77) */
        if (p->distribution != 1) RA_BAD("variant U0 has Uniform traffic only (RandomAccessSimulator.c:57-60)");
        if (p->accessTime != 5) RA_BAD("variant U0 has accessTime 5 hard-coded (RandomAccessSimulator.c:59)");
    }
    if (p->variant == RA_VARIANT_N) {
        /* NOMA.c: Beta traffic only (N:675), rarWindow = 5 >= maxRarWindow is the only path that retransmits (N:453-455) */
        if (p->distribution == 1) RA_BAD("variant N has Beta traffic only (NOMA.c:675)");
        if (p->maxRarWindow > 5) RA_BAD("variant N: maxRarWindow %d > 5 never retransmits in NOMA.c:453-455; not supported", p->maxRarWindow);
        if (p->maxMsg2TxCount < 1) RA_BAD("variant N: maxMsg2TxCount carries maxMsg1ReTx (NOMA.c:46) and must be >= 1");
        /* activeUE draws positions until r > 35 m and gains until >= 1e-7 (NOMA.c:167-172, 185-189): with a radius at or
         * below 35 m the first loop never ends, beyond a few km the second practically never does */
        if (!(p->cellRadius > 35.0f) || !(p->cellRadius <= 5000.0f))
            RA_BAD("variant N: cellRadius %g out of range (35, 5000] m (rejection loops of NOMA.c:167-172, 185-189)", (double)p->cellRadius);
    }
    if (p->nUE < 1 || p->nUE > (1 << 24)) RA_BAD("nUE %d out of range [1, 2^24]", p->nUE);
    if (p->nPreamble < 1 || p->nPreamble > 256) RA_BAD("nPreamble %d out of range [1, 256]", p->nPreamble);
    if (p->backoffIndicator < 1 || p->backoffIndicator > 4096) RA_BAD("backoffIndicator %d out of range [1, 4096]", p->backoffIndicator);
    if (p->nGrantUL < 1) RA_BAD("nGrantUL %d must be >= 1", p->nGrantUL);
    if (p->variant == RA_VARIANT_W && (p->maxRarWindow < 2 || p->maxRarWindow > 256)) RA_BAD("maxRarWindow %d out of range [2, 256] (RAR window 1..255)", p->maxRarWindow);
    if (p->maxMsg2TxCount < 0 || p->maxMsg2TxCount > 255) RA_BAD("maxMsg2TxCount %d out of range [0, 255] (max retx 1..256)", p->maxMsg2TxCount);
    if (p->accessTime < 1 || p->accessTime > 4096) RA_BAD("accessTime %d out of range [1, 4096]", p->accessTime);
    const int h = ra_horizon_ms(p);
    if (h < 1 || h > 65535) RA_BAD("horizon %d ms out of range [1, 65535]", h);
    /* the engines index a replication's move calendar (ring x nUE records of 16 bytes) with 32 bits */
    if (p->variant != RA_VARIANT_U0 && (unsigned long long)ra_host_ring(p) * (unsigned long long)p->nUE >= (1ull << 32))
        RA_BAD("ring %d x nUE %d exceeds 2^32 calendar records per replication (64 GB): lower backoffIndicator / accessTime / nUE",
               ra_host_ring(p), p->nUE);
#undef RA_BAD
    return RA_OK;
}

int ra_host_ring(const ra_params* p) {
    const int a = p->accessTime > 5 ? p->accessTime : 5;
    if (p->variant == RA_VARIANT_N) return next_pow2(p->backoffIndicator + a + 6);   /* occasion <= T + BI + A + 2 */
    /* largest distance from the current ms to a move time: limit branch from a postponed txTime,
     * align(T+1+BI-1) + Wn-1 <= T + BI + A + Wn - 2 (Msg3 restart: T + BI + Wn + 2) -> R must exceed it */
    return next_pow2(p->backoffIndicator + a + p->maxRarWindow);
}

/* arrCum[occ] = activeCheck after the arrival step of ms occ*accessTime */
int ra_host_arrcum(const ra_params* p, int* arrCum, int nOcc) {
    const int h = ra_horizon_ms(p);
    int* arr = new int[h > 0 ? h : 1];
    ra_arrival_schedule(p, arr, h);
    int ac = 0;
    for (int occ = 0; occ < nOcc; ++occ) {
        const int t = occ * p->accessTime;
        if (t < h) ac += arr[t];
        arrCum[occ] = ac;
    }
    delete[] arr;
    return ac;
}

void ra_host_fill_point(RaPointDev* pt) {
    pt->magicBI = ra_magic((unsigned)pt->BI);
    pt->magicP = ra_magic((unsigned)pt->P);
    pt->magicA = ra_magic((unsigned)pt->A);
    pt->modSh = ra_mod_shift((unsigned)pt->BI) | (ra_mod_shift((unsigned)pt->P) << 8) | (ra_mod_shift((unsigned)pt->A) << 16);
    int sh = 0;
    while (((pt->nUE - 1) >> sh) >= RA_HBINS) ++sh;
    pt->hshift = sh;
    ra_layout(*pt);
}

/* variant U0: RaPointDev.G carries nAccessUE = ceil(n*5/60000), at least 1 (U0:60-64); no arrival schedule (nOcc 0) */
void ra_host_point_u0(const ra_params* p, RaPointDev* pt) {
    memset(pt, 0, sizeof *pt);
    pt->nUE = p->nUE; pt->P = p->nPreamble; pt->BI = p->backoffIndicator; pt->A = 5;
    pt->maxTime = ra_horizon_ms(p); pt->seed = p->seed;
    pt->R = next_pow2(p->backoffIndicator + 9);          /* phantom calendar: next match <= time + BI + 3 */
    const int maxTime = 60000, accessTime = 5;
    int nAccessUE = ceil((float)p->nUE * (float)accessTime * 1.0 / (float)maxTime);
    if (nAccessUE == 0) nAccessUE = 1;
    pt->G = nAccessUE;
    ra_host_fill_point(pt);
}

void ra_host_point(const ra_params* p, RaPointDev* pt) {
    if (p->variant == RA_VARIANT_U0) { ra_host_point_u0(p, pt); return; }
    memset(pt, 0, sizeof *pt);
    pt->nUE = p->nUE; pt->P = p->nPreamble; pt->BI = p->backoffIndicator; pt->G = p->nGrantUL;
    pt->Wn = p->maxRarWindow; pt->M = p->maxMsg2TxCount; pt->A = p->accessTime;
    pt->maxTime = ra_horizon_ms(p); pt->geometry = p->geometry ? 1 : 0; pt->R = ra_host_ring(p);
    pt->nOcc = (pt->maxTime + pt->A - 1) / pt->A; pt->seed = p->seed; pt->cellRadius = p->cellRadius;
    ra_host_fill_point(pt);
}

int ra_host_cap3(int variant, const RaPointDev* pt) {
    const long long g = pt->G < pt->nUE + 1 ? pt->G : pt->nUE + 1;
    return (int)((variant == RA_VARIANT_N ? 24 : 2) * g + 4);
}

extern "C" const char* ra_version(void) { return "rach_b200 0.2 (sm_100a; variants W/B, U0, N)"; }
