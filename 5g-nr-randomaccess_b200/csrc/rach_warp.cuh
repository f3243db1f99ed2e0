/*
 * rach_warp.cuh -- "vector form" helpers: code written once that runs as one warp on the device (one lane per
 * element, ballots and shuffles) and as a loop over 32 emulated lanes on the host (tests/emu), so that warp-level
 * formulations can be fuzzed on the CPU against the CPU restatement of the reference (test infrastructure) before they ever run on a GPU.
 *
 *   RW_EACH(l) { ... lane ... x[l] ... }   per-lane statement block: on the device l == 0 and lane is the lane id,
 *                                          on the host l == lane runs over 0..31; per-lane values live in arrays
 *                                          of RW_LANES elements (1 on the device, 32 on the host)
 *   RW_BALLOT(pred)  RW_SHFL(arr, src)  RW_SYNC()  RW_POPC  RW_FFS
 *   rw_sum  rw_min_u32  rw_scan_u32        reductions and the inclusive prefix sum over the lanes
 */
#ifndef RACH_WARP_CUH
#define RACH_WARP_CUH

#ifdef __CUDA_ARCH__
#define RW_LANES 1
#define RW_EACH(l) for (int l = 0, lane = (int)(threadIdx.x & 31u); l < 1 && ((void)lane, true); ++l)
#define RW_BALLOT(arr) __ballot_sync(0xFFFFFFFFu, (arr)[0])
#define RW_SHFL(arr, src) __shfl_sync(0xFFFFFFFFu, (arr)[0], (src))
#define RW_SYNC() __syncwarp()
#define RW_POPC(x) __popc(x)
#define RW_FFS(x) __ffs((int)(x))
#define RW_FN __device__ __forceinline__
RW_FN long long rw_sum(const long long* a) {
    long long v = a[0];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}
RW_FN unsigned rw_min_u32(const unsigned* a) {
    unsigned v = a[0];
    for (int o = 16; o > 0; o >>= 1) { const unsigned t = __shfl_xor_sync(0xFFFFFFFFu, v, o); v = t < v ? t : v; }
    return v;
}
/* incl[lane] = a[0] + ... + a[lane] */
RW_FN void rw_scan_u32(const unsigned* a, unsigned* incl) {
    const int lane = (int)(threadIdx.x & 31u);
    unsigned v = a[0];
    for (int o = 1; o < 32; o <<= 1) { const unsigned t = __shfl_up_sync(0xFFFFFFFFu, v, o); if (lane >= o) v += t; }
    incl[0] = v;
}
#else
#define RW_LANES 32
#define RW_EACH(l) for (int l = 0, lane = 0; l < 32 && ((void)lane, true); ++l, lane = l)
static inline unsigned rw_ballot(const int* a) { unsigned m = 0; for (int i = 0; i < 32; ++i) if (a[i]) m |= 1u << i; return m; }
#define RW_BALLOT(arr) rw_ballot(arr)
#define RW_SHFL(arr, src) ((arr)[(src)])
#define RW_SYNC() ((void)0)
#define RW_POPC(x) __builtin_popcount(x)
#define RW_FFS(x) __builtin_ffs((int)(x))
#define RW_FN static inline
static inline long long rw_sum(const long long* a) { long long v = 0; for (int i = 0; i < 32; ++i) v += a[i]; return v; }
static inline unsigned rw_min_u32(const unsigned* a) { unsigned v = a[0]; for (int i = 1; i < 32; ++i) v = a[i] < v ? a[i] : v; return v; }
static inline void rw_scan_u32(const unsigned* a, unsigned* incl) { unsigned v = 0; for (int i = 0; i < 32; ++i) incl[i] = v += a[i]; }
#endif


#endif /* RACH_WARP_CUH */
