/*
 * rach_emu_hist.cpp -- TEST INFRASTRUCTURE.  The host emulation of rach_emu.cpp, unchanged, with a histogram region:
 * every job the emulation creates starts with RaJobT::hist = ra_emu_hist_base (rach_core.cuh), so the success sites
 * (ra_hist_add) of W/B, N and U0 count into the region armed here.  Built by tests/test_histograms_emulated.py.
 */
#include "rach_emu.cpp"

static std::vector<unsigned> emu_hist_region;

/* a zeroed region of `len` counters (ra_hist_len of the point's horizon) for the next emu_run / emu_run_n / emu_run_u0 */
extern "C" void emu_hist_arm(int len) {
    emu_hist_region.assign((size_t)len, 0u);
    ra_emu_hist_base = emu_hist_region.data();
}
extern "C" const unsigned* emu_hist_data(void) { return emu_hist_region.data(); }
extern "C" int emu_hist_len(int maxTime) { return ra_hist_len(maxTime); }
