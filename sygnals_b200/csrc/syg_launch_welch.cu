// Welch / periodogram kernel instantiations
#include <cstdlib>

#include "syg_launch_common.h"
#include "syg_kernels.cuh"
#include "syg_welch_warp.cuh"

namespace syglaunch {

template <class TL>
static int welch_t(const syg::WelchArgs& a, int sm_count, cudaStream_t st, std::string& err) {
    using SM = sygdev::WelchSmem<TL>;
    static KernelCache kc;
    auto kfn = sygdev::welch_kernel<TL>;
    int blocks_per_sm = 0;
    if (int rc = prepare_kernel(kfn, sygdev::kThreads, SM::bytes, kc, &blocks_per_sm, err)) return rc;
    if (a.g.n_units <= 0) return 0;
    const int grid = (int)std::min<long long>(a.g.n_units, (long long)sm_count * blocks_per_sm);
    g_last.welch_path = SYG_WELCH_BLOCK;
    SYG_LAUNCH(kfn, grid, sygdev::kThreads, SM::bytes, st, a);
    LCK(cudaGetLastError());
    return 0;
}

template <class TL, int NT = 256, int MINB = 2, bool TBLW = false>
static int welch_warp_t(const syg::WelchArgs& a, int sm_count, cudaStream_t st, std::string& err) {
    using WW = sygdev::WelchWarpTile<TL, NT, TBLW>;
    static KernelCache kc;
    auto kfn = sygdev::welch_warp_kernel<TL, NT, MINB, TBLW>;
    int blocks_per_sm = 0;
    if (int rc = prepare_kernel(kfn, NT, WW::bytes, kc, &blocks_per_sm, err)) return rc;
    if (a.g.n_units <= 0) return 0;
    const long long want = (a.g.n_units + NT / 32 - 1) / (NT / 32);
    const int grid = (int)std::min<long long>(want, (long long)sm_count * blocks_per_sm);
    g_last.welch_path = SYG_WELCH_WARP;
    SYG_LAUNCH(kfn, grid, NT, WW::bytes, st, a);
    LCK(cudaGetLastError());
    return 0;
}

int welch(int nfft, const syg::WelchArgs& a, int sm_count, cudaStream_t st, std::string& err) {
    using namespace sygdev;
    static int env = -1;                                                // SYGB200_WELCH_BLOCK=1: the CTA-cooperative kernel for every nfft
    if (env < 0) { const char* e = std::getenv("SYGB200_WELCH_BLOCK"); env = e ? std::atoi(e) : 0; }
    if (!env && nfft <= 2048) {
        switch (ilog2i(nfft / 2)) {
            case 4: return welch_warp_t<FftTile<4, 4>>(a, sm_count, st, err);
            case 5: return welch_warp_t<FftTile<5, 8>>(a, sm_count, st, err);
            case 6: return welch_warp_t<FftTile<6, 8>>(a, sm_count, st, err);
            case 7: return welch_warp_t<FftTile<7, 16>>(a, sm_count, st, err);
            case 8: return welch_warp_t<FftTile<8, 16>>(a, sm_count, st, err);
            case 9: return welch_warp_t<FftTile<9, 32>, 512, 1, true>(a, sm_count, st, err);   // 16 warps + plan tables in one CTA (226 KB)
            case 10: return welch_warp_t<FftTile<10, 32>>(a, sm_count, st, err);
        }
    }
    switch (ilog2i(nfft / 2)) {
        case 4: return welch_t<FftTile<4, 4>>(a, sm_count, st, err);
        case 5: return welch_t<FftTile<5, 8>>(a, sm_count, st, err);
        case 6: return welch_t<FftTile<6, 8>>(a, sm_count, st, err);
        case 7: return welch_t<FftTile<7, 16>>(a, sm_count, st, err);
        case 8: return welch_t<FftTile<8, 16>>(a, sm_count, st, err);
        case 9: return welch_t<FftTile<9, 16>>(a, sm_count, st, err);
        case 10: return welch_t<FftTile<10, 16>>(a, sm_count, st, err);
        case 11: return welch_t<FftTile<11, 16>>(a, sm_count, st, err);
        case 12: return welch_t<FftTile<12, 16>>(a, sm_count, st, err);
    }
    err = "nfft=" + std::to_string(nfft) + ": only powers of two in [32, 8192] are supported";
    return -5;
}

}  // namespace syglaunch
