// dispatch of the warp-synchronous feature kernel over n_fft (included by the warp translation units)
#pragma once

#include <cstdlib>

#include "syg_launch_common.h"
#include "syg_frame_warp.cuh"

#ifndef SYG_NT2048
#define SYG_NT2048 640
#endif

namespace syglaunch {

// plan-specialised instantiations of the n_fft 2048 feature kernel (own translation units: syg_launch_warp_spec*.cu)
int frame_warp_spec44k(const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err);
int frame_warp_spec22k(const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err);
int frame_warp_spec44kl(const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err);
// the same three for ragged launches (STAGE 6; syg_launch_ragged_spec.cu)
int frame_warp_spec44k_ragged(const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err);
int frame_warp_spec22k_ragged(const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err);
int frame_warp_spec44kl_ragged(const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err);

// STAGE 0: features; 6: features of ragged units; 3: STFT output through a CTA tile; 4: STFT magnitude / power through warp-private tiles (see syg_frame_warp.cuh)
template <class TL, bool EXTRA, int NT, int MINB, int STAGE, class SP = sygdev::SpecNone>
static int frame_warp_t(const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err) {
    using WT = sygdev::WarpTile<TL, NT>;
    auto kfn = sygdev::frame_warp_kernel<TL, EXTRA, NT, MINB, STAGE, SP>;
    size_t smem = (size_t)WT::kWarps * WT::FW * WT::RS * sizeof(float);
    const int wide = (STAGE == 3 && a.out_kind == 0) ? 1 : 0;        // complex64 tile
    if (STAGE == 0 || STAGE == 6) smem += WT::table_bytes(a.n_mels, (a.mask & syg::FB_MFCC) ? a.mel_pw_f4 : 0);
    if (STAGE == 3) {
        const int TT = WT::kWarps * WT::FW;
        smem += (size_t)TT * sizeof(long long) + (size_t)(WT::M + 1) * (TT + 1) * (wide ? 8 : 4);
    }
    if (STAGE == 4) smem += (size_t)WT::kWarps * (16 + (((WT::M + 1) * 9 + 1) & ~1)) * sizeof(float)   // per warp: 8 offsets + tile [B][9]
                            + WT::kWinB + WT::kTwB + WT::kTwshB;                                           // window, twiddles, split twiddles
    static KernelCache kc;                                           // the dynamic size depends on the plan (n_mels, taps, complex tile)
    int bps = 0;
    if (int rc = prepare_kernel(kfn, NT, smem, kc, &bps, err)) return rc;
    const int blocks_per_sm_w = bps;
    const long long per_cta = (long long)((STAGE == 4) ? 8 : WT::FW) * WT::kWarps;
    const long long n_rounds = (a.n_frames + per_cta - 1) / per_cta;
    if (n_rounds <= 0) return 0;
    const int grid = (int)std::min<long long>(n_rounds, (long long)sm_count * blocks_per_sm_w);
    SYG_LAUNCH(kfn, grid, NT, smem, st, a);
    LCK(cudaGetLastError());
    return 0;
}

// does the run-time plan equal the compile-time layout of SP (syg_frame_warp.cuh)?  Features that are not requested do not matter.
template <class SP>
static bool spec_matches(const syg::FrameArgs& a) {
    if (!(a.mask & (syg::FB_MFCC | syg::FB_CONTRAST))) return false;
    if (SP::kMask && (a.mask != SP::kMask || a.row_rms != SP::row_rms || a.row_crest != SP::row_crest || a.row_peak != SP::row_peak ||
                      a.row_centroid != SP::row_centroid || a.row_rolloff != SP::row_rolloff)) return false;
    if (a.mask & syg::FB_CONTRAST) {
        if (!SP::kBands || a.nb != SP::nb) return false;
        for (int i = 0; i < SP::nb; ++i)
            if (a.band_lo[i] != SP::band(i, 0) || a.band_cnt[i] != SP::band(i, 1) || a.band_n[i] != SP::band(i, 2)) return false;
    }
    if ((a.mask & syg::FB_MFCC) && !a.mel_iv) {
        if (!SP::kMel || !a.mel_power_is_2 || a.n_mels != 32 * SP::n_sweeps || a.mel_nsweeps != SP::n_sweeps) return false;
        for (int i = 0; i < SP::n_sweeps; ++i)
            if (a.mel_steps[i] != SP::steps(i)) return false;
    }
    return true;
}

template <bool EXTRA, int STAGE>
static int frame_warp_dispatch(int n_fft, const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err) {
    using namespace sygdev;
    constexpr int MINB = 2, NT = 256;
    // STFT stage: the CTA tile couples the warps of a CTA through two barriers per round; 4-warp CTAs (4 per SM) measured
    // 8 % / 5 % faster than 8-warp ones for n_fft 256 / 1024, equal for 512, 15 % slower for 2048 (cfg2, B200)
    constexpr int NT3 = (STAGE == 3) ? 128 : NT, MINB3 = (STAGE == 3) ? 4 : MINB;
    switch (ilog2i(n_fft / 2)) {
        case 4: return frame_warp_t<FftTile<4, 4>, EXTRA, NT, MINB, STAGE>(a, sm_count, st, err);
        case 5: return frame_warp_t<FftTile<5, 8>, EXTRA, NT, MINB, STAGE>(a, sm_count, st, err);
        case 6: return frame_warp_t<FftTile<6, 8>, EXTRA, NT, MINB, STAGE>(a, sm_count, st, err);
        case 7: return frame_warp_t<FftTile<7, 16>, EXTRA, NT3, MINB3, STAGE>(a, sm_count, st, err);
        case 8:
            // warp-private tiles + tables: 16 warps need 226 KB, which fits one 512-thread CTA per SM but not two 256-thread ones
            if constexpr (STAGE == 4) return frame_warp_t<FftTile<8, 16>, EXTRA, 512, 1, STAGE>(a, sm_count, st, err);
            else return frame_warp_t<FftTile<8, 16>, EXTRA, NT, MINB, STAGE>(a, sm_count, st, err);
        case 9:
            if constexpr (STAGE == 4) break;                          // warp-private tiles exist for M <= 256 only
            else return frame_warp_t<FftTile<9, 32>, EXTRA, NT3, MINB3, STAGE>(a, sm_count, st, err);
        case 10:
            if constexpr (STAGE == 4) break;
            // features: one CTA of 16 warps per SM so that the 38 KB of plan tables are held once (leaves ~50 KB of L1)
            if constexpr ((STAGE == 0 || STAGE == 6) && !EXTRA) {
                static int nospec = -1;                               // SYGB200_NO_SPEC=1: always the generic loops (A/B measurements)
                if (nospec < 0) { const char* e = std::getenv("SYGB200_NO_SPEC"); nospec = e ? std::atoi(e) : 0; }
                static int nolay = -1;                                // SYGB200_NO_SPECL=1: skip the layout-specialised instantiation (A/B)
                if (nolay < 0) { const char* e = std::getenv("SYGB200_NO_SPECL"); nolay = e ? std::atoi(e) : 0; }
                constexpr bool rag = (STAGE == 6);
                if (!nospec && !nolay && spec_matches<Spec44kL>(a))
                    return rag ? frame_warp_spec44kl_ragged(a, sm_count, st, err) : frame_warp_spec44kl(a, sm_count, st, err);
                if (!nospec && spec_matches<Spec44k>(a))
                    return rag ? frame_warp_spec44k_ragged(a, sm_count, st, err) : frame_warp_spec44k(a, sm_count, st, err);
                if (!nospec && spec_matches<Spec22k>(a))
                    return rag ? frame_warp_spec22k_ragged(a, sm_count, st, err) : frame_warp_spec22k(a, sm_count, st, err);
            }
            if (STAGE == 0 || STAGE == 6) {
                // 20 warps leave ~40 KB of shared memory for the plan tables: enough for the interval-form mel and for the tap
                // tables of the default banks, not for the long taps of a few wide filters (n_mels 40 or fewer without the
                // interval form, e.g. mel power != 2).  Those plans run 8 warps per CTA.
                const size_t tbl = WarpTile<FftTile<10, 32>, SYG_NT2048>::table_bytes(a.n_mels, (a.mask & syg::FB_MFCC) ? a.mel_pw_f4 : 0);
                int dev = 0, optin = 0;
                LCK(cudaGetDevice(&dev));
                LCK(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
                if (WarpTile<FftTile<10, 32>, SYG_NT2048>::bytes + tbl <= (size_t)optin)
                    return frame_warp_t<FftTile<10, 32>, EXTRA, SYG_NT2048, 1, STAGE>(a, sm_count, st, err);
            }
            return frame_warp_t<FftTile<10, 32>, EXTRA, NT, MINB, STAGE>(a, sm_count, st, err);
    }
    err = "n_fft=" + std::to_string(n_fft) + " has no warp tile";
    return -5;
}

}  // namespace syglaunch
