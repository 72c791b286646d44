// STFT output of the warp-synchronous kernel (n_fft <= 2048): stage 3 = framing + FFT + real split -> transposed CTA tile ->
// contiguous row stores  (dsp.py:167-229 compute_stft; complex64 / magnitude / power)
#include <cstdlib>

#include "syg_launch_warp.h"

namespace syglaunch {
int frame_warp_stft(int n_fft, const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err) {
    // real-valued output of the small transforms: warp-private tiles (no CTA barrier); SYGB200_STFT_CTA_TILE=1 keeps the CTA tile
    static int env = -1;
    if (env < 0) { const char* e = std::getenv("SYGB200_STFT_CTA_TILE"); env = e ? std::atoi(e) : 0; }
    if (a.out_kind != 0 && n_fft <= 512) {
        if (!env) return frame_warp_dispatch<false, 4>(n_fft, a, sm_count, st, err);
        g_last.stft_path = 7;                                           // reached only through the switch
    }
    return frame_warp_dispatch<false, 3>(n_fft, a, sm_count, st, err);
}
}  // namespace syglaunch
