// Mixed-radix kernel instantiations: features / STFT / Welch for transform lengths that are not powers of two (syg_mixed.cuh).
#include "syg_launch_common.h"
#include "syg_mixed.cuh"

namespace syglaunch {

// threads per CTA by transform size: a pass has L / R butterflies, so short transforms take small CTAs (and more of them per SM)
static int mixed_threads(int L) { return L <= 256 ? 64 : (L <= 1024 ? 128 : 256); }

template <int MODE, int NT>
static int frame_mixed_t(const syg::FrameArgs& a, const syg::MixedPlan& mp, int sm_count, cudaStream_t st, std::string& err) {
    auto kfn = sygdev::frame_mixed_kernel<MODE, NT>;
    const size_t smem = sygdev::mixed_layout(mp.L, mp.B, MODE != sygdev::MODE_STFT, NT).bytes;
    static KernelCache kc;
    int blocks_per_sm = 0;
    if (int rc = prepare_kernel(kfn, NT, smem, kc, &blocks_per_sm, err)) return rc;
    if (a.n_frames <= 0) return 0;
    const int grid = (int)std::min<long long>(a.n_frames, (long long)sm_count * blocks_per_sm);
    SYG_LAUNCH(kfn, grid, NT, smem, st, a, mp);
    LCK(cudaGetLastError());
    return 0;
}

template <int MODE>
static int frame_mixed_m(const syg::FrameArgs& a, const syg::MixedPlan& mp, int sm_count, cudaStream_t st, std::string& err) {
    switch (mixed_threads(mp.L)) {
        case 64: return frame_mixed_t<MODE, 64>(a, mp, sm_count, st, err);
        case 128: return frame_mixed_t<MODE, 128>(a, mp, sm_count, st, err);
        default: return frame_mixed_t<MODE, 256>(a, mp, sm_count, st, err);
    }
}

int frame_mixed(int mode, const syg::FrameArgs& a, const syg::MixedPlan& mp, int sm_count, cudaStream_t st, std::string& err) {
    if (mode == sygdev::MODE_FEATURES_RAGGED) return frame_mixed_m<sygdev::MODE_FEATURES_RAGGED>(a, mp, sm_count, st, err);
    return mode == sygdev::MODE_STFT ? frame_mixed_m<sygdev::MODE_STFT>(a, mp, sm_count, st, err)
                                     : frame_mixed_m<sygdev::MODE_FEATURES>(a, mp, sm_count, st, err);
}

template <int NT>
static int welch_mixed_t(const syg::WelchArgs& a, const syg::MixedPlan& mp, int sm_count, cudaStream_t st, std::string& err) {
    auto kfn = sygdev::welch_mixed_kernel<NT>;
    const size_t smem = sygdev::mixed_layout(mp.L, mp.B, false, NT).bytes;
    static KernelCache kc;
    int blocks_per_sm = 0;
    if (int rc = prepare_kernel(kfn, NT, smem, kc, &blocks_per_sm, err)) return rc;
    if (a.g.n_units <= 0) return 0;
    const int grid = (int)std::min<long long>(a.g.n_units, (long long)sm_count * blocks_per_sm);
    SYG_LAUNCH(kfn, grid, NT, smem, st, a, mp);
    LCK(cudaGetLastError());
    return 0;
}

int welch_mixed(const syg::WelchArgs& a, const syg::MixedPlan& mp, int sm_count, cudaStream_t st, std::string& err) {
    switch (mixed_threads(mp.L)) {
        case 64: return welch_mixed_t<64>(a, mp, sm_count, st, err);
        case 128: return welch_mixed_t<128>(a, mp, sm_count, st, err);
        default: return welch_mixed_t<256>(a, mp, sm_count, st, err);
    }
}

}  // namespace syglaunch
