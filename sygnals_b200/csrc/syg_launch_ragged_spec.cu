// plan-specialised n_fft 2048 feature kernels (syg_launch_warp_spec*.cu) for ragged launches (frame_warp_kernel STAGE 6)
#include "syg_launch_warp.h"

namespace syglaunch {
int frame_warp_spec44k_ragged(const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err) {
    return frame_warp_t<sygdev::FftTile<10, 32>, false, SYG_NT2048, 1, 6, sygdev::Spec44k>(a, sm_count, st, err);
}
int frame_warp_spec22k_ragged(const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err) {
    return frame_warp_t<sygdev::FftTile<10, 32>, false, SYG_NT2048, 1, 6, sygdev::Spec22k>(a, sm_count, st, err);
}
int frame_warp_spec44kl_ragged(const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err) {
    return frame_warp_t<sygdev::FftTile<10, 32>, false, SYG_NT2048, 1, 6, sygdev::Spec44kL>(a, sm_count, st, err);
}
}  // namespace syglaunch
