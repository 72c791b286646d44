// Ragged launches (units of their own lengths in one launch): the per-frame {unit, frame in unit} table and the warp-synchronous
// feature kernel instantiations for it (frame_warp_kernel STAGE 6, n_fft <= 2048).
#include "syg_launch_warp.h"

namespace sygdev {

// ut[f] = {u, t, valid[u], starts[u]} for frame f = frame_off[u] - frame_off[0] + t of the chunk.  One thread per frame (grid-stride)
// finds its unit by binary search over frame_off -- the last u with frame_off[u] <= f, never a unit without frames -- so the work is
// even whatever the lengths (one unit of a whole recording or 100 000 short clips).
__global__ void __launch_bounds__(kThreads) ragged_frame_table_kernel(const long long* __restrict__ frame_off,
                                                                      const long long* __restrict__ starts, const int* __restrict__ valid,
                                                                      long long n_units, long long n_frames, int4* __restrict__ ut) {
    const long long base = __ldg(frame_off);
    const long long stride = (long long)gridDim.x * kThreads;
    for (long long f = (long long)blockIdx.x * kThreads + threadIdx.x; f < n_frames; f += stride) {
        long long lo = 0, hi = n_units - 1;
        while (lo < hi) {
            const long long mid = (lo + hi + 1) >> 1;
            if (__ldg(frame_off + mid) - base <= f) lo = mid;
            else hi = mid - 1;
        }
        ut[f] = make_int4((int)lo, (int)(f - (__ldg(frame_off + lo) - base)), __ldg(valid + lo), (int)__ldg(starts + lo));
    }
}

}  // namespace sygdev

namespace syglaunch {

int ragged_frame_table(const long long* frame_off, const long long* starts, const int* valid, long long n_units, long long n_frames,
                       int4* ut, int sm_count, cudaStream_t st, std::string& err) {
    if (n_units <= 0 || n_frames <= 0) return 0;
    const long long want = (n_frames + sygdev::kThreads - 1) / sygdev::kThreads;
    const int grid = (int)std::min<long long>(want, (long long)sm_count * 16);
    SYG_LAUNCH(sygdev::ragged_frame_table_kernel, grid, sygdev::kThreads, 0, st, frame_off, starts, valid, n_units, n_frames, ut);
    LCK(cudaGetLastError());
    return 0;
}

int frame_warp_ragged(int n_fft, bool extra, const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err) {
    return extra ? frame_warp_dispatch<true, 6>(n_fft, a, sm_count, st, err) : frame_warp_dispatch<false, 6>(n_fft, a, sm_count, st, err);
}

}  // namespace syglaunch
