// CTA-synchronous frame kernel instantiations: STFT (all sizes) and features for n_fft 4096 / 8192, plus finalize.
#include <cstdlib>

#include "syg_launch_common.h"
#include "syg_kernels.cuh"
#include "syg_finalize.cuh"

namespace syglaunch {

template <class TL, int MODE>
static int frame_block_t(const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err) {
    using SM = sygdev::FrameSmem<TL>;
    static KernelCache kc;
    auto kfn = sygdev::frame_kernel<TL, MODE>;
    int blocks_per_sm = 0;
    if (int rc = prepare_kernel(kfn, sygdev::kThreads, SM::bytes, kc, &blocks_per_sm, err)) return rc;
    const long long n_rounds = (a.n_frames + TL::F - 1) / TL::F;
    if (n_rounds <= 0) return 0;
    const int grid = (int)std::min<long long>(n_rounds, (long long)sm_count * blocks_per_sm);
    SYG_LAUNCH(kfn, grid, sygdev::kThreads, SM::bytes, st, a);
    LCK(cudaGetLastError());
    return 0;
}

template <class TL, int TT>
static int stft_tile_t(const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err) {
    using SM = sygdev::StftTileSmem<TL, TT>;
    auto kfn = sygdev::stft_tile_kernel<TL, TT>;
    const size_t smem = SM::bytes(a.out_kind == 0);
    static KernelCache kc;
    int blocks_per_sm = 0;
    if (int rc = prepare_kernel(kfn, sygdev::kThreads, smem, kc, &blocks_per_sm, err)) return rc;
    const long long n_tiles = (a.n_frames + TT - 1) / TT;
    if (n_tiles <= 0) return 0;
    const int grid = (int)std::min<long long>(n_tiles, (long long)sm_count * blocks_per_sm);
    SYG_LAUNCH(kfn, grid, sygdev::kThreads, smem, st, a);
    LCK(cudaGetLastError());
    return 0;
}

int frame_block(int n_fft, int mode, const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err) {
    using namespace sygdev;
    const int l = ilog2i(n_fft / 2);
    if (mode == MODE_STFT) {
        static int env = -1;                                            // SYGB200_STFT_BLOCK=1: the per-frame-store kernel (comparison)
        if (env < 0) { const char* e = std::getenv("SYGB200_STFT_BLOCK"); env = e ? std::atoi(e) : 0; }
        if (!env && l == 11) return stft_tile_t<FftTile<11, 16>, 8>(a, sm_count, st, err);
        if (!env && l == 12) return a.out_kind == 0 ? stft_tile_t<FftTile<12, 16>, 4>(a, sm_count, st, err)
                                                     : stft_tile_t<FftTile<12, 16>, 8>(a, sm_count, st, err);
        switch (l) {
            case 4: return frame_block_t<FftTile<4, 4>, MODE_STFT>(a, sm_count, st, err);
            case 5: return frame_block_t<FftTile<5, 8>, MODE_STFT>(a, sm_count, st, err);
            case 6: return frame_block_t<FftTile<6, 8>, MODE_STFT>(a, sm_count, st, err);
            case 7: return frame_block_t<FftTile<7, 16>, MODE_STFT>(a, sm_count, st, err);
            case 8: return frame_block_t<FftTile<8, 16>, MODE_STFT>(a, sm_count, st, err);
            case 9: return frame_block_t<FftTile<9, 16>, MODE_STFT>(a, sm_count, st, err);
            case 10: return frame_block_t<FftTile<10, 16>, MODE_STFT>(a, sm_count, st, err);
            case 11: return frame_block_t<FftTile<11, 16>, MODE_STFT>(a, sm_count, st, err);
            case 12: return frame_block_t<FftTile<12, 16>, MODE_STFT>(a, sm_count, st, err);
        }
    } else if (mode == MODE_FEATURES_RAGGED) {
        switch (l) {
            case 11: return frame_block_t<FftTile<11, 16>, MODE_FEATURES_RAGGED>(a, sm_count, st, err);
            case 12: return frame_block_t<FftTile<12, 16>, MODE_FEATURES_RAGGED>(a, sm_count, st, err);
        }
    } else {
        switch (l) {
            case 11: return frame_block_t<FftTile<11, 16>, MODE_FEATURES>(a, sm_count, st, err);
            case 12: return frame_block_t<FftTile<12, 16>, MODE_FEATURES>(a, sm_count, st, err);
        }
    }
    err = "n_fft=" + std::to_string(n_fft) + ": only powers of two in [32, 8192] are supported";
    return -5;
}

template <int TT, bool RAG>
static int finalize_t(const syg::FinalizeArgs& a, unsigned grid_x, unsigned grid_y, size_t smem, cudaStream_t st, std::string& err) {
    auto kfn = sygdev::finalize_kernel_t<RAG ? (TT | sygdev::kFinRagged) : TT>;
    if (smem > 48 * 1024) {                         // the S_db tile exceeds the default 48 KB for wide mel banks
        static KernelCache kc;
        int nb = 0;
        if (int rc = prepare_kernel(kfn, sygdev::kThreads, smem, kc, &nb, err)) return rc;
    }
    SYG_LAUNCH(kfn, dim3(grid_x, grid_y), dim3(sygdev::kThreads), smem, st, a);
    LCK(cudaGetLastError());
    return 0;
}

// tt = frames per CTA tile: 32 (default) or 64 (narrow mel banks: the CTA is latency bound, twice the frames amortise it)
int finalize(const syg::FinalizeArgs& a, int tt, unsigned grid_x, unsigned grid_y, size_t smem, cudaStream_t st, std::string& err) {
    if (grid_x == 0 || grid_y == 0) return 0;        // no frames: a launch of zero CTAs would fail with an invalid configuration
    if (a.ragged_ut)
        return tt == 64 ? finalize_t<64, true>(a, grid_x, grid_y, smem, st, err) : finalize_t<32, true>(a, grid_x, grid_y, smem, st, err);
    return tt == 64 ? finalize_t<64, false>(a, grid_x, grid_y, smem, st, err) : finalize_t<32, false>(a, grid_x, grid_y, smem, st, err);
}

}  // namespace syglaunch
