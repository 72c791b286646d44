// Unit-resident instantiations of the warp feature kernel (frame_warp_kernel STAGE 5): short units whose mel tile stays on chip
// (BASELINE cfg3: 1 s clips, T = 101 frames, 40 mel bands).  See syg_frame_warp.cuh.
#include "syg_launch_warp.h"

namespace syglaunch {

namespace {
constexpr size_t kSmemPerSm = 227 * 1024;

template <class TL, int NT, int MINB>
struct ResGeom {
    using WT = sygdev::WarpTile<TL, NT>;
    static size_t base_bytes(const syg::FrameArgs& a) {
        return (size_t)WT::kWarps * WT::FW * WT::RS * sizeof(float) + WT::table_bytes(a.n_mels, a.mel_pw_f4);
    }
    static size_t tile_bytes(const syg::FrameArgs& a, int ku) {
        const size_t gf8 = ((size_t)ku * a.T + 7) / 8 * 8;
        return gf8 * ((size_t)sygdev::fin_pitch(a.n_mels) * 4 + 4 + 8) + (size_t)ku * 4 + 16;
    }
    // units per CTA group: the fullest last round of warp tasks among the group sizes that leave room for MINB CTAs per SM
    static int pick_units(const syg::FrameArgs& a) {
        const size_t budget = kSmemPerSm / MINB - 1024;                 // 1 KB per CTA is reserved by the system
        const size_t base = base_bytes(a);
        const int per_round = WT::kWarps * WT::FW;
        double best = 0.0;
        int best_ku = 0;
        for (int ku = 1; ku <= 256; ++ku) {
            if (base + tile_bytes(a, ku) > budget) break;
            const long long gf = (long long)ku * a.T;
            const double eff = (double)gf / (double)(((gf + per_round - 1) / per_round) * per_round);
            if (eff >= best - 0.005) { if (eff > best) best = eff; best_ku = ku; }
        }
        return best_ku;
    }
};

template <class TL, int NT, int MINB>
int res_t(const syg::FrameArgs& a_in, int sm_count, cudaStream_t st, std::string& err) {
    using G = ResGeom<TL, NT, MINB>;
    syg::FrameArgs a = a_in;
    if (a.res_units <= 0) a.res_units = G::pick_units(a);
    if (a.res_units <= 0) return 1;
    auto kfn = sygdev::frame_warp_kernel<TL, false, NT, MINB, 5, sygdev::SpecNone>;
    const size_t smem = G::base_bytes(a) + G::tile_bytes(a, a.res_units);
    static KernelCache kc;
    int bps = 0;
    if (int rc = prepare_kernel(kfn, NT, smem, kc, &bps, err)) return rc;
    const long long n_groups = (a.g.n_units + a.res_units - 1) / a.res_units;
    if (n_groups <= 0) return 0;
    const int grid = (int)std::min<long long>(n_groups, (long long)sm_count * bps);
    g_last.feature_kernel = SYG_FK_RESIDENT;
    SYG_LAUNCH(kfn, grid, NT, smem, st, a);
    LCK(cudaGetLastError());
    return 0;
}
}  // namespace

// units per group the resident kernel would use for this plan (0: the plan does not fit -> the two-kernel path)
int frame_warp_res_units(int n_fft, const syg::FrameArgs& a) {
    using namespace sygdev;
    switch (n_fft) {
        case 256: return ResGeom<FftTile<7, 16>, 256, 2>::pick_units(a);
        case 512: return ResGeom<FftTile<8, 16>, 256, 2>::pick_units(a);
        case 1024: return ResGeom<FftTile<9, 32>, 256, 2>::pick_units(a);
    }
    return 0;
}

int frame_warp_res(int n_fft, const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err) {
    using namespace sygdev;
    switch (n_fft) {
        case 256: return res_t<FftTile<7, 16>, 256, 2>(a, sm_count, st, err);
        case 512: return res_t<FftTile<8, 16>, 256, 2>(a, sm_count, st, err);
        case 1024: return res_t<FftTile<9, 32>, 256, 2>(a, sm_count, st, err);
    }
    return 1;
}

}  // namespace syglaunch
