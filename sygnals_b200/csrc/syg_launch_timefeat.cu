// Remaining per-frame time-domain features (SURVEY.md 8f-2), one warp per frame, straight from the sample buffer:
//   zero_crossing_rate  sygnals/core/audio/features.py:26-71 -> librosa.feature.zero_crossing_rate (EDGE padding when centred,
//                       threshold 1e-10, zero_pos=True, pad=False, mean over the frame)
//   skewness            sygnals/core/features/time_domain.py:67-97   scipy.stats.skew(bias=False); 0 if var < eps
//   kurtosis            time_domain.py:99-126                         scipy.stats.kurtosis(fisher=True, bias=False); 0 if var < eps
//   signal_entropy      time_domain.py:186-227                        numpy.histogram(bins) + scipy.stats.entropy; 0 if constant
// The frames are the zero-padded ones of manager.py:265-273 (np.pad(y, fl//2, 'constant') + librosa.util.frame).
// Moments, histogram edges and bin search are float64 like the reference (the samples are float32 values widened).
#include "syg_launch_common.h"
#include "syg_kernels.cuh"

namespace sygdev {

SYG_DEVICE SYG_INLINE double wsum_d(double v) {
    SYG_UNROLL
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// RAG: ragged launch (a.ragged_ut): the unit and frame index come from the per-frame table, a unit is its own valid samples, rows go
// to [n_rows][n_frames]
template <bool RAG>
SYG_DEVICE SYG_INLINE void time_extra_body(const syg::FrameArgs& a, const int fl, const int entropy_bins) {
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (kThreads / 32);
    const double n = (double)fl;
    for (long long gf = (long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); gf < a.n_frames; gf += warps) {
        const int4 rut = RAG ? __ldg(a.ragged_ut + gf) : make_int4(0, 0, 0, 0);
        const long long u = RAG ? (long long)rut.x : gf / a.T;
        const int t = RAG ? rut.y : (int)(gf - u * a.T);
        const UnitRef ur = RAG ? UnitRef{(long long)rut.w, (long long)rut.z} : unit_ref(a.g, u);
        const float* yb = a.y + ur.start;
        const long long p0 = (long long)t * a.hop - a.cpad;
        float* const orow = RAG ? a.out + gf : a.out + (long long)u * a.n_rows * a.T + t;
        // ---- pass 1: sum, extremes of the zero-padded frame; zero crossings of the edge-padded frame
        double s1 = 0.0;
        float mn = __uint_as_float(0x7f800000u), mx = __uint_as_float(0xff800000u);
        int zc = 0;
        const long long L = RAG ? ur.valid : a.g.unit_len;
        for (int i = lane; i < fl; i += 32) {
            const long long pos = p0 + i;
            const float x = (pos >= 0 && pos < ur.valid) ? __ldg(yb + pos) : 0.0f;
            s1 += (double)x;
            mn = fminf(mn, x);
            mx = fmaxf(mx, x);
            if (a.row_zcr >= 0 && i > 0 && L > 0) {
                // librosa pads the UNIT (its own zero tail included) with its edge values
                long long q = pos < 0 ? 0 : (pos >= L ? L - 1 : pos), q1 = pos - 1 < 0 ? 0 : (pos - 1 >= L ? L - 1 : pos - 1);
                float c = (q < ur.valid) ? __ldg(yb + q) : 0.0f, b = (q1 < ur.valid) ? __ldg(yb + q1) : 0.0f;
                if (fabsf(c) <= 1e-10f) c = 0.0f;
                if (fabsf(b) <= 1e-10f) b = 0.0f;
                zc += ((__float_as_uint(c) ^ __float_as_uint(b)) >> 31) ? 1 : 0;   // np.signbit(c) != np.signbit(b)
            }
        }
        s1 = wsum_d(s1);
        zc = __reduce_add_sync(kFull, zc);
        SYG_UNROLL
        for (int o = 16; o >= 1; o >>= 1) {
            mn = fminf(mn, __shfl_xor_sync(kFull, mn, o));
            mx = fmaxf(mx, __shfl_xor_sync(kFull, mx, o));
        }
        if (lane == 0 && a.row_zcr >= 0) orow[(long long)a.row_zcr * (RAG ? a.ragged_stride : a.T)] = (float)((double)zc / n);
        const bool need_mom = a.row_skew >= 0 || a.row_kurt >= 0;
        const bool need_ent = a.row_entropy >= 0;
        if (!need_mom && !need_ent) continue;
        // ---- pass 2: central moments and the histogram
        const double mu = s1 / n;
        const double first = (double)mn, last = (double)mx;
        const int nb = entropy_bins;
        const double step = (last - first) / (double)nb;                 // numpy.linspace(first, last, nb + 1)
        double m2 = 0.0, m3 = 0.0, m4 = 0.0;
        unsigned long long h0 = 0ull, h1 = 0ull, h2 = 0ull, h3 = 0ull;   // 16 bins x 16-bit lane counters (<= 4 x 4 fields)
        const bool hist = need_ent && nb >= 1 && nb <= 16 && mx > mn;
        for (int i = lane; i < fl; i += 32) {
            const long long pos = p0 + i;
            const float xf = (pos >= 0 && pos < ur.valid) ? __ldg(yb + pos) : 0.0f;
            const double x = (double)xf;
            const double d = x - mu, d2 = d * d;
            m2 += d2; m3 += d2 * d; m4 += d2 * d2;
            if (hist) {
                // numpy.histogram, uniform bins (lib/_histograms_impl.py): index from the scaled offset, then one step of
                // correction against the linspace edges.  linspace rounds idx * step, then adds first: a fused multiply-add
                // moves an edge by an ulp, and the samples lying on it (the zeros of a padded frame) into the next bin
                int idx = (int)(((x - first) / (last - first)) * (double)nb);
                if (idx == nb) idx = nb - 1;
                const double e_lo = (idx == nb) ? last : SYG_DADD_RN(first, SYG_DMUL_RN((double)idx, step));
                if (x < e_lo) idx -= 1;
                else {
                    const double e_hi = (idx + 1 == nb) ? last : SYG_DADD_RN(first, SYG_DMUL_RN((double)(idx + 1), step));
                    if (x >= e_hi && idx != nb - 1) idx += 1;
                }
                const unsigned long long inc = 1ull << (16 * (idx & 3));
                const int w = idx >> 2;
                if (w == 0) h0 += inc; else if (w == 1) h1 += inc; else if (w == 2) h2 += inc; else h3 += inc;
            }
        }
        if (need_mom) {
            m2 = wsum_d(m2) / n; m3 = wsum_d(m3) / n; m4 = wsum_d(m4) / n;
            if (lane == 0) {
                const bool flat = m2 < kEps64;                           // np.var(frame) < eps -> 0.0
                if (a.row_skew >= 0) {
                    double v = 0.0;
                    if (!flat && fl >= 3) v = sqrt((n - 1.0) * n) / (n - 2.0) * m3 / pow(m2, 1.5);
                    orow[(long long)a.row_skew * (RAG ? a.ragged_stride : a.T)] = (float)v;
                }
                if (a.row_kurt >= 0) {
                    double v = 0.0;
                    if (!flat && fl >= 4) v = 1.0 / (n - 2.0) / (n - 3.0) * ((n * n - 1.0) * m4 / (m2 * m2) - 3.0 * (n - 1.0) * (n - 1.0));
                    orow[(long long)a.row_kurt * (RAG ? a.ragged_stride : a.T)] = (float)v;
                }
            }
        }
        if (need_ent) {
            double ent = 0.0;
            if (hist) {
                SYG_UNROLL
                for (int o = 16; o >= 1; o >>= 1) {                       // fields hold <= 64 per lane, <= 2048..8192 after the sum
                    h0 += __shfl_xor_sync(kFull, h0, o); h1 += __shfl_xor_sync(kFull, h1, o);
                    h2 += __shfl_xor_sync(kFull, h2, o); h3 += __shfl_xor_sync(kFull, h3, o);
                }
                if (lane < nb) {
                    const unsigned long long hw = (lane >> 2) == 0 ? h0 : (lane >> 2) == 1 ? h1 : (lane >> 2) == 2 ? h2 : h3;
                    const int c = (int)((hw >> (16 * (lane & 3))) & 0xffffull);
                    if (c > 0) { const double pk = (double)c / n; ent = -pk * log(pk); }
                }
                ent = wsum_d(ent);
            }
            if (lane == 0) orow[(long long)a.row_entropy * (RAG ? a.ragged_stride : a.T)] = (float)ent;
        }
    }
}

__global__ void __launch_bounds__(kThreads) time_extra_kernel(const syg::FrameArgs a, const int fl, const int entropy_bins) {
    time_extra_body<false>(a, fl, entropy_bins);
}
__global__ void __launch_bounds__(kThreads) time_extra_ragged_kernel(const syg::FrameArgs a, const int fl, const int entropy_bins) {
    time_extra_body<true>(a, fl, entropy_bins);
}

}  // namespace sygdev

namespace syglaunch {
int time_extra(const syg::FrameArgs& a, int frame_length, int entropy_bins, int sm_count, cudaStream_t st, std::string& err) {
    if (a.n_frames <= 0) return 0;
    const long long want = (a.n_frames + sygdev::kThreads / 32 - 1) / (sygdev::kThreads / 32);
    const int grid = (int)std::min<long long>(want, (long long)sm_count * 8);
    if (a.ragged_ut) SYG_LAUNCH(sygdev::time_extra_ragged_kernel, grid, sygdev::kThreads, 0, st, a, frame_length, entropy_bins);
    else SYG_LAUNCH(sygdev::time_extra_kernel, grid, sygdev::kThreads, 0, st, a, frame_length, entropy_bins);
    LCK(cudaGetLastError());
    return 0;
}
}  // namespace syglaunch
