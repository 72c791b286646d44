// sygnals_b200/csrc/syg_params.h -- kernel argument blocks (host fills, device reads; passed by value).
#pragma once

#include "syg_platform.h"

namespace sygdev {
constexpr int kThreads = 256;               // threads per CTA of every kernel
constexpr int MODE_FEATURES = 0;            // frame kernel modes
constexpr int MODE_STFT = 1;
constexpr int MODE_FEATURES_RAGGED = 2;     // features of units with their own lengths (FrameArgs::ragged_ut)
constexpr int kFinTT = 32;                  // frames per finalize CTA
// row pitch (floats) of the finalize kernel's S_db tile for N mel bands: >= N and 4 mod 8, so that rows start 16-byte aligned
// and the 8 frames x 4 columns of a DMMA B fragment (and its mirrored columns) fall on 32 distinct banks
#if defined(__CUDACC__)
__host__ __device__
#endif
inline int fin_pitch(int N) { int p = (N + 3) / 4 * 4; while ((p & 7) != 4) p += 4; return p; }
// finalize_kernel: pitch (in doubles) of the folded FP64 rows in shared memory, H = columns of a row.  A multiple of 4 (the DMMA
// k-step) and = 4 (mod 16): the B-fragment read of a half-warp -- 4 frames x 4 consecutive doubles -- then covers 32 distinct banks.
#if defined(__CUDACC__)
__host__ __device__
#endif
inline int fin_pitch_d(int H) { int p = (H + 3) / 4 * 4; while ((p & 15) != 4) p += 4; return p; }
inline size_t fin_smem_bytes(int tt, int n_mels, bool fold) {
    const int H = fold ? (n_mels + 1) / 2 : n_mels;
    return (size_t)(fold ? 2 : 1) * tt * fin_pitch_d(H) * sizeof(double);
}

// shared-memory layout (float words) of the mixed-radix kernels for L complex points, B bins and nt threads per CTA
struct MixedLayout {
    int off_a, off_b, off_pw, off_cand, off_smax, off_dsc_f, total_f;
    size_t bytes;
};
#if defined(__CUDACC__)
__host__ __device__
#endif
inline MixedLayout mixed_layout(int L, int B, bool features, int nt = kThreads) {
    MixedLayout m;
    m.off_a = 0;
    m.off_b = 2 * L;
    m.off_pw = 4 * L;
    m.off_cand = m.off_pw + (features ? (B + (B >> 5) + 1) : 0);
    m.off_smax = m.off_cand + (features ? (nt / 32) * 32 : 0);
    m.off_dsc_f = ((m.off_smax + 4 + 1) / 2) * 2;
    m.total_f = m.off_dsc_f + 2 * (nt / 32 + nt);
    m.bytes = (size_t)m.total_f * 4;
    return m;
}
}  // namespace sygdev

namespace syg {

// feature bits (kernel-internal; the public ids live in include/sygb200.h)
enum : unsigned {
    FB_MFCC = 1u << 0, FB_CONTRAST = 1u << 1, FB_CENTROID = 1u << 2, FB_ROLLOFF = 1u << 3, FB_RMS = 1u << 4,
    FB_CREST = 1u << 5, FB_PEAK = 1u << 6, FB_BANDWIDTH = 1u << 7, FB_FLATNESS = 1u << 8, FB_DOMINANT = 1u << 9,
    FB_ZCR = 1u << 10, FB_MEAN_AMP = 1u << 11, FB_STD_AMP = 1u << 12, FB_SKEW = 1u << 13, FB_KURT = 1u << 14, FB_ENTROPY = 1u << 15,
};
constexpr unsigned FB_SPECTRUM_ANY = FB_MFCC | FB_CONTRAST | FB_CENTROID | FB_ROLLOFF | FB_BANDWIDTH | FB_FLATNESS | FB_DOMINANT;
constexpr unsigned FB_SPECSTATS = FB_CENTROID | FB_ROLLOFF | FB_BANDWIDTH | FB_FLATNESS | FB_DOMINANT;
constexpr unsigned FB_TIME_ANY = FB_RMS | FB_CREST | FB_PEAK | FB_MEAN_AMP | FB_STD_AMP;            // time features of the frame kernels
constexpr unsigned FB_TIME_EXTRA = FB_ZCR | FB_SKEW | FB_KURT | FB_ENTROPY;                           // time_extra_kernel

constexpr int kMaxBands = 12;   // spectral-contrast bands incl. the top one (n_bands + 1)

struct UnitGeom {
    long long n_units;          // units handled by this launch
    long long unit_len;         // padded length of a unit (samples)
    long long unit_stride;      // start_u = u * unit_stride                (if unit_starts == nullptr)
    long long total_len;        // samples in y; valid_u = clamp(total_len - start_u, 0, unit_len)
    const long long* unit_starts;   // optional [n_units] (device)
    const int* unit_valid;          // optional [n_units] (device)
    long long unit0;            // first unit of this launch in the caller's numbering (analytic starts only;
                                // unit_starts / unit_valid are passed already offset)
};

struct FrameArgs {
    const float* y;
    UnitGeom g;
    int T;                      // frames per unit
    int hop;
    int cpad;                   // n_fft/2 when centred, else 0
    int pad_mode;               // 0 constant (zeros), 1 reflect
    long long n_frames;         // g.n_units * T
    const float* window;        // [n_fft], already zero-padded/centred to n_fft
    const float2* tw;           // [M]      exp(-2 pi i k / M)
    const float2* tws;          // [M/2+1]  exp(-2 pi i k / n_fft)
    const float2* twsh;         // [M/2+1]  0.5 exp(-2 pi i k / n_fft)   (split with the halving folded in)
    const float2* tw1k;         // [1024]   exp(-2 pi i k / 1024): sub-transform twiddles of stft_big_kernel (n_fft 4096 / 8192)
    // ---- features
    unsigned mask;
    double bin_hz;              // frequency of bin 1 (numpy rfftfreq step)
    double roll_percent;
    int n_mels;
    const int* mel_start;       // [n_mels] first bin with non-zero weight
    const int* mel_len;         // [n_mels]
    const int* mel_off;         // [n_mels] offset into mel_w
    const float* mel_w;
    const int4* mel_slots;      // [n_mels] {filter, padded start, taps (multiple of 4), offset into mel_pw}, longest first
    const float* mel_pw;        // tap weights in padded-spectrum index space
    int mel_power_is_2;
    float mel_half_power;       // power / 2 (applied to |X|^2)
    int nb;                     // contrast bands incl. top (0 = off)
    int band_lo[kMaxBands];     // first bin
    int band_cnt[kMaxBands];    // bins in the (already "drop last row"-ed) sub-band
    int band_n[kMaxBands];      // quantile count
    // per-frame rows written directly (row < 0: not requested)
    int row_centroid, row_rolloff, row_rms, row_crest, row_peak, row_bandwidth, row_flatness, row_dominant,
        row_zcr, row_mean_amp, row_std_amp, row_skew, row_kurt, row_entropy;
    int n_rows;
    float* out;                 // [n_units][n_rows][T]
    float* melws;               // [n_frames][n_mels]   raw mel energies
    float* cws;                 // [n_frames][2*nb]     contrast peaks | valleys (linear)
    unsigned* unit_max;         // [n_units][4]         bit images of max mel energy, max peak, max valley
    int mel_pw_f4;              // float4 count of mel_pw (for the shared-memory copy of the plan tables)
    int mel_iv;                 // 1: mel_pw holds the interval-form blob (sygplan::MelIntervals) instead of sweep taps
    int mel_nsweeps;            // sweeps of the warp kernel's mel plan and their float4 step counts (host side: lets the launcher
    int mel_steps[8];           // pick a plan-specialised kernel); 0 sweeps = not recorded
    int variant;                // measurement switch (SYGB200_VARIANT, default 0): bit 0 = per-scheduler lock step (see frame_warp_kernel)
    // ---- unit-resident MFCC epilogue (frame_warp_kernel STAGE 5): the finalize arguments + units per CTA group
    int res_units;
    const double* fin_dct;
    int fin_n_mfcc, fin_row_mfcc, fin_dct_fold;
    float fin_amin, fin_top_db;
    // ---- stft
    int out_kind;               // 0 complex64, 1 magnitude, 2 power
    void* stft_out;             // [n_units][B][T]
    // ---- ragged launches (MODE_FEATURES_RAGGED, frame_warp_kernel STAGE 6): units of their own lengths.  ragged_ut[gf] =
    // {unit, frame in unit, unit length, unit start in y} of frame gf (one load, nothing that depends on another load; the chunk's
    // samples span less than 2^31); row r of frame gf goes to out[r * ragged_stride + gf].  T and the tables of g are unused.
    const int4* ragged_ut;      // [n_frames]
    long long ragged_stride;    // >= n_frames
};

// run-time plan of the mixed-radix kernels (syg_mixed.cuh): n real samples per transform, L complex points in shared memory
// (n/2 packed when n is even, n otherwise), B = n/2 + 1 one-sided bins, the radices of the passes in order
struct MixedPlan {
    int n, L, B, packed, npass;
    int radix[24];
};

struct FinalizeArgs {
    long long n_units;
    int T, n_rows;
    int n_mels, n_mfcc, row_mfcc;       // row_mfcc < 0: no mfcc
    const double* dct;                  // [n_mfcc][n_mels] float64 (lifter folded in)
    int dct_fold;                       // 1: DCT-II, row k is (-1)^k symmetric about the centre -> half-length sums
    int nb, row_contrast;               // nb == 0: no contrast
    float amin, top_db;
    const float* melws;
    const float* cws;
    const unsigned* unit_max;
    float* out;
    const int4* ragged_ut;              // ragged launches: [n_frames] {unit, frame in unit, ...} (T unused)
    long long n_frames;                 // ragged launches: frames of the chunk
    long long ragged_stride;            // ragged launches: row r of frame gf at out[r * ragged_stride + gf]
};

struct WelchArgs {
    const float* y;
    UnitGeom g;
    int nperseg, step, nseg;    // sub-segment length (<= nfft), hop, count per unit
    int detrend;                // 1: subtract sub-segment mean
    const float* window;        // [nfft] (nperseg window values then zeros)
    const float2* tw;
    const float2* tws;
    float scale;                // 1/(fs*sum w^2) or 1/(sum w)^2
    int onesided_double;        // 1: double all bins except DC (and Nyquist for even nfft)
    float* psd;                 // [n_units][B]
    float* stats;               // optional [n_units][3]: rms, crest, peak over the unit's unit_len samples
};

}  // namespace syg
