// sygnals_b200/csrc/syg_plan.h -- host-side construction of the constant tables (double precision, rounded once).
//
// Each builder follows the routine the reference calls (librosa / scipy semantics, SURVEY.md Appendix A):
//   window      scipy.signal.get_window(name, win_length, fftbins=True) + librosa.util.pad_center   (A.1)
//   mel basis   librosa.filters.mel(sr, n_fft, n_mels, fmin, fmax, htk=False, norm='slaney', float32) (A.3)
//   dct         scipy.fftpack.dct(type, norm)[:n_mfcc] + librosa lifter                              (A.6)
//   bands       librosa.feature.spectral_contrast octave-band membership and quantile counts         (A.7)
#pragma once

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <string>
#include <vector>

namespace sygplan {

constexpr double kPi = 3.14159265358979323846264338327950288;

inline bool build_window(int window, int win_length, int n_fft, std::vector<float>& out, std::string& err) {
    if (win_length < 1 || win_length > n_fft) { err = "win_length must be in [1, n_fft]"; return false; }
    double a[3] = {0, 0, 0};
    int na = 0;
    switch (window) {
        case 0: a[0] = 0.5; a[1] = 0.5; na = 2; break;                 // hann
        case 1: a[0] = 0.54; a[1] = 0.46; na = 2; break;               // hamming
        case 2: a[0] = 0.42; a[1] = 0.5; a[2] = 0.08; na = 3; break;   // blackman
        case 3: a[0] = 1.0; na = 1; break;                             // boxcar
        default: err = "unsupported window id"; return false;
    }
    out.assign(n_fft, 0.0f);
    const int lpad = (n_fft - win_length) / 2;                         // librosa.util.pad_center
    for (int n = 0; n < win_length; ++n) {
        double w = a[0];
        double sgn = -1.0;
        for (int i = 1; i < na; ++i) { w += sgn * a[i] * std::cos(2.0 * kPi * i * n / (double)win_length); sgn = -sgn; }
        out[lpad + n] = (float)w;
    }
    return true;
}

inline double window_value_d(int window, int win_length, int n) {
    double a[3] = {0, 0, 0};
    int na = 0;
    switch (window) {
        case 0: a[0] = 0.5; a[1] = 0.5; na = 2; break;
        case 1: a[0] = 0.54; a[1] = 0.46; na = 2; break;
        case 2: a[0] = 0.42; a[1] = 0.5; a[2] = 0.08; na = 3; break;
        default: a[0] = 1.0; na = 1; break;
    }
    double w = a[0], sgn = -1.0;
    for (int i = 1; i < na; ++i) { w += sgn * a[i] * std::cos(2.0 * kPi * i * n / (double)win_length); sgn = -sgn; }
    return w;
}

// Radices of the mixed-radix kernels for an L-point transform: fours first, then 2 / 3 / 5 / 7 / 11 / 13.  false if L has a larger
// prime factor (those lengths stay unsupported).
inline bool factorize_smooth(int L, std::vector<int>& radix) {
    radix.clear();
    if (L < 1) return false;
    while (L % 4 == 0) { radix.push_back(4); L /= 4; }
    for (int p : {2, 3, 5, 7, 11, 13})
        while (L % p == 0) { radix.push_back(p); L /= p; }
    return L == 1;
}

// numpy.fft.rfftfreq(n_fft, 1/sr) step, with numpy's operation order
inline double bin_hz(double sr, int n_fft) {
    const double d = 1.0 / sr;
    return 1.0 / ((double)n_fft * d);
}

inline double hz_to_mel(double f) {                       // Slaney (htk=False)
    const double f_sp = 200.0 / 3.0, min_log_hz = 1000.0, min_log_mel = min_log_hz / f_sp;
    const double logstep = std::log(6.4) / 27.0;
    if (f >= min_log_hz) return min_log_mel + std::log(f / min_log_hz) / logstep;
    return f / f_sp;
}
inline double mel_to_hz(double m) {
    const double f_sp = 200.0 / 3.0, min_log_hz = 1000.0, min_log_mel = min_log_hz / f_sp;
    const double logstep = std::log(6.4) / 27.0;
    if (m >= min_log_mel) return min_log_hz * std::exp(logstep * (m - min_log_mel));
    return f_sp * m;
}

struct MelTable {
    int n_mels = 0, n_bins = 0;
    std::vector<int> start, len, off;
    std::vector<float> w;            // concatenated non-zero spans
    std::vector<float> dense;        // optional [n_mels][n_bins]
};

inline bool build_mel(double sr, int n_fft, int n_mels, double fmin, double fmax, bool want_dense, MelTable& t,
                      std::string& err) {
    if (n_mels < 1) { err = "n_mels must be >= 1"; return false; }
    if (fmax <= 0) fmax = sr / 2.0;
    const int B = 1 + n_fft / 2;
    t.n_mels = n_mels; t.n_bins = B;
    t.start.assign(n_mels, 0); t.len.assign(n_mels, 0); t.off.assign(n_mels, 0);
    t.w.clear();
    if (want_dense) t.dense.assign((size_t)n_mels * B, 0.0f);
    const double step_hz = bin_hz(sr, n_fft);
    // mel_frequencies(n_mels + 2): np.linspace(min_mel, max_mel, n) then mel_to_hz
    const int n = n_mels + 2;
    const double mn = hz_to_mel(fmin), mx = hz_to_mel(fmax);
    std::vector<double> mel_f(n);
    const double lstep = (mx - mn) / (double)(n - 1);
    for (int i = 0; i < n; ++i) mel_f[i] = mel_to_hz(i == n - 1 ? mx : mn + lstep * (double)i);
    std::vector<float> row(B);
    for (int i = 0; i < n_mels; ++i) {
        const double fd0 = mel_f[i + 1] - mel_f[i], fd1 = mel_f[i + 2] - mel_f[i + 1];
        const double enorm = 2.0 / (mel_f[i + 2] - mel_f[i]);
        int first = -1, last = -1;
        for (int k = 0; k < B; ++k) {
            const double fk = (double)k * step_hz;
            const double lower = -(mel_f[i] - fk) / fd0;
            const double upper = (mel_f[i + 2] - fk) / fd1;
            double v = lower < upper ? lower : upper;
            if (!(v > 0.0)) v = 0.0;
            float wf = (float)v;                          // weights stored as float32 ...
            wf = (float)((double)wf * enorm);             // ... then `weights *= enorm` (float32 result)
            row[k] = wf;
            if (wf != 0.0f) { if (first < 0) first = k; last = k; }
        }
        t.off[i] = (int)t.w.size();
        if (first >= 0) {
            t.start[i] = first; t.len[i] = last - first + 1;
            for (int k = first; k <= last; ++k) t.w.push_back(row[k]);
        }
        if (want_dense) for (int k = 0; k < B; ++k) t.dense[(size_t)i * B + k] = row[k];
    }
    if (t.w.empty()) t.w.push_back(0.0f);
    return true;
}

// Mel projection in O(bins) per lane ("interval form", frame kernel with more than one frame per warp).  Slaney filters are
// triangles over consecutive mel points f_0 < f_1 < ...: a bin between f_i and f_(i+1) feeds exactly two filters -- filter i with its
// RISING weight and filter i-1 with its FALLING weight.  With the G lanes of a frame owning E contiguous bins each, the projection is
// two running sums per bin (restarted at interval starts and at the lane's first bin) whose interval totals are then combined per
// filter from a short pick list.  The weights are taken from the exact float32 filter table (MelTable::dense), so the result differs
// from the tap sweep only in summation order.
//   blob (float4 units): [0, M/2)            {wr(2i), wf(2i), wr(2i+1), wf(2i+1)} of lane j at index i*G + j   (M = G*E bins)
//                        [M/2, M/2 + n)       per filter one int4 {r0, r1, f0, f1}: word indices of its (at most two) rise totals in CR
//                                             and fall totals in CF; both arrays use the padded spectrum layout k + 4 (k / 32), CF
//                                             starts PSM = M + M/8 words after CR; unused picks point at word 2 PSM (kept zero)
//                        [.., + ceil(G/4))    per lane one uint: bit b set = bin b of the lane continues its predecessor's interval
//                        [.., + 1)            {weight of the Nyquist bin in the last filter, 0, 0, 0}
struct MelIntervals { bool ok = false; std::vector<float> blob; int f4 = 0; };

inline void build_mel_intervals(double sr, int n_fft, int n_mels, double fmin, double fmax, const MelTable& t, int E, int G,
                                MelIntervals& out) {
    out.ok = false;
    const int M = n_fft / 2, B = M + 1;
    if (G * E != M || t.dense.size() != (size_t)n_mels * B || E > 32 || (E & 3)) return;
    if (fmax <= 0) fmax = sr / 2.0;
    const int n = n_mels + 2;
    const double mn = hz_to_mel(fmin), mx = hz_to_mel(fmax), lstep = (mx - mn) / (double)(n - 1), step_hz = bin_hz(sr, n_fft);
    std::vector<double> mel_f(n);
    for (int i = 0; i < n; ++i) mel_f[i] = mel_to_hz(i == n - 1 ? mx : mn + lstep * (double)i);
    std::vector<int> iv(M);                                     // interval of bin k: largest i with mel_f[i] <= f_k (-1: below fmin)
    for (int k = 0; k < M; ++k) {
        const double fk = (double)k * step_hz;
        int i = -1;
        while (i + 1 < n && mel_f[i + 1] <= fk) ++i;
        iv[k] = i;
    }
    auto rise = [&](int k) { return (iv[k] >= 0 && iv[k] <= n_mels - 1) ? iv[k] : -1; };
    auto fall = [&](int k) { return (iv[k] - 1 >= 0 && iv[k] - 1 <= n_mels - 1) ? iv[k] - 1 : -1; };
    // the model must reproduce the filter table exactly: every non-zero weight belongs to the bin's rise or fall filter
    // Nyquist bin: outside the lanes' bins.  Only the LAST filter may weight it (fmax = sr/2: its falling edge ends there; the float
    // table holds rounding dust such as 7.7e-18 for 44.1 kHz / 2048 / 128 mels): the kernel adds that one product explicitly.
    for (int m = 0; m < n_mels; ++m) {
        if (m != n_mels - 1 && t.dense[(size_t)m * B + M] != 0.0f) return;
        for (int k = 0; k < M; ++k)
            if (t.dense[(size_t)m * B + k] != 0.0f && m != rise(k) && m != fall(k)) return;
    }
    const int f4_w = M / 2, f4_p = n_mels, f4_k = (G + 3) / 4;
    if (M % 32) return;
    const int PSM = M + M / 8;                                  // padded length of CR (and of CF)
    auto pad = [](int k) { return k + ((k >> 5) << 2); };
    out.f4 = f4_w + f4_p + f4_k + 1;                            // + one float4: {weight of the Nyquist bin in the last filter, 0, 0, 0}
    out.blob.assign((size_t)out.f4 * 4, 0.0f);
    out.blob[(size_t)(f4_w + f4_p + f4_k) * 4] = t.dense[(size_t)(n_mels - 1) * B + M];
    for (int j = 0; j < G; ++j)
        for (int b = 0; b < E; ++b) {
            const int k = j * E + b;
            const float wr = rise(k) >= 0 ? t.dense[(size_t)rise(k) * B + k] : 0.0f;
            const float wf = fall(k) >= 0 ? t.dense[(size_t)fall(k) * B + k] : 0.0f;
            float* q = &out.blob[((size_t)(b / 2) * G + j) * 4 + (b & 1) * 2];
            q[0] = wr; q[1] = wf;
        }
    int* picks = reinterpret_cast<int*>(&out.blob[(size_t)f4_w * 4]);
    for (int m = 0; m < n_mels; ++m) {
        int nr = 0, nf = 0;
        int* pr = picks + (size_t)m * 4;
        for (int q = 0; q < 4; ++q) pr[q] = 2 * PSM;
        for (int k = 0; k < M; ++k) {
            const bool lane_end = (k % E) == E - 1;
            if (rise(k) == m && (lane_end || k == M - 1 || iv[k + 1] != iv[k])) { if (nr == 2) return; pr[nr++] = pad(k); }
            if (fall(k) == m && (lane_end || k == M - 1 || iv[k + 1] != iv[k])) { if (nf == 2) return; pr[2 + nf++] = PSM + pad(k); }
        }
    }
    unsigned* keep = reinterpret_cast<unsigned*>(&out.blob[(size_t)(f4_w + f4_p) * 4]);
    for (int j = 0; j < G; ++j) {
        unsigned bits = 0;
        for (int b = 1; b < E; ++b)
            if (iv[j * E + b] == iv[j * E + b - 1]) bits |= 1u << b;
        keep[j] = bits;
    }
    out.ok = true;
}

// Mel filters re-expressed for the warp kernel: "slots" sorted by span (longest first, so the 32 lanes of a warp
// sweep filters of similar length), taps indexed in the PADDED power-spectrum space (padi(k) = k + k/32, a zero
// weight at every pad position) and padded to a multiple of 4 taps.  desc = {filter m, padded start, taps, offset}.
struct MelSlots { std::vector<int> desc; std::vector<float> w; };

inline void build_mel_slots(const MelTable& t, MelSlots& s, int n_bins, int gs) {
    // Slots live in the warp kernel's padded spectrum space: ppad(k) = k + 4 * (k / 32) (4 pad words after every 32 bins).
    // Filters are sorted by span and taken gs at a time (gs = 32 / frames-per-warp: the warp sweeps gs filters of each of
    // its frames at once); every slot of a group spans the same number L of float4 steps (the group's longest filter, zero
    // weights elsewhere) so the sweep has a warp-uniform trip count, and the group's taps are interleaved [step][slot] so
    // one 128-bit read per step is contiguous across the lanes.
    //   desc[slot] = {filter, first padded word (multiple of 4), L, offset of the group's taps in float4 units}
    auto ppad = [](int k) { return k + ((k >> 5) << 2); };
    const int ps_words = ((n_bins + 4 * (n_bins >> 5) + 48 + 3) / 4) * 4;     // = WarpTile::PS
    std::vector<int> order(t.n_mels);
    for (int i = 0; i < t.n_mels; ++i) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return t.len[a] > t.len[b]; });
    s.desc.assign((size_t)t.n_mels * 4, 0);
    s.w.clear();
    for (int g0 = 0; g0 < t.n_mels; g0 += gs) {
        const int gn = std::min(gs, t.n_mels - g0);
        int L = 1;
        std::vector<int> pst(gn, 0), len(gn, 1);
        for (int j = 0; j < gn; ++j) {
            const int m = order[g0 + j];
            if (t.len[m] <= 0) continue;
            pst[j] = ppad(t.start[m]) & ~3;
            len[j] = (ppad(t.start[m] + t.len[m] - 1) - pst[j] + 1 + 3) / 4;
            L = std::max(L, len[j]);
        }
        // Bank conflicts: the 8 lanes of a quarter warp read one float4 each per step; they are conflict free when their
        // first float4 indices differ mod 8 (all lanes advance together).  A slot may start up to 7 float4 earlier (zero
        // weights in front), which costs steps only if it pushes the slot beyond the group's longest; per quarter the
        // assignment of residues that minimises that overshoot is found by exhaustive search (8! orders, plan time only).
        for (int q0 = 0; q0 < gn; q0 += 8) {
            const int qn = std::min(8, gn - q0);
            int perm[8] = {0, 1, 2, 3, 4, 5, 6, 7}, best[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            long best_cost = -1;
            do {
                long cost = 0;
                int over = 0;
                for (int j = 0; j < qn; ++j) {
                    const int res = (pst[q0 + j] / 4) & 7;
                    int d = (res - perm[j]) & 7;                          // float4 steps to move the start down
                    if (pst[q0 + j] - 4 * d < 0) d = 0;                    // cannot start before the spectrum: keep (may conflict)
                    over = std::max(over, len[q0 + j] + d);
                    cost += d;
                }
                const long c = (long)std::max(over, L) * 1000 + cost;      // first the group length, then the total padding
                if (best_cost < 0 || c < best_cost) { best_cost = c; for (int j = 0; j < 8; ++j) best[j] = perm[j]; }
            } while (std::next_permutation(perm, perm + 8));
            for (int j = 0; j < qn; ++j) {
                const int res = (pst[q0 + j] / 4) & 7;
                int d = (res - best[j]) & 7;
                if (pst[q0 + j] - 4 * d < 0) d = 0;
                pst[q0 + j] -= 4 * d;
                len[q0 + j] += d;
                L = std::max(L, len[q0 + j]);
            }
        }
        L = (L + 1) / 2 * 2;                                      // the kernel sweeps four steps per iteration plus an optional tail of two
        for (int j = 0; j < gn; ++j) {                              // keep the sweep inside the buffer, and the bank residue with it
            const int limit = ps_words - 4 * L;
            if (pst[j] > limit) {
                const int keep = limit - 4 * (((limit / 4) - (pst[j] / 4)) & 7);
                pst[j] = keep >= 0 ? keep : std::max(0, limit);
            }
        }
        const int goff4 = (int)(s.w.size() / 4);
        s.w.resize(s.w.size() + (size_t)L * gs * 4, 0.0f);
        for (int j = 0; j < gn; ++j) {
            const int m = order[g0 + j];
            for (int i = 0; i < 4 * L; ++i) {
                const int p = pst[j] + i, blk = p / 36, r = p % 36, k = 32 * blk + r;
                float wv = 0.0f;
                if (t.len[m] > 0 && r < 32 && k >= t.start[m] && k < t.start[m] + t.len[m]) wv = t.w[t.off[m] + (k - t.start[m])];
                s.w[((size_t)goff4 + (size_t)(i / 4) * gs + j) * 4 + (i % 4)] = wv;
            }
            int* d = &s.desc[(size_t)(g0 + j) * 4];
            d[0] = m; d[1] = pst[j]; d[2] = L; d[3] = goff4;
        }
    }
    if (s.w.empty()) s.w.assign(4, 0.0f);
}

// rows [n_out][n_mels] of the DCT scipy.fftpack.dct(x, type, norm) restricted to the first n_out outputs,
// with librosa's sinusoidal lifter folded in.
template <class Real>
inline bool build_dct(int n_out, int N, int type, bool ortho, double lifter, int n_mfcc_for_lifter,
                      std::vector<Real>& out, std::string& err) {
    if (n_out < 1 || n_out > N) { err = "n_mfcc must be in [1, n_mels]"; return false; }
    if (lifter < 0) { err = "MFCC lifter must be a non-negative number"; return false; }
    out.assign((size_t)n_out * N, (Real)0);
    for (int k = 0; k < n_out; ++k) {
        double lift = 1.0;
        if (lifter > 0) lift = 1.0 + (lifter / 2.0) * std::sin(kPi * (double)(k + 1) / lifter);
        (void)n_mfcc_for_lifter;
        for (int n = 0; n < N; ++n) {
            double v;
            if (type == 2) {
                v = 2.0 * std::cos(kPi * (double)k * (2.0 * n + 1.0) / (2.0 * N));
                if (ortho) v *= (k == 0) ? std::sqrt(1.0 / (4.0 * N)) : std::sqrt(1.0 / (2.0 * N));
            } else if (type == 3) {
                if (ortho) v = (n == 0) ? 1.0 / std::sqrt((double)N)
                                        : std::sqrt(2.0 / N) * std::cos(kPi * (2.0 * k + 1.0) * n / (2.0 * N));
                else v = (n == 0) ? 1.0 : 2.0 * std::cos(kPi * (2.0 * k + 1.0) * n / (2.0 * N));
            } else if (type == 1 && !ortho && N >= 2) {
                if (n == 0) v = 1.0;
                else if (n == N - 1) v = (k % 2 == 0) ? 1.0 : -1.0;
                else v = 2.0 * std::cos(kPi * (double)k * n / (double)(N - 1));
            } else {
                err = "unsupported dct_type/norm combination";
                return false;
            }
            out[(size_t)k * N + n] = (Real)(v * lift);
        }
    }
    return true;
}

// all_nan: band 0 ([0, fmin]) holds bin 0 only, so its sub-band (the band minus its last row) is empty.  librosa then averages an
// empty slice for that band's peak and valley (NaN), and power_to_db's top_db clamp against the maximum of the whole array spreads
// the NaN to every band of every frame: the reference returns NaN for all contrast rows of the call.
struct Bands { int nb = 0; int lo[16]; int cnt[16]; int nq[16]; bool all_nan = false; };

inline bool build_bands(double sr, int n_fft, int n_bands, double fmin, double quantile, Bands& b, std::string& err) {
    if (n_bands < 1 || n_bands + 1 > 12) { err = "n_bands must be in [1, 11]"; return false; }
    if (!(quantile > 0.0 && quantile < 1.0)) { err = "quantile must lie in the range (0, 1)"; return false; }
    if (!(fmin > 0)) { err = "fmin must be a positive number"; return false; }
    const int B = 1 + n_fft / 2;
    const double step = bin_hz(sr, n_fft);
    std::vector<double> octa(n_bands + 2, 0.0);
    for (int i = 1; i < n_bands + 2; ++i) octa[i] = fmin * std::pow(2.0, (double)(i - 1));
    for (int i = 0; i < n_bands + 1; ++i)
        if (octa[i] >= 0.5 * sr) { err = "Frequency band exceeds Nyquist. Reduce either fmin or n_bands."; return false; }
    b.nb = n_bands + 1;
    b.all_nan = false;
    for (int k = 0; k <= n_bands; ++k) {
        const double lo = octa[k], hi = octa[k + 1];
        int first = -1, last = -1;
        for (int i = 0; i < B; ++i) {
            const double f = (double)i * step;
            if (f >= lo && f <= hi) { if (first < 0) first = i; last = i; }
        }
        if (first < 0) { err = "spectral_contrast band without FFT bins"; return false; }
        if (k > 0) first = (first > 0) ? first - 1 : first;
        if (k == n_bands) last = B - 1;
        const int total = last - first + 1;
        const int rows = total - (k < n_bands ? 1 : 0);
        double q = std::nearbyint(quantile * (double)total);      // np.rint (half to even)
        int nq = (int)(q < 1.0 ? 1.0 : q);
        b.lo[k] = first; b.cnt[k] = rows; b.nq[k] = nq;
        if (rows == 0) b.all_nan = true;                          // band 0 only: a later band always takes its predecessor's last bin
    }
    return true;
}

// segment_fixed_length boundary arithmetic (segmentation.py:62-114)
inline int64_t segment_table(int64_t total, double sr, double sec, double ovl, bool pad, double min_sec,
                             int64_t* seg_len, int64_t* seg_hop, int64_t* starts, int32_t* valid, int64_t cap,
                             std::string& err) {
    if (!(sec > 0)) { err = "segment_length_sec must be positive."; return -1; }
    if (!(ovl >= 0.0 && ovl < 1.0)) { err = "overlap_ratio must be between 0.0 and < 1.0."; return -1; }
    const int64_t seg = (int64_t)(sec * sr);                    // int() truncation (:62)
    if (seg_len) *seg_len = seg;
    if (seg == 0) { if (seg_hop) *seg_hop = 0; return 0; }
    int64_t hop = (int64_t)((double)seg * (1.0 - ovl));         // :67
    if (hop < 1) hop = 1;
    if (seg_hop) *seg_hop = hop;
    const int64_t min_samples = (min_sec >= 0) ? (int64_t)(min_sec * sr) : 0;   // :71
    int64_t n = 0;
    for (int64_t start = 0; start < total; start += hop) {
        const int64_t end = start + seg;
        const int64_t orig = (end < total ? end : total) - start;
        bool keep = false;
        if (min_samples > 0 && orig < min_samples) keep = false;
        else if (end > total) keep = pad;
        else keep = true;
        if (keep) {
            if (starts && n < cap) starts[n] = start;
            if (valid && n < cap) valid[n] = (int32_t)orig;
            ++n;
        }
        if (!pad && start + hop + seg > total) break;            // :113-114
    }
    return n;
}

}  // namespace sygplan
