// sygnals_b200/csrc/syg_kernels.cuh
//
// Kernels of the segment -> features path (reference: sygnals/core/features/manager.py:78-445 and the librosa
// routines it calls, SURVEY.md section 2.3).
//
//   frame_kernel<TL, MODE>   framing (zero / reflect padding by index arithmetic, no frame tensor) -> window ->
//                            packed real FFT in registers + shared memory -> |X|^2 ->
//                              MODE_FEATURES: mel energies, spectral contrast peaks/valleys, centroid, rolloff,
//                                             bandwidth, flatness, dominant frequency, rms, crest, peak, ...
//                              MODE_STFT:     complex / magnitude / power spectrogram  (dsp.py:167-229)
//   finalize_kernel          per unit: power_to_db(ref=max, top_db) + DCT-II -> MFCC rows; contrast dB rows
//   welch_kernel<TL>         per unit: detrend -> window -> FFT -> |X|^2 averaged over sub-segments (+ rms/crest)
#pragma once

#include "syg_device.cuh"
#include "syg_params.h"

namespace sygdev {

constexpr double kEps64 = 2.220446049250313e-16;   // np.finfo(float64).eps: frequency_domain.py:21, time_domain.py:21

template <class TL>
struct FrameSmem {
    static constexpr int F = TL::F;
    static constexpr int off_re = 0;
    static constexpr int off_im = off_re + F * TL::MP;
    static constexpr int off_pw = off_im + F * TL::MP;
    static constexpr int off_cand = off_pw + F * TL::PW;                // 8 warps x 32 floats
    static constexpr int off_smax = off_cand + (kThreads / 32) * 32;    // F x 4 unsigned
    static constexpr int off_dsc_f = ((off_smax + F * 4 + 1) / 2) * 2;   // doubles start (8-byte aligned)
    static constexpr int n_dsc = kThreads / 32 + kThreads;              // group scratch + inclusive-prefix exchange
    static constexpr size_t bytes = (size_t)off_dsc_f * 4 + (size_t)n_dsc * 8;
};

struct UnitRef { long long start; long long valid; };

SYG_DEVICE SYG_INLINE UnitRef unit_ref(const syg::UnitGeom& g, long long u) {
    UnitRef r;
    r.start = g.unit_starts ? g.unit_starts[u] : (u + g.unit0) * g.unit_stride;
    long long v;
    if (g.unit_valid) v = g.unit_valid[u];
    else v = g.total_len - r.start;
    if (v > g.unit_len) v = g.unit_len;
    if (v < 0) v = 0;
    r.valid = v;
    return r;
}

SYG_DEVICE SYG_INLINE long long reflect_index(long long pos, long long L) {
    if (L <= 1) return 0;
    const long long period = 2 * (L - 1);
    long long m = pos % period;
    if (m < 0) m += period;
    return (m >= L) ? period - m : m;
}

// two consecutive samples (pos, pos+1) of a unit, with the padding rule applied
SYG_DEVICE SYG_INLINE float2 load_pair(const float* __restrict__ y, const UnitRef& u, long long pos, int pad_mode) {
    float2 v;
    if (pad_mode == 0) {
        const float* p = y + u.start + pos;
        if (pos >= 0 && pos + 1 < u.valid) {
            if ((reinterpret_cast<uintptr_t>(p) & 7u) == 0) {
                v = __ldg(reinterpret_cast<const float2*>(p));
            } else {
                v.x = __ldg(p);
                v.y = __ldg(p + 1);
            }
        } else {
            v.x = (pos >= 0 && pos < u.valid) ? __ldg(p) : 0.0f;
            v.y = (pos + 1 >= 0 && pos + 1 < u.valid) ? __ldg(p + 1) : 0.0f;
        }
    } else {
        if (u.valid <= 0) { v.x = 0.0f; v.y = 0.0f; return v; }
        v.x = __ldg(y + u.start + reflect_index(pos, u.valid));
        v.y = __ldg(y + u.start + reflect_index(pos + 1, u.valid));
    }
    return v;
}

template <class TL, int MODE>
__global__ void __launch_bounds__(kThreads) frame_kernel(const syg::FrameArgs a) {
    constexpr int E = TL::E, M = TL::M, G = TL::G, F = TL::F, MP = TL::MP, PW = TL::PW;
    using SM = FrameSmem<TL>;
    SYG_DYN_SMEM(smem_raw);
    float* const smf = reinterpret_cast<float*>(smem_raw);
    float* const sre = smf + SM::off_re;
    float* const sim = smf + SM::off_im;
    float* const pw = smf + SM::off_pw;
    float* const cand = smf + SM::off_cand;
    unsigned* const smax = reinterpret_cast<unsigned*>(smf + SM::off_smax);
    double* const dsc = reinterpret_cast<double*>(smf + SM::off_dsc_f);
    double* const dinc = dsc + kThreads / 32;

    const int tid = threadIdx.x;
    const int f = tid / G, j = tid % G;
    const int warp = tid >> 5, lane = tid & 31;
    const long long n_rounds = (a.n_frames + F - 1) / F;
    const int B = M + 1;
    constexpr bool RAG = (MODE == MODE_FEATURES_RAGGED);

    for (long long round = blockIdx.x; round < n_rounds; round += gridDim.x) {
        const long long gf = round * F + f;
        const bool valid = gf < a.n_frames;
        const int4 rut = (RAG && valid) ? __ldg(a.ragged_ut + gf) : make_int4(0, 0, 0, 0);
        const long long u = RAG ? (long long)rut.x : (valid ? gf / a.T : 0);
        const int t = RAG ? rut.y : (valid ? (int)(gf - u * a.T) : 0);
        UnitRef ur = RAG ? UnitRef{(long long)rut.w, (long long)rut.z} : unit_ref(a.g, u);
        if (!valid) ur.valid = 0;
        const long long p0 = (long long)t * a.hop - a.cpad;

        if (MODE != MODE_STFT) {
            for (int i = tid; i < F * 4; i += kThreads) smax[i] = 0u;
        }

        // ---------------- framing + window + time-domain partial statistics ----------------
        float xr[E], xi[E];
        double s_sq = 0.0, s_sum = 0.0, s_abs = 0.0;
        float pk = 0.0f;
        SYG_UNROLL
        for (int r = 0; r < E; ++r) {
            const int c = j + r * G;
            const float2 v = load_pair(a.y, ur, p0 + 2 * c, a.pad_mode);
            const float2 w = __ldg(reinterpret_cast<const float2*>(a.window) + c);
            if (MODE != MODE_STFT) {
                s_sq += (double)v.x * (double)v.x + (double)v.y * (double)v.y;
                s_sum += (double)v.x + (double)v.y;
                s_abs += (double)fabsf(v.x) + (double)fabsf(v.y);
                pk = fmaxf(pk, fmaxf(fabsf(v.x), fabsf(v.y)));
            }
            xr[r] = v.x * w.x;
            xi[r] = v.y * w.y;
        }

        // ---------------- packed real FFT ----------------
        fft_tile_forward<TL>(xr, xi, sre, sim, f, j, a.tw);

        // ---------------- real split -> X[k] ----------------
        {
            const int fb = f * MP;
            const long long ob = (MODE == MODE_STFT) ? ((long long)u * B) * a.T + t : 0;
            SYG_UNROLL
            for (int i = 0; i <= E / 2; ++i) {
                const int k = j + i * G;
                if (i == E / 2 && j != 0) break;          // only the k = M/2 self-pair remains
                const int km = (M - k) & (M - 1);
                const float zkr = SLD(&sre[fb + padi(k)]), zki = SLD(&sim[fb + padi(k)]);
                const float zmr = SLD(&sre[fb + padi(km)]), zmi = SLD(&sim[fb + padi(km)]);
                const float2 w = __ldg(&a.tws[k]);
                float xkr, xki, xmr, xmi;
                real_split(zkr, zki, zmr, zmi, w.x, w.y, xkr, xki, xmr, xmi);
                const int k2 = M - k;                      // k = 0 -> bin M (Nyquist); k = M/2 -> itself
                if (MODE != MODE_STFT) {
                    SST(&pw[f * PW + padi(k)], __fmaf_rn(xkr, xkr, xki * xki));
                    if (k2 != k) SST(&pw[f * PW + padi(k2)], __fmaf_rn(xmr, xmr, xmi * xmi));
                } else if (valid) {
                    if (a.out_kind == 0) {
                        float2* o = reinterpret_cast<float2*>(a.stft_out);
                        o[ob + (long long)k * a.T] = make_float2(xkr, xki);
                        if (k2 != k) o[ob + (long long)k2 * a.T] = make_float2(xmr, xmi);
                    } else {
                        float* o = reinterpret_cast<float*>(a.stft_out);
                        float pk_ = __fmaf_rn(xkr, xkr, xki * xki), pm_ = __fmaf_rn(xmr, xmr, xmi * xmi);
                        if (a.out_kind == 1) { pk_ = sqrt_approx(pk_); pm_ = sqrt_approx(pm_); }   // MUFU.SQRT: 1 ulp, one instruction (sqrtf is ~8)
                        o[ob + (long long)k * a.T] = pk_;
                        if (k2 != k) o[ob + (long long)k2 * a.T] = pm_;
                    }
                }
            }
        }
        if (MODE == MODE_STFT) {
            __syncthreads();        // sre/sim are rewritten by the next round's first pass
            continue;
        }
        __syncthreads();

        float* const orow = RAG ? a.out + gf : a.out + (long long)u * a.n_rows * a.T + t;

        // ---------------- time-domain features (unwindowed, zero-padded frame) ----------------
        if (a.mask & syg::FB_TIME_ANY) {
            const double tsq = group_sum<G>(s_sq, dsc);
            const float tpk = group_max<G>(pk, dsc);
            double tsum = 0.0, tabs = 0.0;
            if (a.mask & (syg::FB_STD_AMP | syg::FB_MEAN_AMP)) {
                tsum = group_sum<G>(s_sum, dsc);
                tabs = group_sum<G>(s_abs, dsc);
            }
            if (j == 0 && valid) {
                const double n = (double)TL::NFFT;
                const double rms = sqrt(tsq / n);
                if (a.row_rms >= 0) orow[(long long)a.row_rms * (RAG ? a.ragged_stride : a.T)] = (float)rms;
                if (a.row_crest >= 0) orow[(long long)a.row_crest * (RAG ? a.ragged_stride : a.T)] = (rms < kEps64) ? 0.0f : (float)((double)tpk / rms);
                if (a.row_peak >= 0) orow[(long long)a.row_peak * (RAG ? a.ragged_stride : a.T)] = tpk;
                if (a.row_mean_amp >= 0) orow[(long long)a.row_mean_amp * (RAG ? a.ragged_stride : a.T)] = (float)(tabs / n);
                if (a.row_std_amp >= 0) {
                    const double mu = tsum / n;
                    double var = tsq / n - mu * mu;
                    if (var < 0.0) var = 0.0;
                    orow[(long long)a.row_std_amp * (RAG ? a.ragged_stride : a.T)] = (float)sqrt(var);
                }
            }
        }

        // ---------------- per-frame spectral statistics ----------------
        if (a.mask & syg::FB_SPECSTATS) {
            // thread j owns the contiguous bins [j*E, j*E + E) (+ bin M for the last thread of the group)
            const float* pf = pw + f * PW;
            const int k0 = j * E;
            const int nk = E + ((j == G - 1) ? 1 : 0);
            double sp = 0.0, sm = 0.0, skm = 0.0, slog = 0.0;
            float vmax = -1.0f;
            int imax = 0;
            for (int i = 0; i < nk; ++i) {
                const float p = SLD(&pf[padi(k0 + i)]);
                const float mg = sqrtf(p);
                sp += (double)p;
                sm += (double)mg;
                skm += (double)mg * (double)(k0 + i);
                if (a.mask & syg::FB_FLATNESS) slog += (double)logf(mg + 2.220446049250313e-16f);
                if (p > vmax) { vmax = p; imax = k0 + i; }
            }
            const double incl = group_scan_incl<G>(sp, dsc);
            __syncthreads();
            dinc[tid] = incl;
            __syncthreads();
            const double total_p = dinc[f * G + G - 1];
            const double prev = (j == 0) ? -1.0 : dinc[tid - 1];
            const double tm = group_sum<G>(sm, dsc);
            const double tkm = group_sum<G>(skm, dsc);
            double centroid_hz = 0.0;
            if (tm >= kEps64) centroid_hz = a.bin_hz * (tkm / tm);
            if (a.row_centroid >= 0 && j == 0 && valid) orow[(long long)a.row_centroid * (RAG ? a.ragged_stride : a.T)] = (float)centroid_hz;
            if (a.row_rolloff >= 0) {
                if (total_p < kEps64) {
                    if (j == 0 && valid) orow[(long long)a.row_rolloff * (RAG ? a.ragged_stride : a.T)] = (float)(a.bin_hz * (double)M);
                } else {
                    const double thr = a.roll_percent * total_p;
                    if (incl >= thr && prev < thr) {           // exactly one thread of the group
                        double c = (j == 0) ? 0.0 : prev;
                        int bin = k0 + nk - 1;
                        for (int i = 0; i < nk; ++i) {
                            c += (double)SLD(&pf[padi(k0 + i)]);
                            if (c >= thr) { bin = k0 + i; break; }
                        }
                        if (valid) orow[(long long)a.row_rolloff * (RAG ? a.ragged_stride : a.T)] = (float)(a.bin_hz * (double)bin);
                    }
                }
            }
            if (a.row_flatness >= 0) {
                const double tl = group_sum<G>(slog, dsc);
                if (j == 0 && valid) {
                    const double am = tm / (double)B;
                    double fl = 0.0;
                    if (am >= kEps64) {
                        fl = exp(tl / (double)B) / am;
                        fl = fl < 0.0 ? 0.0 : (fl > 1.0 ? 1.0 : fl);
                    }
                    orow[(long long)a.row_flatness * (RAG ? a.ragged_stride : a.T)] = (float)fl;
                }
            }
            if (a.row_bandwidth >= 0) {
                double sb = 0.0;
                for (int i = 0; i < nk; ++i) {
                    const double mg = (double)sqrtf(SLD(&pf[padi(k0 + i)]));
                    const double d = a.bin_hz * (double)(k0 + i) - centroid_hz;
                    sb += mg * d * d;
                }
                const double tb = group_sum<G>(sb, dsc);
                if (j == 0 && valid) orow[(long long)a.row_bandwidth * (RAG ? a.ragged_stride : a.T)] = (tm < kEps64) ? 0.0f : (float)sqrt(tb / tm);
            }
            if (a.row_dominant >= 0) {
                // np.argmax: first bin attaining the maximum = smallest index among the threads holding it
                const float gmax = group_max<G>(vmax, dsc);
                float mi = (vmax == gmax) ? -(float)imax : -1.0e9f;
                mi = group_max<G>(mi, dsc);
                if (j == 0 && valid) orow[(long long)a.row_dominant * (RAG ? a.ragged_stride : a.T)] = (float)(a.bin_hz * (double)(-mi));
            }
        }

        // ---------------- mel energies (sparse triangular filters) ----------------
        if (a.mask & syg::FB_MFCC) {
            const int ntask = F * a.n_mels;
            for (int base = 0; base < ntask; base += kThreads) {
                const int task = base + tid;
                const bool act = task < ntask;
                const int ff = act ? task / a.n_mels : 0;
                const int m = act ? task - ff * a.n_mels : 0;
                float acc = 0.0f;
                if (act) {
                    const int st = __ldg(&a.mel_start[m]), ln = __ldg(&a.mel_len[m]);
                    const float* wv = a.mel_w + __ldg(&a.mel_off[m]);
                    const float* pf = pw + ff * PW;
                    if (a.mel_power_is_2) {
                        for (int i = 0; i < ln; ++i) acc = __fmaf_rn(__ldg(&wv[i]), SLD(&pf[padi(st + i)]), acc);
                    } else {
                        for (int i = 0; i < ln; ++i) acc = __fmaf_rn(__ldg(&wv[i]), powf(SLD(&pf[padi(st + i)]), a.mel_half_power), acc);
                    }
                    const long long gff = round * F + ff;
                    if (gff < a.n_frames) a.melws[gff * a.n_mels + m] = acc;
                    else acc = 0.0f;
                }
                // per-frame maximum -> shared slot
                const unsigned bits = __float_as_uint(acc);
                const int ff0 = __shfl_sync(kFull, ff, 0);
                if (__all_sync(kFull, ff == ff0)) {
                    const unsigned mx = __reduce_max_sync(kFull, bits);
                    if (lane == 0) atomicMax(&smax[ff0 * 4 + 0], mx);
                } else if (act) {
                    atomicMax(&smax[ff * 4 + 0], bits);
                }
            }
        }

        // ---------------- spectral contrast: per band mean of the n largest / n smallest magnitudes ----------------
        if (a.mask & syg::FB_CONTRAST) {
            const int ntask = F * a.nb;
            float* mycand = cand + warp * 32;
            for (int task = warp; task < ntask; task += kThreads / 32) {
                const int ff = task / a.nb, bd = task - ff * a.nb;
                const float* pf = pw + ff * PW;
                const float peak = warp_extreme_mean_sqrt<+1>(pf, a.band_lo[bd], a.band_cnt[bd], a.band_n[bd], mycand);
                const float valley = warp_extreme_mean_sqrt<-1>(pf, a.band_lo[bd], a.band_cnt[bd], a.band_n[bd], mycand);
                const long long gff = round * F + ff;
                if (lane == 0 && gff < a.n_frames) {
                    a.cws[gff * (2 * a.nb) + bd] = peak;
                    a.cws[gff * (2 * a.nb) + a.nb + bd] = valley;
                    if (peak == peak) atomicMax(&smax[ff * 4 + 1], __float_as_uint(peak));
                    if (valley == valley) atomicMax(&smax[ff * 4 + 2], __float_as_uint(valley));
                }
            }
        }

        // ---------------- publish per-unit maxima ----------------
        __syncthreads();
        if (a.mask & (syg::FB_MFCC | syg::FB_CONTRAST)) {
            for (int i = tid; i < F * 4; i += kThreads) {
                const int ff = i >> 2, slot = i & 3;
                const long long gff = round * F + ff;
                if (slot < 3 && gff < a.n_frames) {
                    const unsigned v = smax[i];
                    if (v) atomicMax(&a.unit_max[(RAG ? (long long)__ldg(a.ragged_ut + gff).x : gff / a.T) * 4 + slot], v);
                }
            }
        }
    }
}

// --------------------------------------------------------------------------------------------------------
// stft_tile_kernel<TL, TT>: STFT output for the large transforms (n_fft 4096 / 8192; the warp kernel covers the rest).
// A CTA owns TT consecutive frames at a time: its F = kThreads / G frame groups run TT / F rounds of the CTA-cooperative FFT,
// every round drops X / |X| / |X|^2 into a transposed shared-memory tile [B][TT + 1], then the tile leaves as rows of TT
// consecutive frames per bin -- the reference layout is (1 + n_fft/2, T) with frames innermost (dsp.py:167-229), so per-frame
// stores would touch one 32-byte sector for every 4-byte value.
// --------------------------------------------------------------------------------------------------------
template <class TL, int TT>
struct StftTileSmem {
    static constexpr int F = TL::F;
    static constexpr int off_re = 0;
    static constexpr int off_im = off_re + F * TL::MP;
    static constexpr int off_slot = ((off_im + F * TL::MP + 1) / 2) * 2;          // long long [TT]
    static constexpr int off_tile = off_slot + 2 * TT;                             // [B][TT + 1] float (x2 for complex)
    static size_t bytes(bool complex_out) { return ((size_t)off_tile + (size_t)(TL::M + 1) * (TT + 1) * (complex_out ? 2 : 1)) * 4; }
};

template <class TL, int TT>
__global__ void __launch_bounds__(kThreads) stft_tile_kernel(const syg::FrameArgs a) {
    constexpr int E = TL::E, M = TL::M, G = TL::G, F = TL::F, MP = TL::MP, TTP = TT + 1;
    static_assert(TT % F == 0 && kThreads % TT == 0, "tile geometry");
    using SM = StftTileSmem<TL, TT>;
    SYG_DYN_SMEM(smem_raw);
    float* const smf = reinterpret_cast<float*>(smem_raw);
    float* const sre = smf + SM::off_re;
    float* const sim = smf + SM::off_im;
    long long* const slot_off = reinterpret_cast<long long*>(smf + SM::off_slot);
    float* const tile = smf + SM::off_tile;
    const int tid = threadIdx.x;
    const int f = tid / G, j = tid % G;
    const int B = M + 1;
    const long long n_tiles = (a.n_frames + TT - 1) / TT;

    // One CTA per SM (the tile fills shared memory), so nothing else hides the latency of a frame's global loads and most of
    // the register file is idle: the frame-invariant operands (this thread's window taps and split twiddles) stay in registers
    // for the whole kernel and the NEXT frame's samples are fetched while the current frame is transformed.
    float2 wreg[E];
    SYG_UNROLL
    for (int r = 0; r < E; ++r) wreg[r] = __ldg(reinterpret_cast<const float2*>(a.window) + j + r * G);
    float2 twsreg[E / 2 + 1];
    SYG_UNROLL
    for (int i = 0; i <= E / 2; ++i) twsreg[i] = (i < E / 2 || j == 0) ? __ldg(&a.tws[j + i * G]) : make_float2(0.0f, 0.0f);
    float2 vn[E];                                                   // samples of the frame this thread group transforms next
    long long off_n = -1;                                           // its output offset (u, bin 0, t), -1 = past the end
    auto fetch = [&](long long gf) {
        const bool valid = gf < a.n_frames;
        const long long u = valid ? gf / a.T : 0;
        const int t = valid ? (int)(gf - u * a.T) : 0;
        UnitRef ur = unit_ref(a.g, u);
        if (!valid) ur.valid = 0;
        const long long p0 = (long long)t * a.hop - a.cpad;
        SYG_UNROLL
        for (int r = 0; r < E; ++r) vn[r] = load_pair(a.y, ur, p0 + 2 * (j + r * G), a.pad_mode);
        off_n = valid ? ((long long)u * B) * a.T + t : -1;
    };
    fetch((long long)blockIdx.x * TT + f);

    for (long long tl = blockIdx.x; tl < n_tiles; tl += gridDim.x) {
        for (int r0 = 0; r0 < TT; r0 += F) {
            const int slot = r0 + f;
            if (j == 0) slot_off[slot] = off_n;
            float xr[E], xi[E];
            SYG_UNROLL
            for (int r = 0; r < E; ++r) {
                xr[r] = vn[r].x * wreg[r].x;
                xi[r] = vn[r].y * wreg[r].y;
            }
            // prefetch: next round of this tile, or the first round of this CTA's next tile (frames past the end load nothing)
            fetch((r0 + F < TT) ? tl * TT + (r0 + F + f) : (tl + gridDim.x) * TT + f);
            fft_tile_forward<TL>(xr, xi, sre, sim, f, j, a.tw);
            const int fb = f * MP;
            SYG_UNROLL
            for (int i = 0; i <= E / 2; ++i) {
                const int k = j + i * G;
                if (i == E / 2 && j != 0) break;
                const int km = (M - k) & (M - 1);
                const float zkr = SLD(&sre[fb + padi(k)]), zki = SLD(&sim[fb + padi(k)]);
                const float zmr = SLD(&sre[fb + padi(km)]), zmi = SLD(&sim[fb + padi(km)]);
                const float2 w = twsreg[i];
                float xkr, xki, xmr, xmi;
                real_split(zkr, zki, zmr, zmi, w.x, w.y, xkr, xki, xmr, xmi);
                const int k2 = M - k;
                if (a.out_kind == 0) {
                    float2* t2 = reinterpret_cast<float2*>(tile);
                    t2[k * TTP + slot] = make_float2(xkr, xki);
                    if (k2 != k) t2[k2 * TTP + slot] = make_float2(xmr, xmi);
                } else {
                    float pk_ = __fmaf_rn(xkr, xkr, xki * xki), pm_ = __fmaf_rn(xmr, xmr, xmi * xmi);
                    if (a.out_kind == 1) { pk_ = sqrt_approx(pk_); pm_ = sqrt_approx(pm_); }   // MUFU.SQRT: 1 ulp, one instruction (sqrtf is ~8)
                    tile[k * TTP + slot] = pk_;
                    if (k2 != k) tile[k2 * TTP + slot] = pm_;
                }
            }
            __syncthreads();                                        // sre / sim are rewritten by the next round; tile complete after the last
        }
        // rows of TT consecutive frames per bin: thread -> (slot = tid % TT, bins tid / TT + i * kThreads / TT)
        constexpr int KS = kThreads / TT;
        const int sl = tid % TT, kq = tid / TT;
        const long long off = slot_off[sl];
        if (off >= 0) {
            const long long dstep = (long long)KS * a.T;
            if (a.out_kind == 0) {
                const float2* src = reinterpret_cast<const float2*>(tile) + kq * TTP + sl;
                float2* dst = reinterpret_cast<float2*>(a.stft_out) + off + (long long)kq * a.T;
                for (int k = kq; k < B; k += KS, src += KS * TTP, dst += dstep) *dst = *src;
            } else {
                const float* src = tile + kq * TTP + sl;
                float* dst = reinterpret_cast<float*>(a.stft_out) + off + (long long)kq * a.T;
                for (int k = kq; k < B; k += KS, src += KS * TTP, dst += dstep) *dst = *src;
            }
        }
        __syncthreads();                                            // the tile is refilled by the next one
    }
}

// --------------------------------------------------------------------------------------------------------
// Welch / periodogram PSD, one CTA per unit (grid-stride).  scipy.signal.welch semantics (dsp.py:495-560):
// per sub-segment: detrend('constant') -> window -> rfft(nfft) -> |X|^2 * scale; mean over sub-segments;
// one-sided doubling except DC / Nyquist.  Optional per-unit rms / crest / peak over the whole unit
// (time_domain.py:149-184 applied to the unit) for BASELINE config 5.
// --------------------------------------------------------------------------------------------------------
template <class TL>
struct WelchSmem {
    static constexpr int F = TL::F;
    static constexpr int off_re = 0;
    static constexpr int off_im = off_re + F * TL::MP;
    static constexpr int off_acc = off_im + F * TL::MP;
    static constexpr int off_dsc_f = ((off_acc + F * TL::PW + 1) / 2) * 2;
    static constexpr int n_dsc = kThreads / 32 + kThreads;
    static constexpr size_t bytes = (size_t)off_dsc_f * 4 + (size_t)n_dsc * 8;
};

template <class TL>
__global__ void __launch_bounds__(kThreads) welch_kernel(const syg::WelchArgs a) {
    constexpr int E = TL::E, M = TL::M, G = TL::G, F = TL::F, MP = TL::MP, PW = TL::PW;
    using SM = WelchSmem<TL>;
    SYG_DYN_SMEM(smem_raw);
    float* const smf = reinterpret_cast<float*>(smem_raw);
    float* const sre = smf + SM::off_re;
    float* const sim = smf + SM::off_im;
    float* const pacc = smf + SM::off_acc;
    double* const dsc = reinterpret_cast<double*>(smf + SM::off_dsc_f);
    double* const dred = dsc + kThreads / 32;
    const int tid = threadIdx.x;
    const int f = tid / G, j = tid % G;
    const int B = M + 1;

    for (long long u = blockIdx.x; u < a.g.n_units; u += gridDim.x) {
        const UnitRef ur = unit_ref(a.g, u);
        for (int i = tid; i < F * PW; i += kThreads) pacc[i] = 0.0f;
        const int n_rounds = (a.nseg + F - 1) / F;
        for (int round = 0; round < n_rounds; ++round) {
            const int s = round * F + f;
            const bool valid = s < a.nseg;
            UnitRef us = ur;
            if (!valid) us.valid = 0;
            const long long p0 = (long long)s * a.step;
            float xr[E], xi[E];
            double ssum = 0.0;
            SYG_UNROLL
            for (int r = 0; r < E; ++r) {
                const int c = j + r * G;
                float2 v = make_float2(0.0f, 0.0f);
                if (2 * c + 1 < a.nperseg) v = load_pair(a.y, us, p0 + 2 * c, 0);
                else if (2 * c < a.nperseg) v.x = load_pair(a.y, us, p0 + 2 * c, 0).x;
                xr[r] = v.x; xi[r] = v.y;
                ssum += (double)v.x + (double)v.y;
            }
            float mean = 0.0f;
            if (a.detrend) mean = (float)(group_sum<G>(ssum, dsc) / (double)a.nperseg);
            SYG_UNROLL
            for (int r = 0; r < E; ++r) {
                const int c = j + r * G;
                const float2 w = __ldg(reinterpret_cast<const float2*>(a.window) + c);
                xr[r] = (2 * c < a.nperseg) ? (xr[r] - mean) * w.x : 0.0f;
                xi[r] = (2 * c + 1 < a.nperseg) ? (xi[r] - mean) * w.y : 0.0f;
            }
            fft_tile_forward<TL>(xr, xi, sre, sim, f, j, a.tw);
            const int fb = f * MP;
            SYG_UNROLL
            for (int i = 0; i <= E / 2; ++i) {
                const int k = j + i * G;
                if (i == E / 2 && j != 0) break;
                const int km = (M - k) & (M - 1);
                const float zkr = SLD(&sre[fb + padi(k)]), zki = SLD(&sim[fb + padi(k)]);
                const float zmr = SLD(&sre[fb + padi(km)]), zmi = SLD(&sim[fb + padi(km)]);
                const float2 w = __ldg(&a.tws[k]);
                float xkr, xki, xmr, xmi;
                real_split(zkr, zki, zmr, zmi, w.x, w.y, xkr, xki, xmr, xmi);
                const int k2 = M - k;
                if (valid) {
                    pacc[f * PW + padi(k)] += __fmaf_rn(xkr, xkr, xki * xki);
                    if (k2 != k) pacc[f * PW + padi(k2)] += __fmaf_rn(xmr, xmr, xmi * xmi);
                }
            }
            __syncthreads();
        }
        // mean over sub-segments (fixed order -> deterministic)
        const float inv = a.scale / (float)a.nseg;
        for (int k = tid; k < B; k += kThreads) {
            float acc = 0.0f;
            for (int ff = 0; ff < F; ++ff) acc += pacc[ff * PW + padi(k)];
            float v = acc * inv;
            if (a.onesided_double && k != 0 && k != M) v *= 2.0f;
            a.psd[u * B + k] = v;
        }
        if (a.stats) {
            double sq = 0.0;
            float pk = 0.0f;
            for (long long i = tid; i < a.g.unit_len; i += kThreads) {
                const float v = (i < ur.valid) ? __ldg(a.y + ur.start + i) : 0.0f;
                sq += (double)v * (double)v;
                pk = fmaxf(pk, fabsf(v));
            }
            const double tsq = group_sum<kThreads>(sq, dsc);
            const float tpk = group_max<kThreads>(pk, dsc);
            if (tid == 0) {
                const double rms = a.g.unit_len > 0 ? sqrt(tsq / (double)a.g.unit_len) : 0.0;
                a.stats[u * 3 + 0] = (float)rms;
                a.stats[u * 3 + 1] = (rms < kEps64) ? 0.0f : (float)((double)tpk / rms);
                a.stats[u * 3 + 2] = tpk;
            }
        }
        (void)dred;
        __syncthreads();
    }
}

}  // namespace sygdev
