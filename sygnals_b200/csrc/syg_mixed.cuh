// sygnals_b200/csrc/syg_mixed.cuh
//
// Transforms whose length is NOT a power of two (frame_length 400 / 1000 / 1200, the 25 600-sample second of BASELINE config 5,
// odd lengths): one CTA (64 / 128 / 256 threads by length) per frame, a Stockham autosort FFT in shared memory with run-time radices 4 / 2 / 3 / 5 / 7 / 11 / 13.
//
//   frame_mixed_kernel<MODE>   MODE_FEATURES: the feature rows of frame_kernel (syg_kernels.cuh) for any smooth frame_length
//                              MODE_STFT:     complex / magnitude / power spectrogram (dsp.py:167-229)
//   welch_mixed_kernel         scipy.signal.welch / periodogram (dsp.py:434-560) for any smooth nfft up to 29 040
//
// Even lengths are transformed as L = n/2 packed complex points + real split (the layout of every other kernel of the engine);
// odd lengths as L = n complex points with zero imaginary parts.  The pass structure follows the autosort formulation: with Ns
// the product of the radices already applied, butterfly j reads src[j + r L/R], rotates by W_{Ns R}^{r (j mod Ns)} and writes
// dst[(j - j mod Ns) R + (j mod Ns) + r Ns]; after the last pass the spectrum is in natural order.  Twiddles are table entries
// exp(-2 pi i p / L) rounded once from float64 (never recurrences), so the error of the transform stays at the FP32 butterfly
// level for every length.
//
// These kernels serve the shapes the register-FFT kernels cannot; they are written for coverage and parity, not for the roofline:
// the power-of-two family stays on its own kernels.
#pragma once

#include "syg_device.cuh"
#include "syg_kernels.cuh"
#include "syg_params.h"

namespace sygdev {

SYG_DEVICE SYG_INLINE float load_one(const float* __restrict__ y, const UnitRef& u, long long pos, int pad_mode) {
    if (pad_mode == 0) return (pos >= 0 && pos < u.valid) ? __ldg(y + u.start + pos) : 0.0f;
    if (u.valid <= 0) return 0.0f;
    return __ldg(y + u.start + reflect_index(pos, u.valid));
}

SYG_DEVICE SYG_INLINE float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
SYG_DEVICE SYG_INLINE float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }

// R-point forward DFT, natural order in and out.  Radices 2 / 3 / 4 / 5 are written out; larger primes take the O(R^2) sum
// with the exact table entries W_R^j = tw[j L/R].
template <int R>
SYG_DEVICE SYG_INLINE void dft_small(float2* v, const float2* __restrict__ tw, int L) {
    if constexpr (R == 2) {
        const float2 a = v[0], b = v[1];
        v[0] = cadd(a, b);
        v[1] = csub(a, b);
    } else if constexpr (R == 3) {
        const float2 t1 = cadd(v[1], v[2]);
        const float2 m = make_float2(__fmaf_rn(-0.5f, t1.x, v[0].x), __fmaf_rn(-0.5f, t1.y, v[0].y));
        const float2 d = csub(v[1], v[2]);
        const float2 s = make_float2(0.86602540378443865f * d.x, 0.86602540378443865f * d.y);
        v[0] = cadd(v[0], t1);
        v[1] = make_float2(m.x + s.y, m.y - s.x);
        v[2] = make_float2(m.x - s.y, m.y + s.x);
    } else if constexpr (R == 4) {
        const float2 a0 = cadd(v[0], v[2]), a1 = csub(v[0], v[2]), a2 = cadd(v[1], v[3]), a3 = csub(v[1], v[3]);
        v[0] = cadd(a0, a2);
        v[2] = csub(a0, a2);
        v[1] = make_float2(a1.x + a3.y, a1.y - a3.x);
        v[3] = make_float2(a1.x - a3.y, a1.y + a3.x);
    } else if constexpr (R == 5) {
        constexpr float c1 = 0.30901699437494742f, c2 = -0.80901699437494742f, s1 = 0.95105651629515357f, s2 = 0.58778525229247313f;
        const float2 t1 = cadd(v[1], v[4]), t2 = cadd(v[2], v[3]), t3 = csub(v[1], v[4]), t4 = csub(v[2], v[3]);
        const float2 m1 = make_float2(__fmaf_rn(c2, t2.x, __fmaf_rn(c1, t1.x, v[0].x)), __fmaf_rn(c2, t2.y, __fmaf_rn(c1, t1.y, v[0].y)));
        const float2 m2 = make_float2(__fmaf_rn(c1, t2.x, __fmaf_rn(c2, t1.x, v[0].x)), __fmaf_rn(c1, t2.y, __fmaf_rn(c2, t1.y, v[0].y)));
        const float2 n1 = make_float2(__fmaf_rn(s2, t4.x, s1 * t3.x), __fmaf_rn(s2, t4.y, s1 * t3.y));
        const float2 n2 = make_float2(__fmaf_rn(-s1, t4.x, s2 * t3.x), __fmaf_rn(-s1, t4.y, s2 * t3.y));
        v[0] = cadd(v[0], cadd(t1, t2));
        v[1] = make_float2(m1.x + n1.y, m1.y - n1.x);
        v[4] = make_float2(m1.x - n1.y, m1.y + n1.x);
        v[2] = make_float2(m2.x + n2.y, m2.y - n2.x);
        v[3] = make_float2(m2.x - n2.y, m2.y + n2.x);
    } else {
        float2 o[R];
        const int st = L / R;
        SYG_UNROLL
        for (int q = 0; q < R; ++q) {
            float2 acc = v[0];
            SYG_UNROLL
            for (int m = 1; m < R; ++m) {
                const float2 w = __ldg(&tw[((m * q) % R) * st]);
                acc.x = __fmaf_rn(v[m].x, w.x, __fmaf_rn(-v[m].y, w.y, acc.x));
                acc.y = __fmaf_rn(v[m].x, w.y, __fmaf_rn(v[m].y, w.x, acc.y));
            }
            o[q] = acc;
        }
        SYG_UNROLL
        for (int q = 0; q < R; ++q) v[q] = o[q];
    }
}

template <int R, int NT>
SYG_DEVICE SYG_INLINE void mixed_pass(const float2* src, float2* dst, int L, int Ns, const float2* __restrict__ tw, int tid) {
    const int LR = L / R;
    const int tmul = L / (Ns * R);
    for (int j = tid; j < LR; j += NT) {
        const int k = j % Ns;
        float2 v[R];
        SYG_UNROLL
        for (int r = 0; r < R; ++r) v[r] = SLD(&src[j + r * LR]);
        if (Ns > 1) {
            const int ts = k * tmul;                                    // r ts < L: k < Ns, r < R
            SYG_UNROLL
            for (int r = 1; r < R; ++r) {
                const float2 w = __ldg(&tw[r * ts]);
                cmul(v[r].x, v[r].y, w.x, w.y);
            }
        }
        dft_small<R>(v, tw, L);
        const int ob = (j - k) * R + k;
        SYG_UNROLL
        for (int r = 0; r < R; ++r) SST(&dst[ob + r * Ns], v[r]);
    }
}

// all passes of the plan; returns the buffer that holds the spectrum (natural order).  Ends with a CTA barrier.
template <int NT>
SYG_DEVICE SYG_INLINE float2* mixed_fft(float2* a, float2* b, const syg::MixedPlan& mp, const float2* __restrict__ tw, int tid) {
    float2* src = a;
    float2* dst = b;
    int Ns = 1;
    for (int p = 0; p < mp.npass; ++p) {
        const int R = mp.radix[p];
        switch (R) {
            case 2: mixed_pass<2, NT>(src, dst, mp.L, Ns, tw, tid); break;
            case 3: mixed_pass<3, NT>(src, dst, mp.L, Ns, tw, tid); break;
            case 4: mixed_pass<4, NT>(src, dst, mp.L, Ns, tw, tid); break;
            case 5: mixed_pass<5, NT>(src, dst, mp.L, Ns, tw, tid); break;
            case 7: mixed_pass<7, NT>(src, dst, mp.L, Ns, tw, tid); break;
            case 11: mixed_pass<11, NT>(src, dst, mp.L, Ns, tw, tid); break;
            default: mixed_pass<13, NT>(src, dst, mp.L, Ns, tw, tid); break;
        }
        __syncthreads();
        float2* t = src; src = dst; dst = t;
        Ns *= R;
    }
    return src;
}

// Visits every bin of the one-sided spectrum once: fn(k, re, im).  packed: real split of the L-point packed transform (bins
// 0..L); otherwise the first B bins of the n-point transform.
template <int NT, class Fn>
SYG_DEVICE SYG_INLINE void mixed_bins(const float2* z, const syg::MixedPlan& mp, const float2* __restrict__ tws, int tid, Fn fn) {
    const int L = mp.L;
    if (mp.packed) {
        for (int k = tid; k <= L / 2; k += NT) {
            const int km = k ? L - k : 0;
            const float2 zk = SLD(&z[k]), zm = SLD(&z[km]);
            const float2 w = __ldg(&tws[k]);
            float xkr, xki, xmr, xmi;
            real_split(zk.x, zk.y, zm.x, zm.y, w.x, w.y, xkr, xki, xmr, xmi);
            fn(k, xkr, xki);
            if (L - k != k) fn(L - k, xmr, xmi);
        }
    } else {
        for (int k = tid; k < mp.B; k += NT) {
            const float2 v = SLD(&z[k]);
            fn(k, v.x, v.y);
        }
    }
}

template <int MODE, int NT>
__global__ void __launch_bounds__(NT) frame_mixed_kernel(const syg::FrameArgs a, const syg::MixedPlan mp) {
    SYG_DYN_SMEM(smem_raw);
    const int L = mp.L, B = mp.B, N = mp.n;
    const MixedLayout lay = mixed_layout(L, B, MODE != MODE_STFT, NT);
    constexpr bool RAG = (MODE == MODE_FEATURES_RAGGED);
    float* const smf = reinterpret_cast<float*>(smem_raw);
    float2* const bufa = reinterpret_cast<float2*>(smf + lay.off_a);
    float2* const bufb = reinterpret_cast<float2*>(smf + lay.off_b);
    float* const pw = smf + lay.off_pw;
    float* const cand = smf + lay.off_cand;
    unsigned* const smax = reinterpret_cast<unsigned*>(smf + lay.off_smax);
    double* const dsc = reinterpret_cast<double*>(smf + lay.off_dsc_f);
    double* const dinc = dsc + NT / 32;
    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;

    for (long long gf = blockIdx.x; gf < a.n_frames; gf += gridDim.x) {
        const int4 rut = RAG ? __ldg(a.ragged_ut + gf) : make_int4(0, 0, 0, 0);
        const long long u = RAG ? (long long)rut.x : gf / a.T;
        const int t = RAG ? rut.y : (int)(gf - u * a.T);
        const UnitRef ur = RAG ? UnitRef{(long long)rut.w, (long long)rut.z} : unit_ref(a.g, u);
        const long long p0 = (long long)t * a.hop - a.cpad;
        if (MODE != MODE_STFT && tid < 4) smax[tid] = 0u;

        // ---------------- framing + window + time-domain partial statistics ----------------
        double s_sq = 0.0, s_sum = 0.0, s_abs = 0.0;
        float pk = 0.0f;
        if (mp.packed) {
            for (int c = tid; c < L; c += NT) {
                const float2 v = load_pair(a.y, ur, p0 + 2 * c, a.pad_mode);
                const float2 w = __ldg(reinterpret_cast<const float2*>(a.window) + c);
                if (MODE != MODE_STFT) {
                    s_sq += (double)v.x * (double)v.x + (double)v.y * (double)v.y;
                    s_sum += (double)v.x + (double)v.y;
                    s_abs += (double)fabsf(v.x) + (double)fabsf(v.y);
                    pk = fmaxf(pk, fmaxf(fabsf(v.x), fabsf(v.y)));
                }
                SST(&bufa[c], make_float2(v.x * w.x, v.y * w.y));
            }
        } else {
            for (int c = tid; c < L; c += NT) {
                const float v = load_one(a.y, ur, p0 + c, a.pad_mode);
                const float w = __ldg(a.window + c);
                if (MODE != MODE_STFT) {
                    s_sq += (double)v * (double)v;
                    s_sum += (double)v;
                    s_abs += (double)fabsf(v);
                    pk = fmaxf(pk, fabsf(v));
                }
                SST(&bufa[c], make_float2(v * w, 0.0f));
            }
        }
        __syncthreads();
        const float2* const z = mixed_fft<NT>(bufa, bufb, mp, a.tw, tid);

        if (MODE == MODE_STFT) {
            const long long ob = ((long long)u * B) * a.T + t;
            if (a.out_kind == 0) {
                float2* o = reinterpret_cast<float2*>(a.stft_out);
                mixed_bins<NT>(z, mp, a.tws, tid, [&](int k, float re, float im) { o[ob + (long long)k * a.T] = make_float2(re, im); });
            } else {
                float* o = reinterpret_cast<float*>(a.stft_out);
                const bool mag = a.out_kind == 1;
                mixed_bins<NT>(z, mp, a.tws, tid, [&](int k, float re, float im) {
                    const float p = __fmaf_rn(re, re, im * im);
                    o[ob + (long long)k * a.T] = mag ? sqrt_approx(p) : p;
                });
            }
            __syncthreads();                                            // the buffers are refilled by the next frame
            continue;
        }
        mixed_bins<NT>(z, mp, a.tws, tid, [&](int k, float re, float im) { SST(&pw[padi(k)], __fmaf_rn(re, re, im * im)); });
        __syncthreads();

        float* const orow = RAG ? a.out + gf : a.out + (long long)u * a.n_rows * a.T + t;
        // ---------------- time-domain features (unwindowed, zero-padded frame) ----------------
        if (a.mask & syg::FB_TIME_ANY) {
            const double tsq = group_sum<NT>(s_sq, dsc);
            const float tpk = group_max<NT>(pk, dsc);
            double tsum = 0.0, tabs = 0.0;
            if (a.mask & (syg::FB_STD_AMP | syg::FB_MEAN_AMP)) {
                tsum = group_sum<NT>(s_sum, dsc);
                tabs = group_sum<NT>(s_abs, dsc);
            }
            if (tid == 0) {
                const double n = (double)N;
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

        // ---------------- per-frame spectral statistics: thread tid owns the contiguous bins [k0, k1) ----------------
        if (a.mask & syg::FB_SPECSTATS) {
            const int chunk = (B + NT - 1) / NT;
            const int k0 = min(tid * chunk, B), k1 = min(k0 + chunk, B);
            double sp = 0.0, sm = 0.0, skm = 0.0, slog = 0.0;
            float vmax = -1.0f;
            int imax = 0;
            for (int k = k0; k < k1; ++k) {
                const float p = SLD(&pw[padi(k)]);
                const float mg = sqrtf(p);
                sp += (double)p;
                sm += (double)mg;
                skm += (double)mg * (double)k;
                if (a.mask & syg::FB_FLATNESS) slog += (double)logf(mg + 2.220446049250313e-16f);
                if (p > vmax) { vmax = p; imax = k; }
            }
            const double incl = group_scan_incl<NT>(sp, dsc);
            __syncthreads();
            dinc[tid] = incl;
            __syncthreads();
            const double total_p = dinc[NT - 1];
            const double prev = (tid == 0) ? -1.0 : dinc[tid - 1];
            const double tm = group_sum<NT>(sm, dsc);
            const double tkm = group_sum<NT>(skm, dsc);
            double centroid_hz = 0.0;
            if (tm >= kEps64) centroid_hz = a.bin_hz * (tkm / tm);
            if (a.row_centroid >= 0 && tid == 0) orow[(long long)a.row_centroid * (RAG ? a.ragged_stride : a.T)] = (float)centroid_hz;
            if (a.row_rolloff >= 0) {
                if (total_p < kEps64) {
                    if (tid == 0) orow[(long long)a.row_rolloff * (RAG ? a.ragged_stride : a.T)] = (float)(a.bin_hz * (double)(B - 1));
                } else {
                    const double thr = a.roll_percent * total_p;
                    if (incl >= thr && prev < thr) {                    // exactly one thread
                        double c = (tid == 0) ? 0.0 : prev;
                        int bin = k1 - 1;
                        for (int k = k0; k < k1; ++k) {
                            c += (double)SLD(&pw[padi(k)]);
                            if (c >= thr) { bin = k; break; }
                        }
                        orow[(long long)a.row_rolloff * (RAG ? a.ragged_stride : a.T)] = (float)(a.bin_hz * (double)bin);
                    }
                }
            }
            if (a.row_flatness >= 0) {
                const double tl = group_sum<NT>(slog, dsc);
                if (tid == 0) {
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
                for (int k = k0; k < k1; ++k) {
                    const double mg = (double)sqrtf(SLD(&pw[padi(k)]));
                    const double d = a.bin_hz * (double)k - centroid_hz;
                    sb += mg * d * d;
                }
                const double tb = group_sum<NT>(sb, dsc);
                if (tid == 0) orow[(long long)a.row_bandwidth * (RAG ? a.ragged_stride : a.T)] = (tm < kEps64) ? 0.0f : (float)sqrt(tb / tm);
            }
            if (a.row_dominant >= 0) {
                // np.argmax: first bin attaining the maximum = smallest index among the threads holding it
                const float gmax = group_max<NT>(vmax, dsc);
                float mi = (vmax == gmax) ? -(float)imax : -1.0e9f;
                mi = group_max<NT>(mi, dsc);
                if (tid == 0) orow[(long long)a.row_dominant * (RAG ? a.ragged_stride : a.T)] = (float)(a.bin_hz * (double)(-mi));
            }
        }

        // ---------------- mel energies (sparse triangular filters), one filter per thread ----------------
        if (a.mask & syg::FB_MFCC) {
            for (int base = 0; base < a.n_mels; base += NT) {
                const int m = base + tid;
                float acc = 0.0f;
                if (m < a.n_mels) {
                    const int st = __ldg(&a.mel_start[m]), ln = __ldg(&a.mel_len[m]);
                    const float* wv = a.mel_w + __ldg(&a.mel_off[m]);
                    if (a.mel_power_is_2) {
                        for (int i = 0; i < ln; ++i) acc = __fmaf_rn(__ldg(&wv[i]), SLD(&pw[padi(st + i)]), acc);
                    } else {
                        for (int i = 0; i < ln; ++i) acc = __fmaf_rn(__ldg(&wv[i]), powf(SLD(&pw[padi(st + i)]), a.mel_half_power), acc);
                    }
                    a.melws[gf * a.n_mels + m] = acc;
                }
                const unsigned mx = __reduce_max_sync(kFull, __float_as_uint(fmaxf(acc, 0.0f)));
                if (lane == 0 && mx) atomicMax(&smax[0], mx);
            }
        }

        // ---------------- spectral contrast: per band mean of the n largest / n smallest magnitudes, one warp per band ----------------
        if (a.mask & syg::FB_CONTRAST) {
            float* mycand = cand + warp * 32;
            for (int bd = warp; bd < a.nb; bd += NT / 32) {
                const float peak = warp_extreme_mean_sqrt<+1>(pw, a.band_lo[bd], a.band_cnt[bd], a.band_n[bd], mycand);
                const float valley = warp_extreme_mean_sqrt<-1>(pw, a.band_lo[bd], a.band_cnt[bd], a.band_n[bd], mycand);
                if (lane == 0) {
                    a.cws[gf * (2 * a.nb) + bd] = peak;
                    a.cws[gf * (2 * a.nb) + a.nb + bd] = valley;
                    if (peak == peak) atomicMax(&smax[1], __float_as_uint(peak));
                    if (valley == valley) atomicMax(&smax[2], __float_as_uint(valley));
                }
            }
        }

        // ---------------- publish per-unit maxima ----------------
        __syncthreads();
        if ((a.mask & (syg::FB_MFCC | syg::FB_CONTRAST)) && tid < 3) {
            const unsigned v = smax[tid];
            if (v) atomicMax(&a.unit_max[u * 4 + tid], v);
        }
        __syncthreads();                                                // smax / pw / buffers are rewritten by the next frame
    }
}

// --------------------------------------------------------------------------------------------------------
// Welch / periodogram PSD for smooth nfft, one CTA per unit (grid-stride).  Same semantics as welch_kernel (syg_kernels.cuh):
// per sub-segment detrend('constant') -> window -> zero padding to nfft -> rfft -> |X|^2; mean over sub-segments; one-sided
// doubling except DC (and Nyquist when nfft is even).  The running sums live in the unit's own output row (every bin is always
// visited by the same thread), so a 25 600-point periodogram needs shared memory for the two transform buffers only.
// --------------------------------------------------------------------------------------------------------
template <int NT>
__global__ void __launch_bounds__(NT) welch_mixed_kernel(const syg::WelchArgs a, const syg::MixedPlan mp) {
    SYG_DYN_SMEM(smem_raw);
    const int L = mp.L, B = mp.B;
    const MixedLayout lay = mixed_layout(L, B, false, NT);
    float* const smf = reinterpret_cast<float*>(smem_raw);
    float2* const bufa = reinterpret_cast<float2*>(smf + lay.off_a);
    float2* const bufb = reinterpret_cast<float2*>(smf + lay.off_b);
    double* const dsc = reinterpret_cast<double*>(smf + lay.off_dsc_f);
    const int tid = threadIdx.x;

    for (long long u = blockIdx.x; u < a.g.n_units; u += gridDim.x) {
        const UnitRef ur = unit_ref(a.g, u);
        float* const prow = a.psd + u * B;
        for (int s = 0; s < a.nseg; ++s) {
            const long long p0 = (long long)s * a.step;
            float mean = 0.0f;
            if (a.detrend) {
                double ssum = 0.0;
                for (int i = tid; i < a.nperseg; i += NT) ssum += (double)load_one(a.y, ur, p0 + i, 0);
                mean = (float)(group_sum<NT>(ssum, dsc) / (double)a.nperseg);
            }
            if (mp.packed) {
                for (int c = tid; c < L; c += NT) {
                    float2 v = make_float2(0.0f, 0.0f);
                    if (2 * c < a.nperseg) {
                        const float2 w = __ldg(reinterpret_cast<const float2*>(a.window) + c);
                        const float2 x = load_pair(a.y, ur, p0 + 2 * c, 0);
                        v.x = (x.x - mean) * w.x;
                        if (2 * c + 1 < a.nperseg) v.y = (x.y - mean) * w.y;
                    }
                    SST(&bufa[c], v);
                }
            } else {
                for (int c = tid; c < L; c += NT) {
                    float v = 0.0f;
                    if (c < a.nperseg) v = (load_one(a.y, ur, p0 + c, 0) - mean) * __ldg(a.window + c);
                    SST(&bufa[c], make_float2(v, 0.0f));
                }
            }
            __syncthreads();
            const float2* const z = mixed_fft<NT>(bufa, bufb, mp, a.tw, tid);
            const bool first = (s == 0);
            mixed_bins<NT>(z, mp, a.tws, tid, [&](int k, float re, float im) {
                const float p = __fmaf_rn(re, re, im * im);
                prow[k] = first ? p : prow[k] + p;
            });
            __syncthreads();
        }
        const float inv = a.scale / (float)a.nseg;
        const int nyq = (mp.n % 2 == 0) ? B - 1 : -1;
        for (int k = tid; k < B; k += NT) {
            float v = prow[k] * inv;
            if (a.onesided_double && k != 0 && k != nyq) v *= 2.0f;
            prow[k] = v;
        }
        if (a.stats) {
            double sq = 0.0;
            float pk = 0.0f;
            for (long long i = tid; i < a.g.unit_len; i += NT) {
                const float v = (i < ur.valid) ? __ldg(a.y + ur.start + i) : 0.0f;
                sq += (double)v * (double)v;
                pk = fmaxf(pk, fabsf(v));
            }
            const double tsq = group_sum<NT>(sq, dsc);
            const float tpk = group_max<NT>(pk, dsc);
            if (tid == 0) {
                const double rms = a.g.unit_len > 0 ? sqrt(tsq / (double)a.g.unit_len) : 0.0;
                a.stats[u * 3 + 0] = (float)rms;
                a.stats[u * 3 + 1] = (rms < kEps64) ? 0.0f : (float)((double)tpk / rms);
                a.stats[u * 3 + 2] = tpk;
            }
        }
        __syncthreads();
    }
}

}  // namespace sygdev
