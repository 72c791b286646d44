// sygnals_b200/csrc/syg_finalize.cuh -- per-unit epilogues, finalize and mel_store (included by exactly one translation unit)
#pragma once

#include "syg_device.cuh"
#include "syg_params.h"
#include "syg_finalize_dev.cuh"

namespace sygdev {

// --------------------------------------------------------------------------------------------------------
// finalize: grid = (ceil(T/TT), n_units), kThreads threads.
//   MFCC: S_db = 10 log10(max(amin, mel)) - 10 log10(max(amin, max_unit mel)); S_db = max(S_db, max(S_db) - top_db)
//         (librosa.power_to_db(ref=np.max), manager.py:223) then DCT rows (cepstral.py:106-115).
//   contrast: power_to_db(peak) - power_to_db(valley), each clamped to its own unit-wide max - top_db
//         (librosa.feature.spectral_contrast, frequency_domain.py:200-207).
// --------------------------------------------------------------------------------------------------------

// One slot of a tile (finalize and mel_store): frame gf's place in `out` -- (unit, row 0, frame t) of a uniform launch, gf of a ragged
// one -- its unit's maxima, and the unit's reference level and floor of power_to_db(ref=np.max): the maximum of S_db over the unit is
// attained at the maximum energy -> 0 dB.
struct FinSlot {
    long long out;
    const unsigned* um;
    float ref_db, floor_db;
};
template <bool RAG>
SYG_DEVICE SYG_INLINE FinSlot fin_slot(const syg::FinalizeArgs& a, long long gf) {
    const long long u = RAG ? (long long)__ldg(a.ragged_ut + gf).x : gf / a.T;
    const int t = RAG ? 0 : (int)(gf - u * a.T);
    FinSlot s;
    s.um = a.unit_max + u * 4;
    s.out = RAG ? gf : u * (long long)a.n_rows * a.T + t;
    s.ref_db = db10(fmaxf(a.amin, __uint_as_float(s.um[0])));
    s.floor_db = -a.top_db;
    return s;
}

// Persistent: the chunk's frames are one flat sequence cut into tiles of kFinTT consecutive frames (a tile may straddle units:
// every slot carries its own unit, reference level and clamps), CTAs stride over the tiles.  Short units (T = 101 in the
// speech-commands shape) no longer leave partial tiles or one tiny CTA per 32 frames.
// KT = kFinTT | kFinRagged: ragged launch (a.ragged_ut), the chunk's a.n_frames frames, row r of frame gf at
// out[r * ragged_stride + gf]
constexpr int kFinRagged = 1 << 16;
template <int KT>
__global__ void __launch_bounds__(kThreads) finalize_kernel_t(const syg::FinalizeArgs a) {
    constexpr int kFinTT = KT & (kFinRagged - 1);
    constexpr bool RAG = (KT & kFinRagged) != 0;
    SYG_DYN_SMEM(smem_raw);
    __shared__ long long s_out[kFinTT];         // offset of (unit, row 0, frame t) in `out`
    __shared__ float s_ref[kFinTT], s_floor[kFinTT], s_pfloor[kFinTT], s_vfloor[kFinTT];
    const int tid = threadIdx.x;
    const long long total = RAG ? a.n_frames : a.n_units * (long long)a.T;
    const long long n_tiles = (total + kFinTT - 1) / kFinTT;
    const int N = a.n_mels;
    const int H = a.dct_fold ? (N + 1) / 2 : N;
    const int H4 = (H + 3) / 4 * 4;                                     // DMMA k-steps of 4 columns
    // FP64 rows in shared memory, folded on the way in: xe[tt][k] = s[k] + s[N-1-k] (what the even DCT-II coefficients see),
    // xo[tt][k] = s[k] - s[N-1-k] (odd coefficients), k < H = ceil(N/2); other DCT types keep the unfolded row in xe (H = N).
    // The DMMA loop then is one table load, one shared-memory load and one mma per k-step: the float -> double conversions, the
    // fold and their predicates used to sit INSIDE that loop (~45 instructions per k-step; the kernel was issue-bound at 82 %).
    const int PD = fin_pitch_d(H);
    double* const xe = reinterpret_cast<double*>(smem_raw);            // [kFinTT][PD]
    double* const xo = xe + (a.dct_fold ? kFinTT * PD : 0);            // [kFinTT][PD] (folded types only)
    const int warp = tid >> 5, lane = tid & 31;

    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long gf0 = tile * kFinTT;
        const int nt = (int)min((long long)kFinTT, total - gf0);
        if (tid < nt) {
            const FinSlot sl = fin_slot<RAG>(a, gf0 + tid);
            s_out[tid] = sl.out;
            s_ref[tid] = sl.ref_db;
            s_floor[tid] = sl.floor_db;
            s_pfloor[tid] = db10(fmaxf(a.amin, __uint_as_float(sl.um[1]))) - a.top_db;
            s_vfloor[tid] = db10(fmaxf(a.amin, __uint_as_float(sl.um[2]))) - a.top_db;
        }
        __syncthreads();
        if (a.row_mfcc >= 0) {
            const float* const blk = a.melws + gf0 * N;                 // the tile's raw mel energies: ONE contiguous block of nt * N floats
            if (a.dct_fold && (N & 7) == 0) {
                // fast path (N a multiple of 8: H a multiple of 4, every float4 inside one row, 16-byte aligned): a thread takes the
                // chunk k..k+3 of a row and its mirror N-4-k..N-1-k (the CTAs of an SM hide each other's load latency)
                const int cpr = H >> 2;                                 // chunk pairs per row
                const int n_cp = nt * cpr;
                for (int c = tid; c < n_cp; c += kThreads) {
                    const int tt = c / cpr, k = (c - tt * cpr) << 2;
                    const float* row = blk + (size_t)tt * N;
                    const float4 v = __ldg(reinterpret_cast<const float4*>(row + k));
                    const float4 m = __ldg(reinterpret_cast<const float4*>(row + N - 4 - k));
                    const float ref_db = s_ref[tt], floor_db = s_floor[tt];
                    const float x0 = fmaxf(db10(fmaxf(a.amin, v.x)) - ref_db, floor_db), y0 = fmaxf(db10(fmaxf(a.amin, m.w)) - ref_db, floor_db);
                    const float x1 = fmaxf(db10(fmaxf(a.amin, v.y)) - ref_db, floor_db), y1 = fmaxf(db10(fmaxf(a.amin, m.z)) - ref_db, floor_db);
                    const float x2 = fmaxf(db10(fmaxf(a.amin, v.z)) - ref_db, floor_db), y2 = fmaxf(db10(fmaxf(a.amin, m.y)) - ref_db, floor_db);
                    const float x3 = fmaxf(db10(fmaxf(a.amin, v.w)) - ref_db, floor_db), y3 = fmaxf(db10(fmaxf(a.amin, m.x)) - ref_db, floor_db);
                    double2* const pe = reinterpret_cast<double2*>(xe + tt * PD + k);
                    double2* const po = reinterpret_cast<double2*>(xo + tt * PD + k);
                    pe[0] = make_double2((double)x0 + (double)y0, (double)x1 + (double)y1);
                    pe[1] = make_double2((double)x2 + (double)y2, (double)x3 + (double)y3);
                    po[0] = make_double2((double)x0 - (double)y0, (double)x1 - (double)y1);
                    po[1] = make_double2((double)x2 - (double)y2, (double)x3 - (double)y3);
                }
            } else {
                // any N, any DCT type: one (frame, column) per thread and step; columns H..PD-1 are zero (the k-steps run to H4)
                const int n_el = nt * PD;
                for (int i = tid; i < n_el; i += kThreads) {
                    const int tt = i / PD, k = i - tt * PD;
                    double e = 0.0, o = 0.0;
                    if (k < H) {
                        const float* row = blk + (size_t)tt * N;
                        const float ref_db = s_ref[tt], floor_db = s_floor[tt];
                        const float x = fmaxf(db10(fmaxf(a.amin, __ldg(row + k))) - ref_db, floor_db);
                        e = (double)x;
                        if (a.dct_fold) {
                            const int k2 = N - 1 - k;
                            if (k2 != k) {
                                const float y = fmaxf(db10(fmaxf(a.amin, __ldg(row + k2))) - ref_db, floor_db);
                                e = (double)x + (double)y;
                                o = (double)x - (double)y;
                            }                                           // centre of an odd N: once, even coefficients only
                        }
                    }
                    xe[i] = e;
                    if (a.dct_fold) xo[i] = o;
                }
            }
            __syncthreads();
            // DCT as FP64 tensor-core products (mma.sync m8n8k4, DMMA): D[coefficient][frame] += dct[coefficient][n] * S[frame][n].
            // Warp w owns one parity (even coefficients see the folded sums, odd ones the differences) and one n-tile of 8 frames;
            // 8 coefficients of that parity per m-tile.  Per k-step of 4 columns a lane loads ONE table entry and ONE tile entry for
            // 256 multiply-adds of the warp.  Rows of a partial tile beyond nt hold stale values: a B column only feeds its own
            // (unstored) output column.
            {
                const int par = warp & 1;                               // kThreads / 32 = 8 warps: 2 parities x 4 n-tiles of 8 frames (per 32 frames)
                const int g = lane >> 2, q = lane & 3;
                const int n_par = par ? a.n_mfcc / 2 : (a.n_mfcc + 1) / 2;
                const double* const xp = (par && a.dct_fold) ? xo : xe;
                for (int nt8 = (warp >> 1) * 8; nt8 < kFinTT; nt8 += 32)
                for (int m0 = 0; m0 < n_par; m0 += 8) {
                    const double* const xrow = xp + (nt8 + g) * PD + q;  // this lane's frame (B column)
                    const int c_a = par + 2 * (m0 + g);                 // coefficient of this lane's A row
                    const bool a_ok = c_a < a.n_mfcc;
                    const double* const drow = a.dct + (long long)(a_ok ? c_a : 0) * N + q;
                    const int kmax = a_ok ? H - q : 0;                  // table entries of this lane: k0 < kmax
                    double d0 = 0.0, d1 = 0.0;
#ifndef SYG_EMU
#pragma unroll 4
#endif
                    for (int k0 = 0; k0 < H4; k0 += 4) {
                        const double av = (k0 < kmax) ? __ldg(drow + k0) : 0.0;
                        mma_m8n8k4_f64(d0, d1, av, xrow[k0]);
                    }
                    // lane holds D[row g][cols 2q, 2q+1] = coefficient par + 2 (m0 + g) of frames nt8 + 2q, nt8 + 2q + 1
                    if (a_ok) {
                        const int t0 = nt8 + 2 * q;
                        if (t0 < nt) a.out[s_out[t0] + (long long)(a.row_mfcc + c_a) * (RAG ? a.ragged_stride : a.T)] = (float)d0;
                        if (t0 + 1 < nt) a.out[s_out[t0 + 1] + (long long)(a.row_mfcc + c_a) * (RAG ? a.ragged_stride : a.T)] = (float)d1;
                    }
                }
            }
        }
        if (a.nb > 0) {
            for (int i = tid; i < a.nb * kFinTT; i += kThreads) {
                const int bd = i / kFinTT, tt = i - bd * kFinTT;
                if (tt < nt) {
                    const float* c = a.cws + (gf0 + tt) * (2 * a.nb);
                    const float pdb = fmaxf(db10(fmaxf(a.amin, c[bd])), s_pfloor[tt]);
                    const float vdb = fmaxf(db10(fmaxf(a.amin, c[a.nb + bd])), s_vfloor[tt]);
                    a.out[s_out[tt] + (long long)(a.row_contrast + bd) * (RAG ? a.ragged_stride : a.T)] =
                        a.contrast_nan ? __uint_as_float(0x7fc00000u) : pdb - vdb;
                }
            }
        }
        __syncthreads();                                                // the tile buffers are reused
    }
}

// --------------------------------------------------------------------------------------------------------
// mel_store: the epilogue of the mel spectrogram calls, in place of finalize.  The frame kernels left the chunk's mel energies
// frame-major in melws ([frame][n_mels]) and each unit's maximum in unit_max[0]; this kernel writes them frequency-major, as
// S_mel (a.mel_db == 0) or as S_db with finalize's reference level and floor (a.mel_db == 1, store_db): uniform launches
// out[u][m][t] (= s_out + m * T), ragged ones out[m * ragged_stride + gf].  Tiles and slots are finalize's (fin_slot).
//
// A tile's block of nt * N floats is contiguous: it is read in order (16-byte loads when N % 4 == 0) and transposed through
// shared memory tile[m][tt] with a pitch of TT + 1 words (1 mod 32).  A warp's store reads 32 consecutive frames of one band, 32
// distinct banks, and writes one contiguous run of `out`.  On the load side lane L holds bands 4L' .. 4L' + 3 of a frame; writing
// component j in every lane at once would touch 8 banks, so lane L writes its components in the order (j + L / 8) % 4 and each
// write step covers 32 banks wherever a warp's 128 floats lie in one frame (every warp when N is a multiple of 128).
// --------------------------------------------------------------------------------------------------------
// S_db of one mel energy: finalize's power_to_db (db10, amin, the unit's reference level, the -top_db floor) with the subtraction of
// the reference level rounded on its own.  In finalize the compiler fuses it with db10's product into one FMA, which leaves each
// unit's maximum a few 1e-8 dB off 0; here the maximum is exactly 0 dB, as power_to_db(ref=np.max) returns it.  The two differ by
// at most half an ulp of the product (a few 1e-6 dB).
SYG_DEVICE SYG_INLINE float store_db(float x, float amin, float ref_db, float floor_db) {
    return fmaxf(__fadd_rn(db10(fmaxf(amin, x)), -ref_db), floor_db);
}

template <int KT>
__global__ void __launch_bounds__(kThreads) mel_store_kernel(const syg::FinalizeArgs a) {
    constexpr int TT = KT & (kFinRagged - 1);
    constexpr bool RAG = (KT & kFinRagged) != 0;
    constexpr int P = TT + 1;
    SYG_DYN_SMEM(smem_raw);
    float* const tile = reinterpret_cast<float*>(smem_raw);            // [n_mels][P]
    __shared__ long long s_out[TT];
    __shared__ float s_ref[TT];
    const int tid = threadIdx.x;
    const long long total = RAG ? a.n_frames : a.n_units * (long long)a.T;
    const long long n_tiles = (total + TT - 1) / TT;
    const int N = a.n_mels;
    const long long row_stride = RAG ? a.ragged_stride : a.T;
    const float floor_db = -a.top_db;
    const bool db = a.mel_db != 0;

    for (long long ti = blockIdx.x; ti < n_tiles; ti += gridDim.x) {
        const long long gf0 = ti * TT;
        const int nt = (int)min((long long)TT, total - gf0);
        if (tid < nt) {
            const FinSlot sl = fin_slot<RAG>(a, gf0 + tid);
            s_out[tid] = sl.out;
            s_ref[tid] = sl.ref_db;
        }
        __syncthreads();
        const float* const blk = a.melws + gf0 * N;
        if ((N & 3) == 0) {
            // 16-byte aligned: melws is, and every tile starts a multiple of 4 floats into it.  Four loads in flight per thread.
            const int q = N >> 2;                                       // float4 per frame
            const int n4 = nt * q;
            const int rot = (tid >> 3) & 3;                             // = lane / 8
            const float4* const b4 = reinterpret_cast<const float4*>(blk);
            for (int c0 = tid; c0 < n4; c0 += 4 * kThreads) {
                float4 v[4];
#pragma unroll
                for (int r = 0; r < 4; ++r)
                    if (c0 + r * kThreads < n4) v[r] = __ldg(b4 + c0 + r * kThreads);
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const int c = c0 + r * kThreads;
                    if (c >= n4) break;
                    const int tt = c / q, m = (c - tt * q) << 2;
                    if (db) {
                        const float ref_db = s_ref[tt];
                        v[r].x = store_db(v[r].x, a.amin, ref_db, floor_db);
                        v[r].y = store_db(v[r].y, a.amin, ref_db, floor_db);
                        v[r].z = store_db(v[r].z, a.amin, ref_db, floor_db);
                        v[r].w = store_db(v[r].w, a.amin, ref_db, floor_db);
                    }
                    float* const col = tile + m * P + tt;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int k = (j + rot) & 3;
                        col[k * P] = k == 0 ? v[r].x : k == 1 ? v[r].y : k == 2 ? v[r].z : v[r].w;
                    }
                }
            }
        } else {
            const int n_el = nt * N;
            for (int i = tid; i < n_el; i += kThreads) {
                const int tt = i / N, m = i - tt * N;
                const float x = __ldg(blk + i);
                tile[m * P + tt] = db ? store_db(x, a.amin, s_ref[tt], floor_db) : x;
            }
        }
        __syncthreads();
        for (int i = tid; i < N * TT; i += kThreads) {
            const int m = i / TT, tt = i - m * TT;
            if (tt < nt) a.out[s_out[tt] + (long long)m * row_stride] = tile[m * P + tt];
        }
        __syncthreads();                                                // the tile buffers are reused
    }
}

}  // namespace sygdev
