// sygnals_b200/csrc/syg_frame_warp.cuh
//
// frame_warp_kernel<TL, EXTRA>: the feature kernel for n_fft <= 2048 (M = n_fft/2 <= 1024 packed complex points).
//
// Warp-synchronous: G = M/E <= 32 lanes own one frame (E points per lane in registers), a warp owns FW = 32/G frames,
// and nothing in the kernel needs a CTA barrier -- the two radix passes exchange through the warp's private slice of
// shared memory with __syncwarp() only, so the 8 warps of a CTA (and the CTAs of an SM) overlap each other's
// load / butterfly / epilogue phases.  Per frame:
//
//   framing (index arithmetic, zero padding by predicate) -> window -> radix-E DIF in registers -> exchange ->
//   twiddle + radix-R2 in registers -> natural-order Z in smem -> real split -> |X|^2 in smem ->
//   { mel energies, contrast peaks/valleys, centroid, rolloff, rms, crest, peak, [bandwidth, flatness, dominant, ...] }
//
// Shared-memory layout per frame: Z as float2[ZS] (one pad slot every E points: both the stride-E scatter of pass 1 and
// the stride-M/R gather of pass 2 are bank-conflict free for 64-bit accesses) and |X|^2 as float[PS] (one pad word every
// 32 bins: the blocked read of the spectral statistics is conflict free).
//
// Reference semantics: sygnals/core/features/manager.py:177-227,265-345 and the librosa routines of SURVEY.md 2.3.
#pragma once

#include "syg_device.cuh"
#include "syg_kernels.cuh"
#include "syg_params.h"
#include "syg_finalize_dev.cuh"

namespace sygdev {

template <class TL, int NT = kThreads>
struct WarpTile {
    static constexpr int E = TL::E, M = TL::M, G = TL::G, LOG2E = TL::LOG2E;
    static_assert(G <= 32, "warp tile needs at most 32 lanes per frame");
    static_assert(TL::NPASS == 2, "warp tile is a two-pass FFT");
    static constexpr int FW = 32 / G;                         // frames per warp
    static constexpr int R2 = TL::RLAST;                      // radix of pass 2
    static constexpr int ZS = M + (M >> LOG2E) + 1;           // float2 slots per frame
    static constexpr int PS = ((M + 1) + 4 * ((M + 1) >> 5) + 48 + 3) / 4 * 4;  // floats per frame: 4 pad words per 32 bins (ppad) + 48 words of sweep slack
    static constexpr int kWarps = NT / 32;
    // one region per frame, used twice: as the Z exchange buffer of the FFT, then (Z is dead once the real split has pulled
    // its pairs into registers) as the |X|^2 spectrum.  Halves the shared memory per warp, which the SM hands to L1.
    // With FW > 1 the lane groups of a warp store their |X|^2 in the same 32-bit shared-memory access: regions start G banks apart
    // (pitch = G mod 32) so that the groups never collide.
    // the region also holds the two padded running-sum arrays of the interval-form mel projection
    static constexpr int IVW = (M % 32 == 0) ? 2 * (M + M / 8) + 4 : 0;
    static constexpr int RS1 = (2 * ZS > PS ? 2 * ZS : PS);
    static constexpr int RS0 = ((RS1 > IVW ? RS1 : IVW) + 3) / 4 * 4;
    static constexpr int RS = (FW == 1) ? RS0 : ((RS0 - G + 31) / 32 * 32 + G);
    static constexpr int warp_floats = FW * RS;
    static constexpr size_t bytes = (size_t)kWarps * warp_floats * sizeof(float);
    // plan tables kept in shared memory by the fused kernel (all 16-byte multiples): window [2M] floats, tw [M] float2,
    // twsh [M/2+1] float2, mel slots [n_mels] int4, mel taps [mel_pw_f4] float4
    static constexpr int kWinB = 2 * M * 4, kTwB = M * 8, kTwshB = ((M / 2 + 1) * 8 + 15) / 16 * 16;
    SYG_HD static size_t table_bytes(int n_mels, int mel_pw_f4) { return (size_t)kWinB + kTwB + kTwshB + (size_t)n_mels * 16 + (size_t)mel_pw_f4 * 16; }
};

template <int LOG2E>
SYG_DEVICE SYG_INLINE int zpad(int i) { return i + (i >> LOG2E); }

// ---------------------------------------------------------------------------------------------------------------------------
// Plan specialisations of the feature kernel (n_fft 2048).  The spectral-contrast band layout and the mel sweep lengths are plan
// constants; for the layouts below they are ALSO compile-time constants, so the band loop, the selection networks, the pop loops
// and the mel sweeps unroll into straight-line code (no per-band loop overhead, no trip-count loads, no convergence checks in
// front of the warp reductions).  The launcher (syg_launch_warp.h) compares the run-time plan with the spec and falls back to
// SpecNone (the generic loops) on any difference.
//   band(i, 0..2) = {first bin, bins, quantile count}  of sygplan::build_bands(sr, 2048, n_bands=6, fmin=200, quantile=0.02)
//   steps(i)      = float4 steps of mel sweep i of sygplan::build_mel_slots (n_mels = 128, fmin 0, fmax sr/2, 32 filters per sweep)
// ---------------------------------------------------------------------------------------------------------------------------
// kMask != 0: the feature set and the output rows of the non-EXTRA features are compile-time constants too (SpecLayout below)
struct SpecNoLayout {
    static constexpr unsigned kMask = 0u;
    static constexpr int row_rms = -1, row_crest = -1, row_peak = -1, row_centroid = -1, row_rolloff = -1;
};
struct SpecNone : SpecNoLayout {
    static constexpr bool kBands = false, kMel = false;
    static constexpr int nb = 0, n_sweeps = 0;
    SYG_HD static constexpr int band(int, int) { return 0; }
    SYG_HD static constexpr int steps(int) { return 0; }
};
struct Spec44k : SpecNoLayout {                                        // sr 44100 (BASELINE cfg4)
    static constexpr bool kBands = true, kMel = true;
    static constexpr int nb = 7, n_sweeps = 4;
    SYG_HD static constexpr int band(int i, int f) {
        constexpr int t[7][3] = {{0, 9, 1}, {9, 9, 1}, {18, 19, 1}, {37, 37, 1}, {74, 74, 2}, {148, 149, 3}, {297, 728, 15}};
        return t[i][f];
    }
    SYG_HD static constexpr int steps(int i) { constexpr int t[4] = {22, 8, 6, 6}; return t[i]; }
};
struct Spec22k : SpecNoLayout {                                        // sr 22050 (the reference's default sample rate; BASELINE cfg1)
    static constexpr bool kBands = true, kMel = true;
    static constexpr int nb = 7, n_sweeps = 4;
    SYG_HD static constexpr int band(int i, int f) {
        constexpr int t[7][3] = {{0, 18, 1}, {18, 19, 1}, {37, 37, 1}, {74, 74, 2}, {148, 149, 3}, {297, 297, 6}, {594, 431, 9}};
        return t[i][f];
    }
    SYG_HD static constexpr int steps(int i) { constexpr int t[4] = {16, 8, 6, 4}; return t[i]; }
};

// Spec44k + the request of BASELINE cfg4 in the reference's column order: mfcc x13 | contrast x7 | centroid | rolloff | rms | crest.
// The feature-mask branches, the "row requested?" tests and the row offsets fold into the code (launcher: spec_matches).
struct Spec44kL : Spec44k {
    static constexpr unsigned kMask = syg::FB_MFCC | syg::FB_CONTRAST | syg::FB_CENTROID | syg::FB_ROLLOFF | syg::FB_RMS | syg::FB_CREST;
    static constexpr int row_rms = 22, row_crest = 23, row_peak = -1, row_centroid = 20, row_rolloff = 21;
};

template <int G>
SYG_DEVICE SYG_INLINE float lanes_sum(float v) {
    SYG_UNROLL
    for (int o = G / 2; o >= 1; o >>= 1) v += __shfl_xor_sync(kFull, v, o, G);
    return v;
}
template <int G>
SYG_DEVICE SYG_INLINE double lanes_sum(double v) {
    SYG_UNROLL
    for (int o = G / 2; o >= 1; o >>= 1) v += __shfl_xor_sync(kFull, v, o, G);
    return v;
}
template <int G>
SYG_DEVICE SYG_INLINE float lanes_max(float v) {
    SYG_UNROLL
    for (int o = G / 2; o >= 1; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, o, G));
    return v;
}
template <int G>
SYG_DEVICE SYG_INLINE double lanes_scan_incl(double v, int gl) {
    SYG_UNROLL
    for (int o = 1; o < G; o <<= 1) {
        const double n = __shfl_up_sync(kFull, v, o, G);
        if (gl >= o) v += n;
    }
    return v;
}

// STAGE 0: features (framing -> FFT -> |X|^2 in shared memory -> all epilogues).
// STAGE 3: STFT output (framing -> FFT -> real split -> transposed CTA tile -> contiguous row stores).
// STAGE 4: STFT magnitude / power output for M <= 256 (n_fft <= 512): every WARP owns 8 consecutive frames and a private transposed
//          tile [B][8 + 1] -- no CTA barrier at all, the warps of an SM drift apart and overlap each other's load / FFT / store phases.
// STAGE 5: STAGE 0 for SHORT units with the MFCC epilogue on chip (BASELINE cfg3: T = 101 frames, 40 mel bands).  A CTA owns groups of
//          `res_units` consecutive units; the raw mel energies of a group's frames stay in a shared-memory tile, the per-unit maxima
//          in shared words, and after the group's last frame the CTA applies power_to_db(ref = unit max, top_db) and the DCT (FP64
//          DMMA, the code of finalize_kernel) in place and writes the MFCC rows: no mel workspace round trip through HBM, no
//          finalize launch.  Two CTAs per SM alternate between their transform and their epilogue phases.
// STAGE 6: STAGE 0 for ragged units (FrameArgs::ragged_ut): every frame looks its unit and frame index up in the per-frame table,
//          rows go to out[r * ragged_stride + gf].  The row stores spell the stride out at every site: a hoisted
//          64-bit stride changes the register allocation of the uniform instantiations.
// (A two-launch variant -- FFT kernel + 64-register epilogue kernel with the spectra handed over through a workspace -- was
// measured and removed: +4 % at best, see DESIGN.md 4.1 and profiles/r01_t_two_stage_ncu_summary.txt.  CTA barriers between
// the phases of the fused kernel were measured too: +8 % time.)
template <class TL, bool EXTRA, int NT, int MINB, int STAGE, class SP = SpecNone>
__global__ void __launch_bounds__(NT, MINB) frame_warp_kernel(const syg::FrameArgs a) {
    using WT = WarpTile<TL, NT>;
    constexpr int E = WT::E, M = WT::M, G = WT::G, FW = WT::FW, R2 = WT::R2, ZS = WT::ZS, PS = WT::PS, LE = WT::LOG2E;
    constexpr int Q = E / R2;
    constexpr int B = M + 1;
    static_assert(R2 == G, "two-pass warp tile: the last radix equals the lanes per frame");
    constexpr bool kShflSplit = (SYG_SPLIT_SHFL != 0);                  // mirrors of the real split by SHFL (syg_device.cuh: mirror_of)
    constexpr bool kLay = (SP::kMask != 0u);                            // feature set + rows known at compile time
    const unsigned mask = kLay ? SP::kMask : a.mask;
    const int row_rms = kLay ? SP::row_rms : a.row_rms, row_crest = kLay ? SP::row_crest : a.row_crest, row_peak = kLay ? SP::row_peak : a.row_peak;
    const int row_centroid = kLay ? SP::row_centroid : a.row_centroid, row_rolloff = kLay ? SP::row_rolloff : a.row_rolloff;
    // feature stages: pass 2 produces Z/2 (halved twiddle table, element 0 entering with the pending scale 0.5) and the split runs in tangent form (split_power_h)
    constexpr bool kHalfZ = (STAGE == 0 || STAGE == 5 || STAGE == 6) && (SYG_SPLIT_HALF != 0);
    constexpr bool RAG = (STAGE == 6);
    SYG_DYN_SMEM(smem_raw);
    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const int f = lane / G, j = lane % G;
    constexpr int RSS = WT::RS;                                       // floats per frame region
    constexpr int WF = FW * RSS;                                      // floats per warp
    float* const wbase = reinterpret_cast<float*>(smem_raw) + warp * WF;
    // STAGE 3 (STFT output): CTA tile [B][TT + 1] behind the warps' regions, TT = frames of one CTA round; + per-slot output offsets
    constexpr int TT = WT::kWarps * FW, TTP = TT + 1;
    long long* const slot_off = reinterpret_cast<long long*>(reinterpret_cast<float*>(smem_raw) + WT::kWarps * WF);   // [TT]
    float* const tile = reinterpret_cast<float*>(slot_off + TT);                                                    // [B][TTP] float or float2
    // STAGE 4: per-warp block behind the warps' regions: 8 output offsets (long long) + tile [B][9] floats
    constexpr int TT4 = 8, TTP4 = TT4 + 1, SUBS = (STAGE == 4) ? TT4 / FW : 1;
    constexpr int WB4 = 2 * TT4 + ((B * TTP4 + 1) & ~1);               // floats per warp block (even: keeps the offsets 8-byte aligned)
    float* const wblk = reinterpret_cast<float*>(smem_raw) + WT::kWarps * WF + warp * WB4;
    long long* const woff = reinterpret_cast<long long*>(wblk);       // [TT4]
    float* const wtile = wblk + 2 * TT4;                              // [B][TTP4]
    float* const pww = wbase;                                         // [FW][RSS]  Z (float2, zpad layout), later |X|^2 (ppad layout)
    float2* const zs = reinterpret_cast<float2*>(wbase + f * RSS);
    float* const pf = wbase + f * RSS;

    // pad / slack words of the spectra are read (with zero weight) by the mel sweep: they must never hold NaN patterns.  They do
    // hold FFT data of earlier stages (any sign), which is why the power != 2 sweep raises only weighted taps.
    for (int i = lane; i < WF; i += 32) wbase[i] = 0.0f;
    __syncwarp();

    // STAGE 0: the plan tables (window, twiddles, mel taps: ~38 KB for n_fft 2048 / 128 mels) live in shared memory behind the
    // warps' regions -- 116 table loads per lane and frame become LDS with no L1 tag traffic and no misses
    // STAGE 4 keeps window / twiddles / (full-scale) split twiddles there too, behind the per-warp tile blocks: its L1 pipe is the
    // busiest unit (95 %) and 40 of its 56 loads per lane and task were table reads through the L1 tag stage
    constexpr bool TBL = (STAGE == 0 || STAGE == 4 || STAGE == 5 || STAGE == 6);
    unsigned char* const tb = smem_raw + ((size_t)WT::kWarps * WF + (STAGE == 4 ? (size_t)WT::kWarps * WB4 : 0)) * sizeof(float);
    const float2* const t_win = TBL ? reinterpret_cast<const float2*>(tb) : reinterpret_cast<const float2*>(a.window);
    const float2* const t_tw = TBL ? reinterpret_cast<const float2*>(tb + WT::kWinB) : a.tw;
    const float2* const t_twsh = TBL ? reinterpret_cast<const float2*>(tb + WT::kWinB + WT::kTwB) : a.twsh;
    const int4* const t_slots = TBL ? reinterpret_cast<const int4*>(tb + WT::kWinB + WT::kTwB + WT::kTwshB) : a.mel_slots;
    const float4* const t_melw = TBL ? reinterpret_cast<const float4*>(tb + WT::kWinB + WT::kTwB + WT::kTwshB + (size_t)a.n_mels * 16)
                                     : reinterpret_cast<const float4*>(a.mel_pw);
    if (TBL) {
        float2* d_win = const_cast<float2*>(t_win);
        for (int i = tid; i < M; i += NT) d_win[i] = __ldg(reinterpret_cast<const float2*>(a.window) + i);
        float2* d_tw = const_cast<float2*>(t_tw);
        // transposed for the pass-2 access: entry [r][k] = W_M^{r k} (r < R2, k < E; R2 E = M), so that the lanes of a warp
        // (consecutive k) read consecutive words instead of stride-r ones
        for (int i = tid; i < M; i += NT) {
            const float2 w = __ldg(a.tw + (i / E) * (i % E));
            d_tw[i] = kHalfZ ? make_float2(0.5f * w.x, 0.5f * w.y) : w;
        }
        float2* d_twsh = const_cast<float2*>(t_twsh);
        for (int i = tid; i <= M / 2; i += NT) {
            if (kHalfZ) d_twsh[i] = split_twiddle_h(__ldg(a.tws + i), 4 * i < M);
            else d_twsh[i] = __ldg((STAGE == 4 ? a.tws : a.twsh) + i);
        }
        if ((STAGE == 0 || STAGE == 5 || STAGE == 6) && (mask & syg::FB_MFCC)) {
            int4* d_sl = const_cast<int4*>(t_slots);
            for (int i = tid; i < a.n_mels; i += NT) d_sl[i] = __ldg(a.mel_slots + i);
            float4* d_mw = const_cast<float4*>(t_melw);
            for (int i = tid; i < a.mel_pw_f4; i += NT) d_mw[i] = __ldg(reinterpret_cast<const float4*>(a.mel_pw) + i);
        }
        __syncthreads();
    }

    // STAGE 5: behind the tables: tile [GF8][P] of raw mel energies (then S_db), per-frame reference levels and output offsets, per-unit maxima
    constexpr bool RES = (STAGE == 5);
    const int res_P = RES ? fin_pitch(a.n_mels) : 0;
    const int res_GF8 = RES ? (a.res_units * a.T + 7) / 8 * 8 : 0;
    float* const res_tile = reinterpret_cast<float*>(tb + (RES ? WT::table_bytes(a.n_mels, (mask & syg::FB_MFCC) ? a.mel_pw_f4 : 0) : 0));
    float* const res_ref = res_tile + (size_t)res_GF8 * res_P;
    long long* const res_out = reinterpret_cast<long long*>(res_ref + res_GF8);          // res_GF8 is even: 8-byte aligned
    unsigned* const res_umax = reinterpret_cast<unsigned*>(res_out + res_GF8);

    const long long n_tasks = (a.n_frames + FW - 1) / FW;
    // (unit, frame-in-unit) of this lane's frame advance incrementally: one division per kernel instead of one per frame
    const long long stride_tasks = RES ? WT::kWarps : (long long)gridDim.x * WT::kWarps;
    // STAGE 4 walks "super tasks" of 8 consecutive frames (SUBS tasks each) per warp: small steps of FW frames inside one, a
    // large step to the warp's next super task
    const long long stride_frames = (STAGE == 4) ? (stride_tasks - 1) * TT4 + FW : stride_tasks * FW;
    const long long du = RAG ? 0 : stride_frames / a.T;
    const int dt = RAG ? 0 : (int)(stride_frames - du * a.T);
    // STAGE 5: outer loop over this CTA's unit groups (every other stage: one pass)
    const long long n_groups = RES ? (a.g.n_units + a.res_units - 1) / a.res_units : 1;
    for (long long grp = RES ? blockIdx.x : 0; grp < n_groups; grp += RES ? gridDim.x : 1) {
    const long long grp_u0 = RES ? grp * a.res_units : 0;
    const long long grp_f0 = grp_u0 * a.T;                             // first frame of the group
    const long long frame_end = RES ? min(grp_u0 + a.res_units, a.g.n_units) * (long long)a.T : a.n_frames;
    if (RES) {
        if (tid < a.res_units) res_umax[tid] = 0u;
        __syncthreads();
    }
    long long gf_run = RES ? grp_f0 + (long long)warp * FW + f
                           : ((long long)blockIdx.x * WT::kWarps + warp) * ((STAGE == 4) ? TT4 : FW) + f;
    long long u_run = RAG ? 0 : gf_run / a.T;
    int t_run = RAG ? 0 : (int)(gf_run - u_run * a.T);
    // STAGE 6: the table entry of this lane's next frame is loaded one task ahead (its latency hides behind the current task)
    int4 rnext = (RAG && gf_run < frame_end) ? __ldg(a.ragged_ut + gf_run) : make_int4(0, 0, 0, 0);
    const long long task_begin = (STAGE == 4) ? ((long long)blockIdx.x * WT::kWarps + warp) * SUBS : (RES ? 0 : (long long)blockIdx.x * WT::kWarps);
    const long long task_end = (STAGE == 4) ? ((a.n_frames + TT4 - 1) / TT4) * SUBS : (RES ? (frame_end - grp_f0 + FW - 1) / FW : n_tasks);
    // STAGE 0 / 3 / 5: all warps of the CTA run the same number of iterations (tasks past the end are processed as empty frames)
    for (long long task0 = task_begin; task0 < task_end;
         task0 = (STAGE == 4) ? ((((task0 + 1) & (SUBS - 1)) != 0) ? task0 + 1 : task0 + 1 + (stride_tasks - 1) * SUBS) : task0 + stride_tasks) {
        const long long task = (STAGE == 4) ? task0 : task0 + warp;
        const long long tf0 = RES ? grp_f0 + task * FW : task * FW;    // first global frame of this warp's task
        // (measured in round 2: re-aligning the warps of one scheduler with a named barrier once per frame, so that they share
        // instruction fetches of the ~50 KB loop body, costs +2.4 % -- the phase diversity is worth more than the fetches)
        const long long gf = gf_run;
        // one frame per warp and no barrier inside the task (feature stage): a task past the end is simply skipped, and `valid` is a
        // compile-time true for everything below (no predicates on the feature stores, no branches around the workspace rows)
        constexpr bool kSkipInvalid = ((STAGE == 0 || STAGE == 6) && FW == 1);
        const bool valid_rt = gf < frame_end;
        const bool valid = kSkipInvalid ? true : valid_rt;
        const int4 rut = rnext;
        const long long u = RAG ? (long long)rut.x : ((kSkipInvalid || valid) ? u_run : 0);
        const int t = RAG ? rut.y : ((kSkipInvalid || valid) ? t_run : 0);
        if (STAGE == 4 && ((task0 + 1) & (SUBS - 1)) != 0) {          // next task of the same super task: FW frames on
            gf_run += FW;
            t_run += FW;
        } else {
            gf_run += stride_frames;
            u_run += du;
            t_run += dt;
        }
        if (!RAG) while (t_run >= a.T) { t_run -= a.T; ++u_run; }
        if (RAG) rnext = gf_run < frame_end ? __ldg(a.ragged_ut + gf_run) : make_int4(0, 0, 0, 0);
        if (kSkipInvalid && !valid_rt) continue;
        UnitRef ur = RAG ? UnitRef{(long long)rut.w, (long long)rut.z} : unit_ref(a.g, u);
        if (!valid) ur.valid = 0;
        const long long p0 = (long long)t * a.hop - a.cpad;

        float* const orow = RAG ? a.out + gf : a.out + (long long)u * a.n_rows * a.T + t;
        // ---------------- framing + window + time-domain partial statistics ----------------
        float2 z[E];
        float2 sq2 = make_float2(0.0f, 0.0f);
        float pk = 0.0f;
        double s_sum = 0.0, s_abs = 0.0, s_sqd = 0.0;
        {
            const float* src = a.y + ur.start + p0;
            const bool interior = (p0 >= 0) && (p0 + 2 * M <= ur.valid) && ((reinterpret_cast<uintptr_t>(src) & 7u) == 0);
            const float2* w2 = t_win;
            if (__all_sync(kFull, interior)) {
                SYG_UNROLL
                for (int r = 0; r < E; ++r) {
                    const int c = j + r * G;
                    const float2 v = __ldg(reinterpret_cast<const float2*>(src) + c);
                    const float2 w = TBL ? w2[c] : __ldg(w2 + c);
                    sq2 = __ffma2_rn(v, v, sq2);
                    pk = fmaxf(fmaxf(pk, fabsf(v.x)), fabsf(v.y));         // one FMNMX3 (|.| are operand modifiers)
                    if (EXTRA) {
                        s_sum += (double)v.x + (double)v.y;
                        s_abs += (double)fabsf(v.x) + (double)fabsf(v.y);
                        s_sqd += (double)v.x * (double)v.x + (double)v.y * (double)v.y;
                    }
                    z[r] = __fmul2_rn(v, w);
                }
            } else {
                // edge / unaligned frames: predicated loads (zero padding by predicate; reflect padding for STFT).  The frame's valid
                // range is computed once in frame-local 32-bit coordinates [lo, lo + span): one unsigned compare per sample; pairs
                // that lie fully inside an 8-byte aligned frame still load as one LDG.64.
                const long long nv = ur.valid;
                const bool refl = (STAGE == 3) && a.pad_mode == 1 && nv > 0;
                const float* const fb = a.y + ur.start + p0;             // frame base: dereferenced at valid positions only
                const long long lo64 = p0 < 0 ? -p0 : 0, hi64 = nv - p0;
                const int lo = (int)(lo64 < 2 * M ? lo64 : 2 * M);
                const int hi = (int)(hi64 < 0 ? 0 : (hi64 < 2 * M ? hi64 : 2 * M));
                const unsigned span = hi > lo ? (unsigned)(hi - lo) : 0u;
                const bool al = (reinterpret_cast<uintptr_t>(fb) & 7u) == 0;
                SYG_UNROLL
                for (int r = 0; r < E; ++r) {
                    const int c = j + r * G;
                    const unsigned d = (unsigned)(2 * c - lo);
                    float2 v = make_float2(0.0f, 0.0f);
                    if (al && d < span && d + 1u < span) {
                        v = __ldg(reinterpret_cast<const float2*>(fb) + c);
                    } else {
                        if (d < span) v.x = __ldg(fb + 2 * c);
                        else if (refl) v.x = __ldg(a.y + ur.start + reflect_index(p0 + 2 * c, nv));
                        if (d + 1u < span) v.y = __ldg(fb + 2 * c + 1);
                        else if (refl) v.y = __ldg(a.y + ur.start + reflect_index(p0 + 2 * c + 1, nv));
                    }
                    const float2 w = TBL ? w2[c] : __ldg(w2 + c);
                    sq2 = __ffma2_rn(v, v, sq2);
                    pk = fmaxf(fmaxf(pk, fabsf(v.x)), fabsf(v.y));         // one FMNMX3 (|.| are operand modifiers)
                    if (EXTRA) {
                        s_sum += (double)v.x + (double)v.y;
                        s_abs += (double)fabsf(v.x) + (double)fabsf(v.y);
                        s_sqd += (double)v.x * (double)v.x + (double)v.y * (double)v.y;
                    }
                    z[r] = __fmul2_rn(v, w);
                }
            }
        }

        // ---------------- pass 1: radix E, no twiddles; butterfly j scatters to j*E + k' ----------------
        dft_dif_p<E, 1>(z);
        SYG_UNROLL
        for (int kp = 0; kp < E; ++kp) zs[zpad<LE>(j * E + kp)] = z[bitrev(kp, LE)];
        __syncwarp();
        // ---------------- pass 2: Q butterflies of radix R2 per lane, twiddles W_M^{r k} ----------------
        SYG_UNROLL
        for (int q = 0; q < Q; ++q) {
            const int b = j + q * G;
            SYG_UNROLL
            for (int r = 0; r < R2; ++r) {
                z[q * R2 + r] = zs[zpad<LE>(b + r * (M / R2))];
            }
        }
        __syncwarp();
        SYG_UNROLL
        for (int q = 0; q < Q; ++q) {
            const int b = j + q * G;
            const int k = b & (E - 1);                                 // NS = E
            constexpr int SH = TL::LOG2M - ilog2(E * R2);             // = 0: W_{E*R2} = W_M
            SYG_UNROLL
            for (int r = 1; r < R2; ++r) {
                const float2 w = TBL ? t_tw[r * E + k] : __ldg(&t_tw[(r * k) << SH]);
                cmul(z[q * R2 + r].x, z[q * R2 + r].y, w.x, w.y);
            }
            dft_dif_p<R2, 1, kHalfZ>(z + q * R2);
            if constexpr (!kShflSplit) {
                const int ob = (b - k) * R2 + k;
                SYG_UNROLL
                for (int kp = 0; kp < R2; ++kp) {
                    zs[zpad<LE>(ob + kp * E)] = z[q * R2 + bitrev(kp, ilog2(R2))];
                }
            }
        }
        if constexpr (!kShflSplit) __syncwarp();

        // ---------------- real split -> |X[k]|^2 (overwrites the Z region: all pairs are pulled into registers first) ----------------
        // Lane j pairs bin k = j + i G with bin M - k.  All addresses are lane bases plus compile-time offsets: for j >= 1
        // the bins M - iG - j of one step share a pad block, lane 0 (bin M - iG, a block start when iG is a multiple of the
        // block size) sits one pad group further.
        {
            const int jz = (j == 0) ? 1 : 0;
            const float2* const zk0 = zs + j;                           // Z[k]     at zk0[zpad(iG)] (j + iG stays in iG's block: G <= E)
            const float2* const zm0 = zs - j;                           // Z[M - k] at zm0[c1_i], lane 0: + 1 where M - iG starts a block
            const float2* const zm1 = zm0 + jz;
            float2 zk[E / 2 + 1], zm[E / 2 + 1];
            if constexpr (kShflSplit) {
                // the mirrors come from the partner lane's registers (mirror_of): no natural-order Z in shared memory at all
                SYG_UNROLL
                for (int i = 0; i < E / 2; ++i) {
                    zk[i] = z[zreg_of<E, G>(i)];
                    zm[i] = mirror_of<E, G>(z, i, j);
                }
                zk[E / 2] = zm[E / 2] = z[zreg_of<E, G>(E / 2)];          // lane 0 only: bin M/2 pairs with itself
            } else {
                SYG_UNROLL
                for (int i = 0; i <= E / 2; ++i) {
                    const int kk = i * G;                                // compile time after unrolling
                    zk[i] = zk0[kk + (kk >> LE)];
                    const int c1 = (M - kk) + ((M - kk - 1) >> LE);      // zpad(M - kk - j) + j for 1 <= j < G
                    const bool blk = ((M - kk) & (E - 1)) == 0;          // M - kk starts a pad block -> lane 0 is one slot further
                    zm[i] = blk ? zm1[c1] : zm0[c1];
                }
                if (j == 0) zm[0] = zk[0];                               // k = 0 pairs with itself (DC / Nyquist)
                __syncwarp();
            }
            float* const pk0 = pf + j;                                   // P[k]     at pk0[ppad(iG)]
            float* const pm0 = pf - j;                                   // P[M - k] at pm0[q1_i], lane 0: + 4 where M - iG starts a 32-bin block
            float* const pm1 = pm0 + 4 * jz;
            SYG_UNROLL
            for (int i = 0; i <= E / 2; ++i) {
                const int kk = i * G;
                const int k = j + kk;
                if (i == E / 2 && j != 0) break;
                if (STAGE == 4) {
                    const float2 w = t_twsh[k];
                    float xkr, xki, xmr, xmi;
                    real_split(zk[i].x, zk[i].y, zm[i].x, zm[i].y, w.x, w.y, xkr, xki, xmr, xmi);
                    const int slot = (int)(task & (SUBS - 1)) * FW + f;
                    const int k2 = M - k;
                    float pk_ = __fmaf_rn(xkr, xkr, xki * xki), pm_ = __fmaf_rn(xmr, xmr, xmi * xmi);
                    if (a.out_kind == 1) { pk_ = sqrt_approx(pk_); pm_ = sqrt_approx(pm_); }
                    wtile[k * TTP4 + slot] = pk_;
                    if (k2 != k) wtile[k2 * TTP4 + slot] = pm_;
                    continue;
                }
                if (STAGE == 3) {
                    const float2 w = __ldg(&a.tws[k]);
                    float xkr, xki, xmr, xmi;
                    real_split(zk[i].x, zk[i].y, zm[i].x, zm[i].y, w.x, w.y, xkr, xki, xmr, xmi);
                    const int slot = warp * FW + f;
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
                    continue;
                }
                const float2 wh = TBL ? t_twsh[k] : __ldg(&t_twsh[k]);
                float pwk, pwm;
                if constexpr (kHalfZ) split_power_h(4 * i < E, zk[i], zm[i], wh, pwk, pwm);   // k = j + G i < M/4 for every lane iff i < E/4
                else split_power(zk[i], zm[i], wh, pwk, pwm);
                pk0[kk + ((kk >> 5) << 2)] = pwk;
                const int q1 = (M - kk) + (((M - kk - 1) >> 5) << 2);
                const bool blk = ((M - kk) & 31) == 0;
                if (2 * k != M) (blk ? pm1 : pm0)[q1] = pwm;
            }
        }
        __syncwarp();


        if (STAGE == 4) {
            // ---------------- STFT output, warp-private: after the super task's last frames, rows of 8 frames per bin ----------------
            if (j == 0) woff[(int)(task & (SUBS - 1)) * FW + f] = valid ? ((long long)u * B) * a.T + t : -1;
            __syncwarp();
            if (((task0 + 1) & (SUBS - 1)) == 0) {
                const int sl = lane & (TT4 - 1), kq = lane / TT4;       // 4 rows of 8 frames per warp instruction
                const long long off = woff[sl];
                if (off >= 0) {
                    const float* src = wtile + kq * TTP4 + sl;
                    float* dst = reinterpret_cast<float*>(a.stft_out) + off + (long long)kq * a.T;
                    const long long dstep = 4LL * a.T;
                    for (int k = kq; k < B; k += 4, src += 4 * TTP4, dst += dstep) *dst = *src;
                }
                __syncwarp();                                           // the tile is refilled by the warp's next super task
            }
            continue;
        }
        if (STAGE == 3) {
            // ---------------- STFT output: rows of TT consecutive frames per bin leave the CTA as contiguous runs ----------------
            if (j == 0) slot_off[warp * FW + f] = valid ? ((long long)u * B) * a.T + t : -1;
            __syncthreads();
            // thread -> (slot = tid % TT, bins tid / TT + i * NT / TT): the slot, its output offset and the strides are loop constants
            static_assert(NT % TT == 0, "the CTA covers whole tile rows per step");
            constexpr int KS = NT / TT;
            const int sl = tid % TT, kq = tid / TT;
            const long long off = slot_off[sl];
            if (off >= 0) {
                if (a.out_kind == 0) {
                    const float2* src = reinterpret_cast<const float2*>(tile) + kq * TTP + sl;
                    float2* dst = reinterpret_cast<float2*>(a.stft_out) + off + (long long)kq * a.T;
                    const long long dstep = (long long)KS * a.T;
                    for (int k = kq; k < B; k += KS, src += KS * TTP, dst += dstep) *dst = *src;
                } else {
                    const float* src = tile + kq * TTP + sl;
                    float* dst = reinterpret_cast<float*>(a.stft_out) + off + (long long)kq * a.T;
                    const long long dstep = (long long)KS * a.T;
                    for (int k = kq; k < B; k += KS, src += KS * TTP, dst += dstep) *dst = *src;
                }
            }
            __syncthreads();                                        // the tile is refilled by the next round
            continue;
        }
        // ---------------- time-domain features (unwindowed, zero-padded frame) ----------------
        if (mask & syg::FB_TIME_ANY) {
            const float tsq = lanes_sum<G>(sq2.x + sq2.y);
            const float tpk = lanes_max<G>(pk);
            if (j == 0 && valid) {
                const float rms = sqrt_approx(tsq * (1.0f / (float)TL::NFFT));     // MUFU.SQRT (1 ulp) instead of the IEEE sequence; bar: rel 1e-5
                if (row_rms >= 0) orow[(long long)row_rms * (RAG ? a.ragged_stride : a.T)] = rms;
                // eps(float64) = 2^-52 is a float too: the reference's `rms < eps` on the widened value is this float comparison
                if (row_crest >= 0) orow[(long long)row_crest * (RAG ? a.ragged_stride : a.T)] = (rms < 2.220446049250313e-16f) ? 0.0f : __fdividef(tpk, rms);
                if (row_peak >= 0) orow[(long long)row_peak * (RAG ? a.ragged_stride : a.T)] = tpk;
            }
            if (EXTRA) {
                if (mask & (syg::FB_STD_AMP | syg::FB_MEAN_AMP)) {
                    const double tsum = lanes_sum<G>(s_sum), tabs = lanes_sum<G>(s_abs), tsqd = lanes_sum<G>(s_sqd);
                    if (j == 0 && valid) {
                        const double n = (double)TL::NFFT;
                        if (a.row_mean_amp >= 0) orow[(long long)a.row_mean_amp * (RAG ? a.ragged_stride : a.T)] = (float)(tabs / n);
                        if (a.row_std_amp >= 0) {
                            const double mu = tsum / n;
                            double var = tsqd / n - mu * mu;
                            if (var < 0.0) var = 0.0;
                            orow[(long long)a.row_std_amp * (RAG ? a.ragged_stride : a.T)] = (float)sqrt(var);
                        }
                    }
                }
            }
        }

        // ---------------- per-frame spectral statistics (lane j owns bins [j*E, j*E+E), last lane also bin M) ----------------
        if (mask & syg::FB_SPECSTATS) {
            const int k0 = j * E;
            float p[E];
            {
                const float4* pb4 = reinterpret_cast<const float4*>(pf + ppad(k0));   // E is a multiple of 4 and <= 32: one block
                SYG_UNROLL
                for (int i = 0; i < E / 4; ++i) {
                    const float4 v = pb4[i];
                    p[4 * i] = v.x; p[4 * i + 1] = v.y; p[4 * i + 2] = v.z; p[4 * i + 3] = v.w;
                }
            }
            // bin pairs (i, i + 1) in FP32x2: power sums (two packed accumulators), magnitude sums and sum i * mag with the EVEN index
            // as the broadcast multiplier of both halves -- the odd bins' missing "+ 1" is the packed magnitude sum's odd half
            float2 sp2[2] = {make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f)};
            float2 sm2 = make_float2(0.0f, 0.0f), skm2 = make_float2(0.0f, 0.0f);
            float slog = 0.0f, vmax = -1.0f;
            int imax = 0;
            SYG_UNROLL
            for (int i = 0; i < E; i += 2) {
                const float2 mg2 = make_float2(sqrt_approx(p[i]), sqrt_approx(p[i + 1]));
                sp2[(i >> 1) & 1] = __fadd2_rn(sp2[(i >> 1) & 1], make_float2(p[i], p[i + 1]));
                sm2 = __fadd2_rn(sm2, mg2);
                skm2 = __ffma2_rn(mg2, make_float2((float)i, (float)i), skm2);
                if (EXTRA) {
                    SYG_UNROLL
                    for (int h = 0; h < 2; ++h) {
                        if (mask & syg::FB_FLATNESS) slog += logf(sqrtf(p[i + h]) + 2.220446049250313e-16f);
                        if (p[i + h] > vmax) { vmax = p[i + h]; imax = k0 + i + h; }
                    }
                }
            }
            float lsp = (sp2[0].x + sp2[0].y) + (sp2[1].x + sp2[1].y);
            float lsm = sm2.x + sm2.y;
            float lskm = __fmaf_rn(lsm, (float)k0, (skm2.x + skm2.y) + sm2.y);     // sum (k0 + i) mag_i
            const float p_ny = pf[ppad(M)];
            if (j == G - 1) {                                            // bin M (Nyquist)
                const float mg = sqrt_approx(p_ny);
                lsp += p_ny;
                lsm += mg;
                lskm = __fmaf_rn(mg, (float)M, lskm);
                if (EXTRA) {
                    if (mask & syg::FB_FLATNESS) slog += logf(sqrtf(p_ny) + 2.220446049250313e-16f);
                    if (p_ny > vmax) { vmax = p_ny; imax = M; }
                }
            }
            const int nk = E + ((j == G - 1) ? 1 : 0);
            // lane sums are FP32 (pairwise, <= 33 terms); the running sum across lanes is FP64 (reference: float64 cumsum)
            const double incl = lanes_scan_incl<G>((double)lsp, j);
            const double total_p = __shfl_sync(kFull, incl, G - 1, G);
            const float tm = lanes_sum<G>(lsm);
            const float tkm = lanes_sum<G>(lskm);
            double centroid_hz = 0.0;
            if constexpr (EXTRA) {                                       // spectral_bandwidth needs the float64 centroid
                if ((double)tm >= kEps64) centroid_hz = a.bin_hz * ((double)tkm / (double)tm);
                if (row_centroid >= 0 && j == 0 && valid) orow[(long long)row_centroid * (RAG ? a.ragged_stride : a.T)] = (float)centroid_hz;
            } else {
                // the sums are FP32 already; one FP32 division (2^-23 relative against a 1e-5 parity bar) instead of a float64 one
                const float c = (tm >= 2.220446049250313e-16f) ? (float)a.bin_hz * __fdividef(tkm, tm) : 0.0f;
                if (row_centroid >= 0 && j == 0 && valid) orow[(long long)row_centroid * (RAG ? a.ragged_stride : a.T)] = c;
            }
            if (row_rolloff >= 0) {
                // first bin whose cumulative power reaches roll_percent * total (frequency_domain.py:334-346)
                const double thr = a.roll_percent * total_p;
                const unsigned gmask = (G == 32) ? kFull : (((1u << G) - 1u) << (f * G));
                const unsigned hit = __ballot_sync(kFull, incl >= thr) & gmask;
                const int L = hit ? (__ffs((int)hit) - 1 - f * G) : (G - 1);          // crossing lane of this frame's group
                const double prevL = __shfl_sync(kFull, incl - (double)lsp, L, G);
                const float thrl = (float)(thr - prevL);
                // the group's lanes scan lane L's E bins together: R consecutive bins each
                constexpr int R = (E + G - 1) / G;
                const int kL = L * E;
                float v[R], s = 0.0f;
                SYG_UNROLL
                for (int r = 0; r < R; ++r) {
                    const int q = j * R + r;
                    v[r] = (q < E) ? pf[ppad(kL + q)] : 0.0f;
                    s += v[r];
                }
                float inc = s;
                SYG_UNROLL
                for (int o = 1; o < G; o <<= 1) {
                    const float nb_ = __shfl_up_sync(kFull, inc, o, G);
                    if (j >= o) inc += nb_;
                }
                float c = inc - s;
                int pos = -1;
                SYG_UNROLL
                for (int r = 0; r < R; ++r) {
                    c += v[r];
                    if (pos < 0 && j * R + r < E && c >= thrl) pos = j * R + r;
                }
                const unsigned found = __ballot_sync(kFull, pos >= 0) & gmask;
                const int src = found ? (__ffs((int)found) - 1 - f * G) : 0;
                const int posw = __shfl_sync(kFull, pos, src, G);
                if (j == 0 && valid) {
                    int bin;
                    if (total_p < kEps64) bin = M;                                      // silent frame -> freqs[-1]
                    else if (found) bin = kL + posw;
                    else bin = (L == G - 1) ? M : kL + E - 1;                           // only the lane's last element is left
                    orow[(long long)row_rolloff * (RAG ? a.ragged_stride : a.T)] = (float)(a.bin_hz * (double)bin);
                }
            }
            if (EXTRA) {
                if (a.row_flatness >= 0) {
                    const float tl = lanes_sum<G>(slog);
                    if (j == 0 && valid) {
                        const double am = (double)tm / (double)B;
                        double fl = 0.0;
                        if (am >= kEps64) {
                            fl = exp((double)tl / (double)B) / am;
                            fl = fl < 0.0 ? 0.0 : (fl > 1.0 ? 1.0 : fl);
                        }
                        orow[(long long)a.row_flatness * (RAG ? a.ragged_stride : a.T)] = (float)fl;
                    }
                }
                if (a.row_bandwidth >= 0) {
                    double sb = 0.0;
                    SYG_UNROLL
                    for (int i = 0; i < E; ++i) {
                        const double mg = (double)sqrtf(p[i]);
                        const double d = a.bin_hz * (double)(k0 + i) - centroid_hz;
                        sb += mg * d * d;
                    }
                    if (nk > E) {
                        const double d = a.bin_hz * (double)M - centroid_hz;
                        sb += (double)sqrtf(p_ny) * d * d;
                    }
                    const double tb = lanes_sum<G>(sb);
                    if (j == 0 && valid) orow[(long long)a.row_bandwidth * (RAG ? a.ragged_stride : a.T)] = ((double)tm < kEps64) ? 0.0f : (float)sqrt(tb / (double)tm);
                }
                if (a.row_dominant >= 0) {
                    const float gmax = lanes_max<G>(vmax);
                    float mi = (vmax == gmax) ? -(float)imax : -1.0e9f;
                    mi = lanes_max<G>(mi);
                    if (j == 0 && valid) orow[(long long)a.row_dominant * (RAG ? a.ragged_stride : a.T)] = (float)(a.bin_hz * (double)(-mi));
                }
            }
        }

        // ---------------- spectral contrast: per band mean of the n largest / n smallest magnitudes ----------------
        if (mask & syg::FB_CONTRAST) {
            for (int ff = 0; ff < FW; ++ff) {
                const long long gff = tf0 + ff;
                if (!kSkipInvalid && gff >= frame_end) break;
                const float* pp = pww + ff * RSS;
                float pmx = 0.0f, vmx = 0.0f;
                float mine_pv = 0.0f;                                   // lane bd keeps band bd's peak, lane nb + bd its valley
                const int lane_v = lane - a.nb;
                if constexpr (SP::kBands) {
                    SYG_UNROLL
                    for (int bd = 0; bd < SP::nb; ++bd) {               // compile-time band layout: (lo, count, n) fold into the code
                        const float2 pv = band_peak_valley_stream<true>(pp, SP::band(bd, 0), SP::band(bd, 1), SP::band(bd, 2));
                        mine_pv = (lane == bd) ? pv.x : mine_pv;
                        mine_pv = (lane == SP::nb + bd) ? pv.y : mine_pv;
                        pmx = fmaxf(pmx, pv.x);
                        vmx = fmaxf(vmx, pv.y);
                    }
                } else
                for (int bd = 0; bd < a.nb; ++bd) {
                    const int cnt = a.band_cnt[bd];                     // 1 <= band_n <= band_cnt is guaranteed by the plan (syg_api.cu)
                    float2 pv = make_float2(__uint_as_float(0x7fc00000u), __uint_as_float(0x7fc00000u));   // empty band: mean of nothing -> NaN (numpy)
                    if (cnt > 0) pv = band_peak_valley_stream<false>(pp, a.band_lo[bd], cnt, a.band_n[bd]);
                    mine_pv = (lane == bd) ? pv.x : mine_pv;
                    mine_pv = (lane_v == bd) ? pv.y : mine_pv;
                    pmx = fmaxf(pmx, pv.x);                             // fmaxf drops the NaN of an empty band
                    vmx = fmaxf(vmx, pv.y);
                }
                if (lane < 2 * a.nb) a.cws[gff * (2 * a.nb) + lane] = mine_pv;   // one coalesced store per frame (nb <= kMaxBands = 12)
                const long long uff = (FW == 1) ? u : __shfl_sync(kFull, u, ff * G);   // unit of frame ff (FW == 1: warp uniform already)
                const float mx12 = lane ? vmx : pmx;                    // lane 0: peaks -> word 1, lane 1: valleys -> word 2
                if (lane < 2 && mx12 > 0.0f) red_max_u32(a.unit_max + uff * 4 + 1 + lane, __float_as_uint(mx12));
            }
        }
        __syncwarp();                                                   // interval-form mel overwrites the spectrum: contrast has read it
        // ---------------- mel energies: one filter per lane; the warp sweeps GS = 32 / FW filters of each of its frames at once ----------------
        // (Loading a tap vector once for all FW frames of the task -- 32 filters per sweep, frames in an inner loop -- was measured:
        // fewer shared-memory wavefronts but 7 instead of 4 instructions per step and idle lanes in the last sweep; cfg3 +10 % time.)
        if (mask & syg::FB_MFCC) {
            constexpr int GS = 32 / FW;
            const int mf = lane / GS, sl = lane % GS;                   // frame of the warp task, slot within the sweep group
            const long long gmf = tf0 + mf;
            const bool fvalid = kSkipInvalid ? true : (gmf < frame_end);
            // STAGE 5: the energies stay in the CTA tile (row = frame within the group)
            float* const mrow = RES ? res_tile + (size_t)(gmf - grp_f0) * res_P : a.melws + gmf * a.n_mels;
            const float* pfr = pww + mf * RSS;
            const float4* const mw4 = t_melw;
            float fmx = 0.0f;
            if (a.mel_iv) {
                // ---- interval form (sygplan::MelIntervals): lane (f, j) owns the E contiguous bins [jE, jE + E) of its frame.  Two
                // running sums per bin -- the bin's weight in the filter rising through its mel interval and in the one falling
                // through it -- restart at interval starts; their totals land in CR / CF (which take the place of |X|^2: nothing
                // after this stage reads the spectrum in this mode) and every filter adds up its picks.
                static_assert(E % 4 == 0 && E <= 32, "interval form: E bins per lane in one 32-bin block");
                float* const reg = pww + mf * RSS;                      // this frame's region: |X|^2 now, then CR | CF | zero word
                float p[E];
                {
                    const float4* pb4 = reinterpret_cast<const float4*>(reg + ppad(sl * E));
                    SYG_UNROLL
                    for (int i = 0; i < E / 4; ++i) {
                        const float4 v = pb4[i];
                        p[4 * i] = v.x; p[4 * i + 1] = v.y; p[4 * i + 2] = v.z; p[4 * i + 3] = v.w;
                    }
                }
                const float p_nyq = reg[ppad(M)];                       // the Nyquist bin (its word becomes the first of CF)
                __syncwarp();                                           // every lane holds its bins before the region is overwritten
                const float4* const wt = mw4;                           // [E/2][G] {wr, wf, wr, wf}
                const int4* const picks = reinterpret_cast<const int4*>(mw4 + M / 2);
                const unsigned keep = reinterpret_cast<const unsigned*>(mw4 + M / 2 + a.n_mels)[sl];
                constexpr int PSM = M + M / 8;                          // CR at [0, PSM), CF at [PSM, 2 PSM), both in the padded bin layout
                float cr = 0.0f, cf = 0.0f;
                float4* const cr4 = reinterpret_cast<float4*>(reg + ppad(sl * E));
                float4* const cf4 = reinterpret_cast<float4*>(reg + PSM + ppad(sl * E));
                SYG_UNROLL
                for (int q = 0; q < E / 4; ++q) {
                    float r[4], g[4];
                    SYG_UNROLL
                    for (int h = 0; h < 2; ++h) {
                        const float4 w = wt[(2 * q + h) * GS + sl];
                        const int b = 4 * q + 2 * h;
                        const bool k0 = (keep >> b) & 1u, k1 = (keep >> (b + 1)) & 1u;
                        cr = __fmaf_rn(p[b], w.x, k0 ? cr : 0.0f);
                        cf = __fmaf_rn(p[b], w.y, k0 ? cf : 0.0f);
                        r[2 * h] = cr; g[2 * h] = cf;
                        cr = __fmaf_rn(p[b + 1], w.z, k1 ? cr : 0.0f);
                        cf = __fmaf_rn(p[b + 1], w.w, k1 ? cf : 0.0f);
                        r[2 * h + 1] = cr; g[2 * h + 1] = cf;
                    }
                    cr4[q] = make_float4(r[0], r[1], r[2], r[3]);
                    cf4[q] = make_float4(g[0], g[1], g[2], g[3]);
                }
                if (sl == 0) reg[2 * PSM] = 0.0f;                       // the word unused picks point at
                __syncwarp();
                for (int m = sl; m < a.n_mels; m += GS) {
                    const int4 pk4 = picks[m];                          // {r0, r1, f0, f1}
                    float acc = (reg[pk4.x] + reg[pk4.y]) + (reg[pk4.z] + reg[pk4.w]);
                    if (m == a.n_mels - 1) acc = __fmaf_rn(reinterpret_cast<const float*>(mw4 + M / 2 + a.n_mels + (G + 3) / 4)[0], p_nyq, acc);
                    if (fvalid) {
                        mrow[m] = acc;
                        fmx = fmaxf(fmx, acc);
                    }
                }
            } else
            if constexpr (SP::kMel && FW == 1) {
                // plan-specialised sweeps: n_mels = 32 * n_sweeps, every trip count and tap offset is a constant
                int goff = 0;
                SYG_UNROLL
                for (int sw = 0; sw < SP::n_sweeps; ++sw) {
                    const int4 d = t_slots[sw * 32 + sl];                // {filter, first padded word, steps, tap offset}
                    const float4* wv = mw4 + goff + sl;
                    const float4* pp4 = reinterpret_cast<const float4*>(pfr + d.y);
                    float2 m01 = make_float2(0.0f, 0.0f), m23 = m01;
                    SYG_UNROLL
                    for (int i = 0; i < SP::steps(sw); ++i) {
                        const float4 w = wv[32 * i];
                        const float4 q = pp4[i];
                        m01 = __ffma2_rn(make_float2(w.x, w.y), make_float2(q.x, q.y), m01);
                        m23 = __ffma2_rn(make_float2(w.z, w.w), make_float2(q.z, q.w), m23);
                    }
                    const float acc = (m01.x + m01.y) + (m23.x + m23.y);
                    if (fvalid) {
                        mrow[d.x] = acc;
                        fmx = fmaxf(fmx, acc);
                    }
                    goff += 32 * SP::steps(sw);
                }
            } else
            for (int base = 0; base < a.n_mels; base += GS) {
                const int slot = min(base + sl, a.n_mels - 1);
                const int4 d = TBL ? t_slots[slot] : __ldg(&t_slots[slot]);   // {filter, first padded word, steps, tap offset}: steps/offset are warp uniform
                const float4* wv = mw4 + d.w + sl;
                const float4* pp4 = reinterpret_cast<const float4*>(pfr + d.y);
                float acc = 0.0f;
                if (a.mel_power_is_2) {
                    float2 m01 = make_float2(0.0f, 0.0f), m23 = m01;
                    int i = 0;
#ifndef SYG_EMU
#pragma unroll 1
#endif
                    for (; i + 4 <= d.z; i += 4) {                      // steps come in multiples of two (syg_plan.h): fours, then a tail of two
                        SYG_UNROLL
                        for (int c = 0; c < 4; ++c) {
                            const float4 w = TBL ? wv[GS * (i + c)] : __ldg(wv + GS * (i + c));
                            const float4 q = pp4[i + c];
                            m01 = __ffma2_rn(make_float2(w.x, w.y), make_float2(q.x, q.y), m01);
                            m23 = __ffma2_rn(make_float2(w.z, w.w), make_float2(q.z, q.w), m23);
                        }
                    }
                    if (i < d.z) {
                        SYG_UNROLL
                        for (int c = 0; c < 2; ++c) {
                            const float4 w = TBL ? wv[GS * (i + c)] : __ldg(wv + GS * (i + c));
                            const float4 q = pp4[i + c];
                            m01 = __ffma2_rn(make_float2(w.x, w.y), make_float2(q.x, q.y), m01);
                            m23 = __ffma2_rn(make_float2(w.z, w.w), make_float2(q.z, q.w), m23);
                        }
                    }
                    acc = (m01.x + m01.y) + (m23.x + m23.y);
                } else {
                    // Zero-weight taps also cover the pad words of the spectrum, which still hold FFT data from the transform
                    // (negative values too): powf of those is NaN, and 0 * NaN would poison the filter.  Only weighted taps
                    // (always real bins, |X|^2 >= 0) are raised to the power.
                    for (int i = 0; i < d.z; ++i) {
                        const float4 w = TBL ? wv[GS * i] : __ldg(wv + GS * i);
                        const float4 q = pp4[i];
                        acc = __fmaf_rn(w.x, w.x != 0.0f ? powf(q.x, a.mel_half_power) : 0.0f, acc);
                        acc = __fmaf_rn(w.y, w.y != 0.0f ? powf(q.y, a.mel_half_power) : 0.0f, acc);
                        acc = __fmaf_rn(w.z, w.z != 0.0f ? powf(q.z, a.mel_half_power) : 0.0f, acc);
                        acc = __fmaf_rn(w.w, w.w != 0.0f ? powf(q.w, a.mel_half_power) : 0.0f, acc);
                    }
                }
                if (base + sl < a.n_mels && fvalid) {
                    mrow[d.x] = acc;
                    fmx = fmaxf(fmx, acc);
                }
            }
            const float gmx = lanes_max<GS>(fmaxf(fmx, 0.0f));
            const long long umf = (FW == 1) ? u : __shfl_sync(kFull, u, mf * G);   // unit of frame mf (all lanes take part)
            if (sl == 0 && fvalid && gmx > 0.0f) {
                if (RES) atomicMax(&res_umax[(int)(umf - grp_u0)], __float_as_uint(gmx));
                else red_max_u32(a.unit_max + umf * 4, __float_as_uint(gmx));
            }
        }

        __syncwarp();                                                   // smem slices are reused by the next task
    }
    if constexpr (RES) {
        // ---------------- the group's MFCC epilogue, on chip (finalize_kernel's arithmetic on the shared-memory tile) ----------------
        __syncthreads();
        const int gfr = (int)(frame_end - grp_f0);                      // frames of this group
        const int N = a.n_mels, P = res_P;
        for (int fi = tid; fi < gfr; fi += NT) {
            const int ul = fi / a.T, tt = fi - ul * a.T;
            res_ref[fi] = db10(fmaxf(a.fin_amin, __uint_as_float(res_umax[ul])));
            res_out[fi] = (grp_u0 + ul) * (long long)a.n_rows * a.T + tt;
        }
        __syncthreads();
        {
            // A warp item = 8 consecutive frames, BOTH parities (two independent DMMA chains per k-step).  The dB conversion of
            // power_to_db happens on the way into the B fragment: every tile entry is read and converted exactly once.
            const int H = a.fin_dct_fold ? (N + 1) / 2 : N;
            const int H4 = (H + 3) / 4 * 4;
            const int g = lane >> 2, q = lane & 3;
            const int n8 = (gfr + 7) / 8;
            const float floor_db = -a.fin_top_db;
            for (int w = warp; w < n8; w += WT::kWarps) {
                const int nt8 = w * 8;
                const int fr = min(nt8 + g, gfr - 1);                   // this lane's frame (B column); the tail tile repeats the last frame
                const float* const xrow = res_tile + (size_t)fr * P;
                const float ref_db = res_ref[fr];
                const int t0 = nt8 + 2 * q;
                const long long o0 = (t0 < gfr) ? res_out[t0] : 0, o1 = (t0 + 1 < gfr) ? res_out[t0 + 1] : 0;
                const int n_even = (a.fin_n_mfcc + 1) / 2;
                for (int m0 = 0; m0 < n_even; m0 += 8) {
                    const int c_e = 2 * (m0 + g), c_o = c_e + 1;        // coefficients of this lane's A rows (even / odd parity)
                    const bool e_ok = c_e < a.fin_n_mfcc, o_ok = c_o < a.fin_n_mfcc;
                    const double* const drow_e = a.fin_dct + (long long)(e_ok ? c_e : 0) * N + q;
                    const double* const drow_o = a.fin_dct + (long long)(o_ok ? c_o : 0) * N + q;
                    double e0 = 0.0, e1 = 0.0, d0 = 0.0, d1 = 0.0;
                    for (int k0 = 0; k0 < H4; k0 += 4) {
                        const int k = k0 + q;
                        const bool k_ok = k < H;
                        const double av_e = (e_ok && k_ok) ? __ldg(drow_e + k0) : 0.0;
                        const double av_o = (o_ok && k_ok) ? __ldg(drow_o + k0) : 0.0;
                        double bs = 0.0, bd = 0.0;                      // folded: s[k] + s[N-1-k] for even rows, s[k] - s[N-1-k] for odd rows
                        if (k_ok) {
                            const float x = fmaxf(db10(fmaxf(a.fin_amin, xrow[k])) - ref_db, floor_db);
                            bs = bd = (double)x;
                            if (a.fin_dct_fold) {
                                const int k2 = N - 1 - k;
                                if (k2 != k) {
                                    const float x2 = fmaxf(db10(fmaxf(a.fin_amin, xrow[k2])) - ref_db, floor_db);
                                    bs = (double)x + (double)x2;
                                    bd = (double)x - (double)x2;
                                } else {
                                    bd = 0.0;                           // centre of an odd N: once, even rows only
                                }
                            }
                        }
                        mma_m8n8k4_f64(e0, e1, av_e, bs);
                        mma_m8n8k4_f64(d0, d1, av_o, bd);
                    }
                    // lane holds coefficient c of frames nt8 + 2q, nt8 + 2q + 1
                    if (e_ok) {
                        if (t0 < gfr) a.out[o0 + (long long)(a.fin_row_mfcc + c_e) * a.T] = (float)e0;
                        if (t0 + 1 < gfr) a.out[o1 + (long long)(a.fin_row_mfcc + c_e) * a.T] = (float)e1;
                    }
                    if (o_ok) {
                        if (t0 < gfr) a.out[o0 + (long long)(a.fin_row_mfcc + c_o) * a.T] = (float)d0;
                        if (t0 + 1 < gfr) a.out[o1 + (long long)(a.fin_row_mfcc + c_o) * a.T] = (float)d1;
                    }
                }
            }
        }
        __syncthreads();                                                // the tile is refilled by the next group
    }
    }
}

}  // namespace sygdev
