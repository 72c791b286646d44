// sygnals_b200/csrc/syg_api.cu -- the C ABI of libsygb200.so (include/sygb200.h): argument validation, plan
// (constant table) cache, workspace management, chunking and kernel dispatch.  No CPU compute path exists here:
// every entry point either launches the sm_100a kernels of syg_kernels.cuh or fails with an error code.
//
// Reference functions replaced (paths relative to the reference tree):
//   syg_features_*   sygnals/core/features/manager.py:78-445 extract_features() and the per-feature functions
//   syg_stft_*       sygnals/core/dsp.py:167-229 compute_stft()
//   syg_psd_welch_*  sygnals/core/dsp.py:495-560 compute_psd_welch(), :434-493 compute_psd_periodogram()
//   syg_segment_*    sygnals/core/segmentation.py:25-117 segment_fixed_length()
#include "../../include/sygb200.h"

#include <algorithm>
#include <cstdarg>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "syg_launch.h"
#include "syg_plan.h"

// NVTX ranges around every compute entry point (SURVEY.md 5: tracing): visible in nsys / ncu timelines, free when no tool is attached
#ifndef SYG_EMU
#include <nvtx3/nvToolsExt.h>
namespace { struct NvtxRange { explicit NvtxRange(const char* n) { nvtxRangePushA(n); } ~NvtxRange() { nvtxRangePop(); } }; }
#else
namespace { struct NvtxRange { explicit NvtxRange(const char*) {} }; }
#endif
#define SYG_TRACE() NvtxRange nvtx_range_(__func__)

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CK(expr)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (expr);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(e_ == cudaErrorMemoryAllocation ? SYG_E_NOMEM : SYG_E_CUDA, "%s: %s", #expr, \
                        cudaGetErrorString(e_));                                                   \
    } while (0)

// every entry point runs on its context's device and gives the caller's current device back on return
struct DeviceGuard {
    int prev = -1, dev;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int d) : dev(d) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != dev) err = cudaSetDevice(dev);
    }
    ~DeviceGuard() { if (prev >= 0 && prev != dev) cudaSetDevice(prev); }
};
#define ENTER_DEVICE(ctx)                                                                                          \
    DeviceGuard dg_((ctx)->device);                                                                                \
    if (dg_.err != cudaSuccess) return fail(SYG_E_CUDA, "cudaSetDevice(%d): %s", (ctx)->device, cudaGetErrorString(dg_.err))

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return SYG_OK;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = (bytes + 255) / 256 * 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { p = nullptr; return fail(SYG_E_NOMEM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e)); }
        cap = want;
        return SYG_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct PinnedBuf {                 // page-locked host staging owned by a lane (cudaMemcpyAsync from it never stalls the stream)
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return SYG_OK;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        const size_t want = (bytes + 4095) / 4096 * 4096;
        cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
        if (e != cudaSuccess) { p = nullptr; return fail(SYG_E_NOMEM, "cudaHostAlloc(%zu) failed: %s", want, cudaGetErrorString(e)); }
        cap = want;
        return SYG_OK;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

struct Lane {                      // one in-flight chunk of a *_host_* call
    cudaStream_t stream = nullptr;
    DevBuf in, raw, out0, out1, starts, valid, ws, feat;
    PinnedBuf tbl;                 // explicit unit tables of the chunk (starts | valid), reused once tbl_done has passed
    cudaEvent_t tbl_done = nullptr;
    bool tbl_used = false;
};

// what a *_host_* call is handed: float32 mono samples (fmt < 0) or an interleaved PCM payload (SYG_PCM_*, `channels` per frame)
struct InFmt {
    int fmt = -1, channels = 1;
    size_t frame_bytes() const {
        if (fmt < 0) return sizeof(float);
        const size_t bps = fmt == SYG_PCM_U8 ? 1 : (fmt == SYG_PCM_S16 ? 2 : (fmt == SYG_PCM_S24 ? 3 : 4));
        return bps * (size_t)channels;
    }
};

}  // namespace

struct syg_ctx {
    int device = 0;
    int sm_count = 0;
    size_t ws_limit = (size_t)1 << 30;   // 1 GiB: measured best (fewer, fuller launches); 64 MiB chunks keep the workspace in L2 but cost 5 %
    std::mutex mu;
    std::map<std::string, void*> tables;
    std::map<std::string, std::vector<int>> host_ints;
    DevBuf ws;                      // workspace of the device-pointer entry points
    cudaEvent_t ws_done = nullptr;  // recorded after the last kernel that uses `ws`: the next call (any stream) waits on it
    Lane lanes[2];
    // optional per-kernel timing (syg_ctx_profile_*): event pairs around every launch, summed on read
    bool prof_on = false;
    struct ProfPair { cudaEvent_t a, b; int kind; };
    std::vector<ProfPair> prof_pairs;
    double prof_ms[4] = {0, 0, 0, 0};
    long long prof_n[4] = {0, 0, 0, 0};
};

namespace {
enum { PROF_FRAME = 0, PROF_FINALIZE = 1, PROF_WELCH = 2, PROF_OTHER = 3 };   // other = ingest + aggregation
struct ProfScope {
    syg_ctx* c; cudaStream_t st; int kind; cudaEvent_t a = nullptr, b = nullptr;
    ProfScope(syg_ctx* c_, cudaStream_t st_, int kind_) : c(c_), st(st_), kind(kind_) {
        if (c->prof_on && cudaEventCreate(&a) == cudaSuccess && cudaEventCreate(&b) == cudaSuccess) cudaEventRecord(a, st);
        else a = b = nullptr;
    }
    ~ProfScope() {
        if (a && b) { cudaEventRecord(b, st); c->prof_pairs.push_back({a, b, kind}); }
    }
};
}  // namespace

namespace {

bool is_pow2(long long v) { return v > 0 && (v & (v - 1)) == 0; }
int ilog2i(long long v) { int l = 0; while ((1LL << l) < v) ++l; return l; }

// ---------------------------------------------------------------------------------------------- plan tables
template <class T>
int upload_table(syg_ctx* ctx, const std::string& key, const std::vector<T>& host, const T** out) {
    auto it = ctx->tables.find(key);
    if (it != ctx->tables.end()) { *out = reinterpret_cast<const T*>(it->second); return SYG_OK; }
    if (host.empty()) return fail(SYG_E_CUDA, "plan table %s was not built (internal error)", key.c_str());
    void* d = nullptr;
    CK(cudaMalloc(&d, host.size() * sizeof(T)));
    // Pageable-memory cudaMemcpy may return before the DMA has landed and is ordered only against the legacy default stream; the
    // kernels run on the caller's (possibly non-blocking) stream, so wait here: tables are built once per plan.
    cudaError_t e = cudaMemcpy(d, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaStreamSynchronize(cudaStreamLegacy);
    if (e != cudaSuccess) { cudaFree(d); return fail(SYG_E_CUDA, "plan table upload (%s): %s", key.c_str(), cudaGetErrorString(e)); }
    ctx->tables[key] = d;
    *out = reinterpret_cast<const T*>(d);
    return SYG_OK;
}

std::string keyf(const char* fmt, ...) {
    char buf[256];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    return buf;
}

int get_fft_tables(syg_ctx* ctx, int n_fft, const float2** tw, const float2** tws) {
    const int M = n_fft / 2;
    std::string k1 = keyf("tw:%d", n_fft), k2 = keyf("tws:%d", n_fft);
    std::vector<float2> a, b;
    if (!ctx->tables.count(k1)) {                                   // each table under its own key: a failed upload of one cannot poison the other
        a.resize(M);
        for (int k = 0; k < M; ++k) {
            const double ang = -2.0 * sygplan::kPi * (double)k / (double)M;
            a[k] = make_float2((float)std::cos(ang), (float)std::sin(ang));
        }
    }
    if (!ctx->tables.count(k2)) {
        b.resize(M / 2 + 1);
        for (int k = 0; k <= M / 2; ++k) {
            const double ang = -2.0 * sygplan::kPi * (double)k / (double)n_fft;
            b[k] = make_float2((float)std::cos(ang), (float)std::sin(ang));
        }
    }
    int rc = upload_table(ctx, k1, a, tw);
    if (rc) return rc;
    return upload_table(ctx, k2, b, tws);
}

// [n_fft/4 + 1] entries 0.5 exp(-2 pi i k / n_fft): the real split with the halving folded into the twiddle
int get_half_split_twiddles(syg_ctx* ctx, int n_fft, const float2** out) {
    std::string kh = keyf("twsh:%d", n_fft);
    std::vector<float2> h;
    if (!ctx->tables.count(kh)) {
        h.resize(n_fft / 4 + 1);
        for (int k = 0; k <= n_fft / 4; ++k) {
            const double ang = -2.0 * sygplan::kPi * (double)k / (double)n_fft;
            h[k] = make_float2((float)(0.5 * std::cos(ang)), (float)(0.5 * std::sin(ang)));
        }
    }
    return upload_table(ctx, kh, h, out);
}

// ---- transform lengths outside the power-of-two kernels (syg_mixed.cuh): smooth lengths (prime factors <= 13) whose buffers fit
// in one SM's shared memory; powers of two above 8192 take the same route
constexpr size_t kMaxDynSmem = 227 * 1024;
bool native_pow2(long long n) { return is_pow2(n) && n >= 32 && n <= 8192; }

int mixed_plan_of(int n, bool features, syg::MixedPlan& mp, const char* what) {
    std::memset(&mp, 0, sizeof(mp));
    if (n < 8) return fail(SYG_E_UNSUPPORTED, "%s=%d: transform lengths below 8 are not supported", what, n);
    mp.n = n;
    mp.packed = (n % 2 == 0) ? 1 : 0;
    mp.L = mp.packed ? n / 2 : n;
    mp.B = n / 2 + 1;
    std::vector<int> r;
    if (!sygplan::factorize_smooth(mp.L, r) || r.size() > 24)
        return fail(SYG_E_UNSUPPORTED, "%s=%d: only lengths whose prime factors are at most 13 are supported", what, n);
    if (sygdev::mixed_layout(mp.L, mp.B, features).bytes > kMaxDynSmem)
        return fail(SYG_E_UNSUPPORTED, "%s=%d: the transform does not fit in shared memory", what, n);
    mp.npass = (int)r.size();
    for (int i = 0; i < mp.npass; ++i) mp.radix[i] = r[i];
    return SYG_OK;
}

// tw = exp(-2 pi i p / L), p < L, for the mixed-radix passes; tws = real-split twiddles (packed transforms only)
int get_mixed_tables(syg_ctx* ctx, int n, const float2** tw, const float2** tws) {
    if (n % 2 == 0) return get_fft_tables(ctx, n, tw, tws);
    *tws = nullptr;
    std::string k = keyf("twodd:%d", n);
    std::vector<float2> a;
    if (!ctx->tables.count(k)) {
        a.resize(n);
        for (int p = 0; p < n; ++p) {
            const double ang = -2.0 * sygplan::kPi * (double)p / (double)n;
            a[p] = make_float2((float)std::cos(ang), (float)std::sin(ang));
        }
    }
    return upload_table(ctx, k, a, tw);
}

int get_window(syg_ctx* ctx, int window, int win_length, int n_fft, bool centred, const float** out) {
    std::string key = keyf("win:%d:%d:%d:%d", window, win_length, n_fft, (int)centred);
    std::vector<float> w;
    if (!ctx->tables.count(key)) {
        std::string err;
        if (centred) {
            if (!sygplan::build_window(window, win_length, n_fft, w, err)) return fail(SYG_E_BADARG, "%s", err.c_str());
        } else {                                                    // scipy.signal.welch: window then zero padding
            if (window < 0 || window > 3) return fail(SYG_E_UNSUPPORTED, "unsupported window id %d", window);
            w.assign(n_fft, 0.0f);
            for (int n = 0; n < win_length; ++n) w[n] = (float)sygplan::window_value_d(window, win_length, n);
        }
    }
    return upload_table(ctx, key, w, out);
}

// ---------------------------------------------------------------------------------------------- kernel dispatch
// The kernels are instantiated in separate translation units (syg_launch_*.cu, compiled in parallel); they report
// failures as a negative SYG_E_* code plus a message.
int launch_rc(int rc, const std::string& err) { return rc == SYG_OK ? SYG_OK : fail(rc, "%s", err.c_str()); }

int launch_features(int n_fft, const syg::FrameArgs& a_in, int sm_count, cudaStream_t st) {
    std::string err;
    static int variant = -1;
    if (variant < 0) { const char* e = std::getenv("SYGB200_VARIANT"); variant = e ? std::atoi(e) : 0; }
    syg::FrameArgs a = a_in;
    a.variant = variant;
    const bool rag = a.ragged_ut != nullptr;
    const int mode = rag ? sygdev::MODE_FEATURES_RAGGED : sygdev::MODE_FEATURES;
    if (!native_pow2(n_fft)) {
        syg::MixedPlan mp;
        if (int rc = mixed_plan_of(n_fft, true, mp, "frame_length")) return rc;
        return launch_rc(syglaunch::frame_mixed(mode, a, mp, sm_count, st, err), err);
    }
    if (n_fft > 2048) return launch_rc(syglaunch::frame_block(n_fft, mode, a, sm_count, st, err), err);
    if (a.res_units > 0) return launch_rc(syglaunch::frame_warp_res(n_fft, a, sm_count, st, err), err);
    constexpr unsigned extra = syg::FB_BANDWIDTH | syg::FB_FLATNESS | syg::FB_DOMINANT | syg::FB_MEAN_AMP | syg::FB_STD_AMP;
    if (rag) return launch_rc(syglaunch::frame_warp_ragged(n_fft, (a.mask & extra) != 0, a, sm_count, st, err), err);
    return launch_rc(syglaunch::frame_warp(n_fft, (a.mask & extra) != 0, a, sm_count, st, err), err);
}

// frames per warp task of the warp kernel (= WarpTile::FW)
int warp_fw(int n_fft) {
    switch (ilog2i(n_fft / 2)) { case 4: return 8; case 5: return 8; case 6: return 4; case 7: return 4; case 8: return 2; case 9: return 2; default: return 1; }
}

int g_resident_min_groups = -1;     // unit groups a launch needs before the resident kernel is chosen (-1: 4 per SM); tests lower it
int g_last_mel_form = 0;            // 1: the last feature launch with MFCCs used the interval-form mel projection
int g_last_features_resident = 0;   // 1: the last feature launch kept its units on chip (frame_warp_kernel STAGE 5)
long long g_last_feature_frames = 0; // frames the feature kernels processed in the last syg_features_* / syg_segment_vectors_* call
int g_last_stft_path = 0;   // 5 mixed-radix kernel (lengths that are not powers of two), 1 ring (TMA-staged), 2 warp kernel (register-staged), 3 CTA-cooperative kernels, 4 sub-FFT kernel (n_fft 4096 / 8192): last STFT launch

int launch_stft(int n_fft, const syg::FrameArgs& a, int sm_count, cudaStream_t st) {
    std::string err;
    static int env = -1;                                                // SYGB200_STFT_BLOCK=1: the CTA-cooperative kernel for every n_fft
    if (env < 0) { const char* e = std::getenv("SYGB200_STFT_BLOCK"); env = e ? std::atoi(e) : 0; }
    if (!native_pow2(n_fft)) {
        syg::MixedPlan mp;
        if (int rc = mixed_plan_of(n_fft, false, mp, "n_fft")) return rc;
        g_last_stft_path = 5;
        return launch_rc(syglaunch::frame_mixed(sygdev::MODE_STFT, a, mp, sm_count, st, err), err);
    }
    if (n_fft >= 4096 && !env && a.out_kind != 0) {
        g_last_stft_path = 4;
        return launch_rc(syglaunch::stft_big(n_fft, a, sm_count, st, err), err);
    }
    if (n_fft <= 2048 && !env) {
        const int rrc = syglaunch::stft_ring(n_fft, a, sm_count, st, err);      // samples staged by the TMA engine where the layout allows it
        g_last_stft_path = rrc <= 0 ? 1 : 2;
        if (rrc <= 0) return launch_rc(rrc, err);
        return launch_rc(syglaunch::frame_warp_stft(n_fft, a, sm_count, st, err), err);
    }
    g_last_stft_path = 3;
    return launch_rc(syglaunch::frame_block(n_fft, sygdev::MODE_STFT, a, sm_count, st, err), err);
}

int launch_welch(int nfft, const syg::WelchArgs& a, int sm_count, cudaStream_t st) {
    std::string err;
    if (!native_pow2(nfft)) {
        syg::MixedPlan mp;
        if (int rc = mixed_plan_of(nfft, false, mp, "nfft")) return rc;
        return launch_rc(syglaunch::welch_mixed(a, mp, sm_count, st, err), err);
    }
    return launch_rc(syglaunch::welch(nfft, a, sm_count, st, err), err);
}

// ---------------------------------------------------------------------------------------------- validation
int check_units(const syg_units* u) {
    if (!u) return fail(SYG_E_BADARG, "units is NULL");
    if (u->n_units < 0 || u->unit_len < 0 || u->total_len < 0) return fail(SYG_E_BADARG, "negative unit geometry");
    if (!u->unit_starts && u->n_units > 1 && u->unit_stride < 0) return fail(SYG_E_BADARG, "negative unit_stride");
    if (u->unit_len > 0x7fffffffLL) return fail(SYG_E_UNSUPPORTED, "unit_len above 2^31-1 samples");
    return SYG_OK;
}

syg::UnitGeom geom_of(const syg_units* u, long long u0, long long n) {
    syg::UnitGeom g;
    g.n_units = n;
    g.unit_len = u->unit_len;
    g.unit_stride = u->unit_stride;
    g.total_len = u->total_len;
    g.unit_starts = u->unit_starts ? reinterpret_cast<const long long*>(u->unit_starts) + u0 : nullptr;
    g.unit_valid = u->unit_valid ? u->unit_valid + u0 : nullptr;
    g.unit0 = u0;
    return g;
}

struct FeaturePlan {
    syg::FrameArgs fa;             // everything except y, geometry, out, workspaces
    syg::FinalizeArgs fin;
    int n_rows = 0;
    int T = 0;
    size_t ws_per_unit = 0;        // bytes of melws + cws per unit
    int n_fft = 0;
    int entropy_bins = 10;
};

int rows_of(const syg_feature_params* p, int32_t* n_rows) {
    if (!p || !n_rows) return fail(SYG_E_BADARG, "NULL argument");
    if (p->n_features < 0 || p->n_features > SYG_MAX_FEATURES) return fail(SYG_E_BADARG, "n_features out of range");
    int rows = 0;
    unsigned seen = 0;
    for (int i = 0; i < p->n_features; ++i) {
        const int f = p->features[i];
        if (f < 0 || f >= SYG_FEAT_COUNT_) return fail(SYG_E_BADARG, "unknown feature id %d", f);
        if (seen & (1u << f)) return fail(SYG_E_BADARG, "feature id %d requested twice", f);
        seen |= 1u << f;
        if (f == SYG_FEAT_MFCC) {
            if (p->n_mfcc < 1 || p->n_mfcc > 256) return fail(SYG_E_BADARG, "n_mfcc=%d out of range [1, 256]", p->n_mfcc);
            rows += p->n_mfcc;
        } else if (f == SYG_FEAT_SPECTRAL_CONTRAST) {
            if (p->contrast_n_bands < 1 || p->contrast_n_bands > syg::kMaxBands - 1)
                return fail(SYG_E_BADARG, "n_bands=%d out of range [1, %d]", p->contrast_n_bands, syg::kMaxBands - 1);
            rows += p->contrast_n_bands + 1;
        }
        else rows += 1;
    }
    *n_rows = rows;
    return SYG_OK;
}

int build_feature_plan(syg_ctx* ctx, const syg_units* u, const syg_feature_params* p, FeaturePlan& pl) {
    if (!p) return fail(SYG_E_BADARG, "params is NULL");
    if (p->sr <= 0) return fail(SYG_E_BADARG, "sr must be positive");
    const int fl = p->frame_length;
    const bool mixed = !native_pow2(fl);
    if (mixed) {
        syg::MixedPlan mp;
        if (int mrc = mixed_plan_of(fl, true, mp, "frame_length")) return mrc;
    }
    if (p->hop_length < 1) return fail(SYG_E_BADARG, "hop_length must be >= 1");
    int32_t rows = 0;
    int rc = rows_of(p, &rows);
    if (rc) return rc;
    std::memset(&pl.fa, 0, sizeof(pl.fa));
    std::memset(&pl.fin, 0, sizeof(pl.fin));
    syg::FrameArgs& a = pl.fa;
    a.row_centroid = a.row_rolloff = a.row_rms = a.row_crest = a.row_peak = a.row_bandwidth = a.row_flatness =
        a.row_dominant = a.row_zcr = a.row_mean_amp = a.row_std_amp = a.row_skew = a.row_kurt = a.row_entropy = -1;
    pl.fin.row_mfcc = -1;
    pl.fin.row_contrast = -1;
    int row = 0;
    unsigned mask = 0;
    for (int i = 0; i < p->n_features; ++i) {
        switch (p->features[i]) {
            case SYG_FEAT_MFCC: mask |= syg::FB_MFCC; pl.fin.row_mfcc = row; row += p->n_mfcc; break;
            case SYG_FEAT_SPECTRAL_CONTRAST: mask |= syg::FB_CONTRAST; pl.fin.row_contrast = row; row += p->contrast_n_bands + 1; break;
            case SYG_FEAT_SPECTRAL_CENTROID: mask |= syg::FB_CENTROID; a.row_centroid = row++; break;
            case SYG_FEAT_SPECTRAL_ROLLOFF: mask |= syg::FB_ROLLOFF; a.row_rolloff = row++; break;
            case SYG_FEAT_RMS_ENERGY: mask |= syg::FB_RMS; a.row_rms = row++; break;
            case SYG_FEAT_CREST_FACTOR: mask |= syg::FB_CREST; a.row_crest = row++; break;
            case SYG_FEAT_PEAK_AMPLITUDE: mask |= syg::FB_PEAK; a.row_peak = row++; break;
            case SYG_FEAT_SPECTRAL_BANDWIDTH: mask |= syg::FB_BANDWIDTH; a.row_bandwidth = row++; break;
            case SYG_FEAT_SPECTRAL_FLATNESS: mask |= syg::FB_FLATNESS; a.row_flatness = row++; break;
            case SYG_FEAT_DOMINANT_FREQUENCY: mask |= syg::FB_DOMINANT; a.row_dominant = row++; break;
            case SYG_FEAT_MEAN_AMPLITUDE: mask |= syg::FB_MEAN_AMP; a.row_mean_amp = row++; break;
            case SYG_FEAT_STD_DEV_AMPLITUDE: mask |= syg::FB_STD_AMP; a.row_std_amp = row++; break;
            case SYG_FEAT_ZERO_CROSSING_RATE: mask |= syg::FB_ZCR; a.row_zcr = row++; break;
            case SYG_FEAT_SKEWNESS: mask |= syg::FB_SKEW; a.row_skew = row++; break;
            case SYG_FEAT_KURTOSIS: mask |= syg::FB_KURT; a.row_kurt = row++; break;
            case SYG_FEAT_SIGNAL_ENTROPY: mask |= syg::FB_ENTROPY; a.row_entropy = row++; break;
        }
    }
    a.mask = mask;
    a.n_rows = rows;
    pl.n_rows = rows;
    const long long T = syg_frame_count(u->unit_len, fl, p->hop_length, p->center);
    if (T > 0x7fffffffLL) return fail(SYG_E_UNSUPPORTED, "too many frames per unit");
    pl.T = (int)T;
    a.T = (int)T;
    a.hop = p->hop_length;
    a.cpad = p->center ? fl / 2 : 0;
    a.pad_mode = 0;
    a.bin_hz = sygplan::bin_hz((double)p->sr, fl);
    a.roll_percent = p->roll_percent;
    rc = get_window(ctx, p->window, fl, fl, true, &a.window);
    if (rc) return rc;
    rc = mixed ? get_mixed_tables(ctx, fl, &a.tw, &a.tws) : get_fft_tables(ctx, fl, &a.tw, &a.tws);
    if (rc) return rc;
    if (!mixed && (rc = get_half_split_twiddles(ctx, fl, &a.twsh))) return rc;
    size_t ws = 0;
    if (mask & syg::FB_MFCC) {
        if (p->n_mels < 1 || p->n_mels > 256) return fail(SYG_E_UNSUPPORTED, "n_mels=%d: supported range is [1, 256]", p->n_mels);
        if (p->n_mfcc < 1 || p->n_mfcc > p->n_mels) return fail(SYG_E_BADARG, "n_mfcc must be in [1, n_mels]");
        if (!(p->power > 0.0)) return fail(SYG_E_BADARG, "power must be positive");
        const double fmax = p->fmax > 0 ? (double)p->fmax : 0.5 * (double)p->sr;
        std::string key = keyf("mel:%d:%d:%d:%.9g:%.9g", p->sr, fl, p->n_mels, (double)p->fmin, fmax);
        sygplan::MelTable mt;
        if (!ctx->tables.count(key + ":w")) {
            std::string err;
            if (!sygplan::build_mel((double)p->sr, fl, p->n_mels, (double)p->fmin, fmax, false, mt, err))
                return fail(SYG_E_BADARG, "%s", err.c_str());
        }
        if ((rc = upload_table(ctx, key + ":s", mt.start, &a.mel_start))) return rc;
        if ((rc = upload_table(ctx, key + ":l", mt.len, &a.mel_len))) return rc;
        if ((rc = upload_table(ctx, key + ":o", mt.off, &a.mel_off))) return rc;
        if ((rc = upload_table(ctx, key + ":w", mt.w, &a.mel_w))) return rc;
        if (!mixed) {
        sygplan::MelSlots ms;
        if (!ctx->tables.count(key + ":pw")) sygplan::build_mel_slots(mt, ms, fl / 2 + 1, fl <= 2048 ? 32 / warp_fw(fl) : 32);
        std::vector<int4> slots(ms.desc.size() / 4);
        for (size_t i = 0; i < slots.size(); ++i) slots[i] = make_int4(ms.desc[4 * i], ms.desc[4 * i + 1], ms.desc[4 * i + 2], ms.desc[4 * i + 3]);
        if ((rc = upload_table(ctx, key + ":ps", slots, &a.mel_slots))) return rc;
        if ((rc = upload_table(ctx, key + ":pw", ms.w, &a.mel_pw))) return rc;
        {
            std::string kn = key + ":pwn";                       // host side cache: float4 count of the tap table, then the sweep lengths
            if (!ctx->host_ints.count(kn)) {
                const int gs = fl <= 2048 ? 32 / warp_fw(fl) : 32;
                std::vector<int> hv{(int)(ms.w.size() / 4)};
                for (int g0 = 0; g0 < p->n_mels; g0 += gs) hv.push_back(ms.desc[(size_t)g0 * 4 + 2]);
                ctx->host_ints[kn] = hv;
            }
            const std::vector<int>& hv = ctx->host_ints[kn];
            a.mel_pw_f4 = hv[0];
            a.mel_nsweeps = (int)hv.size() - 1 <= 8 ? (int)hv.size() - 1 : 0;
            for (int i = 0; i < a.mel_nsweeps; ++i) a.mel_steps[i] = hv[1 + i];
        }
        a.n_mels = p->n_mels;
        // Interval form of the projection (sygplan::MelIntervals): O(bins) per lane instead of padded tap sweeps.  Default for every
        // warp-kernel transform (n_fft <= 2048); SYGB200_MEL_IV=0 keeps the sweeps, =1 keeps them for n_fft 2048 only (A/B).
        // (Until the plan learnt to carry the Nyquist weight of the last filter it was silently refused for the 44.1 kHz / 2048 / 128
        // bank -- 7.7e-18 of rounding dust in the float table -- and "=2" measured "equal" because it never ran.  It is 10 % of the
        // frame kernel: 5.65 -> 5.10 ms per 2 h.)
        {
            static int iv_env = -1;
            if (iv_env < 0) { const char* e = std::getenv("SYGB200_MEL_IV"); iv_env = e ? std::atoi(e) : 2; }
            // (the frame kernel runs spectral contrast BEFORE the mel stage, so overwriting the spectrum there is safe)
            if (iv_env && fl <= ((iv_env >= 2) ? 2048 : 1024) && fl >= 128 && p->power == 2.0) {
                std::string ki = key + ":iv", kin = key + ":ivn";
                if (!ctx->host_ints.count(kin)) {
                    sygplan::MelTable md;
                    sygplan::MelIntervals iv;
                    std::string err;
                    const int E = fl >= 1024 ? 32 : (fl >= 256 ? 16 : 8);     // = WarpTile::E of the kernel instantiation for this n_fft
                    if (sygplan::build_mel((double)p->sr, fl, p->n_mels, (double)p->fmin, fmax, true, md, err))
                        sygplan::build_mel_intervals((double)p->sr, fl, p->n_mels, (double)p->fmin, fmax, md, E, (fl / 2) / E, iv);
                    if (iv.ok) {
                        const float* d = nullptr;
                        if ((rc = upload_table(ctx, ki, iv.blob, &d))) return rc;
                    }
                    ctx->host_ints[kin] = std::vector<int>{iv.ok ? iv.f4 : 0};
                }
                const int f4 = ctx->host_ints[kin][0];
                if (f4 > 0) {
                    a.mel_iv = 1;
                    a.mel_pw = reinterpret_cast<const float*>(ctx->tables[ki]);
                    a.mel_pw_f4 = f4;
                }
            }
        }
        }                                                            // !mixed: the mixed-radix kernel reads the compact tap table only
        a.n_mels = p->n_mels;
        a.mel_power_is_2 = (p->power == 2.0);
        a.mel_half_power = (float)(0.5 * p->power);
        std::string dk = keyf("dct64:%d:%d:%d:%d:%.9g", p->n_mfcc, p->n_mels, p->dct_type, p->dct_ortho, (double)p->lifter);
        std::vector<double> dct;
        if (!ctx->tables.count(dk)) {
            std::string err;
            if (!sygplan::build_dct(p->n_mfcc, p->n_mels, p->dct_type, p->dct_ortho != 0, (double)p->lifter, p->n_mfcc, dct, err))
                return fail(SYG_E_BADARG, "%s", err.c_str());
        }
        if ((rc = upload_table(ctx, dk, dct, &pl.fin.dct))) return rc;
        pl.fin.n_mels = p->n_mels;
        pl.fin.n_mfcc = p->n_mfcc;
        pl.fin.dct_fold = (p->dct_type == 2) ? 1 : 0;
        ws += (size_t)T * p->n_mels * sizeof(float);
    }
    if (mask & syg::FB_CONTRAST) {
        sygplan::Bands b;
        std::string err;
        if (!sygplan::build_bands((double)p->sr, fl, p->contrast_n_bands, (double)p->contrast_fmin,
                                  (double)p->contrast_quantile, b, err))
            return fail(SYG_E_BADARG, "%s", err.c_str());
        a.nb = b.nb;
        // the kernels rely on 1 <= band_n <= band_cnt for non-empty bands (sortedr[:idx] with idx > rows takes every row)
        for (int i = 0; i < b.nb; ++i) { a.band_lo[i] = b.lo[i]; a.band_cnt[i] = b.cnt[i]; a.band_n[i] = std::max(1, std::min(b.nq[i], std::max(b.cnt[i], 1))); }
        pl.fin.nb = b.nb;
        ws += (size_t)T * 2 * b.nb * sizeof(float);
    }
    pl.n_fft = fl;
    pl.entropy_bins = p->entropy_bins;
    if ((mask & syg::FB_ENTROPY) && (p->entropy_bins < 1 || p->entropy_bins > 16))
        return fail(SYG_E_UNSUPPORTED, "signal_entropy num_bins=%d: supported range is [1, 16]", p->entropy_bins);
    pl.ws_per_unit = ws + 4 * sizeof(unsigned);
    pl.fin.T = (int)T;
    pl.fin.n_rows = rows;
    pl.fin.amin = 1e-10f;
    pl.fin.top_db = 80.0f;
    return SYG_OK;
}

// run the two kernels for units [0, n) of geometry g, writing out rows for those units
int run_features_chunk(syg_ctx* ctx, const FeaturePlan& pl, const float* y, const syg::UnitGeom& g, float* out,
                       void* ws, int n_fft, cudaStream_t st) {
    syg::FrameArgs a = pl.fa;
    a.y = y;
    a.g = g;
    a.n_frames = g.n_units * (long long)pl.T;
    a.out = out;
    char* w = reinterpret_cast<char*>(ws);
    a.unit_max = reinterpret_cast<unsigned*>(w);
    size_t off = ((size_t)g.n_units * 4 * sizeof(unsigned) + 255) / 256 * 256;
    a.melws = reinterpret_cast<float*>(w + off);
    off += ((size_t)a.n_frames * pl.fin.n_mels * sizeof(float) + 255) / 256 * 256;
    a.cws = reinterpret_cast<float*>(w + off);
    // Short units with an MFCC-only epilogue stay on chip (frame_warp_kernel STAGE 5): no mel workspace, no finalize launch.  Needs
    // enough unit groups to fill the GPU; SYGB200_NO_RES=1 keeps the two-kernel path (A/B measurements).
    {
        static int no_res = -1;
        if (no_res < 0) { const char* e = std::getenv("SYGB200_NO_RES"); no_res = e ? std::atoi(e) : 0; }
        constexpr unsigned other = syg::FB_CONTRAST | syg::FB_BANDWIDTH | syg::FB_FLATNESS | syg::FB_DOMINANT | syg::FB_MEAN_AMP | syg::FB_STD_AMP;
        a.res_units = 0;
        if (!no_res && (a.mask & syg::FB_MFCC) && !(a.mask & other) && native_pow2(n_fft) && n_fft <= 1024) {
            const int ku = syglaunch::frame_warp_res_units(n_fft, a);
            const long long min_groups = g_resident_min_groups >= 0 ? g_resident_min_groups : 4LL * ctx->sm_count;
            if (ku > 0 && (g.n_units + ku - 1) / ku >= min_groups) {
                a.res_units = ku;
                a.fin_dct = pl.fin.dct;
                a.fin_n_mfcc = pl.fin.n_mfcc;
                a.fin_row_mfcc = pl.fin.row_mfcc;
                a.fin_dct_fold = pl.fin.dct_fold;
                a.fin_amin = pl.fin.amin;
                a.fin_top_db = pl.fin.top_db;
            }
        }
    }
    g_last_features_resident = a.res_units > 0 ? 1 : 0;
    g_last_feature_frames += a.n_frames;
    if (a.mask & syg::FB_MFCC) g_last_mel_form = a.mel_iv ? 1 : 0;
    const bool need_fin = (a.mask & (syg::FB_MFCC | syg::FB_CONTRAST)) != 0 && a.res_units == 0;
    if (need_fin) CK(cudaMemsetAsync(a.unit_max, 0, (size_t)g.n_units * 4 * sizeof(unsigned), st));
    int rc = SYG_OK;
    if (a.mask & syg::FB_TIME_EXTRA) {                                  // zcr / skewness / kurtosis / entropy: their own streaming kernel
        std::string err;
        ProfScope ps(ctx, st, PROF_FRAME);
        const int trc = syglaunch::time_extra(a, n_fft, pl.entropy_bins, ctx->sm_count, st, err);
        if (trc) return fail(trc, "%s", err.c_str());
    }
    if ((a.mask & ~syg::FB_TIME_EXTRA) == 0) return SYG_OK;             // nothing for the frame kernels
    {
        ProfScope ps(ctx, st, PROF_FRAME);
        rc = launch_features(n_fft, a, ctx->sm_count, st);
    }
    if (rc) return rc;
    if (need_fin) {
        ProfScope ps(ctx, st, PROF_FINALIZE);
        syg::FinalizeArgs f = pl.fin;
        f.n_units = g.n_units;
        f.melws = a.melws;
        f.cws = a.cws;
        f.unit_max = a.unit_max;
        f.out = out;
        static int fin_tt = -1;                                       // SYGB200_FIN_TT=32|64 overrides the tile height (A/B)
        if (fin_tt < 0) { const char* e = std::getenv("SYGB200_FIN_TT"); fin_tt = e ? std::atoi(e) : 0; }
        const int tt = fin_tt == 32 || fin_tt == 64 ? fin_tt : ((f.row_mfcc >= 0 && f.n_mels <= 64) ? 64 : 32);
        const size_t smem = sygdev::fin_smem_bytes(tt, f.n_mels, f.dct_fold != 0);         // folded FP64 S_db rows
        const long long n_tiles = (g.n_units * (long long)pl.T + tt - 1) / tt;
        static int fin_cap = -1;                                      // SYGB200_FIN_CTAS: CTAs per SM of the finalize grid (0 = one CTA per tile)
        if (fin_cap < 0) { const char* e = std::getenv("SYGB200_FIN_CTAS"); fin_cap = e ? std::atoi(e) : 0; }
        const long long cap = fin_cap > 0 ? (long long)ctx->sm_count * fin_cap : 0x7fffffffLL;
        const unsigned grid = (unsigned)std::min<long long>(n_tiles, cap);
        std::string err;
        const int frc = syglaunch::finalize(f, tt, grid, 1u, smem, st, err);
        if (frc) return fail(frc, "%s", err.c_str());
    }
    return SYG_OK;
}

size_t features_ws_bytes(const FeaturePlan& pl, long long n) {
    size_t b = ((size_t)n * 4 * sizeof(unsigned) + 255) / 256 * 256;
    b += ((size_t)n * pl.T * pl.fin.n_mels * sizeof(float) + 255) / 256 * 256;
    b += ((size_t)n * pl.T * 2 * pl.fin.nb * sizeof(float) + 255) / 256 * 256;
    return b + 256;
}

// ---------------------------------------------------------------------------------------------- host pipelines
struct HostChunk {
    long long u0, n;               // units of the chunk
    long long begin, end;          // sample range of y_host covered by the chunk
};

// sample range needed by units [u0, u0 + n)
void chunk_range(const syg_units* u, long long u0, long long n, long long* begin, long long* end) {
    if (!u->unit_starts) {
        long long b = u0 * u->unit_stride;
        long long e = (u0 + n - 1) * u->unit_stride + u->unit_len;
        b = std::min(std::max(b, 0LL), (long long)u->total_len);
        e = std::min(std::max(e, b), (long long)u->total_len);
        *begin = b; *end = e;
        return;
    }
    long long b = u->total_len, e = 0;
    for (long long i = u0; i < u0 + n; ++i) {
        const long long s = u->unit_starts[i];
        long long v = u->unit_valid ? u->unit_valid[i] : u->total_len - s;
        v = std::min<long long>(std::max<long long>(v, 0), u->unit_len);
        if (v > 0) { b = std::min(b, s); e = std::max(e, s + v); }
    }
    if (e < b) { b = 0; e = 0; }
    *begin = b; *end = e;
}

int check_host_units(const syg_units* u) {
    int rc = check_units(u);
    if (rc) return rc;
    if (u->unit_starts) {
        for (long long i = 0; i < u->n_units; ++i) {
            const long long s = u->unit_starts[i];
            long long v = u->unit_valid ? u->unit_valid[i] : u->total_len - s;
            v = std::min<long long>(std::max<long long>(v, 0), u->unit_len);
            if (s < 0 || s + v > u->total_len) return fail(SYG_E_BADARG, "unit %lld lies outside the sample buffer", i);
        }
    }
    return SYG_OK;
}

// Generic chunked host pipeline: H2D of the chunk's samples, `run` on the lane's stream, D2H of up to two outputs.
template <class Run>
int host_pipeline(syg_ctx* ctx, const void* y_host_any, InFmt inf, const syg_units* u, size_t out0_per_unit, void* out0_host,
                  size_t out1_per_unit, void* out1_host, size_t ws_per_unit, long long max_chunk_units, Run run) {
    const unsigned char* y_bytes = reinterpret_cast<const unsigned char*>(y_host_any);
    const size_t fb = inf.frame_bytes();
    if (u->n_units == 0) return SYG_OK;
    const size_t in_target = (size_t)128 << 20, out_target = (size_t)256 << 20;
    long long span = u->unit_starts ? u->unit_len : std::max<long long>(1, std::min(u->unit_stride, u->unit_len));
    long long chunk = std::max<long long>(1, (long long)(in_target / (std::max<long long>(span, 1) * sizeof(float))));
    if (out0_per_unit + out1_per_unit) chunk = std::min<long long>(chunk, std::max<long long>(1, (long long)(out_target / (out0_per_unit + out1_per_unit))));
    if (ws_per_unit) chunk = std::min<long long>(chunk, std::max<long long>(1, (long long)(ctx->ws_limit / ws_per_unit)));
    chunk = std::min(chunk, max_chunk_units);
    if (u->n_units > 1) chunk = std::min<long long>(chunk, (u->n_units + 1) / 2);           // keep both lanes busy
    chunk = std::max<long long>(chunk, 1);
    for (int l = 0; l < 2; ++l) {
        if (!ctx->lanes[l].stream) CK(cudaStreamCreateWithFlags(&ctx->lanes[l].stream, cudaStreamNonBlocking));
        if (!ctx->lanes[l].tbl_done) CK(cudaEventCreateWithFlags(&ctx->lanes[l].tbl_done, cudaEventDisableTiming));
    }
    int li = 0;
    for (long long u0 = 0; u0 < u->n_units; u0 += chunk, li ^= 1) {
        const long long n = std::min(chunk, u->n_units - u0);
        Lane& L = ctx->lanes[li];
        long long b, e;
        chunk_range(u, u0, n, &b, &e);
        int rc;
        if ((rc = L.in.ensure(std::max<size_t>((size_t)(e - b) * sizeof(float), 256)))) return rc;
        if ((rc = L.out0.ensure(std::max<size_t>(out0_per_unit * n, 256)))) return rc;
        if (out1_per_unit && (rc = L.out1.ensure(out1_per_unit * n))) return rc;
        if (ws_per_unit && (rc = L.ws.ensure(ws_per_unit * n + 4096))) return rc;
        // the lane's previous chunk has left its device buffers when this chunk's work reaches them (same stream => ordered)
        if (e > b && inf.fmt < 0) CK(cudaMemcpyAsync(L.in.p, y_bytes + (size_t)b * fb, (size_t)(e - b) * fb, cudaMemcpyHostToDevice, L.stream));
        if (e > b && inf.fmt >= 0) {                                    // PCM payload: fewer PCIe bytes; de-interleaved, averaged and widened on the device
            if ((rc = L.raw.ensure((size_t)(e - b) * fb))) return rc;
            CK(cudaMemcpyAsync(L.raw.p, y_bytes + (size_t)b * fb, (size_t)(e - b) * fb, cudaMemcpyHostToDevice, L.stream));
            std::string err;
            ProfScope ps(ctx, L.stream, PROF_OTHER);
            const int crc = syglaunch::pcm_to_f32(L.raw.p, inf.fmt, inf.channels, e - b, reinterpret_cast<float*>(L.in.p), ctx->sm_count, L.stream, err);
            if (crc) return fail(crc, "%s", err.c_str());
        }
        syg_units cu;
        cu.n_units = n;
        cu.unit_len = u->unit_len;
        cu.unit_starts = nullptr;
        cu.unit_valid = nullptr;
        if (!u->unit_starts) {
            // analytic starts continue inside the chunk: unit i of the chunk starts at (u0+i)*stride - b
            cu.unit_stride = u->unit_stride;
            cu.total_len = e - b;
        } else {
            // the chunk's table goes through the lane's own pinned staging block; it is rewritten only after the copy that read it
            // two chunks ago has completed (an event wait that has practically always passed), so the streams never stall
            const size_t off_valid = ((size_t)n * sizeof(long long) + 15) / 16 * 16;
            if (L.tbl_used) CK(cudaEventSynchronize(L.tbl_done));
            if ((rc = L.tbl.ensure(off_valid + (size_t)n * sizeof(int)))) return rc;
            long long* rel = reinterpret_cast<long long*>(L.tbl.p);
            int* val = reinterpret_cast<int*>(reinterpret_cast<char*>(L.tbl.p) + off_valid);
            for (long long i = 0; i < n; ++i) {
                const long long s = u->unit_starts[u0 + i];
                long long v = u->unit_valid ? u->unit_valid[u0 + i] : u->total_len - s;
                v = std::min<long long>(std::max<long long>(v, 0), u->unit_len);
                rel[i] = v > 0 ? s - b : 0;
                val[i] = (int)v;
            }
            if ((rc = L.starts.ensure(n * sizeof(long long)))) return rc;
            if ((rc = L.valid.ensure(n * sizeof(int)))) return rc;
            CK(cudaMemcpyAsync(L.starts.p, rel, n * sizeof(long long), cudaMemcpyHostToDevice, L.stream));
            CK(cudaMemcpyAsync(L.valid.p, val, n * sizeof(int), cudaMemcpyHostToDevice, L.stream));
            CK(cudaEventRecord(L.tbl_done, L.stream));
            L.tbl_used = true;
            cu.unit_stride = 0;
            cu.total_len = e - b;
            cu.unit_starts = reinterpret_cast<const int64_t*>(L.starts.p);
            cu.unit_valid = reinterpret_cast<const int32_t*>(L.valid.p);
        }
        // analytic chunks: the kernel computes start = (u + unit0) * stride; shift the base pointer instead
        const float* y_dev = reinterpret_cast<const float*>(L.in.p);
        long long shift = 0;
        if (!u->unit_starts) shift = u0 * u->unit_stride - b;        // >= 0: first unit's start relative to the chunk
        rc = run(L, y_dev, cu, shift, u0, n);
        if (rc) return rc;
        CK(cudaMemcpyAsync(reinterpret_cast<char*>(out0_host) + (size_t)u0 * out0_per_unit, L.out0.p, out0_per_unit * n,
                           cudaMemcpyDeviceToHost, L.stream));
        if (out1_per_unit && out1_host)
            CK(cudaMemcpyAsync(reinterpret_cast<char*>(out1_host) + (size_t)u0 * out1_per_unit, L.out1.p, out1_per_unit * n,
                               cudaMemcpyDeviceToHost, L.stream));
    }
    for (int l = 0; l < 2; ++l) CK(cudaStreamSynchronize(ctx->lanes[l].stream));
    return SYG_OK;
}

// geometry of a host chunk on the device: analytic chunks keep (unit0 = 0) and fold the offset into the pointer
syg::UnitGeom chunk_geom(const syg_units& cu, long long shift) {
    syg::UnitGeom g;
    g.n_units = cu.n_units;
    g.unit_len = cu.unit_len;
    g.unit_stride = cu.unit_stride;
    g.total_len = cu.total_len - shift;     // samples available from the (shifted) base
    g.unit_starts = reinterpret_cast<const long long*>(cu.unit_starts);
    g.unit_valid = cu.unit_valid;
    g.unit0 = 0;
    return g;
}

int stft_setup(syg_ctx* ctx, const syg_units* u, int n_fft, int hop, int win_length, int window, int center, int pad_mode,
               int out_kind, syg::FrameArgs& a) {
    const bool mixed = !native_pow2(n_fft);
    if (mixed) {
        syg::MixedPlan mp;
        if (int mrc = mixed_plan_of(n_fft, false, mp, "n_fft")) return mrc;
    }
    if (hop < 1) return fail(SYG_E_BADARG, "hop_length must be >= 1");
    if (win_length < 1 || win_length > n_fft) return fail(SYG_E_BADARG, "win_length must be in [1, n_fft]");
    if (pad_mode != SYG_PAD_CONSTANT && pad_mode != SYG_PAD_REFLECT) return fail(SYG_E_UNSUPPORTED, "unsupported pad_mode %d", pad_mode);
    if (out_kind < 0 || out_kind > 2) return fail(SYG_E_BADARG, "unknown out_kind %d", out_kind);
    if (center && pad_mode == SYG_PAD_REFLECT && u->unit_len <= n_fft / 2 && u->unit_len > 0)
        return fail(SYG_E_SHAPE, "reflect padding needs unit_len > n_fft/2");
    std::memset(&a, 0, sizeof(a));
    const long long T = syg_frame_count(u->unit_len, n_fft, hop, center);
    if (T > 0x7fffffffLL) return fail(SYG_E_UNSUPPORTED, "too many frames per unit");
    a.T = (int)T;
    a.hop = hop;
    a.cpad = center ? n_fft / 2 : 0;
    a.pad_mode = center ? pad_mode : 0;
    a.out_kind = out_kind;
    int rc = get_window(ctx, window, win_length, n_fft, true, &a.window);
    if (rc) return rc;
    if (mixed) return get_mixed_tables(ctx, n_fft, &a.tw, &a.tws);
    if (n_fft >= 4096) {                                                // stft_big_kernel: 1024-point sub-transforms + recombination
        const float2* unused = nullptr;
        if ((rc = get_fft_tables(ctx, 2048, &a.tw1k, &unused))) return rc;
        if ((rc = get_half_split_twiddles(ctx, n_fft, &a.twsh))) return rc;
    }
    return get_fft_tables(ctx, n_fft, &a.tw, &a.tws);
}

struct WelchPlan {
    syg::WelchArgs wa;
    int nfft = 0;
};

int welch_setup(syg_ctx* ctx, const syg_units* u, double fs, int window, int nperseg, int noverlap, int nfft, int detrend,
                int scaling, WelchPlan& pl) {
    if (!(fs > 0)) return fail(SYG_E_BADARG, "fs must be positive");
    if (nperseg < 1) return fail(SYG_E_BADARG, "nperseg must be >= 1");
    if (nfft <= 0) nfft = nperseg;
    if (noverlap < 0) noverlap = nperseg / 2;
    if (noverlap >= nperseg) return fail(SYG_E_BADARG, "noverlap must be less than nperseg.");
    if (nfft < nperseg) return fail(SYG_E_BADARG, "nfft must be greater than or equal to nperseg.");
    const bool mixed = !native_pow2(nfft);
    if (mixed) {
        syg::MixedPlan mp;
        if (int mrc = mixed_plan_of(nfft, false, mp, "nfft")) return mrc;
    }
    if (u->unit_len < nperseg) return fail(SYG_E_SHAPE, "unit_len=%lld shorter than nperseg=%d", (long long)u->unit_len, nperseg);
    if (scaling != SYG_SCALING_DENSITY && scaling != SYG_SCALING_SPECTRUM) return fail(SYG_E_BADARG, "unknown scaling %d", scaling);
    if (window < 0 || window > 3) return fail(SYG_E_UNSUPPORTED, "unsupported window id %d", window);
    std::memset(&pl.wa, 0, sizeof(pl.wa));
    syg::WelchArgs& a = pl.wa;
    pl.nfft = nfft;
    a.nperseg = nperseg;
    a.step = nperseg - noverlap;
    a.nseg = (int)((u->unit_len - noverlap) / a.step);
    a.detrend = detrend ? 1 : 0;
    double s1 = 0.0, s2 = 0.0;
    for (int n = 0; n < nperseg; ++n) { const double w = sygplan::window_value_d(window, nperseg, n); s1 += w; s2 += w * w; }
    a.scale = (float)(scaling == SYG_SCALING_DENSITY ? 1.0 / (fs * s2) : 1.0 / (s1 * s1));
    a.onesided_double = 1;
    int rc = get_window(ctx, window, nperseg, nfft, false, &a.window);
    if (rc) return rc;
    return mixed ? get_mixed_tables(ctx, nfft, &a.tw, &a.tws) : get_fft_tables(ctx, nfft, &a.tw, &a.tws);
}


// ---------------------------------------------------------------------------------------------- ragged batches
// Every unit keeps its own length: unit u is y[starts[u], starts[u] + lengths[u]) with T_u frames, the frame axis is the
// concatenation of the units' frames (frame_off), the feature kernels read a frame's unit, frame index, unit length and start from a
// per-frame table {u, t, len, start} that ragged_frame_table_kernel writes from frame_off and the unit tables.  Chunks are cut by
// cumulative frames and samples, never inside a unit.  A chunk may hold only units without frames: no feature kernel runs for it
// (a launch of zero CTAs is an error), and its segment vectors are the NaN rows of the aggregation.

// validates the tables (host memory) and fills frame_off [n_units + 1]; the plan arguments are checked by build_feature_plan
int check_ragged(const syg_ragged_units* u, int fl, int hop, int center, std::vector<long long>* frame_off) {
    if (!u) return fail(SYG_E_BADARG, "units is NULL");
    if (u->n_units < 0 || u->total_len < 0) return fail(SYG_E_BADARG, "negative unit geometry");
    if (u->n_units > 0 && (!u->starts || !u->lengths)) return fail(SYG_E_BADARG, "unit tables are NULL");
    if (frame_off) frame_off->assign((size_t)u->n_units + 1, 0);
    long long F = 0;
    for (long long i = 0; i < u->n_units; ++i) {
        const long long s = u->starts[i], l = u->lengths[i];
        if (s < 0 || l < 0) return fail(SYG_E_BADARG, "unit %lld: negative start or length", i);
        if (s > u->total_len || l > u->total_len - s) return fail(SYG_E_BADARG, "unit %lld lies outside the sample buffer", i);
        if (l > 0x7fffffffLL) return fail(SYG_E_UNSUPPORTED, "unit %lld: length above 2^31-1 samples", i);
        const long long T = syg_frame_count(l, fl, hop, center);
        if (T > 0x7fffffffLL) return fail(SYG_E_UNSUPPORTED, "unit %lld: more than 2^31-1 frames", i);
        F += T;
        if (frame_off) (*frame_off)[(size_t)i + 1] = F;
    }
    return SYG_OK;
}

size_t al256(size_t b) { return (b + 255) / 256 * 256; }

// device tables of a ragged call, per unit: frame_off (int64, one more entry), starts (int64), lengths (int32), and for the
// aggregation the unit's first frame relative to its chunk (int64) and its frame count (int32)
size_t ragged_tbl_bytes(long long n, bool agg) {
    return al256((size_t)(n + 1) * 8) + al256((size_t)n * 8) + al256((size_t)n * 4) + (agg ? al256((size_t)n * 8) + al256((size_t)n * 4) : 0);
}
struct RaggedTbl { long long* foff; long long* starts; int* valid; long long* seg_off; int* seg_len; };
RaggedTbl ragged_tbl_at(void* base, long long n, bool agg) {
    char* p = reinterpret_cast<char*>(base);
    RaggedTbl t;
    t.foff = reinterpret_cast<long long*>(p); p += al256((size_t)(n + 1) * 8);
    t.starts = reinterpret_cast<long long*>(p); p += al256((size_t)n * 8);
    t.valid = reinterpret_cast<int*>(p); p += al256((size_t)n * 4);
    t.seg_off = agg ? reinterpret_cast<long long*>(p) : nullptr; p += agg ? al256((size_t)n * 8) : 0;
    t.seg_len = agg ? reinterpret_cast<int*>(p) : nullptr;
    return t;
}
// workspace of a chunk of n units and nf frames: unit maxima, mel energies, contrast peaks / valleys, the frame table, and for
// the aggregation the chunk's frame features [n_rows][nf]
size_t ragged_ws_bytes(const FeaturePlan& pl, long long n, long long nf, bool agg) {
    size_t b = al256((size_t)n * 4 * sizeof(unsigned)) + al256((size_t)nf * pl.fin.n_mels * sizeof(float)) +
               al256((size_t)nf * 2 * pl.fin.nb * sizeof(float)) + al256((size_t)nf * sizeof(int4));
    if (agg) b += al256((size_t)nf * pl.n_rows * sizeof(float));
    return b + 256;
}

struct RaggedChunk {
    long long u0, n;               // units
    long long f0, nf;              // frames
    long long b, e;                // samples of y the units cover
};

// host image of the tables of chunk c's units, at entries [at, at + c.n] of t (starts relative to the chunk's first sample, seg_off to
// its first frame)
void ragged_tbl_fill(const RaggedTbl& t, long long at, const syg_ragged_units* u, const std::vector<long long>& foff, const RaggedChunk& c) {
    for (long long i = 0; i <= c.n; ++i) t.foff[at + i] = foff[(size_t)(c.u0 + i)];
    for (long long i = 0; i < c.n; ++i) {
        const long long l = u->lengths[c.u0 + i];
        t.starts[at + i] = l > 0 ? u->starts[c.u0 + i] - c.b : 0;
        t.valid[at + i] = (int)l;
        if (t.seg_off) {
            t.seg_off[at + i] = foff[(size_t)(c.u0 + i)] - c.f0;
            t.seg_len[at + i] = (int)(foff[(size_t)(c.u0 + i + 1)] - foff[(size_t)(c.u0 + i)]);
        }
    }
}

// greedy cut: a chunk takes units while its workspace stays within ws_limit and its samples / frames within the caps; a unit that
// exceeds them alone runs alone
void ragged_chunks(const syg_ragged_units* u, const std::vector<long long>& foff, const FeaturePlan& pl, bool agg, size_t ws_limit,
                   long long max_samples, long long max_frames, std::vector<RaggedChunk>& out) {
    out.clear();
    RaggedChunk c{0, 0, 0, 0, 0, 0};
    long long b = u->total_len, e = 0;
    for (long long i = 0; i < u->n_units; ++i) {
        const long long T = foff[(size_t)i + 1] - foff[(size_t)i];
        const long long s = u->starts[i], l = u->lengths[i];
        const long long nb = l > 0 ? std::min(b, s) : b, ne = l > 0 ? std::max(e, s + l) : e;
        if (c.n > 0 && (ragged_ws_bytes(pl, c.n + 1, c.nf + T, agg) > ws_limit || std::max(ne - nb, 0LL) > max_samples ||
                        c.nf + T > max_frames || c.n + 1 > 0x7fffffffLL)) {
            c.b = e > b ? b : 0; c.e = e > b ? e : 0;
            out.push_back(c);
            c = RaggedChunk{i, 0, foff[(size_t)i], 0, 0, 0};
            b = u->total_len; e = 0;
            if (l > 0) { b = s; e = s + l; }
        } else {
            b = nb; e = ne;
        }
        c.n += 1;
        c.nf += T;
    }
    if (c.n > 0) { c.b = e > b ? b : 0; c.e = e > b ? e : 0; out.push_back(c); }
}

// the feature kernels on one chunk: y and the tables are chunk-relative, rows go to out[r * out_stride + f] (f < nf)
int run_ragged_chunk(syg_ctx* ctx, const FeaturePlan& pl, const float* y, const RaggedTbl& t, long long n, long long nf, float* out,
                     long long out_stride, void* ws, int n_fft, cudaStream_t st) {
    syg::FrameArgs a = pl.fa;
    a.y = y;
    a.g.n_units = n;
    a.g.unit_len = 0x7fffffffLL;           // the kernels take a unit's start and length from the frame table
    a.g.unit_stride = 0;
    a.g.total_len = 0;
    a.g.unit_starts = nullptr;
    a.g.unit_valid = nullptr;
    a.g.unit0 = 0;
    a.T = 0;
    a.n_frames = nf;
    a.out = out;
    a.ragged_stride = out_stride;
    a.res_units = 0;                       // the unit-resident epilogue sizes its tile by units x T: uniform launches only
    char* w = reinterpret_cast<char*>(ws);
    a.unit_max = reinterpret_cast<unsigned*>(w);
    size_t off = al256((size_t)n * 4 * sizeof(unsigned));
    a.melws = reinterpret_cast<float*>(w + off);
    off += al256((size_t)nf * pl.fin.n_mels * sizeof(float));
    a.cws = reinterpret_cast<float*>(w + off);
    off += al256((size_t)nf * 2 * pl.fin.nb * sizeof(float));
    int4* ut = reinterpret_cast<int4*>(w + off);
    a.ragged_ut = ut;
    g_last_features_resident = 0;
    g_last_feature_frames += nf;
    if (a.mask & syg::FB_MFCC) g_last_mel_form = a.mel_iv ? 1 : 0;
    if (nf == 0) return SYG_OK;            // only units without frames: nothing to compute (and no zero-CTA finalize launch)
    std::string err;
    {
        ProfScope ps(ctx, st, PROF_OTHER);
        if (int trc = syglaunch::ragged_frame_table(t.foff, t.starts, t.valid, n, nf, ut, ctx->sm_count, st, err)) return fail(trc, "%s", err.c_str());
    }
    const bool need_fin = (a.mask & (syg::FB_MFCC | syg::FB_CONTRAST)) != 0;
    if (need_fin) CK(cudaMemsetAsync(a.unit_max, 0, (size_t)n * 4 * sizeof(unsigned), st));
    if (a.mask & syg::FB_TIME_EXTRA) {
        ProfScope ps(ctx, st, PROF_FRAME);
        if (int trc = syglaunch::time_extra(a, n_fft, pl.entropy_bins, ctx->sm_count, st, err)) return fail(trc, "%s", err.c_str());
    }
    if ((a.mask & ~syg::FB_TIME_EXTRA) == 0) return SYG_OK;
    {
        ProfScope ps(ctx, st, PROF_FRAME);
        if (int rc = launch_features(n_fft, a, ctx->sm_count, st)) return rc;
    }
    if (!need_fin) return SYG_OK;
    ProfScope ps(ctx, st, PROF_FINALIZE);
    syg::FinalizeArgs f = pl.fin;
    f.n_units = n;
    f.T = 0;
    f.melws = a.melws;
    f.cws = a.cws;
    f.unit_max = a.unit_max;
    f.out = out;
    f.ragged_ut = ut;
    f.n_frames = nf;
    f.ragged_stride = out_stride;
    const int tt = (f.row_mfcc >= 0 && f.n_mels <= 64) ? 64 : 32;     // as run_features_chunk
    const size_t smem = sygdev::fin_smem_bytes(tt, f.n_mels, f.dct_fold != 0);
    const unsigned grid = (unsigned)std::min<long long>((nf + tt - 1) / tt, 0x7fffffffLL);
    if (int frc = syglaunch::finalize(f, tt, grid, 1u, smem, st, err)) return fail(frc, "%s", err.c_str());
    return SYG_OK;
}

int check_agg(const FeaturePlan& pl, const int32_t* agg) {
    if (pl.n_rows > 64) return fail(SYG_E_UNSUPPORTED, "aggregation supports at most 64 rows per call");
    for (int i = 0; i < pl.n_rows; ++i)
        if (agg[i] < SYG_AGG_MEAN || agg[i] > SYG_AGG_MAX) return fail(SYG_E_BADARG, "unknown aggregation id %d", agg[i]);
    return SYG_OK;
}

// agg == nullptr: out is float32 [n_rows][F]; else float64 [n_units][n_rows]
int ragged_dev_impl(syg_ctx* ctx, const float* y_dev, const syg_ragged_units* units, const syg_feature_params* p, const int32_t* agg,
                    void* out_dev, cudaStream_t st) {
    if (!ctx) return fail(SYG_E_BADARG, "ctx is NULL");
    if (!p) return fail(SYG_E_BADARG, "params is NULL");
    std::vector<long long> foff;
    int rc = check_ragged(units, p->frame_length, p->hop_length, p->center, &foff);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ENTER_DEVICE(ctx);
    FeaturePlan pl;
    syg_units pu{};                                   // the plan's per-unit frame count is not used by ragged launches
    if ((rc = build_feature_plan(ctx, &pu, p, pl))) return rc;
    const long long n_units = units->n_units, F = foff.back();
    if (n_units == 0 || F == 0 || pl.n_rows == 0) return SYG_OK;
    if (!y_dev && units->total_len > 0) return fail(SYG_E_BADARG, "y_dev is NULL");
    if (!out_dev) return fail(SYG_E_BADARG, "out_dev is NULL");
    if (agg && (rc = check_agg(pl, agg))) return rc;
    const bool ag = agg != nullptr;
    std::vector<RaggedChunk> chunks;
    ragged_chunks(units, foff, pl, ag, ctx->ws_limit, 0x7fffffffLL, 1LL << 62, chunks);     // starts < 2^31 in the frame table
    size_t ws_max = 0;
    for (const RaggedChunk& c : chunks) ws_max = std::max(ws_max, ragged_ws_bytes(pl, c.n, c.nf, ag));
    const size_t tbl_bytes = ragged_tbl_bytes(n_units, ag);
    // the tables of all units go through lane 0's pinned staging block in one copy; the block is rewritten only after the copy that
    // read it last has completed
    Lane& L = ctx->lanes[0];
    if (!L.tbl_done) CK(cudaEventCreateWithFlags(&L.tbl_done, cudaEventDisableTiming));
    if (L.tbl_used) CK(cudaEventSynchronize(L.tbl_done));
    if ((rc = L.tbl.ensure(tbl_bytes))) return rc;
    const RaggedTbl ht = ragged_tbl_at(L.tbl.p, n_units, ag);
    for (const RaggedChunk& c : chunks) ragged_tbl_fill(ht, c.u0, units, foff, c);
    if (ctx->ws_done) CK(cudaStreamWaitEvent(st, ctx->ws_done, 0));
    else CK(cudaEventCreateWithFlags(&ctx->ws_done, cudaEventDisableTiming));
    if (tbl_bytes + ws_max > ctx->ws.cap) CK(cudaStreamSynchronize(st));   // growing frees the old block: nothing may still use it
    if ((rc = ctx->ws.ensure(tbl_bytes + ws_max))) return rc;
    struct Done { syg_ctx* c; cudaStream_t s; ~Done() { cudaEventRecord(c->ws_done, s); } } done_{ctx, st};
    CK(cudaMemcpyAsync(ctx->ws.p, L.tbl.p, tbl_bytes, cudaMemcpyHostToDevice, st));
    CK(cudaEventRecord(L.tbl_done, st));
    L.tbl_used = true;
    const RaggedTbl dt = ragged_tbl_at(ctx->ws.p, n_units, ag);
    void* ws = reinterpret_cast<char*>(ctx->ws.p) + tbl_bytes;
    for (const RaggedChunk& c : chunks) {
        RaggedTbl ct{dt.foff + c.u0, dt.starts + c.u0, dt.valid + c.u0, ag ? dt.seg_off + c.u0 : nullptr, ag ? dt.seg_len + c.u0 : nullptr};
        float* feat = ag ? reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + ragged_ws_bytes(pl, c.n, c.nf, true) - 256 -
                                                    al256((size_t)c.nf * pl.n_rows * sizeof(float)))
                         : reinterpret_cast<float*>(out_dev) + c.f0;
        if ((rc = run_ragged_chunk(ctx, pl, y_dev + c.b, ct, c.n, c.nf, feat, ag ? c.nf : F, ws, p->frame_length, st))) return rc;
        if (!ag) continue;
        std::string err;
        ProfScope ps(ctx, st, PROF_OTHER);
        const int arc = syglaunch::aggregate(feat, c.n, pl.n_rows, c.nf, ct.seg_off, ct.seg_len, 0, agg,
                                             reinterpret_cast<double*>(out_dev) + (size_t)c.u0 * pl.n_rows, ctx->sm_count, st, err);
        if (arc) return fail(arc, "%s", err.c_str());
    }
    return SYG_OK;
}

// host forms: chunks alternate between the two lanes (H2D of the chunk's samples and tables, kernels, D2H overlapped)
int ragged_host_impl(syg_ctx* ctx, const float* y_host, const syg_ragged_units* units, const syg_feature_params* p, const int32_t* agg,
                     void* out_host) {
    if (!ctx) return fail(SYG_E_BADARG, "ctx is NULL");
    if (!p) return fail(SYG_E_BADARG, "params is NULL");
    std::vector<long long> foff;
    int rc = check_ragged(units, p->frame_length, p->hop_length, p->center, &foff);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ENTER_DEVICE(ctx);
    FeaturePlan pl;
    syg_units pu{};
    if ((rc = build_feature_plan(ctx, &pu, p, pl))) return rc;
    const long long n_units = units->n_units, F = foff.back();
    if (n_units == 0 || F == 0 || pl.n_rows == 0) return SYG_OK;
    if (!y_host && units->total_len > 0) return fail(SYG_E_BADARG, "y_host is NULL");
    if (!out_host) return fail(SYG_E_BADARG, "out_host is NULL");
    if (agg && (rc = check_agg(pl, agg))) return rc;
    const bool ag = agg != nullptr;
    // 128 MiB of samples and 256 MiB of frame features per chunk (host_pipeline's targets); at least two chunks keep both lanes busy
    long long max_frames = std::max<long long>(1, (long long)(((size_t)256 << 20) / ((size_t)pl.n_rows * sizeof(float))));
    if (n_units > 1) max_frames = std::min<long long>(max_frames, std::max<long long>(1, (F + 1) / 2));
    std::vector<RaggedChunk> chunks;
    ragged_chunks(units, foff, pl, ag, ctx->ws_limit, (long long)(((size_t)128 << 20) / sizeof(float)), max_frames, chunks);
    for (int l = 0; l < 2; ++l) {
        if (!ctx->lanes[l].stream) CK(cudaStreamCreateWithFlags(&ctx->lanes[l].stream, cudaStreamNonBlocking));
        if (!ctx->lanes[l].tbl_done) CK(cudaEventCreateWithFlags(&ctx->lanes[l].tbl_done, cudaEventDisableTiming));
    }
    int li = 0;
    for (const RaggedChunk& c : chunks) {
        Lane& L = ctx->lanes[li];
        li ^= 1;
        const size_t tbl_bytes = ragged_tbl_bytes(c.n, ag);
        const size_t out_bytes = ag ? (size_t)c.n * pl.n_rows * sizeof(double) : (size_t)c.nf * pl.n_rows * sizeof(float);
        if ((rc = L.in.ensure(std::max<size_t>((size_t)(c.e - c.b) * sizeof(float), 256)))) return rc;
        if ((rc = L.out0.ensure(std::max<size_t>(out_bytes, 256)))) return rc;
        if ((rc = L.ws.ensure(tbl_bytes + ragged_ws_bytes(pl, c.n, c.nf, ag)))) return rc;
        // the lane's previous chunk has left its device buffers when this chunk's work reaches them (same stream => ordered)
        if (c.e > c.b) CK(cudaMemcpyAsync(L.in.p, y_host + c.b, (size_t)(c.e - c.b) * sizeof(float), cudaMemcpyHostToDevice, L.stream));
        if (L.tbl_used) CK(cudaEventSynchronize(L.tbl_done));
        if ((rc = L.tbl.ensure(tbl_bytes))) return rc;
        ragged_tbl_fill(ragged_tbl_at(L.tbl.p, c.n, ag), 0, units, foff, c);
        CK(cudaMemcpyAsync(L.ws.p, L.tbl.p, tbl_bytes, cudaMemcpyHostToDevice, L.stream));
        CK(cudaEventRecord(L.tbl_done, L.stream));
        L.tbl_used = true;
        const RaggedTbl ct = ragged_tbl_at(L.ws.p, c.n, ag);
        void* ws = reinterpret_cast<char*>(L.ws.p) + tbl_bytes;
        float* feat = ag ? reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + ragged_ws_bytes(pl, c.n, c.nf, true) - 256 -
                                                    al256((size_t)c.nf * pl.n_rows * sizeof(float)))
                         : reinterpret_cast<float*>(L.out0.p);
        if ((rc = run_ragged_chunk(ctx, pl, reinterpret_cast<const float*>(L.in.p), ct, c.n, c.nf, feat, c.nf, ws, p->frame_length,
                                   L.stream)))
            return rc;
        if (ag) {
            std::string err;
            ProfScope ps(ctx, L.stream, PROF_OTHER);
            const int arc = syglaunch::aggregate(feat, c.n, pl.n_rows, c.nf, ct.seg_off, ct.seg_len, 0, agg,
                                                 reinterpret_cast<double*>(L.out0.p), ctx->sm_count, L.stream, err);
            if (arc) return fail(arc, "%s", err.c_str());
            CK(cudaMemcpyAsync(reinterpret_cast<double*>(out_host) + (size_t)c.u0 * pl.n_rows, L.out0.p, out_bytes, cudaMemcpyDeviceToHost,
                               L.stream));
        } else {
            for (int r = 0; r < pl.n_rows; ++r)          // row r of the chunk lands at columns [f0, f0 + nf) of output row r
                CK(cudaMemcpyAsync(reinterpret_cast<float*>(out_host) + (size_t)r * F + c.f0, reinterpret_cast<float*>(L.out0.p) + (size_t)r * c.nf,
                                   (size_t)c.nf * sizeof(float), cudaMemcpyDeviceToHost, L.stream));
        }
    }
    for (int l = 0; l < 2; ++l) CK(cudaStreamSynchronize(ctx->lanes[l].stream));
    return SYG_OK;
}

}  // namespace

// ================================================================================================ C ABI
extern "C" {

const char* syg_version(void) {
#ifdef SYG_EMU
    return "sygb200 0.1.0 (emulator test build)";
#else
    return "sygb200 0.1.0 (sm_100a)";
#endif
}

const char* syg_last_error(void) { return g_err.c_str(); }

int syg_ctx_create(int device, syg_ctx** out) {
    if (!out) return fail(SYG_E_BADARG, "out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0)
        return fail(SYG_E_CUDA, "no CUDA device available (%s); sygb200 has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    if (device < 0 || device >= n) return fail(SYG_E_BADARG, "device %d out of range (0..%d)", device, n - 1);
    DeviceGuard dg_(device);
    if (dg_.err != cudaSuccess) return fail(SYG_E_CUDA, "cudaSetDevice(%d): %s", device, cudaGetErrorString(dg_.err));
    syg_ctx* c = new syg_ctx();
    c->device = device;
    e = cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (e != cudaSuccess || c->sm_count <= 0) { delete c; return fail(SYG_E_CUDA, "cannot query SM count"); }
    *out = c;
    return SYG_OK;
}

void syg_ctx_destroy(syg_ctx* ctx) {
    if (!ctx) return;
    DeviceGuard dg_(ctx->device);
    cudaDeviceSynchronize();
    for (auto& kv : ctx->tables) cudaFree(kv.second);
    ctx->ws.release();
    if (ctx->ws_done) cudaEventDestroy(ctx->ws_done);
    for (auto& l : ctx->lanes) {
        l.in.release(); l.raw.release(); l.out0.release(); l.out1.release(); l.starts.release(); l.valid.release(); l.ws.release(); l.feat.release();
        l.tbl.release();
        if (l.tbl_done) cudaEventDestroy(l.tbl_done);
        if (l.stream) cudaStreamDestroy(l.stream);
    }
    delete ctx;
}

int syg_ctx_set_workspace_limit(syg_ctx* ctx, size_t bytes) {
    if (!ctx) return fail(SYG_E_BADARG, "ctx is NULL");
    if (bytes < ((size_t)1 << 20)) return fail(SYG_E_BADARG, "workspace limit below 1 MiB");
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->ws_limit = bytes;
    return SYG_OK;
}

int syg_ctx_sm_count(const syg_ctx* ctx) { return ctx ? ctx->sm_count : 0; }

int syg_ctx_profile_enable(syg_ctx* ctx, int on) {
    if (!ctx) return fail(SYG_E_BADARG, "ctx is NULL");
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->prof_on = on != 0;
    return SYG_OK;
}

int syg_ctx_profile_read(syg_ctx* ctx, double* ms, int64_t* launches, int reset) {
    if (!ctx) return fail(SYG_E_BADARG, "ctx is NULL");
    std::lock_guard<std::mutex> lk(ctx->mu);
    ENTER_DEVICE(ctx);
    for (auto& pp : ctx->prof_pairs) {
        float t = 0.0f;
        CK(cudaEventSynchronize(pp.b));
        CK(cudaEventElapsedTime(&t, pp.a, pp.b));
        ctx->prof_ms[pp.kind] += (double)t;
        ctx->prof_n[pp.kind] += 1;
        cudaEventDestroy(pp.a);
        cudaEventDestroy(pp.b);
    }
    ctx->prof_pairs.clear();
    for (int i = 0; i < 4; ++i) {
        if (ms) ms[i] = ctx->prof_ms[i];
        if (launches) launches[i] = ctx->prof_n[i];
        if (reset) { ctx->prof_ms[i] = 0; ctx->prof_n[i] = 0; }
    }
    return SYG_OK;
}

void syg_feature_params_default(syg_feature_params* p) {
    if (!p) return;
    std::memset(p, 0, sizeof(*p));
    p->sr = 22050;
    p->frame_length = 2048;       // manager.py:82
    p->hop_length = 512;          // manager.py:83
    p->center = 1;
    p->window = SYG_WINDOW_HANN;
    p->n_mels = 128;              // manager.py:214
    p->fmin = 0.0;
    p->fmax = 0.0;
    p->power = 2.0;
    p->n_mfcc = 13;               // cepstral.py:24
    p->dct_type = 2;
    p->dct_ortho = 1;
    p->lifter = 0.0;
    p->contrast_n_bands = 6;      // frequency_domain.py:150
    p->contrast_fmin = 200.0;
    p->contrast_quantile = 0.02;
    p->roll_percent = 0.85;      // frequency_domain.py:277
    p->entropy_bins = 10;         // time_domain.py:186
}

int syg_features_rows(const syg_feature_params* p, int32_t* n_rows) { return rows_of(p, n_rows); }

int64_t syg_frame_count(int64_t n_samples, int32_t frame_length, int32_t hop_length, int32_t center) {
    if (hop_length < 1 || frame_length < 1 || n_samples < 0) return 0;
    int64_t n = n_samples;
    if (center) n += 2 * (int64_t)(frame_length / 2);
    if (n < frame_length) return 0;
    return 1 + (n - frame_length) / hop_length;
}

int syg_features_f32(syg_ctx* ctx, const float* y_dev, const syg_units* units, const syg_feature_params* p,
                     float* out_dev, void* stream) {
    SYG_TRACE();
    g_last_feature_frames = 0;
    if (!ctx) return fail(SYG_E_BADARG, "ctx is NULL");
    int rc = check_units(units);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ENTER_DEVICE(ctx);
    FeaturePlan pl;
    if ((rc = build_feature_plan(ctx, units, p, pl))) return rc;
    if (units->n_units == 0 || pl.T <= 0 || pl.n_rows == 0) return SYG_OK;
    if (!y_dev && units->total_len > 0) return fail(SYG_E_BADARG, "y_dev is NULL");
    if (!out_dev) return fail(SYG_E_BADARG, "out_dev is NULL");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    long long chunk = std::max<long long>(1, (long long)(ctx->ws_limit / std::max<size_t>(pl.ws_per_unit, 1)));
    chunk = std::min<long long>(chunk, units->n_units);
    // the workspace is shared by every call on this context: order this call's kernels behind the previous user's, whatever
    // stream that was (calls on ONE stream are ordered anyway; two streams would otherwise overwrite each other's mel energies)
    if (ctx->ws_done) CK(cudaStreamWaitEvent(st, ctx->ws_done, 0));
    else CK(cudaEventCreateWithFlags(&ctx->ws_done, cudaEventDisableTiming));
    if (features_ws_bytes(pl, chunk) > ctx->ws.cap) CK(cudaStreamSynchronize(st));   // growing frees the old block: nothing may still use it
    if ((rc = ctx->ws.ensure(features_ws_bytes(pl, chunk)))) return rc;
    struct Done { syg_ctx* c; cudaStream_t s; ~Done() { cudaEventRecord(c->ws_done, s); } } done_{ctx, st};
    for (long long u0 = 0; u0 < units->n_units; u0 += chunk) {
        const long long n = std::min(chunk, units->n_units - u0);
        syg::UnitGeom g = geom_of(units, u0, n);
        rc = run_features_chunk(ctx, pl, y_dev, g, out_dev + (size_t)u0 * pl.n_rows * pl.T, ctx->ws.p, p->frame_length, st);
        if (rc) return rc;
    }
    return SYG_OK;
}

// agg == nullptr: out_host is float32 [n_units][n_rows][T];  else: float64 [n_units][n_rows] (per-row SYG_AGG_* over the frames)
static int features_host_impl(syg_ctx* ctx, const void* y_host, InFmt inf, const syg_units* units, const syg_feature_params* p,
                              const int32_t* agg, void* out_host) {
    NvtxRange nvtx_range_(agg ? "syg_segment_vectors_host" : "syg_features_host");
    g_last_feature_frames = 0;
    if (!ctx) return fail(SYG_E_BADARG, "ctx is NULL");
    if (inf.fmt >= 0 && (inf.fmt > SYG_PCM_F32 || inf.channels < 1 || inf.channels > 64))
        return fail(SYG_E_BADARG, "bad PCM layout (format %d, %d channels)", inf.fmt, inf.channels);
    int rc = check_host_units(units);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ENTER_DEVICE(ctx);
    FeaturePlan pl;
    if ((rc = build_feature_plan(ctx, units, p, pl))) return rc;
    if (units->n_units == 0 || pl.T <= 0 || pl.n_rows == 0) return SYG_OK;
    if (!y_host && units->total_len > 0) return fail(SYG_E_BADARG, "y_host is NULL");
    if (!out_host) return fail(SYG_E_BADARG, "out_host is NULL");
    if (agg) {
        if (pl.n_rows > 64) return fail(SYG_E_UNSUPPORTED, "aggregation supports at most 64 rows per call");
        for (int i = 0; i < pl.n_rows; ++i)
            if (agg[i] < SYG_AGG_MEAN || agg[i] > SYG_AGG_MAX) return fail(SYG_E_BADARG, "unknown aggregation id %d", agg[i]);
    }
    const size_t feat_per_unit = (size_t)pl.n_rows * pl.T * sizeof(float);
    const size_t out_per_unit = agg ? (size_t)pl.n_rows * sizeof(double) : feat_per_unit;
    const int n_fft = p->frame_length;
    // aggregated calls keep the [n, rows, T] block on the device: bound the chunk by it (it replaces the D2H-sized output buffer)
    const long long max_chunk = agg ? std::max<long long>(1, (long long)(((size_t)256 << 20) / feat_per_unit)) : (1LL << 40);
    return host_pipeline(ctx, y_host, inf, units, out_per_unit, out_host, 0, nullptr, features_ws_bytes(pl, 1), max_chunk,
                         [&](Lane& L, const float* y_dev, const syg_units& cu, long long shift, long long, long long n) -> int {
                             int r = L.ws.ensure(features_ws_bytes(pl, n));
                             if (r) return r;
                             float* feat = reinterpret_cast<float*>(L.out0.p);
                             if (agg) {
                                 if ((r = L.feat.ensure(feat_per_unit * n))) return r;
                                 feat = reinterpret_cast<float*>(L.feat.p);
                             }
                             syg::UnitGeom g = chunk_geom(cu, shift);
                             r = run_features_chunk(ctx, pl, y_dev + shift, g, feat, L.ws.p, n_fft, L.stream);
                             if (r || !agg) return r;
                             std::string err;
                             ProfScope ps(ctx, L.stream, PROF_OTHER);
                             const int arc = syglaunch::aggregate(feat, n, pl.n_rows, pl.T, nullptr, nullptr, pl.T, agg,
                                                                  reinterpret_cast<double*>(L.out0.p), ctx->sm_count, L.stream, err);
                             return arc ? fail(arc, "%s", err.c_str()) : SYG_OK;
                         });
}

int syg_features_host_f32(syg_ctx* ctx, const float* y_host, const syg_units* units, const syg_feature_params* p,
                          float* out_host) {
    return features_host_impl(ctx, y_host, InFmt{}, units, p, nullptr, out_host);
}

int syg_features_host_pcm16(syg_ctx* ctx, const int16_t* y_host, const syg_units* units, const syg_feature_params* p,
                            float* out_host) {
    return features_host_impl(ctx, y_host, InFmt{SYG_PCM_S16, 1}, units, p, nullptr, out_host);
}

int syg_features_host_pcm(syg_ctx* ctx, const void* raw_host, int32_t sample_format, int32_t channels, const syg_units* units,
                          const syg_feature_params* p, float* out_host) {
    return features_host_impl(ctx, raw_host, InFmt{sample_format, channels}, units, p, nullptr, out_host);
}

int syg_segment_vectors_host_f32(syg_ctx* ctx, const float* y_host, const syg_units* units, const syg_feature_params* p,
                                 const int32_t* agg, double* out_host) {
    if (!agg) return fail(SYG_E_BADARG, "agg is NULL");
    return features_host_impl(ctx, y_host, InFmt{}, units, p, agg, out_host);
}

int syg_segment_vectors_host_pcm(syg_ctx* ctx, const void* raw_host, int32_t sample_format, int32_t channels,
                                 const syg_units* units, const syg_feature_params* p, const int32_t* agg, double* out_host) {
    if (!agg) return fail(SYG_E_BADARG, "agg is NULL");
    return features_host_impl(ctx, raw_host, InFmt{sample_format, channels}, units, p, agg, out_host);
}

int syg_segment_vectors_f32(syg_ctx* ctx, const float* y_dev, const syg_units* units, const syg_feature_params* p,
                            const int32_t* agg, double* out_dev, void* stream) {
    SYG_TRACE();
    g_last_feature_frames = 0;
    if (!ctx) return fail(SYG_E_BADARG, "ctx is NULL");
    if (!agg) return fail(SYG_E_BADARG, "agg is NULL");
    int rc = check_units(units);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ENTER_DEVICE(ctx);
    FeaturePlan pl;
    if ((rc = build_feature_plan(ctx, units, p, pl))) return rc;
    if (units->n_units == 0 || pl.T <= 0 || pl.n_rows == 0) return SYG_OK;
    if (!y_dev && units->total_len > 0) return fail(SYG_E_BADARG, "y_dev is NULL");
    if (!out_dev) return fail(SYG_E_BADARG, "out_dev is NULL");
    if (pl.n_rows > 64) return fail(SYG_E_UNSUPPORTED, "aggregation supports at most 64 rows per call");
    for (int i = 0; i < pl.n_rows; ++i)
        if (agg[i] < SYG_AGG_MEAN || agg[i] > SYG_AGG_MAX) return fail(SYG_E_BADARG, "unknown aggregation id %d", agg[i]);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    // the frame features of a chunk live in a library-owned block behind the workspace: [chunk][rows][T] never reaches the caller
    const size_t feat_per_unit = (size_t)pl.n_rows * pl.T * sizeof(float);
    long long chunk = std::max<long long>(1, (long long)(ctx->ws_limit / std::max<size_t>(pl.ws_per_unit + feat_per_unit, 1)));
    chunk = std::min<long long>(chunk, units->n_units);
    const size_t ws_bytes = (features_ws_bytes(pl, chunk) + 255) / 256 * 256;
    if (ctx->ws_done) CK(cudaStreamWaitEvent(st, ctx->ws_done, 0));
    else CK(cudaEventCreateWithFlags(&ctx->ws_done, cudaEventDisableTiming));
    if (ws_bytes + feat_per_unit * chunk > ctx->ws.cap) CK(cudaStreamSynchronize(st));
    if ((rc = ctx->ws.ensure(ws_bytes + feat_per_unit * chunk))) return rc;
    struct Done { syg_ctx* c; cudaStream_t s; ~Done() { cudaEventRecord(c->ws_done, s); } } done_{ctx, st};
    float* feat = reinterpret_cast<float*>(reinterpret_cast<char*>(ctx->ws.p) + ws_bytes);
    for (long long u0 = 0; u0 < units->n_units; u0 += chunk) {
        const long long n = std::min(chunk, units->n_units - u0);
        syg::UnitGeom g = geom_of(units, u0, n);
        if ((rc = run_features_chunk(ctx, pl, y_dev, g, feat, ctx->ws.p, p->frame_length, st))) return rc;
        std::string err;
        ProfScope ps(ctx, st, PROF_OTHER);
        const int arc = syglaunch::aggregate(feat, n, pl.n_rows, pl.T, nullptr, nullptr, pl.T, agg, out_dev + (size_t)u0 * pl.n_rows,
                                             ctx->sm_count, st, err);
        if (arc) return fail(arc, "%s", err.c_str());
    }
    return SYG_OK;
}

int64_t syg_ragged_frame_offsets(const syg_ragged_units* units, int32_t frame_length, int32_t hop_length, int32_t center,
                                 int64_t* frame_off) {
    if (frame_length < 1 || hop_length < 1) return fail(SYG_E_BADARG, "frame_length and hop_length must be >= 1");
    std::vector<long long> foff;
    const int rc = check_ragged(units, frame_length, hop_length, center, &foff);
    if (rc) return rc;
    if (frame_off) for (size_t i = 0; i < foff.size(); ++i) frame_off[i] = foff[i];
    return foff.back();
}

int syg_features_ragged_f32(syg_ctx* ctx, const float* y_dev, const syg_ragged_units* units, const syg_feature_params* p,
                            float* out_dev, void* stream) {
    SYG_TRACE();
    g_last_feature_frames = 0;
    return ragged_dev_impl(ctx, y_dev, units, p, nullptr, out_dev, reinterpret_cast<cudaStream_t>(stream));
}

int syg_features_ragged_host_f32(syg_ctx* ctx, const float* y_host, const syg_ragged_units* units, const syg_feature_params* p,
                                 float* out_host) {
    SYG_TRACE();
    g_last_feature_frames = 0;
    return ragged_host_impl(ctx, y_host, units, p, nullptr, out_host);
}

int syg_segment_vectors_ragged_f32(syg_ctx* ctx, const float* y_dev, const syg_ragged_units* units, const syg_feature_params* p,
                                   const int32_t* agg, double* out_dev, void* stream) {
    SYG_TRACE();
    g_last_feature_frames = 0;
    if (!agg) return fail(SYG_E_BADARG, "agg is NULL");
    return ragged_dev_impl(ctx, y_dev, units, p, agg, out_dev, reinterpret_cast<cudaStream_t>(stream));
}

int syg_segment_vectors_ragged_host_f32(syg_ctx* ctx, const float* y_host, const syg_ragged_units* units,
                                        const syg_feature_params* p, const int32_t* agg, double* out_host) {
    SYG_TRACE();
    g_last_feature_frames = 0;
    if (!agg) return fail(SYG_E_BADARG, "agg is NULL");
    return ragged_host_impl(ctx, y_host, units, p, agg, out_host);
}

int syg_ingest_pcm(syg_ctx* ctx, const void* raw_dev, int32_t sample_format, int32_t channels, int64_t n_frames, float* mono_dev,
                   void* stream) {
    SYG_TRACE();
    if (!ctx) return fail(SYG_E_BADARG, "ctx is NULL");
    if (n_frames < 0 || (n_frames > 0 && (!raw_dev || !mono_dev))) return fail(SYG_E_BADARG, "bad PCM buffer");
    if (sample_format < SYG_PCM_U8 || sample_format > SYG_PCM_F32) return fail(SYG_E_BADARG, "unknown PCM sample format %d", sample_format);
    ENTER_DEVICE(ctx);
    std::string err;
    const int rc = syglaunch::pcm_to_f32(raw_dev, sample_format, channels, n_frames, mono_dev, ctx->sm_count,
                                         reinterpret_cast<cudaStream_t>(stream), err);
    return rc ? fail(rc, "%s", err.c_str()) : SYG_OK;
}

int syg_pcm16_to_f32(syg_ctx* ctx, const int16_t* in_dev, float* out_dev, int64_t n, void* stream) {
    SYG_TRACE();
    if (!ctx) return fail(SYG_E_BADARG, "ctx is NULL");
    if (n < 0 || (n > 0 && (!in_dev || !out_dev))) return fail(SYG_E_BADARG, "bad pcm16 buffer");
    ENTER_DEVICE(ctx);
    std::string err;
    const int rc = syglaunch::pcm16_to_f32(reinterpret_cast<const short*>(in_dev), out_dev, n, ctx->sm_count,
                                           reinterpret_cast<cudaStream_t>(stream), err);
    return rc ? fail(rc, "%s", err.c_str()) : SYG_OK;
}

static size_t stft_elem_bytes(int out_kind) { return out_kind == SYG_OUT_COMPLEX ? 2 * sizeof(float) : sizeof(float); }

int syg_stft_f32(syg_ctx* ctx, const float* y_dev, const syg_units* units, int32_t n_fft, int32_t hop_length,
                 int32_t win_length, int32_t window, int32_t center, int32_t pad_mode, int32_t out_kind,
                 void* out_dev, void* stream) {
    SYG_TRACE();
    if (!ctx) return fail(SYG_E_BADARG, "ctx is NULL");
    int rc = check_units(units);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ENTER_DEVICE(ctx);
    syg::FrameArgs a;
    if ((rc = stft_setup(ctx, units, n_fft, hop_length, win_length, window, center, pad_mode, out_kind, a))) return rc;
    if (units->n_units == 0 || a.T <= 0) return SYG_OK;
    if (!y_dev && units->total_len > 0) return fail(SYG_E_BADARG, "y_dev is NULL");
    if (!out_dev) return fail(SYG_E_BADARG, "out_dev is NULL");
    a.y = y_dev;
    a.g = geom_of(units, 0, units->n_units);
    a.n_frames = units->n_units * (long long)a.T;
    a.stft_out = out_dev;
    ProfScope ps(ctx, reinterpret_cast<cudaStream_t>(stream), PROF_FRAME);
    return launch_stft(n_fft, a, ctx->sm_count, reinterpret_cast<cudaStream_t>(stream));
}

int syg_stft_host_f32(syg_ctx* ctx, const float* y_host, const syg_units* units, int32_t n_fft, int32_t hop_length,
                      int32_t win_length, int32_t window, int32_t center, int32_t pad_mode, int32_t out_kind,
                      void* out_host) {
    SYG_TRACE();
    if (!ctx) return fail(SYG_E_BADARG, "ctx is NULL");
    int rc = check_host_units(units);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ENTER_DEVICE(ctx);
    syg::FrameArgs a;
    if ((rc = stft_setup(ctx, units, n_fft, hop_length, win_length, window, center, pad_mode, out_kind, a))) return rc;
    if (units->n_units == 0 || a.T <= 0) return SYG_OK;
    if (!y_host && units->total_len > 0) return fail(SYG_E_BADARG, "y_host is NULL");
    if (!out_host) return fail(SYG_E_BADARG, "out_host is NULL");
    const size_t out_per_unit = (size_t)(n_fft / 2 + 1) * a.T * stft_elem_bytes(out_kind);
    const int sm = ctx->sm_count;
    return host_pipeline(ctx, y_host, InFmt{}, units, out_per_unit, out_host, 0, nullptr, 0, 1LL << 40,
                         [&](Lane& L, const float* y_dev, const syg_units& cu, long long shift, long long, long long n) -> int {
                             syg::FrameArgs c = a;
                             c.y = y_dev + shift;
                             c.g = chunk_geom(cu, shift);
                             c.n_frames = n * (long long)a.T;
                             c.stft_out = L.out0.p;
                             return launch_stft(n_fft, c, sm, L.stream);
                         });
}

int syg_psd_welch_f32(syg_ctx* ctx, const float* y_dev, const syg_units* units, double fs, int32_t window,
                      int32_t nperseg, int32_t noverlap, int32_t nfft, int32_t detrend_constant, int32_t scaling,
                      float* psd_dev, float* stats_dev, void* stream) {
    SYG_TRACE();
    if (!ctx) return fail(SYG_E_BADARG, "ctx is NULL");
    int rc = check_units(units);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ENTER_DEVICE(ctx);
    WelchPlan pl;
    if ((rc = welch_setup(ctx, units, fs, window, nperseg, noverlap, nfft, detrend_constant, scaling, pl))) return rc;
    if (units->n_units == 0) return SYG_OK;
    if (!y_dev || !psd_dev) return fail(SYG_E_BADARG, "NULL device pointer");
    pl.wa.y = y_dev;
    pl.wa.g = geom_of(units, 0, units->n_units);
    pl.wa.psd = psd_dev;
    pl.wa.stats = stats_dev;
    ProfScope ps(ctx, reinterpret_cast<cudaStream_t>(stream), PROF_WELCH);
    return launch_welch(pl.nfft, pl.wa, ctx->sm_count, reinterpret_cast<cudaStream_t>(stream));
}

int syg_psd_welch_host_f32(syg_ctx* ctx, const float* y_host, const syg_units* units, double fs, int32_t window,
                           int32_t nperseg, int32_t noverlap, int32_t nfft, int32_t detrend_constant,
                           int32_t scaling, float* psd_host, float* stats_host) {
    SYG_TRACE();
    if (!ctx) return fail(SYG_E_BADARG, "ctx is NULL");
    int rc = check_host_units(units);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ENTER_DEVICE(ctx);
    WelchPlan pl;
    if ((rc = welch_setup(ctx, units, fs, window, nperseg, noverlap, nfft, detrend_constant, scaling, pl))) return rc;
    if (units->n_units == 0) return SYG_OK;
    if (!y_host || !psd_host) return fail(SYG_E_BADARG, "NULL host pointer");
    const size_t psd_per_unit = (size_t)(pl.nfft / 2 + 1) * sizeof(float);
    const size_t st_per_unit = stats_host ? 3 * sizeof(float) : 0;
    const int sm = ctx->sm_count;
    return host_pipeline(ctx, y_host, InFmt{}, units, psd_per_unit, psd_host, st_per_unit, stats_host, 0, 1LL << 40,
                         [&](Lane& L, const float* y_dev, const syg_units& cu, long long shift, long long, long long) -> int {
                             syg::WelchArgs c = pl.wa;
                             c.y = y_dev + shift;
                             c.g = chunk_geom(cu, shift);
                             c.psd = reinterpret_cast<float*>(L.out0.p);
                             c.stats = st_per_unit ? reinterpret_cast<float*>(L.out1.p) : nullptr;
                             return launch_welch(pl.nfft, c, sm, L.stream);
                         });
}

int syg_aggregate_f32(syg_ctx* ctx, const float* feats_dev, int64_t n_seg, int32_t n_rows, int64_t row_stride,
                      const int64_t* seg_off_dev, const int32_t* seg_len_dev, int32_t fixed_len, const int32_t* agg,
                      double* out_dev, void* stream) {
    SYG_TRACE();
    if (!ctx) return fail(SYG_E_BADARG, "ctx is NULL");
    if (n_seg < 0 || n_rows < 0 || row_stride < 0) return fail(SYG_E_BADARG, "negative aggregation geometry");
    if (n_seg == 0 || n_rows == 0) return SYG_OK;
    if (!feats_dev || !out_dev || !agg) return fail(SYG_E_BADARG, "NULL pointer");
    for (int i = 0; i < n_rows && i < 64; ++i)
        if (agg[i] < SYG_AGG_MEAN || agg[i] > SYG_AGG_MAX) return fail(SYG_E_BADARG, "unknown aggregation id %d", agg[i]);
    ENTER_DEVICE(ctx);
    std::string err;
    const int rc = syglaunch::aggregate(feats_dev, n_seg, n_rows, row_stride, reinterpret_cast<const long long*>(seg_off_dev), seg_len_dev,
                                        fixed_len, agg, out_dev, ctx->sm_count, reinterpret_cast<cudaStream_t>(stream), err);
    return rc ? fail(rc, "%s", err.c_str()) : SYG_OK;
}

int64_t syg_segment_count(int64_t total_samples, double sr, double segment_length_sec, double overlap_ratio,
                          int32_t pad, double min_segment_length_sec, int64_t* seg_len, int64_t* seg_hop) {
    std::string err;
    int64_t n = sygplan::segment_table(total_samples, sr, segment_length_sec, overlap_ratio, pad != 0,
                                       min_segment_length_sec, seg_len, seg_hop, nullptr, nullptr, 0, err);
    if (n < 0) return fail(SYG_E_BADARG, "%s", err.c_str());
    return n;
}

int64_t syg_segment_table(int64_t total_samples, double sr, double segment_length_sec, double overlap_ratio,
                          int32_t pad, double min_segment_length_sec, int64_t* starts, int32_t* valid, int64_t cap) {
    std::string err;
    int64_t n = sygplan::segment_table(total_samples, sr, segment_length_sec, overlap_ratio, pad != 0,
                                       min_segment_length_sec, nullptr, nullptr, starts, valid, cap, err);
    if (n < 0) return fail(SYG_E_BADARG, "%s", err.c_str());
    return n;
}

int syg_mfcc_from_logmel_f64(syg_ctx* ctx, const double* S_dev, int64_t n_units, int32_t n_mels, int64_t T, int32_t n_mfcc,
                             int32_t dct_type, int32_t dct_ortho, double lifter, double* out_dev, void* stream) {
    SYG_TRACE();
    if (!ctx) return fail(SYG_E_BADARG, "ctx is NULL");
    if (n_units < 0 || T < 0 || n_mels < 1 || n_mels > 4096) return fail(SYG_E_BADARG, "bad log-mel matrix geometry");
    if (n_mfcc < 1) return fail(SYG_E_BADARG, "n_mfcc must be positive");
    if (n_units == 0 || T == 0) return SYG_OK;
    if (!S_dev || !out_dev) return fail(SYG_E_BADARG, "NULL device pointer");
    std::lock_guard<std::mutex> lk(ctx->mu);
    ENTER_DEVICE(ctx);
    // scipy's dct(...)[:n_mfcc] keeps min(n_mfcc, n_mels) rows; the table holds exactly those
    const int C = std::min(n_mfcc, n_mels);
    std::string dk = keyf("dct64:%d:%d:%d:%d:%.9g:m%d", C, n_mels, dct_type, dct_ortho, lifter, n_mfcc);
    std::vector<double> dct;
    if (!ctx->tables.count(dk)) {
        std::string err;
        if (!sygplan::build_dct(C, n_mels, dct_type, dct_ortho != 0, lifter, n_mfcc, dct, err)) return fail(SYG_E_BADARG, "%s", err.c_str());
    }
    const double* d_dct = nullptr;
    int rc = upload_table(ctx, dk, dct, &d_dct);
    if (rc) return rc;
    std::string err;
    rc = syglaunch::dct_matrix(S_dev, d_dct, n_units, n_mels, T, C, out_dev, ctx->sm_count, reinterpret_cast<cudaStream_t>(stream), err);
    return rc ? fail(rc, "%s", err.c_str()) : SYG_OK;
}

int syg_spectral_contrast_from_mag_f32(syg_ctx* ctx, const float* S_dev, int32_t n_bins, int64_t T, double sr, int32_t n_bands,
                                       double fmin, double quantile, float* out_dev, void* stream) {
    SYG_TRACE();
    if (!ctx) return fail(SYG_E_BADARG, "ctx is NULL");
    if (n_bins < 2 || T < 0) return fail(SYG_E_BADARG, "bad spectrogram geometry");
    if (T == 0) return SYG_OK;
    if (!S_dev || !out_dev) return fail(SYG_E_BADARG, "NULL device pointer");
    std::lock_guard<std::mutex> lk(ctx->mu);
    ENTER_DEVICE(ctx);
    sygplan::Bands b;
    std::string err;
    if (!sygplan::build_bands(sr, 2 * (n_bins - 1), n_bands, fmin, quantile, b, err)) return fail(SYG_E_BADARG, "%s", err.c_str());
    int nq[syg::kMaxBands];
    for (int i = 0; i < b.nb; ++i) nq[i] = std::max(1, std::min(b.nq[i], std::max(b.cnt[i], 1)));
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    // workspace: unit maxima (one "unit" = the whole matrix: power_to_db clamps 80 dB below the array maximum) + linear peaks / valleys
    const size_t need = 256 + (size_t)T * 2 * b.nb * sizeof(float);
    if (ctx->ws_done) CK(cudaStreamWaitEvent(st, ctx->ws_done, 0));
    else CK(cudaEventCreateWithFlags(&ctx->ws_done, cudaEventDisableTiming));
    if (need > ctx->ws.cap) CK(cudaStreamSynchronize(st));
    int rc = ctx->ws.ensure(need);
    if (rc) return rc;
    struct Done { syg_ctx* c; cudaStream_t s; ~Done() { cudaEventRecord(c->ws_done, s); } } done_{ctx, st};
    unsigned* um = reinterpret_cast<unsigned*>(ctx->ws.p);
    float* cws = reinterpret_cast<float*>(reinterpret_cast<char*>(ctx->ws.p) + 256);
    CK(cudaMemsetAsync(um, 0, 4 * sizeof(unsigned), st));
    rc = syglaunch::contrast_spectrum(S_dev, n_bins, T, b.nb, b.lo, b.cnt, nq, cws, um, ctx->sm_count, st, err);
    if (rc) return fail(rc, "%s", err.c_str());
    syg::FinalizeArgs f;
    std::memset(&f, 0, sizeof(f));
    f.n_units = 1; f.T = (int)T; f.n_rows = b.nb; f.row_mfcc = -1; f.nb = b.nb; f.row_contrast = 0; f.amin = 1e-10f; f.top_db = 80.0f;
    f.cws = cws; f.unit_max = um; f.out = out_dev;
    if (T > 0x7fffffffLL) return fail(SYG_E_UNSUPPORTED, "too many frames");
    const long long n_tiles = (T + sygdev::kFinTT - 1) / sygdev::kFinTT;
    rc = syglaunch::finalize(f, sygdev::kFinTT, (unsigned)std::min<long long>(n_tiles, 0x7fffffffLL), 1u, 256, st, err);
    return rc ? fail(rc, "%s", err.c_str()) : SYG_OK;
}

int syg_debug_last_stft_path(void) { return g_last_stft_path; }
int syg_debug_last_features_resident(void) { return g_last_features_resident; }
int64_t syg_debug_last_feature_frames(void) { return g_last_feature_frames; }
int syg_debug_last_mel_form(void) { return g_last_mel_form; }
void syg_debug_set_resident_min_groups(int n) { g_resident_min_groups = n; }

int syg_debug_window(int32_t window, int32_t win_length, int32_t n_fft, float* out) {
    if (!out) return fail(SYG_E_BADARG, "out is NULL");
    std::vector<float> w;
    std::string err;
    if (!sygplan::build_window(window, win_length, n_fft, w, err)) return fail(SYG_E_BADARG, "%s", err.c_str());
    std::memcpy(out, w.data(), w.size() * sizeof(float));
    return SYG_OK;
}

int syg_debug_mel_basis(int32_t sr, int32_t n_fft, int32_t n_mels, double fmin, double fmax, float* out) {
    if (!out) return fail(SYG_E_BADARG, "out is NULL");
    sygplan::MelTable mt;
    std::string err;
    if (!sygplan::build_mel((double)sr, n_fft, n_mels, (double)fmin, fmax > 0 ? (double)fmax : 0.5 * sr, true, mt, err))
        return fail(SYG_E_BADARG, "%s", err.c_str());
    std::memcpy(out, mt.dense.data(), mt.dense.size() * sizeof(float));
    return SYG_OK;
}

int syg_debug_dct(int32_t n_mfcc, int32_t n_mels, int32_t dct_type, int32_t ortho, double lifter, float* out) {
    if (!out) return fail(SYG_E_BADARG, "out is NULL");
    std::vector<float> d;
    std::string err;
    if (!sygplan::build_dct(n_mfcc, n_mels, dct_type, ortho != 0, (double)lifter, n_mfcc, d, err))
        return fail(SYG_E_BADARG, "%s", err.c_str());
    std::memcpy(out, d.data(), d.size() * sizeof(float));
    return SYG_OK;
}

int syg_debug_contrast_bands(int32_t sr, int32_t n_fft, int32_t n_bands, double fmin, double quantile, int32_t* lo,
                             int32_t* cnt, int32_t* nq) {
    sygplan::Bands b;
    std::string err;
    if (!sygplan::build_bands((double)sr, n_fft, n_bands, (double)fmin, (double)quantile, b, err))
        return fail(SYG_E_BADARG, "%s", err.c_str());
    for (int i = 0; i < b.nb; ++i) {
        if (lo) lo[i] = b.lo[i];
        if (cnt) cnt[i] = b.cnt[i];
        if (nq) nq[i] = b.nq[i];
    }
    return SYG_OK;
}

int syg_host_alloc(void** p, size_t bytes) {
    if (!p) return fail(SYG_E_BADARG, "p is NULL");
    *p = nullptr;
    CK(cudaHostAlloc(p, std::max<size_t>(bytes, 1), cudaHostAllocDefault));
    return SYG_OK;
}

int syg_host_free(void* p) {
    if (!p) return SYG_OK;
    CK(cudaFreeHost(p));
    return SYG_OK;
}

}  // extern "C"
