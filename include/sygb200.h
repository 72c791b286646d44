/*
 * sygb200.h -- C ABI of libsygb200.so, the B200 (sm_100a) engine for the Sygnals segment->features hot path.
 *
 * The reference (araray/sygnals v1.0.0) is pure Python and defines no FFI; these entry points are what a binding
 * for this path replaces, one per reference function (paths relative to the reference tree):
 *
 *   syg_features_*        sygnals/core/features/manager.py:78-445  extract_features()
 *                         + sygnals/core/features/cepstral.py:20-120 mfcc()
 *                         + sygnals/core/features/frequency_domain.py:24-74 spectral_centroid(), :147-212
 *                           spectral_contrast(), :274-351 spectral_rolloff(), :76-145 spectral_bandwidth(),
 *                           :214-271 spectral_flatness(), :354-386 dominant_frequency()
 *                         + sygnals/core/features/time_domain.py:128-147 peak_amplitude(), :149-184 crest_factor(),
 *                           :23-58 mean_amplitude()/std_dev_amplitude()
 *                         + sygnals/core/audio/features.py:73-131 rms_energy()
 *                         applied to a batch of "units" (clips, or fixed-length segments of one recording).
 *   syg_stft_*            sygnals/core/dsp.py:167-229  compute_stft()
 *   syg_psd_welch_*       sygnals/core/dsp.py:495-560  compute_psd_welch(), :434-493 compute_psd_periodogram()
 *   syg_segment_count /   sygnals/core/segmentation.py:25-117  segment_fixed_length() (boundary arithmetic; the
 *   syg_segment_table     samples themselves are never copied: kernels frame segments by index)
 *   syg_frame_count       sygnals/core/features/manager.py:149-157 / librosa.stft frame count
 *
 * Conventions: plain pointers and sizes; every function returns SYG_OK (0) or a negative SYG_E_* code and never
 * throws; syg_last_error() gives a thread-local message.  "_dev" pointers are device pointers on the context's
 * device, "_host" pointers are host memory (pinned for full copy speed).  `stream` is a cudaStream_t passed as
 * void* (NULL = default stream).  All device work is asynchronous on `stream`; the *_host_* variants return after
 * the results are in host memory.  There is NO CPU fallback: without a CUDA device every call fails.
 */
#ifndef SYGB200_H
#define SYGB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SYG_OK 0
#define SYG_E_BADARG (-1)
#define SYG_E_SHAPE (-2)
#define SYG_E_CUDA (-3)
#define SYG_E_NOMEM (-4)
#define SYG_E_UNSUPPORTED (-5)

typedef struct syg_ctx syg_ctx;

/* feature ids, in the reference's names (manager.py:38-69) */
enum {
    SYG_FEAT_MFCC = 0,               /* n_mfcc rows  mfcc_0..                       */
    SYG_FEAT_SPECTRAL_CONTRAST = 1,  /* n_bands+1 rows contrast_band_i, contrast_delta */
    SYG_FEAT_SPECTRAL_CENTROID = 2,
    SYG_FEAT_SPECTRAL_ROLLOFF = 3,
    SYG_FEAT_RMS_ENERGY = 4,
    SYG_FEAT_CREST_FACTOR = 5,
    SYG_FEAT_PEAK_AMPLITUDE = 6,
    SYG_FEAT_SPECTRAL_BANDWIDTH = 7,
    SYG_FEAT_SPECTRAL_FLATNESS = 8,
    SYG_FEAT_DOMINANT_FREQUENCY = 9,
    SYG_FEAT_MEAN_AMPLITUDE = 10,
    SYG_FEAT_STD_DEV_AMPLITUDE = 11,
    SYG_FEAT_ZERO_CROSSING_RATE = 12, /* audio/features.py:26-71 (librosa: edge padding, threshold 1e-10) */
    SYG_FEAT_SKEWNESS = 13,           /* time_domain.py:67-97   scipy.stats.skew(bias=False)               */
    SYG_FEAT_KURTOSIS = 14,           /* time_domain.py:99-126  scipy.stats.kurtosis(fisher, bias=False)   */
    SYG_FEAT_SIGNAL_ENTROPY = 15,     /* time_domain.py:186-227 numpy.histogram(num_bins) + entropy        */
    SYG_FEAT_COUNT_ = 16
};

enum { SYG_WINDOW_HANN = 0, SYG_WINDOW_HAMMING = 1, SYG_WINDOW_BLACKMAN = 2, SYG_WINDOW_BOXCAR = 3 };
enum { SYG_PAD_CONSTANT = 0, SYG_PAD_REFLECT = 1 };
enum { SYG_OUT_COMPLEX = 0, SYG_OUT_MAGNITUDE = 1, SYG_OUT_POWER = 2 };
enum { SYG_SCALING_DENSITY = 0, SYG_SCALING_SPECTRUM = 1 };

#define SYG_MAX_FEATURES 16

/* A batch of units inside one sample buffer y.  Unit u covers y[start_u, start_u + valid_u) followed by zeros up
 * to unit_len (segment_fixed_length(pad=True) semantics, segmentation.py:90-94).
 *   analytic:  start_u = u * unit_stride, valid_u = clamp(total_len - start_u, 0, unit_len)
 *   explicit:  unit_starts[u], unit_valid[u]   (device pointers for *_f32, host pointers for *_host_f32)      */
typedef struct {
    int64_t n_units;
    int64_t unit_len;
    int64_t unit_stride;
    int64_t total_len;
    const int64_t* unit_starts; /* optional */
    const int32_t* unit_valid;  /* optional */
} syg_units;

/* extract_features(y, sr, features, frame_length, hop_length, center, window, feature_params)  manager.py:78-88 */
typedef struct {
    int32_t sr;
    int32_t frame_length; /* = n_fft = win_length (manager.py:184-187); a power of two in 32..8192, or any
                           * length >= 8 with prime factors <= 13 that fits in shared memory (mixed-radix kernels) */
    int32_t hop_length;
    int32_t center;       /* 1: zero-pad frame_length/2 both sides */
    int32_t window;       /* SYG_WINDOW_* */
    int32_t n_features;
    int32_t features[SYG_MAX_FEATURES]; /* ordered SYG_FEAT_* ids; rows follow this order (manager.py:230) */
    /* feature_params['mfcc'] (manager.py:213-217, cepstral.py:24-27) */
    int32_t n_mels;       /* 128 */
    double fmin;          /* 0 */
    double fmax;          /* <= 0: sr/2 */
    double power;         /* 2.0 */
    int32_t n_mfcc;       /* 13 */
    int32_t dct_type;     /* 2 */
    int32_t dct_ortho;    /* 1 */
    double lifter;        /* 0 */
    /* feature_params['spectral_contrast'] (frequency_domain.py:147-153) */
    int32_t contrast_n_bands; /* 6 */
    double contrast_fmin;     /* 200 */
    double contrast_quantile; /* 0.02 (double: rint(quantile * n_bins) must round as numpy does) */
    /* feature_params['spectral_rolloff'] (frequency_domain.py:277) */
    double roll_percent;      /* 0.85 */
    /* feature_params['signal_entropy'] (time_domain.py:186) */
    int32_t entropy_bins;     /* 10; supported range 1..16 */
} syg_feature_params;

const char* syg_version(void);
const char* syg_last_error(void);

int syg_ctx_create(int device, syg_ctx** out);
void syg_ctx_destroy(syg_ctx* ctx);
/* upper bound for the context-owned intermediate workspace (default 1 GiB); units are processed in chunks */
int syg_ctx_set_workspace_limit(syg_ctx* ctx, size_t bytes);
int syg_ctx_sm_count(const syg_ctx* ctx);
/* optional per-kernel timing for bench.py: CUDA events around every kernel launch on the launching stream.
 * read: ms[4] / launches[4] = {frame kernel (FFT + features or STFT), finalize kernel, welch kernel, other (ingest +
 * aggregation)}, summed since the last reset; synchronises on the recorded events. */
int syg_ctx_profile_enable(syg_ctx* ctx, int on);
int syg_ctx_profile_read(syg_ctx* ctx, double* ms, int64_t* launches, int reset);

void syg_feature_params_default(syg_feature_params* p);
/* number of output rows for the requested features (mfcc -> n_mfcc, spectral_contrast -> n_bands+1, else 1) */
int syg_features_rows(const syg_feature_params* p, int32_t* n_rows);
/* librosa / manager frame count: center ? 1 + n/hop (even frame_length) : n >= fl ? 1 + (n - fl)/hop : 0 */
int64_t syg_frame_count(int64_t n_samples, int32_t frame_length, int32_t hop_length, int32_t center);

/* out_dev: float32 [n_units][n_rows][T], T = syg_frame_count(unit_len, ...) */
int syg_features_f32(syg_ctx* ctx, const float* y_dev, const syg_units* units, const syg_feature_params* p,
                     float* out_dev, void* stream);
/* same, host buffers: chunked H2D / kernels / D2H overlapped on internal streams */
int syg_features_host_f32(syg_ctx* ctx, const float* y_host, const syg_units* units, const syg_feature_params* p,
                          float* out_host);

/* PCM16 ingest (the step before the path: sygnals/core/audio/io.py:84-95 load_audio -> librosa.load hands the reference
 * float samples = int16 / 32768).  Same as syg_features_host_f32 for 16-bit mono PCM in host memory: half the PCIe bytes, the
 * widening runs on the device.  syg_pcm16_to_f32 is the device-side conversion alone. */
int syg_features_host_pcm16(syg_ctx* ctx, const int16_t* y_host, const syg_units* units, const syg_feature_params* p,
                            float* out_host);
int syg_pcm16_to_f32(syg_ctx* ctx, const int16_t* in_dev, float* out_dev, int64_t n, void* stream);

/* General ingest = load_audio(file, sr=None, mono=True) (sygnals/core/audio/io.py:38-102 -> librosa.load -> soundfile.read(dtype=
 * float32) + librosa.to_mono) for the payload of a WAV 'data' chunk: `n_frames` interleaved frames of `channels` samples.
 * Normalisation as libsndfile: u8 (x-128)/128, s16 x/2^15, s24 x/2^23 (little endian), s32 x/2^31, f32 unchanged; channel mean as
 * numpy's np.mean(axis=0) on float32 (sequential float32 sum, one division).  Bit-exact against that arithmetic.
 * The header is parsed on the host (sygnals_b200/core/audio/io.py); resampling (sr != native) stays on the reference path. */
enum { SYG_PCM_U8 = 0, SYG_PCM_S16 = 1, SYG_PCM_S24 = 2, SYG_PCM_S32 = 3, SYG_PCM_F32 = 4 };
int syg_ingest_pcm(syg_ctx* ctx, const void* raw_dev, int32_t sample_format, int32_t channels, int64_t n_frames,
                   float* mono_dev, void* stream);
/* syg_features_host_f32 for a PCM payload in host memory: the raw bytes cross PCIe, ingest runs on the device.  `units` counts
 * FRAMES of the payload (one frame = `channels` samples = one mono sample after the mix-down). */
int syg_features_host_pcm(syg_ctx* ctx, const void* raw_host, int32_t sample_format, int32_t channels, const syg_units* units,
                          const syg_feature_params* p, float* out_host);

/* Segment vectors: extract_features() per unit followed by format_feature_vectors_per_segment() (sygnals/core/ml_utils/
 * formatters.py:51-163, the consumer in `sygnals save dataset`, sygnals/cli/save_cmd.py:140-190) with every unit as one segment:
 * out [n_units][n_rows] float64, agg[r] in SYG_AGG_* per feature row (host array).  The frame features [n_units][n_rows][T] stay
 * in a library-owned block on the device: the result that crosses PCIe (host forms) or NVLink (the final gather) is T times smaller. */
int syg_segment_vectors_f32(syg_ctx* ctx, const float* y_dev, const syg_units* units, const syg_feature_params* p,
                            const int32_t* agg, double* out_dev, void* stream);
int syg_segment_vectors_host_f32(syg_ctx* ctx, const float* y_host, const syg_units* units, const syg_feature_params* p,
                                 const int32_t* agg, double* out_host);
int syg_segment_vectors_host_pcm(syg_ctx* ctx, const void* raw_host, int32_t sample_format, int32_t channels,
                                 const syg_units* units, const syg_feature_params* p, const int32_t* agg, double* out_host);

/* Ragged batches: units of their own lengths in one call (a folder of clips, the variable-length segments of one recording).
 * Unit u is exactly y[starts[u], starts[u] + lengths[u]): no padding to a common length; units may overlap or leave gaps.  It has
 * T_u = syg_frame_count(lengths[u], ...) frames (0 allowed); F_0 = 0, F_{u+1} = F_u + T_u, F = F_{n_units}.
 * Features: float32 [n_rows][F], row r of frame t of unit u at out[r * F + F_u + t] -- the reference's features_dict over a
 * concatenated frame axis with (F_u, F_{u+1}) as segment indices (formatters.py:51-163).  Columns F_u .. F_{u+1}-1 equal, bit for
 * bit, syg_features_host_f32 on that unit alone (its own power_to_db reference level included).
 * Segment vectors: float64 [n_units][n_rows], agg[r] in SYG_AGG_* over the unit's T_u frames (T_u = 0: a NaN row).
 * The tables are HOST memory for the device and the host forms alike; the call stages them before it returns.
 * Errors: SYG_E_BADARG for a negative start or length, a unit outside the sample buffer or NULL tables (n_units > 0);
 * SYG_E_UNSUPPORTED for lengths[u] or T_u above 2^31-1; plan errors as syg_features_*.  n_units = 0 or F = 0: nothing to do. */
typedef struct {
    int64_t n_units;
    int64_t total_len;          /* samples in y */
    const int64_t* starts;      /* [n_units] host memory */
    const int64_t* lengths;     /* [n_units] host memory */
} syg_ragged_units;

/* F (>= 0) or a negative SYG_E_*; frame_off (optional, [n_units + 1]) receives F_0 .. F_{n_units} */
int64_t syg_ragged_frame_offsets(const syg_ragged_units* units, int32_t frame_length, int32_t hop_length, int32_t center,
                                 int64_t* frame_off);
int syg_features_ragged_f32(syg_ctx* ctx, const float* y_dev, const syg_ragged_units* units, const syg_feature_params* p,
                            float* out_dev, void* stream);
int syg_features_ragged_host_f32(syg_ctx* ctx, const float* y_host, const syg_ragged_units* units, const syg_feature_params* p,
                                 float* out_host);
int syg_segment_vectors_ragged_f32(syg_ctx* ctx, const float* y_dev, const syg_ragged_units* units, const syg_feature_params* p,
                                   const int32_t* agg, double* out_dev, void* stream);
int syg_segment_vectors_ragged_host_f32(syg_ctx* ctx, const float* y_host, const syg_ragged_units* units,
                                        const syg_feature_params* p, const int32_t* agg, double* out_host);

/* compute_stft(): out [n_units][1 + n_fft/2][T]; complex64 (interleaved) / float32 magnitude / float32 power */
int syg_stft_f32(syg_ctx* ctx, const float* y_dev, const syg_units* units, int32_t n_fft, int32_t hop_length,
                 int32_t win_length, int32_t window, int32_t center, int32_t pad_mode, int32_t out_kind,
                 void* out_dev, void* stream);
int syg_stft_host_f32(syg_ctx* ctx, const float* y_host, const syg_units* units, int32_t n_fft, int32_t hop_length,
                      int32_t win_length, int32_t window, int32_t center, int32_t pad_mode, int32_t out_kind,
                      void* out_host);

/* compute_psd_welch() per unit: psd [n_units][1 + nfft/2]; stats (optional) [n_units][3] = rms, crest, peak of
 * the unit.  noverlap < 0: nperseg/2; nfft <= 0: nperseg (a power of two in 32..8192, or
 * any length >= 8 with prime factors <= 13 up to 28 800: the mixed-radix kernels). */
int syg_psd_welch_f32(syg_ctx* ctx, const float* y_dev, const syg_units* units, double fs, int32_t window,
                      int32_t nperseg, int32_t noverlap, int32_t nfft, int32_t detrend_constant, int32_t scaling,
                      float* psd_dev, float* stats_dev, void* stream);
int syg_psd_welch_host_f32(syg_ctx* ctx, const float* y_host, const syg_units* units, double fs, int32_t window,
                           int32_t nperseg, int32_t noverlap, int32_t nfft, int32_t detrend_constant,
                           int32_t scaling, float* psd_host, float* stats_host);

/* format_feature_vectors_per_segment() (sygnals/core/ml_utils/formatters.py:51-163): NaN-aware aggregation of each segment's
 * frames, per row agg[r] in SYG_AGG_* (formatters.py:39-45).  Element (s, r, i) = feats_dev[off_s + r * row_stride + i],
 * i < len_s, with off_s = seg_off_dev ? seg_off_dev[s] : s * n_rows * row_stride and len_s = seg_len_dev ? seg_len_dev[s] :
 * fixed_len (len_s <= 0: NaN row, the reference's skipped segment).  out_dev: float64 [n_seg][n_rows].  agg is a HOST array. */
enum { SYG_AGG_MEAN = 0, SYG_AGG_STD = 1, SYG_AGG_MEDIAN = 2, SYG_AGG_MIN = 3, SYG_AGG_MAX = 4 };
int syg_aggregate_f32(syg_ctx* ctx, const float* feats_dev, int64_t n_seg, int32_t n_rows, int64_t row_stride,
                      const int64_t* seg_off_dev, const int32_t* seg_len_dev, int32_t fixed_len, const int32_t* agg,
                      double* out_dev, void* stream);

/* segment_fixed_length() boundary arithmetic (segmentation.py:62-114).  seg_len/seg_hop receive the integer
 * lengths; returns the number of segments (>= 0) or a negative error. */
int64_t syg_segment_count(int64_t total_samples, double sr, double segment_length_sec, double overlap_ratio,
                          int32_t pad, double min_segment_length_sec, int64_t* seg_len, int64_t* seg_hop);
int64_t syg_segment_table(int64_t total_samples, double sr, double segment_length_sec, double overlap_ratio,
                          int32_t pad, double min_segment_length_sec, int64_t* starts, int32_t* valid, int64_t cap);

/* plan tables, exported for the tests (window [n_fft]; mel basis dense [n_mels][1 + n_fft/2]; dct [n][n_mels]) */
/* Matrix-level forms of the boundary: the reference functions that take a spectrogram (frequency-major, rows x frames).
 * mfcc(S=log-mel) (sygnals/core/features/cepstral.py:94-117 -> scipy.fftpack.dct(S, axis=-2, type, norm)[:n_mfcc], lifter
 * M *= 1 + (lifter/2) sin(pi (1..n_mfcc) / lifter)): S [n_units][n_mels][T] float64 -> out [n_units][min(n_mfcc, n_mels)][T] float64.
 * spectral_contrast(S=|X|) (sygnals/core/features/frequency_domain.py:147-212, librosa defaults: quantile 0.02, dB output, each
 * of peak / valley clamped 80 dB below its own maximum): S [n_bins][T] float32 magnitudes of an n_fft = 2 (n_bins - 1) transform
 * -> out [n_bands + 1][T] float32. */
int syg_mfcc_from_logmel_f64(syg_ctx* ctx, const double* S_dev, int64_t n_units, int32_t n_mels, int64_t T, int32_t n_mfcc,
                             int32_t dct_type, int32_t dct_ortho, double lifter, double* out_dev, void* stream);
int syg_spectral_contrast_from_mag_f32(syg_ctx* ctx, const float* S_dev, int32_t n_bins, int64_t T, double sr, int32_t n_bands,
                                       double fmin, double quantile, float* out_dev, void* stream);

/* which kernel family the last syg_stft_* call of this process launched: 1 TMA-staged ring kernel, 2 register-staged warp
 * kernel, 3 CTA-cooperative kernels, 4 sub-FFT kernel for n_fft 4096 / 8192 (tests and bench.py report it) */
int syg_debug_last_stft_path(void);
/* 1 when the last feature launch kept its (short) units on chip: mel tile + dB + DCT inside the frame kernel, no finalize launch */
int syg_debug_last_features_resident(void);
/* frames the feature kernels processed in the last syg_features_* / syg_segment_vectors_* call, all chunks (n_units * T for the
 * uniform forms, F for the ragged ones) */
int64_t syg_debug_last_feature_frames(void);
/* mel projection of the last feature launch with MFCCs: 1 interval form (running sums per mel interval + picks), 0 padded tap sweeps
 * (the form is refused for banks its planner cannot represent; tests pin it for the BASELINE banks so that a refusal is not silent) */
int syg_debug_last_mel_form(void);
/* unit groups a launch needs before the resident kernel is chosen (default -1: four per SM); tests set 1 to drive it with few units */
void syg_debug_set_resident_min_groups(int n);
int syg_debug_window(int32_t window, int32_t win_length, int32_t n_fft, float* out);
int syg_debug_mel_basis(int32_t sr, int32_t n_fft, int32_t n_mels, double fmin, double fmax, float* out);
int syg_debug_dct(int32_t n_mfcc, int32_t n_mels, int32_t dct_type, int32_t ortho, double lifter, float* out);
int syg_debug_contrast_bands(int32_t sr, int32_t n_fft, int32_t n_bands, double fmin, double quantile,
                             int32_t* lo, int32_t* cnt, int32_t* nq);

/* pinned host memory helpers for callers without their own allocator */
int syg_host_alloc(void** p, size_t bytes);
int syg_host_free(void* p);

#ifdef __cplusplus
}
#endif
#endif /* SYGB200_H */
