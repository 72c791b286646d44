// PCM16 ingest: int16 samples -> float32 in [-1, 1) exactly as libsndfile / soundfile.read(dtype='float32') normalises them
// (x / 32768), which is what librosa.load hands the reference (sygnals/core/audio/io.py:84-95).
#include "syg_launch_common.h"
#include "syg_device.cuh"

namespace sygdev {
__global__ void __launch_bounds__(kThreads) pcm16_to_f32_kernel(const short* __restrict__ in, float* __restrict__ out, long long n) {
    const long long stride = (long long)gridDim.x * kThreads;
    const long long n8 = n >> 3;                                    // 8 samples (16 bytes in, 32 bytes out) per thread step
    const bool aligned = ((reinterpret_cast<uintptr_t>(in) & 15u) == 0) && ((reinterpret_cast<uintptr_t>(out) & 15u) == 0);
    long long done = 0;
    if (aligned) {
        const int4* in4 = reinterpret_cast<const int4*>(in);
        float4* out4 = reinterpret_cast<float4*>(out);
        for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n8; i += stride) {
            const int4 v = __ldg(in4 + i);
            const int w[4] = {v.x, v.y, v.z, v.w};
            float f[8];
            SYG_UNROLL
            for (int k = 0; k < 4; ++k) {
                f[2 * k] = (float)(short)(w[k] & 0xffff) * (1.0f / 32768.0f);
                f[2 * k + 1] = (float)(short)((unsigned)w[k] >> 16) * (1.0f / 32768.0f);
            }
            out4[2 * i] = make_float4(f[0], f[1], f[2], f[3]);
            out4[2 * i + 1] = make_float4(f[4], f[5], f[6], f[7]);
        }
        done = n8 << 3;
    }
    for (long long i = done + (long long)blockIdx.x * kThreads + threadIdx.x; i < n; i += stride)
        out[i] = (float)in[i] * (1.0f / 32768.0f);
}

// General ingest (load_audio(mono=True), sygnals/core/audio/io.py:38-102 -> librosa.load -> soundfile.read(dtype=float32) + to_mono):
// interleaved PCM frames of `channels` samples -> one float32 per frame.  Normalisation as libsndfile does it (u8: (x - 128) / 128,
// s16: x / 2^15, s24: x / 2^23, s32: x / 2^31, f32: unchanged); the channel mean as numpy computes np.mean(y, axis=0) on a float32
// array: float32 sum over the channels in numpy's order (sequential below 8 channels, its 8-way pairwise scheme from 8 on), then one
// float32 division by the count.  FMT: 0 u8, 1 s16, 2 s24, 3 s32, 4 f32.
// SMEM: p points into shared memory (the planar kernel's staged tile), where the read-only global load does not apply
template <bool SMEM, class T>
SYG_DEVICE SYG_INLINE T pcm_load(const unsigned char* p) {
    if (SMEM) return *reinterpret_cast<const T*>(p);
    return __ldg(reinterpret_cast<const T*>(p));
}

template <int FMT, bool SMEM = false>
SYG_DEVICE SYG_INLINE float pcm_sample(const unsigned char* __restrict__ p) {
    if (FMT == 0) return ((float)(int)pcm_load<SMEM, unsigned char>(p) - 128.0f) * (1.0f / 128.0f);
    if (FMT == 1) return (float)pcm_load<SMEM, short>(p) * (1.0f / 32768.0f);
    if (FMT == 2) {
        const int v = (int)pcm_load<SMEM, unsigned char>(p) | ((int)pcm_load<SMEM, unsigned char>(p + 1) << 8) |
                      ((int)(signed char)pcm_load<SMEM, unsigned char>(p + 2) << 16);   // little endian, sign from the top byte
        return (float)v * (1.0f / 8388608.0f);
    }
    if (FMT == 3) return (float)pcm_load<SMEM, int>(p) * (1.0f / 2147483648.0f);
    return pcm_load<SMEM, float>(p);
}

template <int FMT>
__global__ void __launch_bounds__(kThreads) pcm_ingest_kernel(const unsigned char* __restrict__ raw, int channels, long long n_frames,
                                                              float* __restrict__ out) {
    constexpr int BPS = FMT == 0 ? 1 : (FMT == 1 ? 2 : (FMT == 2 ? 3 : 4));
    const long long stride = (long long)gridDim.x * kThreads;
    const float cnt = (float)channels;
    for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n_frames; i += stride) {
        const unsigned char* p = raw + i * (long long)(channels * BPS);
        float acc;
        if (channels < 8) {
            acc = pcm_sample<FMT>(p);
            for (int c = 1; c < channels; ++c) acc += pcm_sample<FMT>(p + c * BPS);
        } else {
            // numpy's pairwise_sum along the contiguous axis (the channels of one frame after librosa's transpose): eight running
            // sums over blocks of eight, combined as a tree, then the tail added one by one (channels <= 64 < its 128 block size)
            float r[8];
            SYG_UNROLL
            for (int k = 0; k < 8; ++k) r[k] = pcm_sample<FMT>(p + k * BPS);
            int c = 8;
            for (; c + 8 <= channels; c += 8) {
                SYG_UNROLL
                for (int k = 0; k < 8; ++k) r[k] += pcm_sample<FMT>(p + (c + k) * BPS);
            }
            acc = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
            for (; c < channels; ++c) acc += pcm_sample<FMT>(p + c * BPS);
        }
        out[i] = channels > 1 ? acc / cnt : acc;
    }
}

// Planar ingest (load_audio(mono=False)): interleaved frames of `channels` samples -> float32 planes out[c * pitch + i], the same
// normalisation as above and no mix-down.  A tiled transpose: a CTA stages kPlanarTile frames (contiguous payload bytes, 16-byte
// loads when the tile is 16-byte aligned, byte loads otherwise) into shared memory, then consecutive threads write consecutive
// frames of one channel.  Staged rows are padded to an odd number of 32-bit words, so the threads of a warp, which read one channel
// of 32 consecutive frames, hit 32 different banks.  Only frames i < n_frames of each plane are written.
constexpr int kPlanarTile = 128;
constexpr int kPlanarRowMax = 64 * 4 + 4;                       // bytes of a padded row: 64 channels of 4 bytes, one pad word

template <int FMT>
__global__ void __launch_bounds__(kThreads) pcm_planar_kernel(const unsigned char* __restrict__ raw, int channels, long long n_frames,
                                                              long long pitch, float* __restrict__ out) {
    constexpr int BPS = FMT == 0 ? 1 : (FMT == 1 ? 2 : (FMT == 2 ? 3 : 4));
    __shared__ int4 tile4[kPlanarTile * kPlanarRowMax / 16];
    unsigned char* tile = reinterpret_cast<unsigned char*>(tile4);
    const int fb = channels * BPS;
    const int rs = (((fb + 3) / 4) | 1) * 4;                    // padded row stride in bytes
    const long long n_tiles = (n_frames + kPlanarTile - 1) / kPlanarTile;
    for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const long long f0 = t * kPlanarTile;
        const int nf = n_frames - f0 < kPlanarTile ? (int)(n_frames - f0) : kPlanarTile;
        const unsigned char* src = raw + f0 * fb;
        const int bytes = nf * fb;
        __syncthreads();                                        // the previous tile has been read
        if ((reinterpret_cast<uintptr_t>(src) & 15u) == 0 && fb % 4 == 0) {
            const int fw = fb / 4;                              // 32-bit words per frame: a word never straddles two rows
            const int n16 = bytes / 16;
            for (int k = threadIdx.x; k < n16; k += kThreads) {
                const int4 v = __ldg(reinterpret_cast<const int4*>(src) + k);
                const int w[4] = {v.x, v.y, v.z, v.w};
                SYG_UNROLL
                for (int j = 0; j < 4; ++j) {
                    const int wi = 4 * k + j;
                    *reinterpret_cast<int*>(tile + (wi / fw) * rs + (wi % fw) * 4) = w[j];
                }
            }
            for (int wi = 4 * n16 + threadIdx.x; wi < bytes / 4; wi += kThreads)
                *reinterpret_cast<int*>(tile + (wi / fw) * rs + (wi % fw) * 4) = __ldg(reinterpret_cast<const int*>(src) + wi);
        } else {
            for (int b = threadIdx.x; b < bytes; b += kThreads) tile[(b / fb) * rs + b % fb] = __ldg(src + b);
        }
        __syncthreads();
        for (int k = threadIdx.x; k < channels * nf; k += kThreads) {
            const int c = k / nf, i = k - c * nf;
            out[(long long)c * pitch + f0 + i] = pcm_sample<FMT, true>(tile + i * rs + c * BPS);
        }
    }
}
}  // namespace sygdev

namespace syglaunch {
int pcm16_to_f32(const short* in, float* out, long long n, int sm_count, cudaStream_t st, std::string& err);
int pcm_to_f32(const void* raw, int fmt, int channels, long long n_frames, float* out, int sm_count, cudaStream_t st, std::string& err) {
    if (n_frames <= 0) return 0;
    if (channels < 1 || channels > 64) { err = "channels must be in [1, 64]"; return -1; }
    if (fmt == 1 && channels == 1) return pcm16_to_f32(reinterpret_cast<const short*>(raw), out, n_frames, sm_count, st, err);   // vectorised
    const unsigned char* r = reinterpret_cast<const unsigned char*>(raw);
    const int grid = (int)std::min<long long>((n_frames + sygdev::kThreads - 1) / sygdev::kThreads, (long long)sm_count * 16);
    switch (fmt) {
        case 0: SYG_LAUNCH(sygdev::pcm_ingest_kernel<0>, grid, sygdev::kThreads, 0, st, r, channels, n_frames, out); break;
        case 1: SYG_LAUNCH(sygdev::pcm_ingest_kernel<1>, grid, sygdev::kThreads, 0, st, r, channels, n_frames, out); break;
        case 2: SYG_LAUNCH(sygdev::pcm_ingest_kernel<2>, grid, sygdev::kThreads, 0, st, r, channels, n_frames, out); break;
        case 3: SYG_LAUNCH(sygdev::pcm_ingest_kernel<3>, grid, sygdev::kThreads, 0, st, r, channels, n_frames, out); break;
        case 4: SYG_LAUNCH(sygdev::pcm_ingest_kernel<4>, grid, sygdev::kThreads, 0, st, r, channels, n_frames, out); break;
        default: err = "unknown PCM sample format " + std::to_string(fmt); return -1;
    }
    LCK(cudaGetLastError());
    return 0;
}

int pcm_to_planes(const void* raw, int fmt, int channels, long long n_frames, long long pitch, float* out, int sm_count, cudaStream_t st,
                  std::string& err) {
    if (n_frames <= 0) return 0;
    if (channels < 1 || channels > 64) { err = "channels must be in [1, 64]"; return -1; }
    const unsigned align = fmt == 1 ? 2u : (fmt == 3 || fmt == 4 ? 4u : 1u);
    if (channels == 1 && (reinterpret_cast<uintptr_t>(raw) & (align - 1)) == 0)        // mono: the one plane is the mono ingest
        return pcm_to_f32(raw, fmt, 1, n_frames, out, sm_count, st, err);
    const unsigned char* r = reinterpret_cast<const unsigned char*>(raw);
    const int grid = (int)std::min<long long>((n_frames + sygdev::kPlanarTile - 1) / sygdev::kPlanarTile, (long long)sm_count * 6);
    switch (fmt) {
        case 0: SYG_LAUNCH(sygdev::pcm_planar_kernel<0>, grid, sygdev::kThreads, 0, st, r, channels, n_frames, pitch, out); break;
        case 1: SYG_LAUNCH(sygdev::pcm_planar_kernel<1>, grid, sygdev::kThreads, 0, st, r, channels, n_frames, pitch, out); break;
        case 2: SYG_LAUNCH(sygdev::pcm_planar_kernel<2>, grid, sygdev::kThreads, 0, st, r, channels, n_frames, pitch, out); break;
        case 3: SYG_LAUNCH(sygdev::pcm_planar_kernel<3>, grid, sygdev::kThreads, 0, st, r, channels, n_frames, pitch, out); break;
        case 4: SYG_LAUNCH(sygdev::pcm_planar_kernel<4>, grid, sygdev::kThreads, 0, st, r, channels, n_frames, pitch, out); break;
        default: err = "unknown PCM sample format " + std::to_string(fmt); return -1;
    }
    LCK(cudaGetLastError());
    return 0;
}

int pcm16_to_f32(const short* in, float* out, long long n, int sm_count, cudaStream_t st, std::string& err) {
    if (n <= 0) return 0;
    const long long want = (n / 8 + sygdev::kThreads - 1) / sygdev::kThreads + 1;
    const int grid = (int)std::min<long long>(want, (long long)sm_count * 8);
    SYG_LAUNCH(sygdev::pcm16_to_f32_kernel, grid, sygdev::kThreads, 0, st, in, out, n);
    LCK(cudaGetLastError());
    return 0;
}
}  // namespace syglaunch
