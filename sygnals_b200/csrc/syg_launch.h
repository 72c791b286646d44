// sygnals_b200/csrc/syg_launch.h -- host-side launch interface between syg_api.cu and the kernel translation units.
#pragma once

#include <string>

#include "../../include/sygb200.h"
#include "syg_params.h"

namespace syglaunch {
// what the last launch of each kernel family ran, for the syg_debug_last_* getters: one host store per launch
struct LastLaunch {
    int feature_kernel = 0;        // SYG_FK_*
    int stft_path = 0;             // syg_debug_last_stft_path
    int welch_path = 0;            // SYG_WELCH_*
    int mixed_threads = 0;         // threads per CTA of the last mixed-radix launch
    int fin_tt = 0;                // finalize: frames per tile, CTAs, tiles
    long long fin_ctas = 0, fin_tiles = 0;
};
extern LastLaunch g_last;

// all return 0 or a negative SYG_E_* code (-3 CUDA, -5 unsupported) with a message in err
int frame_block(int n_fft, int mode, const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err);
int frame_warp(int n_fft, bool extra, const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err);
// TMA-staged ring kernel; returns 1 when the call is not eligible (the caller then launches frame_warp_stft / frame_block)
int stft_ring(int n_fft, const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err);
// n_fft 4096 / 8192, real-valued output: 1024-point sub-FFTs per warp + recombination (syg_stft_big.cuh)
int stft_big(int n_fft, const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err);
// unit-resident feature kernel (short units, MFCC epilogue on chip): units per CTA group for this plan (0 = not eligible), launch
int frame_warp_res_units(int n_fft, const syg::FrameArgs& a);
int frame_warp_res(int n_fft, const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err);
// ragged launches (FrameArgs::ragged_ut, syg_launch_ragged.cu): the per-frame table {unit, frame in unit, length, start} from frame
// offsets frame_off[n_units + 1] and the unit tables (starts < 2^31: relative to the chunk's samples), and the warp feature kernel
// (STAGE 6).  frame_block / frame_mixed / time_extra / finalize take MODE_FEATURES_RAGGED / ragged_ut themselves.
int ragged_frame_table(const long long* frame_off, const long long* starts, const int* valid, long long n_units, long long n_frames,
                       int4* ut, int sm_count, cudaStream_t st, std::string& err);
int frame_warp_ragged(int n_fft, bool extra, const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err);
int frame_warp_stft(int n_fft, const syg::FrameArgs& a, int sm_count, cudaStream_t st, std::string& err);
int finalize(const syg::FinalizeArgs& a, int tt, unsigned grid_x, unsigned grid_y, size_t smem, cudaStream_t st, std::string& err);
// mel spectrogram epilogue (mel_store_kernel): a chunk's mel energies to [unit][n_mels][T] / [n_mels][ragged_stride], S_mel or S_db
int mel_store(const syg::FinalizeArgs& a, int sm_count, cudaStream_t st, std::string& err);
int aggregate(const float* feats, long long n_seg, int n_rows, long long row_stride, const long long* seg_off, const int* seg_len,
              int fixed_len, const int* agg_host, double* out, int sm_count, cudaStream_t st, std::string& err);
int time_extra(const syg::FrameArgs& a, int frame_length, int entropy_bins, int sm_count, cudaStream_t st, std::string& err);
int pcm_to_f32(const void* raw, int fmt, int channels, long long n_frames, float* out, int sm_count, cudaStream_t st, std::string& err);
int pcm16_to_f32(const short* in, float* out, long long n, int sm_count, cudaStream_t st, std::string& err);
// interleaved PCM -> float32 planes out[c * pitch + i] (i < n_frames), one per channel; channels == 1 takes pcm_to_f32
int pcm_to_planes(const void* raw, int fmt, int channels, long long n_frames, long long pitch, float* out, int sm_count, cudaStream_t st,
                  std::string& err);
int dct_matrix(const double* S, const double* D, long long n_units, int N, long long T, int C, double* out, int sm_count, cudaStream_t st,
               std::string& err);
int contrast_spectrum(const float* S, int B, long long T, int nb, const int* lo, const int* cnt, const int* nq, float* cws, unsigned* unit_max,
                      int sm_count, cudaStream_t st, std::string& err);
// transform lengths that are not powers of two (syg_mixed.cuh): mode = MODE_FEATURES / MODE_STFT
int frame_mixed(int mode, const syg::FrameArgs& a, const syg::MixedPlan& mp, int sm_count, cudaStream_t st, std::string& err);
int welch_mixed(const syg::WelchArgs& a, const syg::MixedPlan& mp, int sm_count, cudaStream_t st, std::string& err);
int welch(int nfft, const syg::WelchArgs& a, int sm_count, cudaStream_t st, std::string& err);
}  // namespace syglaunch
