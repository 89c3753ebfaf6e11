// Host-side plan + launch descriptors of the fused log-mel kernel (see mel_kernels.cu).
#pragma once

#include "fa_common.cuh"
#include "resample_plan.h"
#include <cuda_runtime.h>
#include <vector>

namespace fa {
namespace mel {

struct cpx;

// Mirrors the parameters of AudioMelSpectrogram.init (AudioMelSpectrogram.swift:59-70).
struct MelConfig {
    int32_t sample_rate;
    int32_t n_mels;
    int32_t n_fft;
    int32_t hop_length;
    int32_t win_length;
    float preemph;
    int32_t pad_to;
    float log_floor;
    int32_t log_floor_mode;    // 0 additive log(x + floor), 1 clamped log(max(x, floor))
    int32_t window_periodic;
};

// One unit of work = a run of frames of one clip.  A long clip is cut into several units so that H2D copies,
// kernels and D2H copies of successive units overlap; a batch of clips is simply many units in one launch.
struct MelUnit {
    long long audio_off;     // float offset of the clip's sample 0 inside the audio buffer (multiple of 4 for TMA)
    long long n;             // samples in the clip
    long long out_off;       // float offset of the clip's output inside the output buffer
    long long out_stride;    // mel-major layout: row stride (= padded frame count); unused for time-major
    long long frame_begin;   // first frame of this unit
    long long frame_count;   // frames in this unit
    float last;              // lastAudioSample (pre-emphasis state), x[-1]
    int tile_begin;          // first tile index of this unit inside its launch
};

struct MelLaunch {
    const float *audio;
    float *out;
    const MelUnit *units;
    int num_units;
    int total_tiles;
    int hop;
    int pad;            // audio index of buffer position j of frame f is f*hop + j - pad
    float preemph;
    int n_mels;
    float log_floor;
    int log_clamped;
    int ot_stride;      // floats per row of the staged output tile: n_mels + 4 (16-byte aligned rows) or n_mels + 1
    int vec_out;        // time-major copy-out in float4 stores: n_mels % 4 == 0 and every unit's output 16-byte aligned
    int log_normal;     // log_floor is a normal float: the denormal handling of the device log can be skipped
    int layout;         // 0 time-major [T x nMels], 1 mel-major [nMels x stride]
    const void *lane_tab;   // [32] LaneTables<V> of the launch's window placement and precision (mel_core.cuh)
    const float *win_tab;
    const uint8_t *in_tab;
    const float *fb_w;
    const int *fb_lo;
    const int *fb_hi;
    const int *fb_off;
    const int4 *fb_slots;   // mel512_kernel's filterbank schedule: {first bin, quads, weight offset, mel bin or -1} per slot
    int n_slots;
    int fb_nnz, fb_cap;
    int pt_len, pt_cap, raw_cap;
    int use_tma;
    int mid_full;          // window covers buffer positions [64, 448): pass 1 skips the in-window select for slots 1..6
    unsigned inv_n_mels;   // ceil(2^32 / n_mels): idx / n_mels == umulhi(idx, inv) for idx < 2^16 (n_mels > 1)
    int inline_unit;       // single-unit launch: the descriptor travels in the kernel parameters (unit0), units is not read
    MelUnit unit0;
};

struct MelPlan {
    MelConfig cfg{};
    std::vector<float> window;       // [win]
    std::vector<float> filterbank;   // [n_mels x 257] dense, as the reference exposes it (getFilterbank)
    int fb_nnz = 0, fb_cap = 0;
    int pt_len = 0, pt_cap = 0, raw_cap = 0;
    size_t smem_bytes = 0;
    int num_sms = 0;
    long long launches = 0;          // kernels launched through this plan (bench.py reports it)
    int precision = 0;               // transform arithmetic: 0 = FP64 (one frame per warp), 1 = packed float32 pairs
    int pipeline_chunks = 24;        // units a long host-buffer call is cut into (H2D / kernel / D2H overlap)
    bool zero_copy_out = false;      // time-major output in a pinned host buffer: the kernel stores straight into it
                                     // (measured SLOWER than the staged copy on B200 + PCIe 5: 4.72 vs 4.53 ms per hour; opt-in)
    bool inline_unit = false;        // next launch() passes its (single) unit in the kernel parameters
    bool generic = false;            // nFFT != 512 or odd hop: mel_generic_kernel (FP64 transform whatever `precision`)
    int generic_warps = 0, generic_prow = 0, generic_log2n = 0;
    void *d_generic_tw = nullptr;    // FP64 twiddles W_n^k, k < n/2

    void *d_lane_tab[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};   // [window placement][precision]
    float *d_win_tab_mode[2] = {nullptr, nullptr};
    uint8_t *d_in_tab_mode[2] = {nullptr, nullptr};
    float *d_fb_w = nullptr;
    int *d_fb_lo = nullptr, *d_fb_hi = nullptr, *d_fb_off = nullptr;
    void *d_fb_slots = nullptr;
    int n_slots = 0;

    MelUnit *d_units = nullptr, *h_units = nullptr;
    int units_cap = 0;
    float *d_audio = nullptr, *d_out = nullptr;   // staging for the host-buffer entry points
    size_t d_audio_cap = 0, d_out_cap = 0;
    // AudioConverter stage ahead of the kernel (fa_audio_to_mel): raw PCM staging + the polyphase table of the last ratio
    void *d_pcm = nullptr;
    size_t d_pcm_cap = 0;
    resample::Design rs_design;
    double rs_in = 0.0, rs_out = 0.0;
    float *d_rs_tab = nullptr;
    cudaStream_t streams[3] = {nullptr, nullptr, nullptr};   // h2d, compute, d2h
    std::vector<cudaEvent_t> events;
    cudaEvent_t timer[2] = {nullptr, nullptr};   // fa_mel_timer_*: events on the compute stream

    ~MelPlan();
    void release();
    int init(const MelConfig &c);
    long long frame_count(long long n, int mode, long long expected) const;
    int ensure_units(int count);
    int ensure_staging(size_t audio_floats, size_t out_floats);
    int ensure_events(size_t count);
    // kernel launch over units [first, first+count) already resident in d_units
    int launch(const float *d_audio_base, float *d_out_base, int first, int count, int total_tiles, int mode,
               int layout, cudaStream_t stream, bool aligned16);

    // mode: 0 .center, 1 .prePadded, 2 legacy compute(); layout: 0 time-major, 1 mel-major
    int compute_device(const float *d_in, long long n, float last, int mode, long long expected, int layout,
                       float *d_out_buf, long long out_len, long long *mel_length, long long *num_frames,
                       cudaStream_t stream);
    int compute_host(const float *audio, long long n, float last, int mode, long long expected, int layout,
                     float *out, long long out_len, long long *mel_length, long long *num_frames);
    // PCM in any AudioFormat (host) -> [device: mixdown + resample to cfg.sample_rate] -> log-mel (host).  Only the raw
    // PCM crosses PCIe on the way in (int16 halves the bytes); *resampled = samples at the model rate.
    int compute_host_pcm(const void *pcm, long long frames, const resample::AudioFormat &f, float last, int mode,
                         int layout, float *out, long long out_len, long long *mel_length, long long *num_frames,
                         long long *resampled);
    int ensure_resampler(double in_rate, double out_rate);
    int compute_batch_host(const float *audio, const long long *offsets, int count, const float *last, int mode,
                           int layout, float *out, const long long *out_offsets, long long *mel_lengths,
                           long long *num_frames);
    int compute_batch_device(const float *d_in, const long long *offsets, int count, const float *last, int mode,
                             int layout, float *d_out_buf, const long long *out_offsets, long long *mel_lengths,
                             long long *num_frames, cudaStream_t stream);
};

// mel_adapters.cu: device epilogues for the callers directly behind AudioMelSpectrogram (host buffers in and out)
int normalize_per_feature_host(float *x, long long T, int M, long long valid);   // mel_adapters.cu
int unified_features(MelPlan &p, const float *window, long long n, long long valid_count, float *out, long long out_len,
                     long long *total_frames, int *valid_frames);
int lseend_features(MelPlan &p, const float *chunk, long long n, float *cmn_mean, long long *cmn_count, float *out,
                    long long out_len, long long *frames);

void build_window(int length, bool periodic, std::vector<float> &w);
void build_filterbank(int n_fft, int n_mels, int sample_rate, std::vector<float> &fb);

} // namespace mel
} // namespace fa
