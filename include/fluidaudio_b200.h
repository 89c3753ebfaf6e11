/* fluidaudio_b200 — C ABI of the B200-native (sm_100a) implementation of FluidAudio's two CPU hot paths.
 *
 * Every entry point is what a Swift/cgo/ctypes FFI binding for that piece of the reference would bind:
 * plain pointers and sizes, caller-owned buffers, an int status, no exception ever crosses the boundary
 * (same conventions as the reference's only C boundary, Sources/FastClusterWrapper/include/FastClusterWrapper.h).
 * There is NO CPU fallback: without an sm_100a device every compute call returns FA_NO_DEVICE.
 *
 * Reference interfaces replaced (paths relative to the FluidAudio repository):
 *   fa_mel_*             Sources/FluidAudio/Shared/AudioMelSpectrogram.swift:18-121 (class + init),
 *                        :132 compute, :185 computeFlat, :299/:325 computeFlatTransposed, :486-493 getters
 *   fa_audio_resample / fa_audio_to_mel / fa_resample_output_count
 *                        Sources/FluidAudio/Shared/AudioConverter.swift:60-71 (resample), :299-370 (convertBuffer),
 *                        :388-442 (linearResample) — the converter stage on the GPU, fused ahead of the log-mel kernel
 *   fa_linear_resample   Sources/FluidAudio/Shared/AudioConverter.swift:388-442 (linearResample; the converter stage's linear kernel)
 *   fa_l2_normalize_rows Sources/FluidAudio/Diarizer/Offline/Clustering/AHCClustering.swift:70-105
 *   fastcluster_compute_centroid_linkage  (declared in FastClusterWrapper.h, same symbol as the reference)
 *   fa_ahc_cluster       AHCClustering.swift:20-67  (AHCClustering.cluster)
 *   fa_dendrogram_cut    AHCClustering.swift:112-121,124-210
 *   fa_vbx_refine        Sources/FluidAudio/Diarizer/Offline/Clustering/VBxClustering.swift:41-165 (refine)
 *   fa_compute_centroids Sources/FluidAudio/Diarizer/Offline/Core/OfflineDiarizerManager.swift:613-691
 *   fa_assign_embeddings OfflineDiarizerManager.swift:789-822
 *   fa_diarize_cluster   OfflineDiarizerManager.swift:270-384 (cluster(_:), clustering phase)
 *   fa_constrained_assign / fa_hungarian_solve / fa_build_chunk_assignments
 *                        ConstrainedClusterAssignment.swift:20-42, HungarianAssignment.swift:8-97, :885-911
 *   fa_kmeans_cluster / fa_speaker_constraints_resolve
 *                        KMeansClustering.swift:39-130,212-223, SpeakerCountConstraints.swift:27-85,
 *                        VBxClustering.swift:685-733 (refineWithConstraints)
 *   fa_build_segments    Diarizer/Offline/Utils/OfflineReconstruction.swift:24-253, 359-505
 *   fa_export_*          OfflineDiarizerManager.swift:913-955 (exportEmbeddings: the JSON dump of TimedEmbedding +
 *                        cluster, OfflineDiarizerTypes.swift:706-716) — the backend's on-disk input format
 */
#ifndef FLUIDAUDIO_B200_H
#define FLUIDAUDIO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    FA_STATUS_OK = 0,
    FA_STATUS_INVALID_ARGUMENT = 1,
    FA_STATUS_INDEX_OVERFLOW = 2,
    FA_STATUS_OUTPUT_TOO_SMALL = 3,
    FA_STATUS_ALLOCATION_FAILURE = 4,
    FA_STATUS_RUNTIME_ERROR = 5,   /* e.g. NaN distance, as the reference's nan_error */
    FA_STATUS_NO_DEVICE = 6,       /* no sm_100a GPU visible: there is deliberately no CPU fallback */
    FA_STATUS_CUDA_ERROR = 7,
    FA_STATUS_UNSUPPORTED = 8,
    FA_STATUS_UNKNOWN_ERROR = 255
} fa_status;

/* ---- runtime ------------------------------------------------------------------------------------------- */
const char *fa_version(void);
const char *fa_last_error(void);            /* thread-local text of the last failure */
int32_t fa_device_count(void);              /* sm_100a devices visible */
fa_status fa_set_device(int32_t ordinal);   /* binds the calling thread; one process per GPU is the intended use */
fa_status fa_device_synchronize(void);
int64_t fa_kernel_launch_count(void);       /* kernels this library has launched in this process */

/* Pinned host memory and device memory for callers that want the copy engines / resident buffers. */
fa_status fa_host_alloc(size_t bytes, void **out);
fa_status fa_host_free(void *p);
fa_status fa_device_alloc(size_t bytes, void **out);
fa_status fa_device_free(void *p);
fa_status fa_memcpy_h2d(void *dst_device, const void *src_host, size_t bytes);
fa_status fa_memcpy_d2h(void *dst_host, const void *src_device, size_t bytes);

/* Bare copy-engine probe: `reps` rounds of one H2D copy (h2d_bytes from host_src) and one D2H copy (d2h_bytes into
 * host_dst) issued together on two streams; *ms_per_round = wall clock per round.  The floor under every host-buffer
 * ("end to end") number: what PCIe and the host memory path deliver with no kernel in between. */
fa_status fa_memcpy_probe(const void *host_src, size_t h2d_bytes, void *host_dst, size_t d2h_bytes, int32_t reps,
                          float *ms_per_round);

/* Device-side timing of a region on the library's default stream (CUDA events). */
fa_status fa_timer_start(void);
fa_status fa_timer_stop_ms(float *elapsed_ms);

/* ---- log-mel frontend ---------------------------------------------------------------------------------- */
typedef struct {
    int32_t sample_rate;     /* 16000 */
    int32_t n_mels;          /* 128 (reference default); 80 in BASELINE config 2 */
    int32_t n_fft;           /* 512 */
    int32_t hop_length;      /* 160 */
    int32_t win_length;      /* 400 */
    float preemph;           /* 0.97 */
    int32_t pad_to;          /* 0 -> 1 */
    float log_floor;         /* 2^-24 */
    int32_t log_floor_mode;  /* 0 = additive log(x+floor), 1 = clamped log(max(x,floor)) */
    int32_t window_periodic; /* 0 = symmetric Hann, 1 = periodic */
} fa_mel_config;

enum { FA_MEL_PAD_CENTER = 0, FA_MEL_PAD_PREPADDED = 1, FA_MEL_LEGACY_COMPUTE = 2 };
enum { FA_MEL_TIME_MAJOR = 0 /* [T x nMels], computeFlatTransposed */, FA_MEL_MEL_MAJOR = 1 /* [nMels x T], computeFlat / compute */ };

typedef struct fa_mel fa_mel;   /* one handle per stream of calls: like the Swift class it is not thread-safe */

void fa_mel_default_config(fa_mel_config *cfg);
fa_status fa_mel_create(const fa_mel_config *cfg, fa_mel **out);
void fa_mel_destroy(fa_mel *mel);
fa_status fa_mel_get_window(const fa_mel *mel, float *out, size_t len);       /* getHannWindow(): win_length floats */
fa_status fa_mel_get_filterbank(const fa_mel *mel, float *out, size_t len);   /* getFilterbank(): n_mels x (n_fft/2+1) */
/* frames the reference would produce; expected_frames < 0 means nil */
int64_t fa_mel_frame_count(const fa_mel *mel, int64_t sample_count, int32_t padding_mode, int64_t expected_frames);

/* Arithmetic of the 512-point transform (window product, |.|^2, filterbank and log are float32 in both, like the reference):
 *   FA_MEL_PRECISION_F64  (default) DFT evaluated in FP64 and rounded once — the implementation-independent value,
 *                         reproduces the oracle to ~5e-6 in the log domain whatever the signal's dynamic range;
 *   FA_MEL_PRECISION_F32  DFT in float32 like the reference's own vDSP_DFT_zop (AudioMelSpectrogram.swift:459-481), two
 *                         frames per warp on packed FFMA2/FADD2: ~2x the throughput; carries the float32 noise floor of
 *                         any float32 FFT (measured max |delta log-mel| 6e-5 over BASELINE's hour of audio). */
enum { FA_MEL_PRECISION_F64 = 0, FA_MEL_PRECISION_F32 = 1 };
fa_status fa_mel_set_precision(fa_mel *mel, int32_t precision);
int32_t fa_mel_get_precision(const fa_mel *mel);
/* Host-buffer calls on long clips are cut into `chunks` units whose H2D copy, kernels and D2H copy overlap on three
 * streams (default 24; 1 = no overlap).  Results do not depend on it. */
fa_status fa_mel_set_pipeline_chunks(fa_mel *mel, int32_t chunks);
/* When the caller's time-major output buffer is pinned host memory (fa_host_alloc / cudaHostAlloc), the kernel stores its rows
 * straight into it over PCIe instead of staging them in HBM and copying.  Default OFF: on B200 + PCIe 5 the SM-issued posted writes
 * measured slower than the copy engine (4.72 vs 4.53 ms per audio-hour, profiles/r02_mel.md); pageable buffers always take the copy. */
fa_status fa_mel_set_zero_copy_output(fa_mel *mel, int32_t enabled);

/* Host buffers in and out (the drop-in call).  On return *mel_length = valid frames, *num_frames = padded frames;
 * out receives num_frames*n_mels floats in `layout`.  Mirrors computeFlatTransposed / computeFlat / compute. */
fa_status fa_mel_compute(fa_mel *mel, const float *audio, size_t sample_count, float last_audio_sample,
                         int32_t padding_mode, int64_t expected_frames, int32_t layout, float *out, size_t out_len,
                         int64_t *mel_length, int64_t *num_frames);
/* Same with buffers already resident in HBM (asynchronous on the library stream). */
fa_status fa_mel_compute_device(fa_mel *mel, const float *d_audio, size_t sample_count, float last_audio_sample,
                                int32_t padding_mode, int64_t expected_frames, int32_t layout, float *d_out,
                                size_t out_len, int64_t *mel_length, int64_t *num_frames);
/* Batch of independent clips.  Clip i is audio[offsets[i] .. offsets[i+1]); its output starts at out_offsets[i]
 * and holds num_frames[i]*n_mels floats (use fa_mel_frame_count to size it).  last_samples may be NULL. */
fa_status fa_mel_compute_batch(fa_mel *mel, const float *audio, const int64_t *offsets, int32_t clip_count,
                               const float *last_samples, int32_t padding_mode, int32_t layout, float *out,
                               const int64_t *out_offsets, int64_t *mel_lengths, int64_t *num_frames);
fa_status fa_mel_compute_batch_device(fa_mel *mel, const float *d_audio, const int64_t *offsets, int32_t clip_count,
                                      const float *last_samples, int32_t padding_mode, int32_t layout, float *d_out,
                                      const int64_t *out_offsets, int64_t *mel_lengths, int64_t *num_frames);

/* CUDA-event timer on the stream the mel kernels run on: bracket any number of fa_mel_compute*_device calls. */
fa_status fa_mel_timer_start(fa_mel *mel);
fa_status fa_mel_timer_stop_ms(fa_mel *mel, float *elapsed_ms);

/* Callers directly behind AudioMelSpectrogram, with their post-processing as device epilogues of the mel kernel.
 * fa_mel_unified_features = UnifiedMelExtractor.features(window:validCount:) (ASR/Parakeet/Unified/
 *   UnifiedMelExtractor.swift:52-113): the handle must be configured like its AudioMelSpectrogram (:31-40);
 *   total_frames = window_samples / hop + 1, valid_frames = min(valid_count / hop, total_frames); out receives the
 *   per-feature-normalised log-mel packed [n_mels x total_frames] (the MLMultiArray [1, nMels, T]).
 * fa_mel_lseend_features = LSEENDPreprocessor.processAudioQueue (Diarizer/LS-EEND/LSEENDPreprocessor.swift:249-283):
 *   the handle configured as :70-81 (preemph 0, periodic Hann, clamped floor 1e-10); out receives [frames x n_mels]
 *   log10-scaled, cumulative-mean-normalised features; cmn_mean[n_mels] / cmn_count are the running state, updated. */
fa_status fa_mel_unified_features(fa_mel *mel, const float *window, size_t window_samples, size_t valid_count,
                                  float *out, size_t out_len, int64_t *total_frames, int32_t *valid_frames);
fa_status fa_mel_lseend_features(fa_mel *mel, const float *chunk, size_t n, float *cmn_mean, int64_t *cmn_count,
                                 float *out, size_t out_len, int64_t *frames);


/* NeMo per-feature normalisation of a time-major [frames x n_mels] buffer, in place (host buffer).
 * UnifiedMelExtractor.normalizePerFeature, Sources/FluidAudio/ASR/Parakeet/Unified/UnifiedMelExtractor.swift:88-113 */
fa_status fa_mel_normalize_per_feature(float *x, int64_t frames, int32_t n_mels, int64_t valid_frames);

/* ---- AudioConverter stage on the GPU ---------------------------------------------------------------------
 * PCM in any of the layouts AVAudioPCMBuffer / a WAV file hands over -> mono float32 at out_rate.
 *   algorithm AUTO follows AudioConverter.convertBuffer (:299-305): more than two channels take linearResample
 *   (:388-442, reproduced BIT FOR BIT: mean mixdown, src = i * ratio in double, two-tap float32 lerp); one or two
 *   channels take the AVAudioConverter path, whose arithmetic is closed — replaced by a documented Kaiser-windowed-sinc
 *   polyphase filter (24 zero crossings, beta 12, pass band 0.94 of the lower Nyquist; fluidaudio_b200/csrc/
 *   resample_plan.h), "parity unpinned" against Apple's sample values.  in_rate == out_rate is the identity on the
 *   samples (:66-68), after mixdown / int16 widening (v / 32768) when the input is not already mono float32.
 *   Output length = Int(Double(frames) / (in_rate / out_rate)) (:417-418) for both algorithms: the reference's tests
 *   accept +-1 % (AudioConverterTests.swift:129-176). */
enum { FA_PCM_F32 = 0, FA_PCM_I16 = 1 };
enum { FA_RESAMPLE_AUTO = 0, FA_RESAMPLE_SINC = 1, FA_RESAMPLE_LINEAR = 2 };
typedef struct {
    double in_rate;        /* e.g. 48000 */
    double out_rate;       /* 16000 (AudioConverter's default target) */
    int32_t channels;      /* >= 1 */
    int32_t format;        /* FA_PCM_F32 / FA_PCM_I16 */
    int32_t interleaved;   /* 1: [frames x channels] (WAV); 0: planar [channels x frames] (floatChannelData) */
    int32_t algorithm;     /* FA_RESAMPLE_* */
} fa_audio_format;
int64_t fa_resample_output_count(const fa_audio_format *fmt, int64_t frames);
/* AudioConverter.resample / resampleBuffer: host PCM in, host float32 mono out (conversion runs on the GPU). */
fa_status fa_audio_resample(const void *pcm, int64_t frames, const fa_audio_format *fmt, float *out, int64_t out_cap,
                            int64_t *out_count);
/* AudioConverter.resample followed by AudioMelSpectrogram.computeFlatTransposed / computeFlat as ONE device pipeline:
 * only the raw PCM crosses PCIe on the way in (int16 halves the bytes of the float path), the converted samples never
 * leave HBM.  fmt->out_rate must equal the handle's sample_rate.  *resampled_count (may be NULL) = samples at out_rate. */
fa_status fa_audio_to_mel(fa_mel *mel, const void *pcm, int64_t frames, const fa_audio_format *fmt,
                          float last_audio_sample, int32_t padding_mode, int32_t layout, float *out, size_t out_len,
                          int64_t *mel_length, int64_t *num_frames, int64_t *resampled_count);

/* AudioConverter.linearResample: planar [channels x frames] -> mono at out_rate.  Returns the sample count
 * through *out_count; call with out == NULL to size the buffer. */
fa_status fa_linear_resample(const float *planar, int64_t frames, int32_t channels, double in_rate, double out_rate,
                             float *out, int64_t out_cap, int64_t *out_count);

/* ---- offline clustering backend ------------------------------------------------------------------------ */
fa_status fa_l2_normalize_rows(const double *x, size_t rows, size_t dim, double *out);

/* AHCClustering.cluster: rows are NOT yet normalised; labels are canonical (first appearance order). */
fa_status fa_ahc_cluster(const double *features, size_t count, size_t dim, double threshold, int32_t *labels);

/* Device time of the calling thread's most recent linkage: [0] initial nearest-neighbour pass, [1] heapify + copies,
 * [2] persistent merge kernel, [3] total (ms).  Diagnostics only. */
void fa_ahc_last_stage_ms(float *out4);

/* Placement the calling thread's most recent linkage ran with, as six values:
 *   [0] master level: 3 = heap, nearest neighbours and slot table in shared memory, 2 = heap and nearest neighbours,
 *       1 = heap only (all three with 16-bit heap indices), 0 = all in global memory (32-bit heap indices)
 *   [1] 1 = node vectors resident in the workers' shared memory, 0 = streamed from global memory
 *   [2] worker CTAs   [3] node slots per worker CTA (resident only, else 0)
 *   [4] initial nearest-neighbour pass: 0 = exact, 1 = float32 filter with the per-row pass 2, 2 = float32 filter with
 *       the tiled pass 2, 3 = filter abandoned for the exact pass (non-finite input or too many candidates)
 *   [5] SMs of the device
 * All zeros before the thread's first linkage.  Diagnostics only: needs no device and changes no result. */
void fa_ahc_last_placement(int32_t *out6);

/* Swift-side dendrogram cut + relabel on a SciPy-format linkage Z [(count-1) x 4]. */
fa_status fa_dendrogram_cut(const double *Z, size_t count, double threshold, int32_t *labels);

typedef struct {
    double Fa;               /* 0.07 */
    double Fb;               /* 0.8 */
    int32_t max_iterations;  /* 20 */
    double epsilon;          /* 1e-4 */
    double init_smoothing;   /* 7.0 */
} fa_vbx_config;
void fa_vbx_default_config(fa_vbx_config *cfg);

/* VBxClustering.refine.  rho: T x D; psi: psi_len doubles (identity if psi_len != D); initial: T labels.
 * speakers = number of distinct initial labels (the caller sizes gamma [T x speakers], pi [speakers],
 * elbos [max(max_iterations,1)], hard [T]).  *iterations receives the number of EM iterations run. */
fa_status fa_vbx_refine(const double *rho, size_t T, size_t D, const double *psi, size_t psi_len,
                        const int32_t *initial, int32_t speakers, const fa_vbx_config *cfg, double *gamma,
                        double *pi, double *elbos, int32_t *hard, int32_t *iterations);

/* computeCentroids (gamma/pi weighted, speakers with pi > 1e-7).  centroids capacity speakers x dim.
 * *centroid_count receives K. */
fa_status fa_compute_centroids(const double *embeddings, size_t T, size_t dim, const double *gamma, const double *pi,
                               int32_t speakers, double *centroids, int32_t *centroid_count);

/* assignEmbeddings: cosine against every centroid, first maximum wins.  scores may be NULL (else N x K). */
fa_status fa_assign_embeddings(const double *embeddings, size_t N, size_t dim, const double *centroids, int32_t K,
                               int32_t *labels, double *scores);

#define FA_NO_VALUE INT32_MIN   /* an absent optional count (Swift nil) in fa_cluster_config / fa_speaker_constraints_resolve */

typedef struct {
    double threshold;        /* 0.6  OfflineDiarizerConfig.clusteringThreshold */
    fa_vbx_config vbx;       /* warmStartFa/Fb, VBx.maxIterations, convergenceTolerance */
    /* OfflineDiarizerConfig.Clustering.numSpeakers / minSpeakers / maxSpeakers (OfflineDiarizerTypes.swift);
     * FA_NO_VALUE = nil (zero and negative counts are legal inputs, the reference clamps them to 1).
     * When the count VBx arrives at violates them the embeddings are re-clustered with K-Means (n_init 10, seeds 0..9,
     * 100 iterations) and assigned by plain argmax (VBxClustering.swift:685-733, OfflineDiarizerManager.swift:354-375). */
    int32_t num_speakers, min_speakers, max_speakers;
    int32_t reserved;
} fa_cluster_config;
void fa_cluster_default_config(fa_cluster_config *cfg);

typedef struct {
    int32_t training_count;    /* embeddings that survived the NaN/Inf filter */
    int32_t initial_clusters;  /* AHC cluster count (= VBx speaker count S) */
    int32_t vbx_iterations;
    int32_t centroid_count;    /* K */
    float ms_normalize, ms_ahc, ms_cut, ms_vbx, ms_assign, ms_total;   /* device/host stage times */
    int32_t was_adjusted;      /* VBxOutput.wasAdjusted: K-Means replaced the VBx clusters */
    int32_t detected_clusters; /* VBxOutput.assignedClusterCount before the adjustment */
} fa_cluster_info;

/* OfflineDiarizerManager.cluster(_:) lines 286-375 (unconstrained argmax assignment):
 *   emb256: N x emb_dim float32; rho: N x rho_dim float64; psi: rho_dim doubles, or NULL for the identity (pass NULL
 *   when the PLDA parameters have another length: VBxClustering.swift:71-76).  labels: N final assignments.
 * Optional outputs (may be NULL): initial [N] AHC labels of the training rows (-1 for filtered rows),
 * centroids [max_centroids x emb_dim], info. */
fa_status fa_diarize_cluster(const float *emb256, const double *rho, size_t N, size_t emb_dim, size_t rho_dim,
                             const double *psi, const fa_cluster_config *cfg, int32_t *labels, int32_t *initial,
                             double *centroids, int32_t max_centroids, fa_cluster_info *info);

/* Same with the reference's DEFAULT assignment (OfflineDiarizerConfig.Clustering.constrainedAssignment = true,
 * OfflineDiarizerManager.swift:357-369): chunk_index[N] is TimedEmbedding.chunkIndex; local speakers that share a chunk
 * are matched to distinct clusters (labels[i] = -2 when a chunk has more local speakers than clusters).
 * chunk_index == NULL, or a single centroid, falls back to the plain argmax like the reference. */
fa_status fa_diarize_cluster_chunks(const float *emb256, const double *rho, size_t N, size_t emb_dim, size_t rho_dim,
                                    const double *psi, const fa_cluster_config *cfg, const int32_t *chunk_index,
                                    int32_t *labels, int32_t *initial, double *centroids, int32_t max_centroids,
                                    fa_cluster_info *info);

/* HungarianAssignment.solve / maxScoreAssignment (HungarianAssignment.swift:8-61, :67-97),
 * ConstrainedClusterAssignment.assign (ConstrainedClusterAssignment.swift:20-42) and
 * OfflineDiarizerManager.buildChunkAssignments (:885-911).  Exact integer logic on tiny per-chunk matrices: host. */
fa_status fa_hungarian_solve(const int64_t *cost_square, int32_t n, int32_t *assignment);
fa_status fa_max_score_assignment(const double *scores, int32_t rows, int32_t cols, int32_t *assignment);
fa_status fa_constrained_assign(const double *scores, size_t N, int32_t K, const int32_t *chunk_index, int32_t *labels);
fa_status fa_build_chunk_assignments(const int32_t *chunk_index, const int32_t *speaker_index, const int32_t *assignments,
                                     size_t N, int32_t num_chunks, int32_t num_speakers, int32_t cluster_count,
                                     int32_t *matrix);

/* OfflineReconstruction.buildSegments (Diarizer/Offline/Utils/OfflineReconstruction.swift:24-253): the step after
 * fa_build_chunk_assignments in OfflineDiarizerManager.cluster(_:).  speaker_weights: SegmentationOutput.speakerWeights
 * flattened [num_chunks x num_frames x num_speakers]; chunk_offsets: SegmentationOutput.chunkOffsets (offsets_count may
 * be smaller than num_chunks: missing chunks start at chunk * window_duration); hard_clusters: the matrix returned by
 * fa_build_chunk_assignments [hard_rows x num_speakers] (-2 = inactive); centroid_count: centroids.count.
 * Output: *segment_count segments sorted by start (speakerId = "S<cluster+1>", embedding = centroid[cluster]); when
 * segment_cap is too small the first segment_cap are written and FA_STATUS_OUTPUT_TOO_SMALL is returned.  Host code; the
 * zero-vote re-embed pass (off by default, needs the embedding model) is not part of it. */
typedef struct {
    double frame_duration, window_duration, min_gap_duration, seg_min_duration_off, seg_min_duration_on, min_segment_duration;
    int32_t exclusive_segments;
    int32_t reserved;
} fa_reconstruct_config;
void fa_reconstruct_default_config(fa_reconstruct_config *cfg);   /* OfflineDiarizerConfig defaults, frame_duration = 0 */
fa_status fa_build_segments(const float *speaker_weights, int32_t num_chunks, int32_t num_frames, int32_t num_speakers,
                            const double *chunk_offsets, int32_t offsets_count, const int32_t *hard_clusters,
                            int32_t hard_rows, int32_t centroid_count, const fa_reconstruct_config *cfg,
                            int32_t *seg_cluster, float *seg_start, float *seg_end, float *seg_quality,
                            int32_t segment_cap, int32_t *segment_count);

/* OfflineReconstruction.buildSpeakerDatabase (:296-357): database [K x dim] = per speaker the float32 mean of its segments'
 * embeddings (a segment's embedding is Float(centroids[cluster])); segment_counts [K]; speakers without segment stay zero. */
fa_status fa_build_speaker_database(const int32_t *seg_cluster, int32_t segment_count, const double *centroids, int32_t K,
                                    int32_t dim, float *database, int32_t *segment_counts);

/* KMeansClustering.clusterWithCentroidsNInit (Diarizer/Offline/Clustering/KMeansClustering.swift:39-130) on raw
 * embeddings [N x D]: labels [N], centroids (normalised space) [min(num_clusters, N) x D] -> *centroid_rows rows;
 * *best_init = index of the winning seed.  n_init <= 1 runs the single seeded clustering (:39-92).
 * fa_speaker_constraints_resolve = SpeakerCountConstraints.resolve (SpeakerCountConstraints.swift:27-71);
 * FA_NO_VALUE = nil. */
fa_status fa_kmeans_cluster(const double *embeddings, size_t N, size_t D, int32_t num_clusters, int32_t max_iterations,
                            int32_t n_init, uint64_t base_seed, int32_t *labels, double *centroids,
                            int32_t centroid_cap, int32_t *centroid_rows, int32_t *best_init);
fa_status fa_speaker_constraints_resolve(int64_t num_embeddings, int64_t num_speakers, int64_t min_speakers,
                                         int64_t max_speakers, int64_t *resolved_min, int64_t *resolved_max);

/* Embedding-export files (JSON array written by the reference when OfflineDiarizerConfig.embeddingExportPath is set):
 * {chunkIndex, speakerIndex, startFrame, endFrame, startTime, endTime, embedding256[], rho128[], cluster} per entry.
 * fa_export_shape parses the file and reports the entry count and vector lengths; fa_export_read fills caller-owned
 * arrays (any output pointer may be NULL); fa_export_write produces a file the reference's Codable struct decodes.
 * float32 values round-trip bit-exactly (shortest-form decimal <-> strtof). */
fa_status fa_export_shape(const char *path, size_t *count, size_t *emb_dim, size_t *rho_dim);
fa_status fa_export_read(const char *path, size_t count, size_t emb_dim, size_t rho_dim, int32_t *chunk_index,
                         int32_t *speaker_index, int32_t *start_frame, int32_t *end_frame, double *start_time,
                         double *end_time, float *emb, double *rho, int32_t *cluster);
fa_status fa_export_write(const char *path, size_t count, size_t emb_dim, size_t rho_dim, const int32_t *chunk_index,
                          const int32_t *speaker_index, const int32_t *start_frame, const int32_t *end_frame,
                          const double *start_time, const double *end_time, const float *emb, const double *rho,
                          const int32_t *cluster);

/* Many independent embedding sets (meetings) on this GPU.  Set m is rows [set_offsets[m], set_offsets[m+1]).
 * Several sets are clustered concurrently on disjoint SM partitions. */
fa_status fa_diarize_cluster_batch(const float *emb256, const double *rho, const int64_t *set_offsets,
                                   int32_t set_count, size_t emb_dim, size_t rho_dim, const double *psi,
                                   const fa_cluster_config *cfg, int32_t *labels, fa_cluster_info *infos);

/* Same with the reference's default constrained assignment in every set (OfflineDiarizerManager.swift:357-369):
 * chunk_index[row] is TimedEmbedding.chunkIndex of that row, numbered inside its own set; NULL = plain argmax. */
fa_status fa_diarize_cluster_batch_chunks(const float *emb256, const double *rho, const int64_t *set_offsets,
                                          int32_t set_count, size_t emb_dim, size_t rho_dim, const double *psi,
                                          const fa_cluster_config *cfg, const int32_t *chunk_index, int32_t *labels,
                                          fa_cluster_info *infos);

#ifdef __cplusplus
}
#endif
#endif /* FLUIDAUDIO_B200_H */
