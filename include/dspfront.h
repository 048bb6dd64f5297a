/*
 * dspfront.h -- C ABI of libdspfront.so, the B200 (sm_100a) implementation of
 * DSP-AudioRecLabs' data-parallel front end and KNN classify step.
 *
 * The reference has no FFI of its own: its boundary is the Python module
 * surface of src/audio_processing.py, src/feature_extraction.py and the 'knn'
 * branch of src/models.py (SURVEY.md section 8(b)).  Every entry point below
 * names the reference interface (file:line under /root/reference) it stands
 * in for; the ctypes binding a maintainer would add is shown in
 * INTEGRATION.md and shipped as dsp_audioreclabs_b200/_capi.py.
 *
 * Conventions: plain pointers and sizes only; every function returns
 * DSP_OK (0) or a negative dsp_status and leaves a message for
 * dsp_last_error(); outputs are caller-allocated; "host" entry points take
 * host pointers and return only when the outputs are filled; "device" entry
 * points take device pointers, enqueue on the context's stream and return
 * immediately (dsp_sync() waits).  There is no CPU implementation behind any
 * of these calls: without a CUDA device dsp_create() fails.
 */
#ifndef DSPFRONT_H_
#define DSPFRONT_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSPFRONT_ABI_VERSION 2

typedef enum {
  DSP_OK = 0,
  DSP_ERR_INVALID = -1,   /* bad argument (the Python shims raise ValueError) */
  DSP_ERR_CUDA = -2,      /* CUDA runtime failure */
  DSP_ERR_NO_DEVICE = -3, /* no usable sm_100 device */
  DSP_ERR_UNSUPPORTED = -4,
  DSP_ERR_NOMEM = -5
} dsp_status;

/* sample encodings accepted by the front end (what load_wav can produce,
 * src/audio_processing.py:31-44, plus the float arrays the per-call API takes) */
typedef enum {
  DSP_S16 = 0, /* 16-bit PCM, value/32768.0      (:35-38) */
  DSP_U8 = 1,  /* 8-bit PCM, uint8(value-128)/128.0: the reference's uint8 subtraction wraps (:31-34) */
  DSP_F32 = 2, /* float samples, used as-is (widened to float64) */
  DSP_F64 = 3  /* float64 samples, used as-is */
} dsp_dtype;

/* create_window, src/audio_processing.py:278-296 */
typedef enum { DSP_WIN_RECTANGULAR = 0, DSP_WIN_HAMMING = 1, DSP_WIN_HANNING = 2 } dsp_window_type;

/* per-utterance status written by the front end */
#define DSP_UTT_OK 0
#define DSP_UTT_EMPTY 1      /* no audio after endpoint detection: ValueError at :388-389 */
#define DSP_UTT_NO_FRAMES 2  /* zero frames: ValueError at feature_extraction.py:27-28 */
#define DSP_UTT_EXACT 0x100  /* flag bit: result came from the float64 replay kernel */

/* Parameters of process_audio_file (src/audio_processing.py:336-343) with the
 * config.py names (config.py:35-45). */
typedef struct {
  int32_t frame_length;        /* config.FRAME_LENGTH, samples */
  int32_t frame_shift;         /* config.FRAME_SHIFT, samples */
  int32_t window;              /* dsp_window_type */
  int32_t do_endpoint_detection;
  double energy_high_ratio;    /* config.ENERGY_HIGH_RATIO */
  double energy_low_ratio;     /* config.ENERGY_LOW_RATIO */
  double zcr_threshold_ratio;  /* config.ZCR_THRESHOLD_RATIO */
  int32_t channels;            /* 1, or 2 = interleaved stereo averaged per frame (:43-44) */
  int32_t force_exact;         /* 1: run every utterance through the float64 replay kernel */
  int32_t aligned16;           /* device entry point only, optional hint: 1 = every utterance starts on a 16-byte
                                * boundary (offsets multiples of 8 samples, 16-byte aligned buffer).  Since ABI 2
                                * nothing depends on it for the pipelined kernel -- packed CSR batches of any
                                * length run at full speed, its producer realigns them on chip; the hint only
                                * selects between two builds of the older resident kernel for other geometries */
} dsp_frontend_params;

/* Output pointers of one front-end batch.  Any pointer may be NULL to skip
 * that output.  Ragged outputs are addressed through the offsets computed by
 * dsp_frontend_plan(): utterance b owns [feat_offsets[b], feat_offsets[b+1])
 * of energy/magnitude/zcr (n_frames[b] entries are valid) and
 * [epd_offsets[b], epd_offsets[b+1]) of epd_energy/epd_zcr. */
typedef struct {
  int32_t* start;        /* [B] start_point                 (endpoint_detection :272) */
  int32_t* end;          /* [B] end_point                   (:273) */
  int32_t* n_epd_frames; /* [B] len(energy_list)            (:166) */
  int32_t* n_frames;     /* [B] len(frames)                 (frame_signal :299-333) */
  int32_t* status;       /* [B] DSP_UTT_* */
  float* energy;         /* ragged, extract_frame_features 'energy'    (feature_extraction.py:34-37) */
  float* magnitude;      /* ragged, 'magnitude' */
  float* zcr;            /* ragged, 'zcr' (integer valued) */
  float* stats;          /* [B,15] extract_statistical_features (:65-88) */
  double* epd_energy;    /* ragged, energy_list of endpoint_detection (:183) */
  float* epd_zcr;        /* ragged, zcr_list (:184) */
  /* ABI 2: the same results as the reference holds them, in float64.  Requesting ANY of these routes the
   * whole batch through the float64 replay kernel, whose values are bit-identical to the NumPy path
   * (the drop-in process_audio_file / extract_features_from_frames use them; the float outputs above
   * are the throughput path, held to the north star's 1e-5 relative). */
  double* energy_f64;    /* ragged like `energy` */
  double* magnitude_f64; /* ragged like `magnitude` */
  double* zcr_f64;       /* ragged like `zcr` */
  double* stats_f64;     /* [B,15] */
  double* epd_zcr_f64;   /* ragged like `epd_zcr` */
  double* frames_f64;    /* dense windowed frames of frame_signal (:299-333): row feat_offsets[b] + t holds
                          * frame t of utterance b, frame_length values each -- only for callers that really
                          * read the (F, fl) matrix process_audio_file returns */
} dsp_frontend_outputs;

typedef struct dsp_context dsp_context;

/* ---- context ----------------------------------------------------------- */
int dsp_abi_version(void);
const char* dsp_last_error(void);
/* device: CUDA ordinal.  Fails with DSP_ERR_NO_DEVICE when there is no GPU. */
int dsp_create(int device, dsp_context** out);
int dsp_destroy(dsp_context* ctx);
/* Enqueue all device entry points on an existing CUDA stream (e.g. torch's current stream; a NULL
 * handle is CUDA's legacy default stream).  dsp_use_own_stream() returns to the context's own. */
int dsp_set_stream(dsp_context* ctx, void* cuda_stream);
int dsp_use_own_stream(dsp_context* ctx);
int dsp_sync(dsp_context* ctx);
/* Tuning knobs (not needed for correctness): "pcm_variant" = -1 automatic, 0..9 one build of the
 * fused kernel (0, 8, 9 shared-memory resident; 1-7 streaming, for 16-byte aligned utterances), 10 the
 * pipelined kernel (build 0 where its plan does not fit); "tma_chunk" = bytes per bulk copy;
 * "stagger_ns" = start-up delay per co-resident CTA; "knn_prune" = 0 off, 1 automatic, 2 always. */
int dsp_set_tuning(dsp_context* ctx, const char* key, int value);
/* kernels launched by this context since creation (bench.py's gpu_launches) */
int64_t dsp_launch_count(dsp_context* ctx);
int dsp_device_sm_count(dsp_context* ctx);

/* ---- front end --------------------------------------------------------- */
/* Batch layout: utterance b starts at element offsets[b] of the sample buffer (elements =
 * samples of one channel times `channels`).  lengths == NULL: packed CSR, utterance b is
 * [offsets[b], offsets[b+1]).  lengths != NULL: utterance b holds lengths[b] elements and
 * offsets[b+1] - offsets[b] >= lengths[b] may include padding -- e.g. every start rounded up to
 * a multiple of 8 samples so that the aligned (TMA / streaming) loads apply to ragged data.
 *
 * dsp_frontend_plan: host arithmetic only.  Fills feat_offsets[B+1] / epd_offsets[B+1]
 * (capacities: frame counts of the untrimmed utterances, SURVEY.md A.2) and returns the longest
 * utterance. */
int dsp_frontend_plan(const int64_t* offsets, const int32_t* lengths, int64_t n_utts,
                      const dsp_frontend_params* p, int64_t* feat_offsets, int64_t* epd_offsets,
                      int64_t* max_len);

/* create_window (src/audio_processing.py:278-296): float64 window of `length`. */
int dsp_window(int window_type, int32_t length, double* out);

/* process_audio_file minus the WAV decode + extract_features_from_frames
 * ('statistical'), batched (src/audio_processing.py:364-394,
 * src/feature_extraction.py:91-112).  All pointers are DEVICE pointers. */
int dsp_frontend_batch_device(dsp_context* ctx, const void* samples, int dtype,
                              const int64_t* offsets, const int32_t* lengths, const int64_t* feat_offsets,
                              const int64_t* epd_offsets, int64_t n_utts, int64_t max_len,
                              const dsp_frontend_params* p, const dsp_frontend_outputs* out);

/* Same with HOST pointers: stages through pinned memory in chunks, overlapping
 * upload, kernels and download.  This is the call the Python shims make. */
int dsp_frontend_batch_host(dsp_context* ctx, const void* samples, int dtype,
                            const int64_t* offsets, const int32_t* lengths, int64_t n_utts,
                            const dsp_frontend_params* p, const dsp_frontend_outputs* out);

/* preprocess = remove_dc + normalize_audio (src/audio_processing.py:49-90) for one
 * float64 signal; mode 0 = remove_dc only, 1 = normalize only, 2 = both.  Host pointers. */
int dsp_preprocess_host(dsp_context* ctx, const double* x, int64_t n, int mode, double* out);

/* endpoint_detection on an already pre-processed float64 signal
 * (src/audio_processing.py:135-275).  Host pointers; energy_list/zcr_list hold
 * (n-fl)/fs+1 entries when n >= fl. */
int dsp_endpoint_detection_host(dsp_context* ctx, const double* x, int64_t n,
                                const dsp_frontend_params* p, int32_t* start, int32_t* end,
                                int32_t* n_epd_frames, double* energy_list, double* zcr_list);

/* frame_signal (src/audio_processing.py:299-333): frames_out is [n_frames, frame_length]
 * float64 with n_frames from dsp_frame_count().  Host pointers. */
int64_t dsp_frame_count(int64_t n, int32_t frame_length, int32_t frame_shift);
int dsp_frame_signal_host(dsp_context* ctx, const double* x, int64_t n, int32_t frame_length,
                          int32_t frame_shift, int window_type, double* frames_out);

/* extract_frame_features + compute_statistics on an arbitrary float64 frame matrix
 * (src/feature_extraction.py:12-88; with n_frames == 1 these are
 * compute_short_time_energy/magnitude/zero_crossing_rate, audio_processing.py:93-132).
 * energy/magnitude/zcr: [n_frames] float64, stats: [15] float64 (may be NULL). */
int dsp_frame_features_host(dsp_context* ctx, const double* frames, int64_t n_frames,
                            int32_t frame_length, double* energy, double* magnitude, double* zcr,
                            double* stats);

/* compute_statistics (src/feature_extraction.py:46-62) of one float64 sequence -> 5 values. */
int dsp_sequence_stats_host(dsp_context* ctx, const double* seq, int64_t n, double* out5);

/* normalize_features (src/feature_extraction.py:157-181).  fit != 0 computes mean/std
 * (population) over axis 0 of the C-ordered [n, d] x into mean/std first, in NumPy's summation
 * order for the caller's original layout: fit = 1 adds the rows one after another (np.mean over
 * axis 0 of a C-ordered array), fit = 2 sums every column pairwise (np.mean of each column as a
 * 1-D array: 1-D, (n, 1) and Fortran-ordered inputs).  std == 0 is replaced by 1 when applying
 * (the returned std keeps the replacement, as the reference does). */
int dsp_zscore_host(dsp_context* ctx, const double* x, int64_t n, int32_t d, int fit, double* mean,
                    double* std, double* out);
int dsp_zscore_device(dsp_context* ctx, const double* x, int64_t n, int32_t d, int fit, double* mean,
                      double* std, double* out);
/* Apply only, on the float32 [n,15] statistics the fused front end writes (dsp_frontend_outputs.stats): each value
 * is widened exactly and normalised with the given float64 mean / std (std == 0 counts as 1) -- the step between
 * the front end and dsp_knn_predict_device in the batched pipeline (train_model.py:147-148).  Device pointers. */
int dsp_zscore_apply_f32_device(dsp_context* ctx, const float* x, int64_t n, int32_t d, const double* mean,
                                const double* std, double* out);

/* ---- KNN classify (src/models.py:33-35,52-58 -> sklearn KNeighborsClassifier) ---- */
typedef struct dsp_knn dsp_knn;
/* fit: keeps a device copy of train[n,d] (float64, row major) and labels[n].
 * index_base is added to local row numbers in every reported neighbour index
 * (row-sharded multi-GPU: the shard's first global row). */
int dsp_knn_fit_host(dsp_context* ctx, const double* train, const int32_t* labels, int64_t n,
                     int32_t d, int32_t k, int64_t index_base, dsp_knn** out);
int dsp_knn_fit_device(dsp_context* ctx, const double* train, const int32_t* labels, int64_t n,
                       int32_t d, int32_t k, int64_t index_base, dsp_knn** out);
int dsp_knn_free(dsp_knn* knn);
/* k nearest train rows of each query by exact float64 squared Euclidean distance, ties to
 * the lower index: nbr_idx[m,k] (global), nbr_sqdist[m,k], nbr_label[m,k]; any may be NULL. */
int dsp_knn_topk_host(dsp_knn* knn, const double* queries, int64_t m, int64_t* nbr_idx,
                      double* nbr_sqdist, int32_t* nbr_label);
int dsp_knn_topk_device(dsp_knn* knn, const double* queries, int64_t m, int64_t* nbr_idx,
                        double* nbr_sqdist, int32_t* nbr_label);
/* The same for a ROW SHARD of the train set when the caller knows, per query, an upper bound on the squared distance of
 * its k-th neighbour in the WHOLE train set (row-sharded KNN: the k-th distance within the shard that owns the query,
 * src/models.py:56-58 semantics unchanged): the shard returns its rows inside that radius -- possibly fewer than k,
 * the rest of a query's slots are (-1, +inf, -1) -- and never has to discover a threshold of its own.  Exact like
 * dsp_knn_topk_device: every row of the shard within the bound (ties included) is returned or displaced by k better
 * ones.  bound_sqdist: float64 [m], +inf = no bound; NULL = dsp_knn_topk_device. */
int dsp_knn_topk_bounded_device(dsp_knn* knn, const double* queries, int64_t m, const double* bound_sqdist, int64_t* nbr_idx,
                                double* nbr_sqdist, int32_t* nbr_label);
/* predict = topk + majority vote, vote ties to the smallest label. */
int dsp_knn_predict_host(dsp_knn* knn, const double* queries, int64_t m, int32_t* labels_out);
/* Diagnostics of the last topk / predict call on this handle (waits for it): how many queries the
 * float64 certificate sent to the exhaustive float64 rescan, and which candidate scan ran
 * (0 = none: float64 only, 1 = fp32 tiled scan, 2 = tensor-core scan of wide features, 3 = tensor-core filter for
 * d <= 15 with the fp32 scan standing in when a query leaves its range).  Results never depend on it. */
int dsp_knn_last_stats(dsp_knn* knn, int64_t* rescanned, int32_t* scan_kind);
int dsp_knn_predict_device(dsp_knn* knn, const double* queries, int64_t m, int32_t* labels_out);
/* Merge R candidate lists (as gathered from R row shards, layout [R,m,k]) into the global
 * top-k and vote.  Device pointers. */
int dsp_knn_merge_vote_device(dsp_context* ctx, const double* cand_sqdist, const int64_t* cand_idx,
                              const int32_t* cand_label, int32_t n_lists, int64_t m, int32_t k,
                              int32_t* labels_out, int64_t* nbr_idx_out, double* nbr_sqdist_out);

/* ---- MFCC + DTW template matching (BASELINE config 5; SURVEY.md 8 a11 / f4) -------------
 * NOT in the reference (compare_feature_methods.py has no spectral features and no template
 * matching): a self-specified variant, defined by oracle/mfcc_dtw_oracle.py ("self-oracle").  It
 * composes with the path above: pre-processing as src/audio_processing.py:49-90, the trimmed
 * segment [start, end) from endpoint_detection (:135-275), frames by frame_signal's rule
 * (:299-333), then pre-emphasis, window, power spectrum of an n_fft-point FFT, the caller's
 * mel filterbank [n_mels][n_fft/2+1], log(max(., log_floor)) and the caller's DCT matrix
 * [n_ceps][n_mels].  mfcc_offsets[B+1] (in frames, from dsp_frame_count(end-start, ...))
 * addresses the ragged output [frames][n_ceps]. */
typedef struct {
  int32_t frame_length, frame_shift, n_fft, n_mels, n_ceps;
  int32_t window;        /* dsp_window_type */
  double pre_emphasis;   /* y[i] = x[i] - pre_emphasis * x[i-1] inside the segment */
  double log_floor;
} dsp_mfcc_params;

int dsp_mfcc_batch_host(dsp_context* ctx, const int16_t* samples, const int64_t* offsets,
                        const int32_t* lengths, const int32_t* seg_start, const int32_t* seg_end,
                        int64_t n_utts, const dsp_mfcc_params* params, const float* filterbank,
                        const float* dct, const int64_t* mfcc_offsets, float* mfcc_out,
                        int32_t* n_frames_out);
/* DTW (Euclidean local distance, steps (1,0) (0,1) (1,1), accumulated cost D[n-1][m-1]) of every
 * query sequence against every template sequence -- one CTA per pair, anti-diagonal wavefront --
 * and the k cheapest templates per query (ties to the lower index).  Sequences are ragged
 * [frames][dim] float32 with offsets in frames.  cost_out (optional) receives the full
 * [nq][nt] matrix.  index_base lets row-sharded template sets be merged like KNN candidates. */
int dsp_dtw_topk_host(dsp_context* ctx, const float* q_feats, const int64_t* q_offsets, int64_t nq,
                      const float* t_feats, const int64_t* t_offsets, const int32_t* t_labels,
                      int64_t nt, int32_t dim, int32_t k, int64_t index_base, float* cost_out,
                      double* nbr_cost, int64_t* nbr_idx, int32_t* nbr_label);

/* ---- batched WAV ingest (SURVEY.md 8 f1) ----------------------------------
 * Replaces the per-file `wave.open` / `readframes` / `np.frombuffer` of load_wav
 * (src/audio_processing.py:21-40) for whole file lists.  Host-only I/O: no CUDA device is
 * needed for dsp_wav_scan / dsp_wav_read.  The chunk walk accepts and rejects what CPython's
 * `wave` module does; dsp_wav_info.status says why a file was refused (the callers of the
 * reference skip such files, run_experiments.py:109-111).  Sample widths other than 1 and 2
 * parse fine and are refused by the caller like load_wav does (ValueError, :39-40). */
typedef enum {
  DSP_WAV_OK = 0,
  DSP_WAV_ERR_OPEN = 1,      /* cannot open / stat the file */
  DSP_WAV_ERR_NOT_RIFF = 2,  /* wave.Error: file does not start with RIFF id */
  DSP_WAV_ERR_NOT_WAVE = 3,  /* wave.Error: not a WAVE file */
  DSP_WAV_ERR_FORMAT = 4,    /* wave.Error: unknown format / unknown extended format */
  DSP_WAV_ERR_WIDTH = 5,     /* wave.Error: bad sample width */
  DSP_WAV_ERR_CHANNELS = 6,  /* wave.Error: bad # of channels */
  DSP_WAV_ERR_ORDER = 7,     /* wave.Error: data chunk before fmt chunk */
  DSP_WAV_ERR_MISSING = 8,   /* wave.Error: fmt chunk and/or data chunk missing */
  DSP_WAV_ERR_TRUNCATED = 9  /* EOFError inside the fmt chunk, or the payload could not be read */
} dsp_wav_status;

typedef struct {
  int32_t status;        /* dsp_wav_status */
  int32_t channels;      /* getnchannels() */
  int32_t sample_width;  /* getsampwidth(), bytes */
  int32_t sample_rate;   /* getframerate() */
  int64_t n_frames;      /* getnframes() */
  int64_t data_offset;   /* file offset of the PCM payload */
  int64_t data_bytes;    /* len(readframes(getnframes())): what the file really holds */
} dsp_wav_info;

/* Parse the headers of n_files files with `threads` host threads. */
int dsp_wav_scan(const char* const* paths, int64_t n_files, int32_t threads, dsp_wav_info* info);
/* Read the PCM payload of every file with status DSP_WAV_OK to dst + dst_byte_offsets[i]
 * (data_bytes[i] bytes each, as stored: little-endian int16 / uint8, interleaved channels).
 * dst is normally pinned memory from dsp_host_alloc, laid out for dsp_frontend_batch_host. */
int dsp_wav_read(const char* const* paths, int64_t n_files, int32_t threads, dsp_wav_info* info,
                 const int64_t* dst_byte_offsets, void* dst, int64_t dst_bytes);
/* Page-locked host memory for staging buffers (cudaHostAlloc / cudaFreeHost). */
int dsp_host_alloc(int64_t bytes, void** out);
int dsp_host_free(void* p);

#ifdef __cplusplus
}
#endif
#endif /* DSPFRONT_H_ */
