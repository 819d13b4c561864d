/*
 * wdx_b200.h — C ABI of the B200-native WarpDemuX classification path.
 *
 * Drop-in boundary: these entry points are what a ctypes/cffi binding inside
 * the reference would call instead of its CPU code.  Plain pointers and sizes,
 * no torch / numpy / C++ types.  Every data pointer may be HOST memory
 * (pageable or pinned) or DEVICE memory of the model's device; the library
 * asks the driver (cudaPointerGetAttributes) and stages copies itself.
 *
 * Return value: 0 on success, a negative wdx_status otherwise; the message is
 * available from wdx_last_error() (thread-local).  The library never aborts
 * and never falls back to a CPU implementation: without a usable CUDA device
 * every compute entry point returns WDX_ERR_CUDA.
 *
 * Thread-safety: a wdx_model handle owns device buffers and one internal
 * stream; calls on the SAME handle are serialised by an internal mutex, calls
 * on different handles run concurrently.  (The reference is re-entrant and is
 * called from worker processes / 4 live threads: one handle per worker.)
 */
#ifndef WDX_B200_H
#define WDX_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct wdx_model wdx_model;

typedef enum {
    WDX_OK = 0,
    WDX_ERR_INVALID = -1, /* bad argument (shape, dtype, NULL, k out of range) */
    WDX_ERR_CUDA = -2,    /* CUDA runtime error / no device */
    WDX_ERR_NOMEM = -3,
    WDX_ERR_UNSUPPORTED = -4
} wdx_status;

/* dtype tags for untyped buffers */
enum { WDX_F64 = 0, WDX_F32 = 1 };

/* Arithmetic mode of the DTW recurrence.
 *  EXACT_F64        float64, no FMA contraction: distances bit-identical to the
 *                   CPU restatement of dtaidistance's dtw_distance.
 *  FAST_F32         float32 with FMA: distances within 1e-5 relative.
 *  FAST_F32_GUARDED FAST_F32, then every read whose confidence margin lies
 *                   within `guard` of its threshold, or whose top-2 class
 *                   probabilities are within `guard`, is recomputed in
 *                   EXACT_F64 — labels/threshold decisions equal EXACT's. */
enum { WDX_MODE_EXACT_F64 = 0, WDX_MODE_FAST_F32 = 1, WDX_MODE_FAST_F32_GUARDED = 2 };

/* per-read status bits written to `flags` */
enum {
    WDX_FLAG_NONFINITE = 1, /* fingerprint or a kernel value was NaN/inf (sklearn would raise) */
    WDX_FLAG_RECOMPUTED = 2, /* GUARDED mode: this read was redone in EXACT_F64 */
    WDX_FLAG_GUARD_OVERFLOW = 4 /* GUARDED mode: more than max(4096, n/64) reads of a launch were near a
                                  boundary; this one kept its FAST_F32 result (re-run it in EXACT_F64) */
};

/* ---- model -------------------------------------------------------------
 * Replaces the state the reference keeps in a pickled DTW_SVM:
 *   warpdemux/models/dtw_base.py:13-25 (model, _X, label_mapper, thresholds,
 *   window, penalty), warpdemux/models/dtw_svm.py:26-30 (gamma, pwr_dist),
 *   sklearn SVC arrays walked by svm.cpp:2868-2896.
 *
 *   sv          [n_sv, L]        float64, support vectors, class-sorted (DTW_SVM._X)
 *   n_sv_class  [k]              SVC._n_support
 *   dual_coef   [k-1, n_sv]      SVC._dual_coef_, row-major
 *   rho         [k(k-1)/2]       -SVC._intercept_
 *   probA/probB [k(k-1)/2]       Platt coefficients
 *   thresholds  [k]              per-class confidence thresholds (DTW_SVM.thresholds)
 *   label_map   [k]              class index -> barcode label (noise = -1)
 *   window      Sakoe-Chiba window as dtaidistance defines it (|i-j| <= window-1); 0 = none
 *   penalty     NOT squared here (the library squares it, like dtaidistance)
 * All arrays are HOST pointers and are copied.  2 <= k <= 16, 1 <= L <= 64. */
int wdx_model_create(const double* sv, int n_sv, int L, const int32_t* n_sv_class, int k,
                     const double* dual_coef, const double* rho, const double* probA,
                     const double* probB, const double* thresholds, const int64_t* label_map,
                     int window, double penalty, double gamma, int pwr_dist, int device,
                     wdx_model** out);

void wdx_model_destroy(wdx_model* m);

/* Guard band of WDX_MODE_FAST_F32_GUARDED (default 5e-5; measured |conf_fast - conf_exact| <= 2e-6). */
int wdx_model_set_guard(wdx_model* m, double guard);

/* Reads per internal launch (default 2^22); bounds the scratch for the
 * one-vs-one decision sums (k(k-1)/2 doubles per read). */
int wdx_model_set_chunk_reads(wdx_model* m, int64_t chunk_reads);

/* How many contiguous ranges the support-vector list is cut into (grid.y).
 * 0 (default) = automatic: 1 for large batches, more for small ones so that a
 * 512-read live batch still fills the GPU.  With 1 the one-vs-one decision
 * sums are accumulated in exactly libsvm's order. */
int wdx_model_set_sv_splits(wdx_model* m, int splits);

/* ---- predict -------------------------------------------------------------
 * Replaces DTW_SVM.predict (warpdemux/models/dtw_svm.py:54-98):
 * distance_matrix_to (parallel_distances.py:58-67) -> pdist_kernel
 * (dtw_svm.py:21-22) -> SVC.predict_proba (svm.cpp:2921-2964) -> process_probs
 * (models/utils.py:45-61), fused on the device; the distance matrix is never
 * written to HBM unless `dist` is given.
 *
 *   X       [n, L]     fingerprints, x_dtype WDX_F64 or WDX_F32
 *   labels  [n]        int64 barcode labels (-1 = below threshold / noise)    (required)
 *   conf    [n]        float64 top1-top2 probability margin                    (or NULL)
 *   prob    [n, k]     float64 class probabilities                             (or NULL)
 *   flags   [n]        uint8 WDX_FLAG_* bits                                   (or NULL)
 *   dist    [n, n_sv]  float32 DTW distances as the reference casts them       (or NULL; debug/secondary seam)
 *   stream  cudaStream_t to launch on, or NULL for the handle's own stream.
 * The call returns after the results are complete, except when EVERY buffer
 * is device memory and `stream` is non-NULL: then the work is only enqueued
 * on `stream` (no host synchronisation).  Host input is staged through pinned
 * memory in chunks, the copy of chunk c+1 overlapping the kernels of chunk c. */
int wdx_predict(wdx_model* m, const void* X, int64_t n, int x_dtype, int mode,
                int64_t* labels, double* conf, double* prob, uint8_t* flags,
                float* dist, void* stream);

/* ---- distance matrix (secondary seam) ------------------------------------
 * Replaces warpdemux.parallel_distances.distance_matrix_to
 * (parallel_distances.py:48-84): DTW between every row of X [nX,L] and every
 * row of Y [nY,L] (float64 in), window/penalty as above.
 *   out_dtype WDX_F32: float32 [nX,nY], the reference's return dtype;
 *   out_dtype WDX_F64: float64 [nX,nY], the values before that cast
 *                      (bit-exact vs the CPU restatement in EXACT mode). */
int wdx_distance_matrix_to(const double* X, int64_t nX, const double* Y, int64_t nY, int L,
                           int window, double penalty, int mode, void* out, int out_dtype,
                           int device, void* stream);

/* ---- fingerprint extraction ------------------------------------------------
 * Replaces, for a whole minibatch at once, the reference's per-read loop over
 * barcode_fpt_wrapper -> detect_results_to_fpt (warpdemux/file_proc.py:418-428,
 * 188-224; warpdemux/sig_proc.py:394-605, non-consensus path): extract_adapter
 * (sig_proc.py:382-391), MAD winsorisation (:421-431), windowed t-test
 * (segmentation/_c_segmentation.pyx:124-161), scipy find_peaks + top-num_events
 * change points (sig_proc.py:176-198), segment means (_c_segmentation.pyx:41-53),
 * mean/std normalisation (sig_proc.py:99-111, 546-552), last barcode_num_events
 * (:569-594) and the six adapter statistics (:562-567).
 *
 * Configuration = the keys of the reference's SigProcConfig this path reads
 * (config/config_files/rna004_130bps@v1.0.toml:5-14; adapted
 * rna004_130bps@v0.2.4.toml:7).  Only sig_extract.normalization = "none",
 * segmentation.normalization = "mean", accept_less_cpts = false and
 * consensus_refinement = false are implemented (every shipped DTW-SVM model). */
typedef struct {
    int32_t padding;            /* sig_extract.padding                 (100) */
    double outlier_thresh;      /* core.sig_norm_outlier_thresh        (5.0) */
    int32_t min_obs_per_base;   /* segmentation.min_obs_per_base       (6)   */
    int32_t running_stat_width; /* segmentation.running_stat_width     (12)  */
    int32_t num_events;         /* segmentation.num_events             (110), <= 254 */
    int32_t barcode_num_events; /* segmentation.barcode_num_events     (25)  */
    int32_t max_slice_len;      /* longest adapter slice (adapter_end - adapter_start + 2*padding) to size the
                                   per-read shared memory for (14 B per sample; smaller = more reads per SM);
                                   0 = derive it from the batch: a host loop over host-resident bounds, or a
                                   small device reduction + 4-byte read back (a host sync) for device-resident
                                   bounds.  Hard limit 16000 samples. */
} wdx_fp_config;

/* per-read status written to `status` (0 = ReadResult.success) */
enum {
    WDX_FP_OK = 0,
    WDX_FP_FAIL_SEGMENTATION = 1, /* "event segmentation failed" (sig_proc.py:537-544): < num_events peaks */
    WDX_FP_FAIL_DETECT = 2,       /* detect_ok[r] == 0 (sig_proc.py:400-407) */
    WDX_FP_FAIL_NORMALIZE = 3,    /* "segment normalization failed" (sig_proc.py:553-560): NaN inside the adapter slice */
    WDX_FP_FAIL_TOO_LONG = 4,     /* adapter slice longer than the shared-memory limit */
    WDX_FP_FAIL_CONSENSUS = 5     /* "consensus query outlier" (sig_proc.py:500-521), consensus-guided mode only */
};

typedef struct wdx_fp wdx_fp;

int wdx_fp_create(const wdx_fp_config* cfg, int device, wdx_fp** out);
void wdx_fp_destroy(wdx_fp* f);
/* Second capacity for the rare long adapters (the LLR fallback can place an adapter end anywhere below
 * core.max_obs_trace, the CNN only below core.max_obs_adapter): with wdx_fp_config.max_slice_len > 0 and
 * len > max_slice_len, reads that do not fit the first pass are redone by a second launch with this capacity
 * instead of failing with WDX_FP_FAIL_TOO_LONG; all other reads keep the occupancy of the small capacity.  0 = off. */
int wdx_fp_set_long_slice_len(wdx_fp* f, int32_t len);
/* One-shot: the fingerprint pass of the NEXT wdx_fp_extract* / wdx_fp_predict call only revisits the reads whose entry in
 * `status` (device memory, written by an earlier call over the same batch) equals `status`; all other reads keep their
 * fingerprints and status.  Lets a caller fingerprint the reads that passed the boundary validation while the LLR
 * re-detection of the failed ones (combined.py:222-296) still runs, and come back for the rescued reads
 * (status WDX_FP_FAIL_DETECT = 2) afterwards.  0 = off. */
int wdx_fp_set_resume_status(wdx_fp* f, int32_t status);
/* Scalar promotion of the winsorisation bounds med -+ outlier_thresh * mad (warpdemux/sig_proc.py:421-431), where med and
 * mad are np.float32 scalars and outlier_thresh a Python float.  on = 0 (default): numpy >= 2 semantics (NEP 50), every
 * step in float32 — the numpy of this image, which the golden fixtures were written with.  on != 0: numpy < 2 semantics
 * (the reference's environment.yml pins numpy 1.26.4): the bounds are formed in float64 and rounded to float32 once by
 * np.clip.  The two differ by one float32 ulp of a bound for a fraction of the reads. */
int wdx_fp_set_numpy1_promotion(wdx_fp* f, int on);

/*   signals        [n, stride] float32 calibrated pA signal, one read per row (the reference's minibatch,
 *                  file_proc.py:333-354).  Rows may be NaN-padded at the end; the first NaN ends the read.
 *   sig_len        [n] int32 valid samples per row, or NULL
 *   adapter_start/adapter_end [n] int64   DetectResults.adapter_start / adapter_end
 *   detect_ok      [n] uint8 DetectResults.success, or NULL (all true)
 *   clip_in_place  != 0: write the winsorised adapter slice back into `signals`, as the reference's
 *                  in-place np.clip on its view does (sig_proc.py:426-431)
 *   fpt            [n, barcode_num_events] float64 (NaN rows for failed reads)           (required)
 *   dwell          [n, barcode_num_events] int64 dwell times of the kept events          (or NULL)
 *   stats          [n, 6] float64 adapter_dt_med, adapter_dt_mad, adapter_event_mean,
 *                  adapter_event_std, adapter_event_med, adapter_event_mad                (or NULL)
 *   status         [n] int32 WDX_FP_*                                                     (required)
 * Buffers may be host or device memory, as for wdx_predict. */
int wdx_fp_extract(wdx_fp* f, const float* signals, int64_t n, int64_t stride, const int32_t* sig_len,
                   const int64_t* adapter_start, const int64_t* adapter_end, const uint8_t* detect_ok,
                   int clip_in_place, double* fpt, int64_t* dwell, double* stats, int32_t* status,
                   void* stream);

/* ---- consensus-guided barcode refinement ("next" row: the tRNA fingerprint, BASELINE configs[3]) ----
 * Replaces `segment_signal_with_consensus_guided_barcode_refinement` + the consensus branch of
 * `detect_results_to_fpt` (warpdemux/sig_proc.py:257-378, 451-521; configuration
 * rna004_130bps@v1.0_tRNA.toml:13-29, refinement_optimal_cpts = false): adapter segmentation into
 * num_events + 1 events -> sub-sequence alignment of the consensus query against the mean-normalised
 * event means (dtaidistance warping_paths with penalty and start relaxation psi = (q, 0, s, 0), no
 * window; SubsequenceAlignment.best_match) -> sig_barcode_start -> second change-point selection on
 * the tail of the t-test scores (barcode_segm_events points, uncapped min_obs_per_base /
 * running_stat_width) -> event means normalised with the ADAPTER events' mean / std (normalize_wrt)
 * -> the last wdx_fp_config.barcode_num_events (= barcode_num_events[1]) -> outlier filter on the
 * match position.  After wdx_fp_set_consensus every wdx_fp_extract* / wdx_fp_predict call on the
 * handle runs this variant; query_len = 0 (or NULL) switches back.
 * Two inputs on which the reference itself raises instead of returning are reported as failed reads:
 * NaN padding inside the slice (WDX_FP_FAIL_NORMALIZE) and adapters so short that the adapter window
 * is narrower than running_stat_width (WDX_FP_FAIL_SEGMENTATION). */
typedef struct {
    const double* query;         /* warpdemux._consensus.ALL[consensus_model], HOST pointer (copied) */
    int32_t query_len;           /* <= 128 (84 for rna004_130bps_v1_0) */
    int32_t barcode_segm_events; /* segmentation.barcode_num_events[0]               (25)  */
    double penalty;              /* consensus_subseq_match_penalty                   (1.5) */
    int32_t psi_query_begin;     /* consensus_subseq_match_psi[0]                    (5)   */
    int32_t psi_series_begin;    /* consensus_subseq_match_psi[2]                    (40)  */
    int32_t ub_start;            /* consensus_subseq_match_ub_start                  (18)  */
    int32_t lb_end;              /* consensus_subseq_match_lb_end                    (69)  */
    int32_t ub_end;              /* consensus_subseq_match_ub_end                    (97)  */
} wdx_fp_consensus;

int wdx_fp_set_consensus(wdx_fp* f, const wdx_fp_consensus* c);

/* wdx_fp_extract plus `cons` [n, 3] int32: seg_cons_query_start, seg_cons_query_end, sig_barcode_start
 * (ReadResult fields, sig_proc.py:595-604); NULL unless the handle is in consensus-guided mode. */
int wdx_fp_extract_ex(wdx_fp* f, const float* signals, int64_t n, int64_t stride, const int32_t* sig_len,
                      const int64_t* adapter_start, const int64_t* adapter_end, const uint8_t* detect_ok,
                      int clip_in_place, double* fpt, int64_t* dwell, double* stats, int32_t* status,
                      int32_t* cons, void* stream);

/* Fused minibatch step (file_proc.py:418-450): fingerprints never leave the
 * device between extraction and wdx_predict.  Failed reads get label -1, NaN
 * confidence/probabilities and WDX_FLAG_NONFINITE.  `fpt` may be NULL. */
int wdx_fp_predict(wdx_fp* f, wdx_model* m, const float* signals, int64_t n, int64_t stride,
                   const int32_t* sig_len, const int64_t* adapter_start, const int64_t* adapter_end,
                   const uint8_t* detect_ok, int mode, int64_t* labels, double* conf, double* prob,
                   uint8_t* flags, double* fpt, int32_t* status, void* stream);

/* Device time (ms) and launch count of the fingerprint kernel in the last call on this handle. */
int wdx_fp_enable_timing(wdx_fp* f, int on);
int wdx_fp_last_kernel_ms(wdx_fp* f, double* ms, int* launches);

/* ---- adapter / poly(A) boundary CNN ("next" row: the step before the fingerprint stage) -------------
 * Replaces adapted.detect.cnn.cnn_detect (warpdemux/adapted/adapted/detect/cnn.py:165-183) for a whole
 * minibatch: prepare_data (cnn.py:71-85: zero-padded block-mean downscaling, downscale.py:4-41; float32
 * nanmedian / MAD normalisation; NaN -> -5), the BoundariesCNN forward (cnn.py:16-52) and cnn_predict
 * (cnn.py:104-162: argmax of channel 0 over the adapter range, masked argmax of channel 1, scipy
 * find_peaks(distance=5) on the FLATTENED batch, top polya_cand_k peaks per read, including the
 * reference's row shift when a read has no peak).
 *
 * Weights are the tensors of the reference's torch state dict (adapted/models/rna004_130bps@v0.2.4.pth),
 * float32, torch layouts, HOST pointers (copied):
 *   w0 [64,1,7] b0 [64]   Conv1d(1,64,7,stride 3,padding 3)
 *   w1 [64,64,7] b1 [64]  Conv1d(64,64,7,padding 3)
 *   w2 [64,64,7] b2 [64]  Conv1d(64,64,7,padding 3)
 *   w3 [64,2,7] b3 [2]    ConvTranspose1d(64,2,7,stride 3,padding 3)
 * Only this architecture (channels 64, kernel 7) is implemented. */
typedef struct {
    int32_t min_obs_adapter;   /* core.min_obs_adapter            (1000) */
    int32_t max_obs_adapter;   /* core.max_obs_adapter            (6500) */
    int32_t downscale_factor;  /* core.downscale_factor           (10), <= 128 */
    int32_t polya_cand_k;      /* cnn_boundaries.polya_cand_k     (5 for WarpDemuX, 10 for ADAPTed), 2..16 */
    int32_t channels;          /* 64 */
    int32_t kernel_size;       /* 7  */
} wdx_cnn_config;

/* Arithmetic of the two 64->64 convolutions (97 % of the work):
 *  EXACT_F32   float32 FMA on the CUDA cores (the reference computes in float32 on the CPU; results
 *              agree to summation order).
 *  FAST_TC     tcgen05 tensor cores: activations and weights split into fp16 high + low parts, three
 *              products per term accumulated in float32 (error ~2^-21 relative, float32-class).
 *  GUARDED     FAST_TC, then every read whose argmax decisions have a top-2 margin below the guard, or
 *              whose activations left the fp16 range, is recomputed in EXACT_F32. */
enum { WDX_CNN_EXACT_F32 = 0, WDX_CNN_FAST_TC = 1, WDX_CNN_GUARDED = 2 };

/* per-read bits written to `flags` */
enum {
    WDX_CNN_FLAG_NONFINITE = 1,  /* a score was NaN/inf (degenerate input, e.g. MAD = 0) */
    WDX_CNN_FLAG_RECOMPUTED = 2, /* GUARDED: redone in EXACT_F32 */
    WDX_CNN_FLAG_CHAIN = 4,      /* peak-distance suppression depended on samples beyond the 64-sample halo
                                    around the read; candidates of this read may differ from scipy's */
    WDX_CNN_FLAG_RANGE = 8       /* FAST_TC: an activation exceeded the fp16 range (re-run in EXACT_F32) */
};

typedef struct wdx_cnn wdx_cnn;

int wdx_cnn_create(const wdx_cnn_config* cfg, const float* w0, const float* b0, const float* w1, const float* b1,
                   const float* w2, const float* b2, const float* w3, const float* b3, int device, wdx_cnn** out);
void wdx_cnn_destroy(wdx_cnn* c);

/*   signals [n, stride] float32 calibrated pA rows, NaN padded (the reference's minibatch, file_proc.py:241-262)
 *   preds   [n, 1 + polya_cand_k] int64: adapter end, poly(A) end candidates (samples; 0 = none)   (required)
 *   scores  [n, 2, To] float32 raw CNN output, To = 3*((T-1)/3+1)-2, T = ceil((stride-min_obs_adapter)/factor)  (or NULL)
 *   flags   [n] uint8 WDX_CNN_FLAG_*                                                               (or NULL)
 * Buffers may be host or device memory.  The whole call is ONE flattened batch for the peak search. */
int wdx_cnn_detect(wdx_cnn* c, const float* signals, int64_t n, int64_t stride, int mode, int64_t* preds,
                   float* scores, uint8_t* flags, void* stream);
/* prepare_data alone (cnn.py:71-85): x [n, T] float32, the CNN input (bit-identical to the numpy chain). */
int wdx_cnn_prepare(wdx_cnn* c, const float* signals, int64_t n, int64_t stride, float* x, void* stream);
/* cnn_predict alone (cnn.py:104-162) on given scores [n, 2, t_out] float32.  scaled == 0: downscaled positions as
 * cnn_predict returns them; scaled != 0: samples, with the == min_obs_adapter -> 0 rule of cnn_detect (cnn.py:176-181). */
int wdx_cnn_predict(wdx_cnn* c, const float* scores, int64_t n, int32_t t_out, int scaled, int64_t* preds, uint8_t* flags,
                    void* stream);
/* Length To of the score rows for a given row stride. */
int wdx_cnn_score_len(wdx_cnn* c, int64_t stride, int32_t* t_in, int32_t* t_out);
int wdx_cnn_set_guard(wdx_cnn* c, double guard);
/* Device time (ms) of the convolution kernels in the last wdx_cnn_detect on this handle, and their launch count. */
int wdx_cnn_enable_timing(wdx_cnn* c, int on);
int wdx_cnn_last_kernel_ms(wdx_cnn* c, double* ms, int* launches);

/* ---- validation of the CNN's boundary predictions (the step between wdx_cnn_detect and wdx_fp_extract) ----
 * Replaces adapted.detect.combined.validate_boundaries (warpdemux/adapted/adapted/detect/combined.py:409-683)
 * as combined_detect_cnn calls it for every read of a minibatch (combined.py:211-221):
 *   validate_boundaries(signal[:full_signal_len], Boundaries(0, pred[0], pred[1], pred[1:]), spc, full_signal_len)
 * i.e. adapter median / MAD range check, open-pore detection (anomalies.py:16-35: adapter_start moves to the last
 * open-pore sample), real_range_check (real_range.py:34-63), mean_var_shift_polyA_check over the poly(A)
 * candidates (mvs.py:42-159) and the optional median-shift check.  mvs_detect_overwrite = true is not implemented
 * (WDX_ERR_UNSUPPORTED); the partition statistics of DetectResults come from wdx_validate_run_ex.
 * Reads that fail are the ones the reference hands to its LLR fallback (combined.py:222-290) - that stays with the
 * caller.  Ranges are [lo, hi] with -INFINITY / INFINITY for "None". */
typedef struct {
    int32_t min_obs_adapter;          /* core.min_obs_adapter                     (1000) */
    int32_t detect_open_pores;        /* real_range.detect_open_pores             (1) */
    int32_t real_signal_check;        /* real_range.real_signal_check             (1) */
    int32_t mean_window;              /* real_range.mean_window                   (300) */
    int32_t max_obs_local_range;      /* real_range.max_obs_local_range           (5000) */
    int32_t open_pore_min_obs_diff;   /* find_open_pores(min_obs_diff)            (10) */
    double open_pore_min;             /* find_open_pores(sig_range[0])            (200.0) */
    double mean_start_range[2], mean_end_range[2], local_range[2], adapter_mad_range[2];
    int32_t mvs_detect_check;         /* mvs_polya.mvs_detect_check               (1) */
    int32_t mvs_detect_overwrite;     /* must be 0 */
    int32_t pA_mean_window;           /* (20) */
    int32_t pA_var_window;            /* (100) */
    int32_t median_shift_window;      /* (1000) */
    int32_t detect_med_shift;         /* med_shift.detect_med_shift               (0) */
    int32_t med_shift_window;         /* (2000) */
    int32_t reserved;
    double pA_var_range[2], median_shift_range[2], polyA_med_range[2], polyA_local_range[2];
    double pA_mean_range[2];                     /* used when not (-inf, inf) */
    double pA_mean_adapter_med_scale_range[2];   /* else this range times the adapter median (combined.py:505-519) */
    double med_shift_range[2];
} wdx_validate_config;

/* info[.][0]: 0 = success, else the reference's fail_reason */
enum {
    WDX_VAL_OK = 0,
    WDX_VAL_NO_ADAPTER = 1,     /* "No adapter detected (primary)" */
    WDX_VAL_ADAPTER_MAD = 2,    /* "adapter MAD check failed" */
    WDX_VAL_OPEN_PORE = 3,      /* "Open pore too close to boundary" */
    WDX_VAL_REAL_RANGE = 4,     /* "Real signal check failed" */
    WDX_VAL_NO_POLYA = 5,       /* "No polya detected (primary)" */
    WDX_VAL_MVS_NO_SIGNAL = 6,  /* "MVS polya check failed: not enough signal" */
    WDX_VAL_MVS_CHECKS = 7,     /* "MVS polya check failed: " + names of the checks whose bit in info[.][1] is clear */
    WDX_VAL_MED_SHIFT = 8,      /* "Median shift check failed" */
    WDX_VAL_HAS_NAN = 9         /* the ValueError of combined.py:416-418 ("Signal contains nan values") */
};
#define WDX_VAL_NVALS 12

typedef struct wdx_validate wdx_validate;

int wdx_validate_create(const wdx_validate_config* cfg, int device, wdx_validate** out);
void wdx_validate_destroy(wdx_validate* v);
/*   signals  [n, stride] float32 calibrated pA rows, NaN padded (file_proc.py:241-262)
 *   full_len [n] int32 full_signal_lens (may exceed stride)
 *   preds    [n, ld] int64 wdx_cnn_detect's output: adapter end, poly(A) end candidates (0 = none)
 *   success  [n] uint8 DetectResults.success
 *   info     [n, 4] int32: fail code (WDX_VAL_*), check bits (bit0 mean, 1 var, 2 med, 3 range, 4 shift: set = passed),
 *            number of open pores kept, 0
 *   bounds   [n, 3] int64 adapter_start, adapter_end, polya_end (DetectResults fields)
 *   vals     [n, WDX_VAL_NVALS] float64 or NULL: adapter median, adapter MAD (as thresholded), real_adapter_mean_start,
 *            real_adapter_mean_end, real_adapter_local_range, mvs_detect_mean_at_loc, mvs_detect_var_at_loc,
 *            mvs_detect_polya_med, mvs_detect_polya_local_range, mvs_detect_med_shift, adapter_rna_median_shift, NaN;
 *            NaN where the reference leaves None
 * Buffers may be host or device memory; stride * 4 bytes must fit in shared memory (<= ~54 000 samples). */
int wdx_validate_run(wdx_validate* v, const float* signals, int64_t n, int64_t stride, const int32_t* full_len,
                     const int64_t* preds, int32_t ld, uint8_t* success, int32_t* info, int64_t* bounds, double* vals,
                     void* stream);
/* As wdx_validate_run, plus the partition statistics of DetectResults (adapted/partition/signal_partitions.py:65-96,
 * combined.py:631-636) when `parts` is not NULL:
 *   parts [n, WDX_VAL_NPART] float64: for the adapter [adapter_start, adapter_end), poly(A) [adapter_end, polya_end) and
 *   preloaded-RNA [polya_end, len) partitions: start, len, mean, std, med, mad (float32 numpy arithmetic, widened);
 *   NaN where the reference leaves None (empty partition, or the NaN-signal error). */
#define WDX_VAL_NPART 18
int wdx_validate_run_ex(wdx_validate* v, const float* signals, int64_t n, int64_t stride, const int32_t* full_len,
                        const int64_t* preds, int32_t ld, uint8_t* success, int32_t* info, int64_t* bounds, double* vals,
                        double* parts, void* stream);
/* As wdx_validate_run_ex, plus DetectResults.open_pores when `open_pores` is not NULL (the column of the reference's
 * detected_boundaries_*.csv.gz / failed_reads_*.csv.gz, adapted/output.py:26-51):
 *   open_pores [n, WDX_VAL_PORES_LD] int32: [0] = number of positions find_open_pores(...).ravel() returns
 *   (anomalies.py:16-35, combined.py:469-477; -1 = None: the step did not run for this read), [1 ..] the positions in
 *   ascending order (at most WDX_VAL_PORES_LD - 1 of them are stored). */
#define WDX_VAL_PORES_LD 64
int wdx_validate_run_report(wdx_validate* v, const float* signals, int64_t n, int64_t stride, const int32_t* full_len,
                            const int64_t* preds, int32_t ld, uint8_t* success, int32_t* info, int64_t* bounds, double* vals,
                            double* parts, int32_t* open_pores, void* stream);
/* on != 0: stop at the first failing poly(A) candidate.  success and bounds are unchanged (the reference never sets
 * `success` back to True after a failed candidate, combined.py:540-610); the fail code, check bits and mvs_* values are
 * those of the FIRST failing candidate instead of the last one evaluated.  For callers that only need the verdict (the
 * fingerprint stage); default off = reference-identical report. */
int wdx_validate_set_verdict_only(wdx_validate* v, int on);
/* One-shot, for the NEXT wdx_validate_run*: right behind the first validation pass — before the LLR re-detection of the
 * failed reads (wdx_validate_set_llr) is queued — `success` is copied to `success_snapshot` ([n] uint8, device memory) and
 * `event` (a cudaEvent_t, may be NULL) is recorded on the call's stream.  The reads that passed are final at that point
 * (the re-detection only revisits failed reads: combined.py:222), so a caller may hand them to the next stage on another
 * stream while the tail still runs.  NULL, NULL = off. */
int wdx_validate_set_early(wdx_validate* v, uint8_t* success_snapshot, void* event);
int wdx_validate_enable_timing(wdx_validate* v, int on);
int wdx_validate_last_kernel_ms(wdx_validate* v, double* ms, int* launches);

/* ---- LLR fallback of the boundary detection -------------------------------------------------------------------
 * Replaces the re-detection branch of adapted.detect.combined.combined_detect_cnn
 * (warpdemux/adapted/adapted/detect/combined.py:222-296) for the reads whose CNN boundaries fail validation:
 *   normalize_signal(row[:min(max_obs_trace, full_len)])                          detect/normalize.py:15-63
 *   "hail mary" (cnn_boundaries.fallback_to_llr_short_reads, combined.py:232-274): for short reads with a long
 *       CNN poly(A) stretch the poly(A) end is re-detected on [cnn adapter_end, cnn polya_end) by an LLR trace
 *       (detect/llr.py:243-334, _c_llr.pyx:66-88) + detect_full_polya_trace_peak_with_spike (llr.py:385-455);
 *       the re-validated result REPLACES the read's result, success or not
 *   full LLR (cnn_boundaries.fallback_to_llr, combined.py:275-290): detect_llr_on_downscaled_signal
 *       (combined.py:39-129: adapter end = first peak of the LLR trace by scipy find_peaks(width, prominence x nanstd,
 *       rel_height), corrected for plateaus and split peaks, llr.py:124-240; poly(A) end as above); its validated
 *       result replaces the read's result only if it SUCCEEDS.
 * After wdx_validate_set_llr(v, cfg) every wdx_validate_run / wdx_validate_run_ex call performs this branch on the
 * device behind the validation of the given boundaries (two llr_kernel + two masked validate_kernel launches, no
 * host round trip); cfg = NULL switches it off again.  info[.][3] then reports, per read:
 *   bits 0-1  which boundaries the reported result validated: 0 = the given (CNN) ones, 1 = hail mary, 2 = full LLR
 *             (for 1 and 2 DetectResults.llr_adapter_end / llr_polya_end are bounds[.][1] / bounds[.][2] and the
 *             reference's primary_method of that result is "llr")
 *   bit 2     the hail-mary re-detection ran, bit 3 the full LLR detection ran.
 * Two more fail codes appear in info[.][0]: */
enum {
    WDX_VAL_MAD_ZERO = 10,   /* "MAD normalization failed: scale is 0" (normalize.py:55-58), the read's whole result */
    WDX_VAL_LLR_ERROR = 11   /* reserved: other exceptions of the fallback branch */
};
typedef struct {
    int32_t max_obs_trace;             /* core.max_obs_trace                       (10000 WarpDemuX, 16000 ADAPTed) */
    int32_t min_obs_adapter;           /* core.min_obs_adapter                     (1000) */
    int32_t max_obs_adapter;           /* core.max_obs_adapter                     (6500) */
    int32_t downscale_factor;          /* core.downscale_factor                    (10) */
    double sig_norm_outlier_thresh;    /* core.sig_norm_outlier_thresh             (5.0) */
    double adapter_peak_prominence;    /* llr_boundaries.adapter_peak_prominence   (1.0) */
    double adapter_peak_rel_height;    /* llr_boundaries.adapter_peak_rel_height   (1.0) */
    int32_t adapter_peak_width;        /* llr_boundaries.adapter_peak_width        (1000) */
    int32_t fallback_to_llr;           /* cnn_boundaries.fallback_to_llr           (1) */
    int32_t fallback_to_llr_short_reads; /* cnn_boundaries.fallback_to_llr_short_reads (1) */
    int32_t reserved;
} wdx_llr_config;
int wdx_validate_set_llr(wdx_validate* v, const wdx_llr_config* cfg);

/* ---- raw ADC samples -> calibrated pA minibatch rows on the device --------------------------------------------
 * The reference's loader hands float32 pA rows to the worker (pod5 `signal_pa` = (adc + calibration_offset) *
 * calibration_scale in float32, rows NaN padded to sig_preload_size; file_proc.py:227-262).  Shipping the int16 ADC
 * samples and calibrating after the upload halves the bytes that cross PCIe; results are bit-identical.
 *   adc [n, stride_in] int16, n_valid [n] int32 samples present per row, offset / scale [n] float32,
 *   out [n, stride_out] float32 (NaN from n_valid on).  DEVICE pointers; asynchronous on `stream`. */
int wdx_calibrate_rows(const int16_t* adc, int64_t n, int64_t stride_in, const int32_t* n_valid, const float* offset,
                       const float* scale, float* out, int64_t stride_out, int device, void* stream);

/* ---- pod5 VBZ signal -> int16 ADC rows on the device ----------------------------------------------------------
 * A pod5 signal chunk is zstd( streamvbyte16( zigzag( delta( int16 )))), one zstd frame per chunk (RFC 8878).  The
 * chunks go to the device still compressed; one warp decodes one frame, one CTA turns one read's chunks into its row.
 * Supported zstd subset: one frame per chunk (single-segment or with a window descriptor, with or without
 * Frame_Content_Size), raw / RLE / compressed blocks, raw / RLE / Huffman (1 or 4 streams) / treeless literals,
 * predefined / RLE / FSE / repeat sequence tables.  Anything else is a per-chunk status, never a fault: */
enum {
    WDX_VBZ_OK = 0,
    WDX_VBZ_BAD_MAGIC = 1,   /* not a zstd frame */
    WDX_VBZ_DICTIONARY = 2,  /* the frame names a dictionary */
    WDX_VBZ_CHECKSUM = 3,    /* content checksum flag set (not verified, so not accepted) */
    WDX_VBZ_RESERVED = 4,    /* reserved header bit, block type or field */
    WDX_VBZ_TRUNCATED = 5,   /* the input ends inside the frame */
    WDX_VBZ_CORRUPT = 6,     /* inconsistent table description, bitstream, offset or size */
    WDX_VBZ_TOO_LARGE = 7,   /* content larger than the output capacity (rows: the svb16 bound ceil(s/8) + 2 s) */
    WDX_VBZ_FRAMES = 8,      /* skippable frame, or bytes after the frame (a second frame) */
    WDX_VBZ_SAMPLES = 9,     /* rows: the key / data lengths disagree with the chunk's `samples` */
    WDX_VBZ_SCRATCH = 10     /* rows: a chunk's scratch region is misaligned or smaller than it needs */
};
/* Decompress m frames: frame i = src[chunk_off[i], chunk_off[i+1]) -> scratch[scratch_off[i], scratch_off[i+1]).
 * Decoding stops once limit[i] bytes exist (a prefix); content that exceeds the region while limit[i] is larger is
 * WDX_VBZ_TOO_LARGE.  produced [m] int64 = bytes written (0 unless status is WDX_VBZ_OK), status [m] int32.
 * DEVICE pointers; asynchronous on `stream`. */
int wdx_zstd_decompress(const uint8_t* src, const int64_t* chunk_off, int64_t m, const int64_t* limit, uint8_t* scratch,
                        const int64_t* scratch_off, int64_t* produced, int32_t* status, int device, void* stream);
/* n reads of VBZ chunks -> int16 rows [n, stride]: read r = chunks [read_chunks[r], read_chunks[r+1]) in order, chunk c
 * holds samples[c] samples; each chunk's delta sum restarts at 0 (pod5 decodes chunks independently).  Only the prefix
 * of a chunk the row needs is decompressed.  Chunk c's scratch region [scratch_off[c], scratch_off[c+1]) must start
 * 16-byte aligned and hold 16 + ceil(s/8) + 2 min(s, stride - first sample of c) bytes.  n_valid [n] int32 =
 * min(sum of the read's samples, stride); samples beyond it are 0.  status [n] int32 = the first WDX_VBZ_* of the
 * read's chunks; a read with a non-zero status has n_valid 0 and a zero row.  DEVICE pointers; asynchronous. */
int wdx_vbz_decode_rows(const uint8_t* src, const int64_t* chunk_off, const int32_t* samples, int64_t m, const int64_t* read_chunks,
                        int64_t n, uint8_t* scratch, const int64_t* scratch_off, int16_t* rows, int64_t stride, int32_t* n_valid,
                        int32_t* status, int device, void* stream);

/* ---- introspection -------------------------------------------------------- */
const char* wdx_last_error(void);
int wdx_device_count(void);
/* Kernels launched by this library in this process so far (for bench accounting). */
int64_t wdx_kernel_launch_count(void);
/* Device time (ms) the dominant fused DTW+SVC kernel took in the last
 * wdx_predict on this handle, and how many launches that covered; measured
 * with CUDA events on the handle's stream when timing is enabled. */
int wdx_model_enable_timing(wdx_model* m, int on);
int wdx_model_last_kernel_ms(wdx_model* m, double* ms, int* launches);
/* Same, restricted to the launches of one arithmetic (exact != 0: EXACT_F64
 * launches, e.g. the GUARDED re-run; exact == 0: FAST_F32 launches). */
int wdx_model_last_kernel_ms_mode(wdx_model* m, int exact, double* ms, int* launches);
const char* wdx_version(void);

#ifdef __cplusplus
}
#endif
#endif /* WDX_B200_H */
