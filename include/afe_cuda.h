/*
 * afe_cuda.h — C ABI of the B200-native MFCC front end (libafe_cuda.so).
 *
 * Drop-in boundary for the ONE hot path of mankeyboy/ASR-FeatExt-OpenCL:
 *   int16 PCM -> segment+window -> real FFT -> |X|/N2 -> mel+log -> DCT-II(+lifter) -> delta/delta-delta -> CMN/CVN/MINMAX.
 * Every entry point names the reference interface it replaces (paths relative to the reference tree).
 * Plain pointers and sizes only; no C++/torch types. All functions return 0 on success, non-zero on error
 * (message via afe_last_error(), thread local) unless documented otherwise. No exceptions cross this boundary;
 * the C++ mirror classes in asr-featext-opencl_b200/host/ rethrow std::runtime_error with the reference's messages.
 *
 * There is NO CPU fallback: every compute entry point fails loudly when no CUDA device / kernel image is usable.
 * Handles are not thread-safe; one CUDA stream per handle (reference: one in-order queue per object, mfccopencl.cpp:149).
 */
#ifndef AFE_CUDA_H_
#define AFE_CUDA_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* 2: Normalizer-owned corpus verbs (afe_normalizer_accumulate / allreduce / finalize / apply; afe_normalizer_allreduce now takes
 *    the Normalizer, afe_batch_normalizer() hands out the batch's), pre-emphasis setters, afe_build_flags, the streaming
 *    object runs on the fused kernel, AFE_BATCH_WS_KERNEL / AFE_BATCH_FAST_MATH removed. */
/* 3: the tensor-core phase-2 flag (64) removed; afe_batch_set_options refuses flag bits outside AFE_BATCH_Q1_EXACT |
 *    AFE_BATCH_NO_TMA | AFE_BATCH_UNFUSED_NORM | AFE_BATCH_NO_CLUSTER. */
#define AFE_ABI_VERSION 3

/* normalizer.h:5 */
enum afe_norm { AFE_NORM_NONE = 0, AFE_NORM_CMN = 1, AFE_NORM_CVN = 2, AFE_NORM_MINMAX = 3 };
/* parambase.h:9 */
enum afe_dyn { AFE_DYN_NONE = 0, AFE_DYN_DELTA = 1, AFE_DYN_ACC = 2 };

/* The 15 constructor arguments of MfccBase / MfccOpenCL in declaration order (mfccbase.h:21-35, mfccopencl.h:45-60). */
typedef struct afe_params {
    int input_buffer_size; /* samples per set_input() block ("sample_limit") */
    int window_size;       /* W, samples */
    int shift;             /* S, samples */
    int num_banks;
    float sample_rate;
    float low_freq;
    float high_freq;
    int ceps_len;          /* 0 -> log-mel (FBANK) output */
    int want_c0;           /* c0 is the LAST static column (mfcccpu.cpp:133-135) */
    float lift_coef;
    int norm;              /* enum afe_norm */
    int dyn;               /* enum afe_dyn */
    int delta_l1;
    int delta_l2;
    int norm_after_dyn;
} afe_params;

const char *afe_last_error(void);
int afe_abi_version(void);
/* bit 0: built with -DAFE_DEVTOOLS (timing hooks read from the environment; never in a product build) */
int afe_build_flags(void);
/* number of visible CUDA devices; 0 with an error string when the driver/runtime is unusable */
int afe_device_count(void);

/* ------------------------------------------------------------------------------------------------------------------
 * Host-side table builders (pure host code; same float/double expression order as the reference so that filter
 * edges can never disagree). Usable without a GPU.
 * ---------------------------------------------------------------------------------------------------------------- */
/* ParamBase::estimated_window_count (parambase.cpp:16-19) */
int afe_estimated_window_count(int samples, int window_size, int shift);
/* MfccBase::get_output_data_width (mfccbase.cpp:33-43) */
int afe_output_width(const afe_params *p);
/* ceil2(window_size) (mfcccpu.cpp:10-20,94) */
int afe_fft_size(int window_size);
/* window synthesis of the reference driver (ASR_OCL.cpp:149-152): (0.56-0.46cos(2 pi i/W))/32768 */
void afe_make_window(float *window, int window_size);
/* MfccCpu::refresh_filters (mfcccpu.cpp:24-60): edges[num_banks+2], filters[2*N2] (even/odd interleaved rows) */
int afe_build_filters(const afe_params *p, float alpha, int *edges, float *filters);
/* DCT-II + lifter matrix (mfcccpu.cpp:118-136): dct[num_banks][dct_len], dct_len = ceps_len + want_c0 */
int afe_build_dct(const afe_params *p, float *dct);

/* ------------------------------------------------------------------------------------------------------------------
 * Streaming MFCC object — replaces `new MfccOpenCL(... 15 args ..., cl_device_id)` (mfccopencl.h:45-73) and is
 * driven exactly like ParamBase (parambase.h:23-32): set_window -> {set_input -> [set_alpha ->] apply ->
 * get_output}* -> flush -> apply -> get_output (ASR_OCL.cpp:152,234-243,268-278).
 * Numerics follow the CPU class MfccCpu (the OpenCL class is not a valid oracle, SURVEY F3), including the
 * single-block flush quirk Q1 unless AFE_OPT_FIX_FLUSH_STATICS is set.
 * ---------------------------------------------------------------------------------------------------------------- */
typedef struct afe_mfcc afe_mfcc;

int afe_mfcc_create(const afe_params *p, int cuda_device, afe_mfcc **out);        /* MfccOpenCL::MfccOpenCL */
void afe_mfcc_destroy(afe_mfcc *h);                                               /* ~MfccOpenCL */
int afe_mfcc_set_window(afe_mfcc *h, const float *window);                        /* ParamBase::set_window */
int afe_mfcc_set_alpha(afe_mfcc *h, float alpha);                                 /* ParamBase::set_alpha (VTLN) */
/* Per-frame pre-emphasis before the window: y[j] = x[j] - c*x[j-1], y[0] = (1-c)*x[0]. The reference has none
 * (segmentercpu.cpp:21-27): the default 0 is its behaviour, bit for bit. 0 <= c < 1. */
int afe_mfcc_set_preemphasis(afe_mfcc *h, float coefficient);
int afe_mfcc_input_buffer_size(const afe_mfcc *h);                                /* ParamBase::get_input_buffer_size */
int afe_mfcc_estimated_window_count(const afe_mfcc *h, int samples);              /* ParamBase::estimated_window_count */
int afe_mfcc_output_width(const afe_mfcc *h);                                     /* get_output_data_width */
/* *frames = rows ready (0 allowed). Data is copied before return. Error if samples > input_buffer_size
 * ("Can't process data, buffer is too small", mfcccpu.cpp:338-339). */
int afe_mfcc_set_input(afe_mfcc *h, const int16_t *data, int samples, int *frames);
int afe_mfcc_flush(afe_mfcc *h, int *frames);                                     /* ParamBase::flush; second call -> 0 */
int afe_mfcc_apply(afe_mfcc *h);                                                  /* ParamBase::apply */
/* out: caller-owned frames*width floats, row-major [static | delta | delta-delta] (mfcccpu.cpp:427-444).
 * Error "Window count too high" if frames exceeds the object's capacity. */
int afe_mfcc_get_output(afe_mfcc *h, float *out, int frames);
/* The reference never clears m_last_block (Q3): one object per utterance. reset() makes the handle reusable. */
int afe_mfcc_reset(afe_mfcc *h);
enum afe_mfcc_option {
    AFE_OPT_FIX_FLUSH_STATICS = 1,
    AFE_OPT_STAGED_KERNELS = 2     /* A-B test: one kernel per reference stage instead of the fused kernel; before set_window */
};
int afe_mfcc_set_option(afe_mfcc *h, int option, int value);
/* 1 when the object's blocks run through the fused kernel (one launch per apply()), 0 when the parameter set needs the
 * staged kernels (FFT sizes other than 256/512, odd shift, normalisation before the deltas, ...). Both run on the GPU. */
int afe_mfcc_uses_fused_kernel(const afe_mfcc *h);
int afe_mfcc_kernel_launches(const afe_mfcc *h); /* fused-kernel launches since creation */

/* ------------------------------------------------------------------------------------------------------------------
 * Stage objects with device buffers (the `cl_mem` arguments of the OpenCL variants become device pointers).
 * ---------------------------------------------------------------------------------------------------------------- */
typedef struct afe_segmenter afe_segmenter;   /* SegmenterOpenCL (segmenteropencl.h:27-42) */
int afe_segmenter_create(int window_size, int shift, int window_limit, int deltasize, int cuda_device,
                         afe_segmenter **out);                                    /* ::init */
void afe_segmenter_destroy(afe_segmenter *s);                                     /* ::cleanup */
int afe_segmenter_set_window(afe_segmenter *s, const float *window);
int afe_segmenter_set_preemphasis(afe_segmenter *s, float coefficient);           /* see afe_mfcc_set_preemphasis */
/* d_out: DEVICE float[window_count_no_delta][ceil2(W)], zero padded beyond W */
int afe_segmenter_set_input(afe_segmenter *s, const int16_t *data_in, float *d_out, int samples,
                            int *window_count, int *window_count_no_delta);
int afe_segmenter_flush(afe_segmenter *s, float *d_out, int *window_count, int *window_count_no_delta);
int afe_segmenter_remaining_samples(const afe_segmenter *s);
int afe_segmenter_samples(const afe_segmenter *s);
int afe_segmenter_is_flushed(const afe_segmenter *s);
int afe_segmenter_was_flushed(const afe_segmenter *s);

typedef struct afe_delta afe_delta;           /* DeltaOpenCL (deltaopencl.h:17-22) */
int afe_delta_create(int dim, int window_limit, int delta_size, int cuda_device, afe_delta **out);
void afe_delta_destroy(afe_delta *d);
/* d_data: DEVICE float[window_count + 2*delta_size][dim]; result in afe_delta_output() [window_count][dim] */
int afe_delta_apply(afe_delta *d, const float *d_data, int window_count);
float *afe_delta_output(afe_delta *d);        /* DEVICE pointer (get_output_buffer) */

typedef struct afe_normalizer afe_normalizer; /* NormalizerOpenCL (normalizeropencl.h:25-28) */
int afe_normalizer_create(int norm_type, int dim, int cuda_device, afe_normalizer **out);
void afe_normalizer_destroy(afe_normalizer *n);
/* in place on DEVICE float[window_count][dim] starting `offset` floats into d_data; stats in double */
int afe_normalizer_normalize(afe_normalizer *n, float *d_data, int offset, int window_count, int use_last_stats);
/* Corpus-level CMVN: the three kernels of NormalizerOpenCL::normalize (norm.cl kernelSum :1-40, kernelFinalizeSum :42-78,
 * kernelNormalize :80-125; normalizeropencl.cpp:123-158) as separate verbs on the Normalizer's running record, with the
 * ONE collective of the path between the first two. Record = sum[dim] | sumsq[dim] | count | min[dim] | max[dim] doubles.
 *   reset -> accumulate (any number of blocks / shards) -> allreduce (all ranks) -> finalize -> apply (any number of blocks) */
int afe_normalizer_stats_len(const afe_normalizer *n);                            /* 4*dim + 1 */
int afe_normalizer_reset(afe_normalizer *n);
int afe_normalizer_accumulate(afe_normalizer *n, const float *d_data, int offset, int window_count);
/* in-place NCCL all-reduce of the record over the communicator's ranks (ncclComm_t as void*): sums and count with ncclSum,
 * minima with ncclMin, maxima with ncclMax, one NCCL group; asynchronous on the Normalizer's stream */
int afe_normalizer_allreduce(afe_normalizer *n, void *nccl_comm);
int afe_normalizer_finalize(afe_normalizer *n);                                   /* normalizercpu.cpp:31-66 on the record */
int afe_normalizer_apply(afe_normalizer *n, float *d_data, int offset, int window_count);
int afe_normalizer_get_stats(afe_normalizer *n, double *h_stats);                 /* HOST double[stats_len] */
int afe_normalizer_set_stats(afe_normalizer *n, const double *h_stats);           /* e.g. sums reduced by another transport */

/* small helpers so stage objects can be driven from C / ctypes without another CUDA binding */
int afe_device_malloc(int cuda_device, size_t bytes, void **d_ptr);
int afe_device_free(int cuda_device, void *d_ptr);
int afe_memcpy_h2d(int cuda_device, void *d_dst, const void *h_src, size_t bytes);
int afe_memcpy_d2h(int cuda_device, void *h_dst, const void *d_src, size_t bytes);

/* ------------------------------------------------------------------------------------------------------------------
 * Batch extractor — the fused hot path. The per-object streaming API above cannot fill a B200; this runs a whole
 * shard of utterances through ONE fused kernel (segment+window -> FFT -> |X| -> mel+log -> DCT -> delta/delta-delta,
 * with per-utterance / corpus column statistics as a by-product) plus a light normalise pass when norm != NONE.
 * Each utterance is processed as the reference driver processes a file that fits one block
 * (ASR_OCL.cpp:227-301 with sample_limit >= N): T = estimated_window_count(N) rows per utterance.
 * ---------------------------------------------------------------------------------------------------------------- */
typedef struct afe_batch afe_batch;

enum afe_stats_scope {
    AFE_STATS_REFERENCE_BLOCK = 0, /* per utterance over the first T-(l1+l2) rows, as the reference block does (Q2) */
    AFE_STATS_UTTERANCE = 1,       /* per utterance over all T rows */
    AFE_STATS_CORPUS = 2           /* one set of statistics for all utterances of all ranks (NCCL all-reduce) */
};
enum afe_batch_flags {
    AFE_BATCH_Q1_EXACT = 1,        /* reproduce the single-block flush quirk Q1 (statics of the last D rows) */
    AFE_BATCH_NO_TMA = 2,          /* stage PCM with plain vector loads instead of cp.async.bulk (debug / A-B test) */
    AFE_BATCH_UNFUSED_NORM = 8,    /* normalise with the separate K2/K3 kernels instead of inside the fused kernel (A-B test) */
    AFE_BATCH_NO_CLUSTER = 32      /* fused normalisation through the ticket scheme (last tile of an utterance normalises it in
                                      place via L2) instead of thread-block clusters + distributed shared memory (A-B test) */
};

int afe_batch_create(const afe_params *p, int cuda_device, afe_batch **out);
void afe_batch_destroy(afe_batch *b);
int afe_batch_set_window(afe_batch *b, const float *window);
int afe_batch_set_alpha(afe_batch *b, float alpha);
int afe_batch_set_preemphasis(afe_batch *b, float coefficient);                   /* see afe_mfcc_set_preemphasis */
int afe_batch_set_options(afe_batch *b, int stats_scope, int flags);              /* flags: afe_batch_flags; other bits fail */
/* Use the caller's CUDA stream (cudaStream_t / CUstream as void*); NULL -> the handle's own stream. */
int afe_batch_set_stream(afe_batch *b, void *cuda_stream);
/* sample_offsets / sample_lengths: HOST int64[n_utts], start (in samples, even) and length of each utterance inside
 * the packed PCM buffer. Every offset should be a multiple of 8 samples (16 B) for the TMA path; otherwise the
 * plain-load path is used. Builds the tile table and uploads it. total_frames receives sum of T. */
int afe_batch_plan(afe_batch *b, const int64_t *sample_offsets, const int64_t *sample_lengths, int n_utts,
                   int64_t *total_frames);
/* Segments of longer streams (time sharding, f4): entry u covers the samples [offset, offset + length) = T frames and produces only
 * the rows of its frames [first_frame[u], first_frame[u] + n_frames[u]); frames outside that range are real delta context.
 * Normalisation over segments needs the AFE_STATS_CORPUS scope (extract_device -> corpus_stats -> allreduce -> normalize_device). */
int afe_batch_plan_segments(afe_batch *b, const int64_t *sample_offsets, const int64_t *sample_lengths, const int *first_frame,
                            const int *n_frames, int n_segments, int64_t *total_frames);
/* HOST int64[n_utts+1] first output row of each utterance */
int afe_batch_frame_offsets(const afe_batch *b, int64_t *frame_offsets);
int afe_batch_num_tiles(const afe_batch *b);
int afe_batch_kernel_launches(const afe_batch *b); /* kernels launched by the last run */
const char *afe_batch_kernel_name(const afe_batch *b); /* the instantiation that runs, e.g. "k_fused_mfcc<512,13,8,5,false>" */
/* d_pcm: DEVICE int16 buffer covering every [offset, offset+length) (+16 B slack after the last sample),
 * d_out: DEVICE float[total_frames][width]. Asynchronous on the handle's stream. */
int afe_batch_run_device(afe_batch *b, const int16_t *d_pcm, float *d_out);
/* Two-pass pieces for corpus statistics: extract raw features + per-tile column statistics ... */
int afe_batch_extract_device(afe_batch *b, const int16_t *d_pcm, float *d_out);
/* ... reduce them to corpus sums on the device (DEVICE double[stats_len], record layout at afe_cmvn_finalize_host) ... */
int afe_batch_corpus_stats(afe_batch *b, double **d_stats, int *stats_len);
/* ... which live in the batch's corpus Normalizer (NULL unless the scope is AFE_STATS_CORPUS and norm != NONE; owned by the
 * batch, valid until the next afe_batch_plan / destroy): all-reduce them over the ranks with
 * afe_normalizer_allreduce(afe_batch_normalizer(b), comm) — the ONE collective of the path ... */
afe_normalizer *afe_batch_normalizer(afe_batch *b);
/* ... or merge externally reduced sums (HOST double[stats_len]), e.g. from a gloo all-reduce in CPU tests ... */
int afe_batch_set_corpus_stats(afe_batch *b, const double *h_stats, int stats_len);
/* ... then finalise mean / scale and normalise d_out in place. */
int afe_batch_normalize_device(afe_batch *b, float *d_out);
int afe_batch_synchronize(afe_batch *b);
/* End to end with HOST buffers: H2D of PCM, run, D2H of features, all inside the call (pinned staging, chunked). */
int afe_batch_run_host(afe_batch *b, const int16_t *h_pcm, float *h_out);

/* Host-only statistics helpers (no GPU needed): the finalize formulas of normalizercpu.cpp:31-66 on double sums. */
/* stats record (also the layout of afe_batch_corpus_stats): sum[width], sumsq[width], count, min[width], max[width]
 * => 4*width+1 doubles; the first 2*width+1 all-reduce with SUM, then MIN, then MAX. */
int afe_cmvn_finalize_host(int norm_type, int width, const double *stats, float *mean, float *scale);
/* contiguous utterance ranges balanced by samples: rank r owns utterances [starts[r], starts[r+1]); starts[n_ranks+1] */
int afe_shard_utterances(const int64_t *sample_lengths, int n_utts, int n_ranks, int *starts);

/* One stream over n_ranks GPUs by time: rank r produces the frames [first[r], first[r] + count[r]) from the samples
 * [sample_begin[r], sample_begin[r] + sample_count[r]) (its frames + delta_frames of context per side, the reference's
 * (W - S) + 2 D S carry-over, segmentercpu.cpp:69-73,90-92); local_first[r] is its first frame inside that sample range.
 * Feed each rank's range to afe_batch_plan_segments; corpus scope + afe_normalizer_allreduce give stream-level CMN / CVN. */
int afe_shard_stream(int64_t total_samples, int window_size, int shift, int delta_frames, int n_ranks, int64_t *sample_begin,
                     int64_t *sample_count, int64_t *first, int *count, int *local_first);

/* NCCL plumbing (libnccl is dlopen'ed; these fail loudly if it is missing). unique id = 128 bytes. */
int afe_nccl_get_unique_id(void *id128);
int afe_nccl_comm_init(const void *id128, int n_ranks, int rank, int cuda_device, void **comm);
int afe_nccl_comm_destroy(void *comm);

#ifdef __cplusplus
}
#endif
#endif /* AFE_CUDA_H_ */
