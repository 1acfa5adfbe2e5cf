/*
 * ktf_b200.h -- C ABI of libktf_b200.so: hand-written sm_100a CUDA kernels for the
 * wav -> x-vector hot path of shahruk10/kaldi-tflite.
 *
 * The reference has no FFI of its own: its boundary is the tf.keras Layer protocol
 * (SURVEY.md 8b).  Each entry point below therefore replaces the `call()` body of one
 * reference layer (cited per function as file:line under
 * /root/reference/kaldi_tflite/lib/), and is what a ctypes / cgo / JNI stub would bind.
 *
 * Conventions
 *   - every function returns 0 on success, a negative KTF_E* code on failure;
 *     `ktf_last_error()` returns a thread-local message for the last failure.
 *   - all `*_dev` pointers are device pointers on the current CUDA device, owned by
 *     the caller (the Python host lets torch allocate them); `*_host` are host pointers.
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream); all work is
 *     enqueued asynchronously on it, nothing synchronises.
 *   - handles own constant tables / packed weights on the device on which they were created.
 *     ktf_frontend handles are immutable after creation and may be shared by threads.  ktf_affine
 *     handles created with KTF_PREC_BF16, ktf_tdnn_stack and float32 ktf_plda handles additionally own a grow-only
 *     device workspace that forward calls write: ONE such handle serves one stream / thread at a
 *     time (create one handle per stream for concurrent use).
 *   - tensors are row-major, innermost dimension contiguous; float32 unless stated.
 *   - there is no CPU fallback anywhere in this library.
 */
#ifndef KTF_B200_H_
#define KTF_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KTF_OK 0
#define KTF_EINVAL (-1)    /* bad argument / unsupported configuration */
#define KTF_ECUDA (-2)     /* CUDA runtime error (message has the cudaError string) */
#define KTF_ENOMEM (-3)

/* Thread-local description of the last error returned on this thread. */
const char* ktf_last_error(void);
/* ABI version of this header (major * 100 + minor). */
int ktf_version(void);
/* Compute capability of the current device as major*10+minor (e.g. 100), <0 on error. */
int ktf_device_arch(void);
/* Total number of kernel launches enqueued by this library since load (bench bookkeeping). */
int64_t ktf_launch_count(void);

/* ------------------------------------------------------------------------------------
 * Context: one per (process, device) for hosts that do not bring their own CUDA runtime binding (SURVEY.md 8b).  It owns
 * a non-blocking stream (pass ktf_ctx_stream(ctx) as the `stream` of any entry point below), gives such hosts device
 * memory and copies, and carries the NCCL communicator of the one collective this path has.  The Python host does not
 * need it: torch supplies the device memory, the streams and the process group.  Contexts are independent of each other;
 * one context serves one host thread at a time.
 * ---------------------------------------------------------------------------------- */
typedef struct ktf_ctx ktf_ctx;
int ktf_ctx_create(int32_t device, ktf_ctx** out);
void ktf_ctx_destroy(ktf_ctx* ctx);
int32_t ktf_ctx_device(const ktf_ctx* ctx);
void* ktf_ctx_stream(const ktf_ctx* ctx);            /* cudaStream_t */
int ktf_ctx_synchronize(ktf_ctx* ctx);               /* waits for the context's stream */
int ktf_ctx_malloc(ktf_ctx* ctx, int64_t bytes, void** dev_out);
int ktf_ctx_free(ktf_ctx* ctx, void* dev);
/* asynchronous on the context's stream */
int ktf_ctx_memcpy_h2d(ktf_ctx* ctx, void* dst_dev, const void* src_host, int64_t bytes);
/* enqueued on the context's stream; returns when the host buffer is valid */
int ktf_ctx_memcpy_d2h(ktf_ctx* ctx, void* dst_host, const void* src_dev, int64_t bytes);

/* The only collective of the hot path (SURVEY.md 8e): PLDA all-vs-all scoring shards the ENROLLED vectors over the GPUs
 * and all-gathers the transformed TEST vectors, after which every rank scores its own (n_test x n_enroll / G) block with
 * ktf_plda_score -- layers/plda/plda.py:247-263 scores one set against itself on one device.  NCCL is bound at run time
 * (libnccl.so.2, or the path in $KTF_NCCL_LIB); ktf_nccl_available() says whether it could be.
 *   rank 0: ktf_nccl_unique_id(id)  ->  the host ships the KTF_NCCL_UNIQUE_ID_BYTES bytes to every rank (file, socket, MPI)
 *   every rank: ktf_nccl_comm_init(ctx, nranks, rank, id)   (collective: all ranks must call it)
 *   ktf_nccl_allgather_xvec: recv_dev[(r * rows_per_rank + i) * dim + d] = rank r's send_dev[i * dim + d]; every rank
 *   contributes rows_per_rank rows (pad the last shard), elem_bytes = 4 (float32) or 8 (float64) per element.
 *   stream NULL = the context's stream.  A context without a communicator is a world of one rank (the gather is a copy). */
#define KTF_NCCL_UNIQUE_ID_BYTES 128
int ktf_nccl_available(void);
int ktf_nccl_unique_id(void* id_out_host);
int ktf_nccl_comm_init(ktf_ctx* ctx, int32_t nranks, int32_t rank, const void* id_host);
int ktf_nccl_comm_destroy(ktf_ctx* ctx);
int ktf_nccl_allgather_xvec(ktf_ctx* ctx, const void* send_dev, void* recv_dev, int64_t rows_per_rank, int32_t dim,
                            int32_t elem_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * Front-end: Framing + Windowing + FilterBank + DCT/MFCC in ONE fused kernel.
 * Replaces layers/dsp/framing.py:243-265, windowing.py:180-209, filterbank.py:225-242,
 * dct.py:175-176 and mfcc.py:197-244.  Frames are never materialised in HBM.
 * ---------------------------------------------------------------------------------- */

enum { KTF_OUT_MFCC = 0, KTF_OUT_FBANK = 1, KTF_OUT_WINDOWED = 2 };

typedef struct {
  int32_t frame_width;      /* samples gathered per frame = 2*(frame_size/2) (framing.py:107-109) */
  int32_t frame_shift;      /* samples between frame starts; == frame_width for pre-framed input */
  int32_t fft_length;       /* next power of two >= frame_width (filterbank.py:133-136,156): 256 .. 4096 */
  int32_t num_mels;         /* columns of mel_bank */
  int32_t num_ceps;         /* columns of dct (<= num_mels); ignored unless KTF_OUT_MFCC */
  int32_t output;           /* KTF_OUT_* */
  int32_t remove_dc_offset; /* windowing.py:186-189 */
  int32_t raw_energy;       /* windowing.py:192-193 / :205-206 */
  int32_t use_energy;       /* MFCC: coefficient 0 <- log-energy (mfcc.py:214-228);
                               WINDOWED: also write log-energy */
  int32_t use_power;        /* filterbank.py:234-235 */
  int32_t use_log_fbank;    /* filterbank.py:239-240 */
  int32_t apply_lifter;     /* mfcc.py:211-212 */
  float preemphasis;        /* windowing.py:195-200; <= 0 disables */
  float energy_floor;       /* lower clip of the LOG energy (windowing.py:177) */
  float epsilon;            /* added before log (windowing.py:176, filterbank.py:240) */
  float dither;             /* windowing.py:182-183: every FRAMED sample gets its own dither * N(0,1) (frames that overlap
                               do not share noise), drawn inside the kernel from a counter-based generator
                               (Philox4x32-7 keyed by the seed below, counter = (frame, sample); Box-Muller).  Random by
                               construction: statistically matched to the reference, never bit-matched; 0 disables */
} ktf_frontend_cfg;

/* Seed of the dither generator (process-wide): forward call number n after this call draws from stream seed + n, so two
 * runs that set the same seed and issue the same calls produce the same features.  Default seed 0. */
int ktf_set_dither_seed(uint64_t seed);

typedef struct ktf_frontend ktf_frontend;

/* Tables are the constants the reference layers precompute in build():
 *   window_host   [frame_width]                       windowing.py:130-156
 *   mel_bank_host [(fft_length/2+1) x num_mels]       filterbank.py:141-189 (may be NULL for WINDOWED)
 *   dct_host      [num_mels x num_ceps]               dct.py:98-143        (NULL unless MFCC)
 *   lifter_host   [num_ceps]                          mfcc.py:146-159      (NULL unless apply_lifter)
 * The bank is applied in sparse form: for every filter only the FFT bins between its first and
 * last non-zero weight are visited. */
int ktf_frontend_create(const ktf_frontend_cfg* cfg, const float* window_host,
                        const float* mel_bank_host, const float* dct_host,
                        const float* lifter_host, ktf_frontend** out);
void ktf_frontend_destroy(ktf_frontend* fe);

/* Frames produced for `num_samples` samples: 1 + (num_samples - frame_width) / frame_shift
 * (framing.py:231-235), 0 if num_samples < frame_width. */
int64_t ktf_frontend_num_frames(const ktf_frontend* fe, int64_t num_samples);
/* Output feature dimension (num_ceps, num_mels or frame_width depending on `output`). */
int32_t ktf_frontend_out_dim(const ktf_frontend* fe);

/* Uniform batch: wav_dev[b * wav_stride + i], i < num_samples, b < batch.
 * out_dev is (batch, T, out_dim) with T = ktf_frontend_num_frames(num_samples).
 * energy_dev (batch, T) is written only for KTF_OUT_WINDOWED with use_energy (else may be NULL). */
int ktf_frontend_forward(const ktf_frontend* fe, const float* wav_dev, int64_t batch,
                         int64_t num_samples, int64_t wav_stride, float* out_dev,
                         float* energy_dev, void* stream);

/* Ragged batch: utterance b occupies wav_dev[sample_offsets[b] .. sample_offsets[b+1]) and its
 * frames go to rows frame_offsets[b] .. frame_offsets[b+1]) of out_dev (total_frames, out_dim).
 * Both offset arrays are HOST arrays of batch+1 int64 (frame_offsets is an OUTPUT, filled here). */
int ktf_frontend_forward_ragged(const ktf_frontend* fe, const float* wav_dev, int64_t batch,
                                const int64_t* sample_offsets_host, int64_t* frame_offsets_host,
                                float* out_dev, float* energy_dev, void* stream);

/* Ingest options of the step BEFORE the reference path (SURVEY.md 8f rank 1):
 *   sample_format  KTF_SAMPLE_F32: float32 samples in int16 scale (the reference's input convention,
 *                  models/kaldi/xvector_extractor.py:90-91); KTF_SAMPLE_S16: raw int16 PCM as stored in a wav file --
 *                  replaces the loaders' int16 -> float32 step (testdata/feats/feats.py:31-34) and halves the bytes
 *                  that cross PCIe and HBM.  int16 needs the fused 400-sample / 512-point MFCC / fbank kernel
 *                  or fft_length 1024..4096 (every output kind, dithered or not).
 *   snip_edges     1: frames as in framing.py:231-239 (no padding).  0: Kaldi's default snip-edges=false -- the
 *                  utterance is mirror-padded on both sides INSIDE the kernel (index reflection while staging), which
 *                  replaces kaldi_numpy.PadWaveform (kaldi_numpy/frame_extraction.py:54-89) on the host;
 *                  (num_samples + shift/2) / shift frames.
 * ktf_frontend_forward / _ragged are the (F32, snip_edges=1) special cases. */
enum { KTF_SAMPLE_F32 = 0, KTF_SAMPLE_S16 = 1 };
int64_t ktf_frontend_num_frames_ex(const ktf_frontend* fe, int64_t num_samples, int32_t snip_edges);
int ktf_frontend_forward_ex(const ktf_frontend* fe, const void* wav_dev, int32_t sample_format,
                            int32_t snip_edges, int64_t batch, int64_t num_samples, int64_t wav_stride,
                            float* out_dev, float* energy_dev, void* stream);
int ktf_frontend_forward_ragged_ex(const ktf_frontend* fe, const void* wav_dev, int32_t sample_format,
                                   int32_t snip_edges, int64_t batch, const int64_t* sample_offsets_host,
                                   int64_t* frame_offsets_host, float* out_dev, float* energy_dev,
                                   void* stream);

/* Framing alone (only when a caller really wants frames in HBM): out (batch, T, frame_width). */
int ktf_framing_forward(const float* wav_dev, int64_t batch, int64_t num_samples,
                        int64_t wav_stride, int32_t frame_width, int32_t frame_shift,
                        float* out_dev, void* stream);

/* ------------------------------------------------------------------------------------
 * VAD -- layers/dsp/vad.py:156-203 (+ the gather_nd compaction of
 * models/kaldi/xvector_extractor.py:163-165).  Integer-exact vote; the per-utterance mean
 * log-energy is accumulated in a fixed order.
 * ---------------------------------------------------------------------------------- */
typedef struct {
  float energy_threshold;
  float energy_mean_scale;
  float proportion_threshold;
  int32_t frames_context;
  int32_t energy_coeff;
} ktf_vad_cfg;

/* feats_dev (total_frames, dim); utterance b = rows frame_offsets_dev[b]..[b+1) (device int64,
 * batch+1).  mask_dev (total_frames) float 0/1. */
int ktf_vad_mask(const ktf_vad_cfg* cfg, const float* feats_dev, int32_t dim,
                 const int64_t* frame_offsets_dev, int64_t batch, int64_t total_frames,
                 float* mask_dev, void* stream);

/* Stable compaction of the rows with mask != 0 (per utterance):
 *   out_offsets_dev (batch+1 int64, device): compacted frame offsets,
 *   index_dev (total_frames int64, device): row index (into feats) of each kept frame,
 *   out_feats_dev (>= kept frames, dim) may be NULL to skip the gather.
 * workspace_dev must hold ktf_vad_compact_workspace(batch, total_frames) bytes. */
int64_t ktf_vad_compact_workspace(int64_t batch, int64_t total_frames);
/* The kept-row count stays on the device (out_offsets_dev[batch]); index_dev / out_feats_dev hold that many
 * meaningful rows. */
int ktf_vad_compact(const float* feats_dev, int32_t dim, const float* mask_dev,
                    const int64_t* frame_offsets_dev, int64_t batch, int64_t total_frames,
                    int64_t* out_offsets_dev, int64_t* index_dev, float* out_feats_dev,
                    void* workspace_dev, void* stream);

/* ------------------------------------------------------------------------------------
 * Sliding-window CMVN -- layers/normalization/cmvn.py:186-250 (center=True only, like the
 * reference).  in/out (total_frames, dim); ragged through frame_offsets_dev (batch+1).
 * padding_valid: keep only frames [N/2, T-(N-1)/2) of each utterance longer than the
 * window (cmvn.py:230-237); out rows then follow out_offsets_dev (batch+1, device).
 * max_frames: any upper bound on the longest utterance (sizes the grid; the lengths themselves
 * are read on the device, so a VAD-compacted batch needs no host round trip).
 * ---------------------------------------------------------------------------------- */
int ktf_cmvn_forward(const float* in_dev, int32_t dim, const int64_t* frame_offsets_dev,
                     int64_t batch, int64_t total_frames, int64_t max_frames, int32_t window,
                     int32_t norm_vars, int32_t padding_valid, const int64_t* out_offsets_dev,
                     float* out_dev, void* stream);

/* ------------------------------------------------------------------------------------
 * TDNN affine (+ ReLU + BatchNorm + statistics) -- layers/tdnn/tdnn.py:251-280,
 * keras ReLU (models/kaldi/sequential.py:71-72), layers/normalization/batchnorm.py:81-88,
 * and the reduce-all branch of layers/stats/stats_pooling.py:211-240 fused as an epilogue.
 *   y[t, u] = bn_scale[u] * act( sum_k sum_d x[clamp(t + ctx_k), d] * W[u, k*D + d] + bias[u] )
 *             + bn_offset[u]
 * ---------------------------------------------------------------------------------- */
#define KTF_MAX_CONTEXT 16
enum { KTF_PREC_F32 = 0, KTF_PREC_BF16 = 1 };
enum { KTF_ACT_NONE = 0, KTF_ACT_RELU = 1 };

typedef struct {
  int32_t in_dim;                     /* D */
  int32_t out_dim;                    /* U */
  int32_t num_context;                /* K */
  int32_t context[KTF_MAX_CONTEXT];   /* sorted offsets (tdnn.py:108) */
  int32_t subsampling_factor;         /* tdnn.py:239 */
  int32_t padding_valid;              /* 0 = SAME (edge clamp, tdnn.py:244-247), 1 = VALID */
  int32_t activation;                 /* KTF_ACT_* applied before BatchNorm */
  int32_t precision;                  /* KTF_PREC_* : operand precision of the contraction */
} ktf_affine_cfg;

typedef struct ktf_affine ktf_affine;

/* weights_host: Kaldi <LinearParams> layout (U, K*D), i.e. W[u, k*D + d]
 *   (layers/tdnn/utils.py:22-28 maps it to the TF kernel[0,k,d,u]);
 * bias_host (U) or NULL; bn_scale_host/bn_offset_host (U) or NULL:
 *   scale = gamma / sqrt(var + eps), offset = -mean * scale (batchnorm.py:81-88). */
int ktf_affine_create(const ktf_affine_cfg* cfg, const float* weights_host, const float* bias_host,
                      const float* bn_scale_host, const float* bn_offset_host, ktf_affine** out);
void ktf_affine_destroy(ktf_affine* a);

/* Rows produced for an utterance of T input rows (tdnn.py:224-239). */
int64_t ktf_affine_out_rows(const ktf_affine* a, int64_t T);

/* x_dev (total_in_rows, D); utterance b = rows in_offsets_dev[b]..[b+1); output rows follow
 * out_offsets_dev (for SAME padding and subsampling 1 the two arrays are identical).
 * total_in_rows / total_out_rows may be UPPER BOUNDS of in_offsets_dev[batch] / out_offsets_dev[batch]
 * (they size grids and scratch; the offsets are read on the device), so a VAD-compacted batch needs no
 * host round trip for its kept-row count; rows past the actual count are then undefined in y_dev.
 * Both precisions support every mode of the reference layer: KTF_PREC_BF16 runs padding="VALID" and
 * subsampling_factor > 1 (tdnn.py:224-249) as a splice of the evaluated time steps + one tcgen05 GEMM.
 * y_dev (total_out_rows, U) may be NULL when only statistics are wanted.
 * stats_dev, if not NULL, is (batch, 2, U) float32 and receives sum_t y and sum_t y^2 per
 * utterance (it is zeroed by this call). */
int ktf_affine_forward(const ktf_affine* a, const float* x_dev, const int64_t* in_offsets_dev,
                       const int64_t* out_offsets_dev, int64_t batch, int64_t total_in_rows,
                       int64_t total_out_rows, float* y_dev, float* stats_dev, void* stream);

/* Whole network on the tcgen05 engine: [affine(+ReLU+BN)] x n1 -> StatsPooling(reduce-all,
 * stats_pooling.py:211-240) -> [affine(+ReLU+BN)] x n2, i.e. the keras Sequential built by
 * models/kaldi/sequential.py:86-143.  All layers must have been created with KTF_PREC_BF16,
 * padding SAME and subsampling 1.  Activations stay on the device in bf16 between layers (fp32
 * accumulation in TMEM); the splice of every layer is implicit (shifted TMA loads).
 * stats_after_layer = index of the layer whose output is pooled over time (-1: no pooling);
 * layers after it must have context [0].  The pooled layer runs with its operands swapped and
 * accumulates the per-utterance sum / sum of squares in its epilogue (fp32), so its activation is
 * never stored; the sums are centred on the BatchNorm moving mean of each unit (-offset / scale), so a unit
 * whose post-ReLU values sit far above zero keeps its pooled std (no E[r^2] - E[r]^2 cancellation in fp32).
 * Empty utterances (offsets_dev[b] == offsets_dev[b+1]) are allowed: one produces no per-frame rows, a pooled
 * row of NaN (the mean over zero frames, as the reference's reduce_mean) that later layers compute from, and
 * leaves the other utterances' results unchanged; nothing outside the caller's rows of feats_dev is read.
 * The same holds for a KTF_PREC_BF16 ktf_affine_forward.
 * The stack borrows the layer handles and owns a grow-only device workspace:
 * forward calls on ONE stack handle must be issued on one stream at a time. */
typedef struct ktf_tdnn_stack ktf_tdnn_stack;
int ktf_tdnn_stack_create(ktf_affine* const* layers, int32_t num_layers, int32_t stats_after_layer,
                          int32_t include_std, float stats_epsilon, ktf_tdnn_stack** out);
void ktf_tdnn_stack_destroy(ktf_tdnn_stack* s);
int32_t ktf_tdnn_stack_out_dim(const ktf_tdnn_stack* s);
/* feats_dev (total_rows, D0) fp32, utterance b = rows offsets_dev[b]..[b+1) (device int64, batch+1).
 * total_rows may be an UPPER BOUND of offsets_dev[batch] (see ktf_affine_forward): every per-frame kernel
 * reads the actual row count on the device.
 * out_dev: (batch, out_dim) fp32 when the stack pools over time, else (total_rows, out_dim). */
int ktf_tdnn_stack_forward(ktf_tdnn_stack* s, const float* feats_dev, const int64_t* offsets_dev,
                           int64_t batch, int64_t total_rows, float* out_dev, void* stream);

/* wav -> x-vector form of the stack (models/kaldi/xvector_extractor.py:162-171): the VAD compaction (tf.gather_nd, :163-165),
 * the sliding CMVN (layers/normalization/cmvn.py:186-250 with center=True, norm_vars=False, padding SAME) and the splice
 * of the first layer are ONE pre-pass kernel in front of the GEMMs -- the kept rows are gathered into shared memory
 * through the VAD index list, normalised there and leave as the bf16 operand of the first layer.
 *   feats_dev   (all_rows, D0) un-normalised features (MFCCs before VAD)
 *   index_dev   row index (into feats_dev) of every kept frame, in compacted order (ktf_vad_compact), or NULL when
 *               feats_dev already holds the compacted rows
 *   offsets_dev compacted frame offsets (batch + 1, device); total_rows >= offsets_dev[batch] (upper bound)
 *   max_frames  any upper bound on the longest compacted utterance (sizes the grid)
 * Requires a first layer with consecutive contexts and a tile that fits (ktf_tdnn_stack_vad_prepass_fits); other CMVN
 * modes: ktf_cmvn_forward + ktf_tdnn_stack_forward. */
int ktf_tdnn_stack_forward_vad(ktf_tdnn_stack* s, const float* feats_dev, const int64_t* index_dev,
                               const int64_t* offsets_dev, int64_t batch, int64_t total_rows, int64_t max_frames,
                               int32_t cmvn_window, float* out_dev, void* stream);

/* 1 when ktf_tdnn_stack_forward_vad accepts (cmvn_window, max_frames): a first layer with consecutive contexts within
 * +-4, and a pre-pass tile of 32..256 frames whose rows (tile + window + 8 halo frames) fit in shared memory.  With 30-dim
 * features windows up to 800 fit; with 80-dim features up to 262.  0 otherwise: run ktf_vad_compact with the gather,
 * ktf_cmvn_forward and ktf_tdnn_stack_forward instead. */
int32_t ktf_tdnn_stack_vad_prepass_fits(const ktf_tdnn_stack* s, int32_t cmvn_window, int64_t max_frames);

/* Element-wise helpers for callers that use ReLU / BatchNorm as stand-alone layers. */
int ktf_relu_forward(const float* x_dev, int64_t n, float* y_dev, void* stream);
int ktf_scale_offset_forward(const float* x_dev, int64_t rows, int32_t dim,
                             const float* scale_dev, const float* offset_dev, float* y_dev,
                             void* stream);

/* ------------------------------------------------------------------------------------
 * StatsPooling -- layers/stats/stats_pooling.py:211-316.
 * ---------------------------------------------------------------------------------- */
/* (batch, 2, U) sums -> (batch, U or 2U) mean || std; counts_dev = frames per utterance
 * taken from offsets_dev (batch+1).  std = sqrt(relu(E[x^2]-mean^2) + eps). */
int ktf_stats_finalize(const float* sums_dev, const int64_t* offsets_dev, int64_t batch,
                       int32_t dim, int32_t include_std, float epsilon, int32_t input_period,
                       float* out_dev, void* stream);
/* General reduce-all (any input_period): x (total_rows, dim) -> out (batch, dim or 2*dim). */
int ktf_stats_reduce(const float* x_dev, const int64_t* offsets_dev, int64_t batch, int32_t dim,
                     int32_t input_period, int32_t include_std, float epsilon, float* out_dev,
                     void* stream);
/* Windowed mode for ONE uniform batch (batch, T, dim) -> (batch, T_out, dim or 2*dim);
 * eval step t_j = t_start + j*output_period, window offsets range(left, right_excl, input_period),
 * out-of-range taps masked (stats_pooling.py:179-209,266-295); repeat = output_period for SAME. */
int ktf_stats_windows(const float* x_dev, int64_t batch, int64_t T, int32_t dim, int32_t left,
                      int32_t right_excl, int32_t input_period, int64_t t_start, int64_t num_eval,
                      int32_t output_period, int32_t repeat, int32_t include_std, float epsilon,
                      float* out_dev, void* stream);

/* ------------------------------------------------------------------------------------
 * x-vector back-end -- models/kaldi/xvector_extractor.py:174-181:
 *   y = (x - mean) @ L^T + o ; y *= sqrt(out_dim) / ||y||     transform (out_dim, in_dim+1) = [L | o]
 * ---------------------------------------------------------------------------------- */
int ktf_lda_forward(const float* x_dev, int64_t batch, int32_t in_dim, int32_t out_dim,
                    const float* mean_dev, const float* transform_dev, int32_t length_norm,
                    float* y_dev, void* stream);

/* ------------------------------------------------------------------------------------
 * PLDA -- layers/plda/plda.py:163-263.  dtype_bytes = 4 (float32) or 8 (float64 parameters
 * and arithmetic, the reference default).
 * ---------------------------------------------------------------------------------- */
typedef struct ktf_plda ktf_plda;
int ktf_plda_create(int32_t dim, const double* mean_host, const double* transform_host,
                    const double* psi_host, int32_t normalize_length, int32_t simple_length_norm,
                    int32_t dtype_bytes, ktf_plda** out);
/* num_examples (SURVEY.md 8f rank 3): the enrolled vectors scored through this handle are averages over that many
 * utterances -- plda.py:163-182 (covariance psi + I/n in the length normalisation) and :228-231 (class mean
 * n psi / (n psi + 1) u, variance 1 + psi / (n psi + 1)).  ktf_plda_create is the n = 1 case. */
int ktf_plda_create_ex(int32_t dim, const double* mean_host, const double* transform_host,
                       const double* psi_host, int32_t normalize_length, int32_t simple_length_norm,
                       int32_t dtype_bytes, double num_examples, ktf_plda** out);
void ktf_plda_destroy(ktf_plda* p);
/* x (n, dim) float32 -> u (n, dim) of dtype_bytes each: u = T x - T m, length-normalised
 * (plda.py:184-196). */
int ktf_plda_transform(const ktf_plda* p, const float* x_dev, int64_t n, void* u_dev, void* stream);
/* scores[i, j] = LLR(test u_i | enrolled u_j) (plda.py:215-245) for i < n_test, j < n_enroll;
 * scores_dev is (n_test, ld) of dtype_bytes each.  Evaluated as A_i + B_j + u_i^T diag(c) u_j. */
int ktf_plda_score(const ktf_plda* p, const void* u_test_dev, int64_t n_test,
                   const void* u_enroll_dev, int64_t n_enroll, void* scores_dev, int64_t ld,
                   void* stream);

/* Compact score output (SURVEY.md 8f rank 3): at dim 128 the score matrix is bound by its own HBM write (4 bytes per
 * trial, 64 FLOP per byte), so callers that rank or threshold trials can take the scores as bfloat16 (2 bytes per trial,
 * relative rounding 2^-9): the fp32-equivalent value A_i + B_j + u_i^T diag(c) u_j is formed in TMEM / registers exactly
 * as for KTF_SCORES_NATIVE and rounded once on the way out.  KTF_SCORES_BF16 needs a float32 handle; scores_dev is then
 * (n_test, ld) bfloat16.  KTF_SCORES_NATIVE == ktf_plda_score (plda.py:215-245). */
enum { KTF_SCORES_NATIVE = 0, KTF_SCORES_BF16 = 1 };
int ktf_plda_score_ex(const ktf_plda* p, const void* u_test_dev, int64_t n_test, const void* u_enroll_dev,
                      int64_t n_enroll, void* scores_dev, int64_t ld, int32_t score_format, void* stream);

/* Best trial per test vector (SURVEY.md 8f rank 3, the top-k = 1 form of the compact output): best_score_dev[i] =
 * max_j LLR(test u_i | enrolled u_j) and best_index_dev[i] = the j that attains it (the lowest j on a tie; -1 and -inf
 * when n_enroll == 0), with the same fp32-equivalent arithmetic as the score matrix entry (plda.py:215-245) -- the
 * (n_test, n_enroll) matrix is never written, so the call is bound by the operand stream instead of a 4-byte-per-trial
 * HBM write.  Needs a float32 handle (the tcgen05 score GEMM). */
int ktf_plda_score_top1(const ktf_plda* p, const void* u_test_dev, int64_t n_test, const void* u_enroll_dev,
                        int64_t n_enroll, float* best_score_dev, int64_t* best_index_dev, void* stream);

/* k best trials per test vector (the top-k form of ktf_plda_score_top1), 1 <= k <= KTF_PLDA_TOPK_MAX:
 * scores_dev / index_dev are (n_test, k) row-major; row i holds the k largest entries of row i of the score matrix
 * ktf_plda_score would write -- the same fp32-equivalent values, bit for bit -- and their enrolled columns, sorted by
 * score, descending; on equal scores the lower column comes first (a stable descending sort of the row).  When
 * k > n_enroll, entries n_enroll .. k-1 are (-inf, -1); n_enroll == 0 gives (-inf, -1) everywhere.  The matrix is never
 * written.  Needs a float32 handle (the tcgen05 score GEMM) and n_enroll < 2^32; k outside 1 .. KTF_PLDA_TOPK_MAX is
 * KTF_EINVAL.  No host synchronisation: the scratch (partial lists of every row) lives in the handle's grow-only
 * workspace, so once it has grown for a shape the call can be captured in a CUDA graph.  As every call that uses that
 * workspace, calls on one handle must not run concurrently on different streams. */
#define KTF_PLDA_TOPK_MAX 32
int ktf_plda_score_topk(const ktf_plda* p, const void* u_test_dev, int64_t n_test, const void* u_enroll_dev,
                        int64_t n_enroll, int32_t k, float* scores_dev, int64_t* index_dev, void* stream);
/* Merge of per-row top-k lists, e.g. of enrolled shards scored on different GPUs (indexes offset to the global
 * numbering): scores_in_dev / index_in_dev are (num_lists, n_rows, k_in); entries with index < 0 are skipped, lists need
 * not be sorted.  Output (n_rows, k), 1 <= k <= KTF_PLDA_TOPK_MAX: the k best candidates of every row with the ordering
 * and padding of ktf_plda_score_topk (score descending, lower index first on equal scores, (-inf, -1) past the last
 * candidate). */
int ktf_topk_merge(const float* scores_in_dev, const int64_t* index_in_dev, int32_t num_lists, int64_t n_rows,
                   int32_t k_in, int32_t k, float* scores_dev, int64_t* index_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* KTF_B200_H_ */
