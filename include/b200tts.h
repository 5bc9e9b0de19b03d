/*
 * b200tts.h -- C ABI of libb200tts.so: the sm_100a replacement for the hot paths of
 * lturing/tacotronv2_wavernn_chinese.
 *
 * The reference is pure Python and has no FFI of its own (SURVEY.md section 8b); the
 * boundary that a maintainer binds is therefore the body of three Python methods.
 * Each entry point below names the reference interface it replaces
 * (paths relative to the reference root):
 *
 *   b200tts_wavernn_create     <- WaveRNN.__init__ + WaveRNN.load      wavernn/models/fatchord_version.py:93-129, :414-417
 *   b200tts_wavernn_upsample   <- UpsampleNetwork.forward (+pad_tensor) wavernn/models/fatchord_version.py:82-89, :185-186, :281-291
 *   b200tts_wavernn_generate   <- WaveRNN.generate (unbatched branch)   wavernn/models/fatchord_version.py:169-264
 *                                 incl. decode_mu_law                   wavernn/utils/dsp.py:98-103
 *   b200tts_wavernn_generate_host  same, HOST buffers in/out (what wavernn_gen.py:41 sees end to end)
 *   gen_opts.fold_target/_overlap  <- fold_with_overlap + xfade_and_unfold  fatchord_version.py:293-405 (--batched)
 *
 * Conventions
 *   - plain C types only; no torch / CUDA types in any signature (`stream` is a cudaStream_t passed as void*).
 *   - all `d_*` pointers are DEVICE pointers on the context's device, all `h_*` pointers are HOST pointers;
 *     the caller owns every buffer it passes, the library owns only what *_create allocates.
 *   - every function returns 0 on success or a negative B200TTS_E* code; the message is available from
 *     b200tts_last_error() (thread local).  Nothing aborts or throws across the ABI.
 *   - work is enqueued on `stream` and is asynchronous unless stated; a context is bound to one device and
 *     its calls must be serialised by the caller (one context per GPU per process).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with B200TTS_ECUDA.
 */
#ifndef B200TTS_H_
#define B200TTS_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200TTS_ABI_VERSION 3

enum {
  B200TTS_OK = 0,
  B200TTS_EINVAL = -1,   /* bad argument / unsupported configuration            */
  B200TTS_ECUDA = -2,    /* CUDA runtime error (message carries the CUDA string) */
  B200TTS_ENOMEM = -3,   /* device or host allocation failed                    */
  B200TTS_EMISSING = -4, /* a required weight tensor was not supplied           */
  B200TTS_ESHAPE = -5    /* a weight tensor has the wrong shape                 */
};

/* Model dimensions = the constructor arguments of the reference WaveRNN (fatchord_version.py:93-95),
 * filled from wavernn_hparams.py:18-41,50. */
typedef struct {
  int32_t rnn_dims;            /* voc_rnn_dims     512 */
  int32_t fc_dims;             /* voc_fc_dims      512 */
  int32_t bits;                /* bits             10  -> n_classes = 1 << bits */
  int32_t pad;                 /* voc_pad          2   */
  int32_t feat_dims;           /* num_mels         80  */
  int32_t compute_dims;        /* voc_compute_dims 128 */
  int32_t res_out_dims;        /* voc_res_out_dims 128 (aux_dims = res_out_dims / 4) */
  int32_t res_blocks;          /* voc_res_blocks   10  */
  int32_t n_upsample;          /* len(voc_upsample_factors), <= 4 */
  int32_t upsample_factors[4]; /* (5, 5, 11) */
  int32_t hop_length;          /* 275 == prod(upsample_factors) */
} b200tts_wavernn_cfg;

/* One named fp32 weight tensor in HOST memory, contiguous row-major; names are the reference
 * state_dict keys ("I.weight", "rnn1.weight_ih_l0", "upsample.resnet.layers.3.batch_norm1.running_var", ...).
 * The library copies and repacks; the caller may free the data after *_create returns. */
typedef struct {
  const char* name;
  const float* data;
  int32_t ndim;
  int64_t shape[4];
} b200tts_tensor;

/* Sampling noise for `Categorical(softmax(logits)).sample()` (fatchord_version.py:232-235), which the
 * reference evaluates as argmax_i(p_i / q_i), q_i ~ Exp(1).  The kernels evaluate the equivalent
 * argmax_i(logit_i - log q_i). */
enum {
  B200TTS_RNG_PHILOX = 0,          /* q from Philox4x32-10 keyed by (seed, global utterance, step, class) */
  B200TTS_RNG_EXT_EXPONENTIAL = 1  /* q read from d_q[S][B][n_classes] (tests: noise shared with the oracle) */
};
typedef struct {
  int32_t mode;
  uint64_t seed;
  uint64_t utterance_offset; /* global index of row 0 (multi-GPU shards keep results independent of the split) */
  const float* d_q;          /* EXT_EXPONENTIAL only */
  const uint64_t* d_utterance_ids; /* optional [B] (ABI 2): global index of EVERY row, for batches whose rows are not consecutive
                                      utterances (length-sorted chunks of a ragged set, pipeline.py); overrides utterance_offset */
} b200tts_rng;

enum {
  B200TTS_KERNEL_AUTO = 0,
  B200TTS_KERNEL_UTTERANCE = 1, /* one CTA per group of utterances, weights streamed from L2      */
  B200TTS_KERNEL_GRID = 2,      /* weight-stationary persistent cooperative grid, all SMs per step */
  B200TTS_KERNEL_TC = 3         /* layer-stationary tensor-core pipeline (tcgen05, split-fp16 operands), 33-256 rows */
};
typedef struct {
  int32_t kernel;             /* B200TTS_KERNEL_*                                                      */
  int32_t mu_law;             /* hp.mu_law (wavernn_hparams.py:28); non-zero -> decode_mu_law          */
  const int16_t* d_teacher;   /* optional [B][S]: fed back instead of the sampled label (teacher forcing) */
  float* d_logits;            /* optional [S][B][n_classes]: fc3 outputs of every step (debug / parity) */
  int32_t max_steps;          /* 0 = all S = T*hop steps; otherwise stop early (no wave is produced)   */
  int32_t fold_target;        /* > 0: fold-with-overlap batched generation of ONE utterance (fatchord_version.py:188-190,
                                 :250-251, :293-405; hp.voc_target).  Then B must be 1, d_labels (if given) is
                                 [n_folds][fold_len] (see b200tts_wavernn_fold_geometry) and d_wave is the cross-faded wave */
  int32_t fold_overlap;       /* hp.voc_overlap                                                          */
  const int32_t* d_utt_frames;/* optional [B]: true frame count of each row of a zero-padded ragged batch; row b of d_wave is then
                                 truncated and faded at (frames_b - 1)*hop like a batch-1 run, and zero beyond      */
  /* PACKED generation of a ragged set (ABI 3; no counterpart in the reference, which is batch-1).  The B utterances of d_mel are
   * not one row each: `pack_rows` (<= 32) kernel rows each run a QUEUE of utterances back to back -- segment k of row r is
   * utterance d_pack_utt[r*pack_segs + k] (< 0: none) and occupies lock-steps [d_pack_start[r*(pack_segs+1) + k],
   * d_pack_start[r*(pack_segs+1) + k + 1]); a row restarts from the zero state (fatchord_version.py:194-196) at every segment
   * start and the noise is keyed by (utterance, step within the utterance), so every utterance gets bit for bit the labels of a
   * stand-alone run.  Lock-steps are spent on samples that are needed instead of on padding.  d_labels stays [B][S], d_wave
   * [B][(T-1)*hop] (give d_utt_frames).  Requires the push kernel (rnn_dims = fc_dims = 512), PHILOX noise, no debug buffers. */
  const int32_t* d_pack_utt;
  const int32_t* d_pack_start;
  int32_t pack_rows, pack_segs, pack_steps;   /* pack_steps = last segment end over all rows */
} b200tts_gen_opts;

typedef struct b200tts_wavernn b200tts_wavernn;

int b200tts_abi_version(void);
const char* b200tts_last_error(void);
/* number of CUDA devices visible, or a negative error */
int b200tts_device_count(void);

int b200tts_wavernn_create(b200tts_wavernn** out, int device, const b200tts_wavernn_cfg* cfg,
                           const b200tts_tensor* weights, int n_weights);
void b200tts_wavernn_destroy(b200tts_wavernn* ctx);

/* d_mel [B][feat][T] (unpadded, as generate() receives it) ->
 *   d_mels_up    [B][T*hop][feat]     (may be NULL)
 *   d_aux_frames [B][T][res_out]      (may be NULL; aux is constant within a hop, so it is kept at frame rate)
 *   d_aux_full   [B][T*hop][res_out]  (may be NULL; the reference's materialised layout) */
int b200tts_wavernn_upsample(b200tts_wavernn* ctx, const float* d_mel, int B, int T, float* d_mels_up,
                             float* d_aux_frames, float* d_aux_full, void* stream);

/* d_mel [B][feat][T] -> d_labels [B][S] (S = T*hop, may be NULL), d_wave [B][(T-1)*hop] float64 mu-law decoded,
 * truncated and faded exactly like fatchord_version.py:243-258 (may be NULL).  Needs T >= 21 when d_wave != NULL. */
int b200tts_wavernn_generate(b200tts_wavernn* ctx, const float* d_mel, int B, int T, const b200tts_rng* rng,
                             const b200tts_gen_opts* opts, int16_t* d_labels, double* d_wave, void* stream);

/* STREAMING.  d_mel [B][feat][T] -> the same labels / wave as b200tts_wavernn_generate, and while the kernel runs, the final wave
 * samples in h_wave [B][(T-1)*hop] (PINNED host memory the device can write, e.g. cudaHostAlloc / torch pin_memory); *h_progress =
 * lock-steps whose samples are in h_wave (published every chunk_steps steps and at the end; < 0: the kernel gave up).  Sample n of
 * every row is final once *h_progress > n.  The call stores 0 to *h_progress before it enqueues anything; both buffers must stay
 * alive until the stream has passed the call.  Push kernel only: 1..32 rows, no folding, no packed rows, max_steps == 0, kernel
 * auto or grid; everything else -> B200TTS_EINVAL (no counterpart in the reference, which returns audio only at the end). */
int b200tts_wavernn_generate_stream(b200tts_wavernn* ctx, const float* d_mel, int B, int T, const b200tts_rng* rng,
                                    const b200tts_gen_opts* opts, int chunk_steps, double* h_wave, int64_t* h_progress,
                                    int16_t* d_labels, double* d_wave, void* stream);
/* Host-only helper: acquire-loads *h_progress until it is >= at_least or < 0 or timeout_ms passes; returns B200TTS_OK and the
 * last value seen in *progress (the caller decides what a timeout means).  Releases nothing, launches nothing, needs no device. */
int b200tts_wavernn_stream_wait(const int64_t* h_progress, int64_t at_least, int timeout_ms, int64_t* progress);

/* n_folds and fold_len = target + 2*overlap of fold_with_overlap (fatchord_version.py:319-330) for a T-frame utterance. */
int b200tts_wavernn_fold_geometry(int T, int hop, int target, int overlap, int* n_folds, int* fold_len);

/* Same with HOST buffers: copies h_mel to the device, generates, copies labels / wave back, synchronises. */
int b200tts_wavernn_generate_host(b200tts_wavernn* ctx, const float* h_mel, int B, int T, const b200tts_rng* rng,
                                  const b200tts_gen_opts* opts, int16_t* h_labels, double* h_wave);

/* The Exp(1) noise the PHILOX mode uses for (utterance, step, class): d_q[n_steps][B][n_classes].
 * Lets a test hand the production noise stream to the oracle. */
int b200tts_philox_exponential(int device, uint64_t seed, uint64_t utterance_offset, int B, int step0, int n_steps,
                               int n_classes, float* d_q, void* stream);

/* Number of kernel launches the library has issued on this context since creation (bench.py: gpu_launches). */
int64_t b200tts_wavernn_launch_count(const b200tts_wavernn* ctx);
/* Milliseconds (CUDA events on the launch stream) spent in the per-sample generation kernel by the most recent
 * generate call; blocks until that kernel has finished.  Negative on error. */
double b200tts_wavernn_last_kernel_ms(b200tts_wavernn* ctx);
/* Which step kernel the last generate call ran: 1 utterance, 2 wide grid, 3 push, 4 multi-group push, 5 tensor-core pipeline
 * (0: none yet).  Instrumentation for bench.py's roofline; no reference counterpart. */
int b200tts_wavernn_last_kernel(const b200tts_wavernn* ctx);

/* Synchronises the device and reports whether the most recent generate call on this context completed: the persistent
 * generation kernels spin on data written by peer thread blocks and give up after ~2 s (B200TTS_ECUDA, the wave of that call
 * is filled with NaN).  The stream-ordered b200tts_wavernn_generate cannot report this itself; callers that hand audio to a
 * user (WaveRNN.generate <- fatchord_version.py:169, wavernn_gen.py:41) call this after their own synchronisation point. */
int b200tts_wavernn_check(b200tts_wavernn* ctx);

/* Measured fp32 CUDA-core ceiling of `device` in TFLOP/s (register-only packed FFMA2 loop on every SM): the denominator
 * of bench.py's FLOP-form roofline. */
int b200tts_debug_fp32_peak(int device, double* tflops);

/* ------------------------------------------------------------------------------------------------------------------
 * Tacotron-2 forward-attention decoder loop (secondary hot path).
 *   b200tts_taco_create  <- the decoder-side variables tf.train.Saver restores (tacotron_synthesize.py:76-78), by their
 *                           checkpoint names minus the "Tacotron_model/inference/" prefix
 *   b200tts_taco_decode  <- dynamic_decode(CustomDecoder(TacotronDecoderCell, TacoTestHelper)) tacotron/models/tacotron.py:99-103
 *                           = Architecture_wrappers.py:175-218 + attention.py:119-231 + modules.py:114-142,240-251,304,334-342
 *                           + custom_decoder.py:105-135 + helpers.py:36-66
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t num_mels;         /* 80   tacotron_hparams.py num_mels                */
  int32_t prenet_units;     /* 256  prenet_layers = [256, 256]                  */
  int32_t lstm_units;       /* 256  decoder_lstm_units (checkpoint kernels are [768+256,1024] and [512,1024]) */
  int32_t enc_dim;          /* 512  2 * encoder_lstm_units                      */
  int32_t attn_dim;         /* 128  attention_dim                               */
  int32_t attn_filters;     /* 32   attention_filters                           */
  int32_t attn_kernel;      /* 31   attention_kernel                            */
  float zoneout;            /* 0.1  tacotron_zoneout_rate                       */
} b200tts_taco_cfg;

enum { B200TTS_TACO_DROPOUT_PHILOX = 0, B200TTS_TACO_DROPOUT_EXT = 1 };
typedef struct {
  int32_t mode;
  uint64_t seed;
  uint64_t utterance_offset;
  const uint8_t* d_masks;   /* EXT: keep flags [B][max_steps][2][prenet_units]; prenet dropout is ON at inference (modules.py:249) */
} b200tts_taco_dropout;

typedef struct b200tts_taco b200tts_taco;

int b200tts_taco_create(b200tts_taco** out, int device, const b200tts_taco_cfg* cfg, const b200tts_tensor* weights, int n_weights);
void b200tts_taco_destroy(b200tts_taco* ctx);

/* d_memory [B][Tx_max][enc_dim] encoder outputs, d_lengths [B] (<= Tx_max <= 512).  Every sentence runs until its own
 * stop token exceeds 0.5 or max_steps.  window != 0 enables the inference attention window of forward_attention.py:171-215.
 * Outputs: d_frames [B][max_steps][num_mels] raw decoder outputs (before the clip of tacotron.py:111), d_stop [B][max_steps],
 * d_align [B][max_steps][Tx_max] (may be NULL), d_nsteps [B] = frames produced (the last one is the frame whose stop fired). */
int b200tts_taco_decode(b200tts_taco* ctx, const float* d_memory, const int32_t* d_lengths, int B, int Tx_max,
                        const b200tts_taco_dropout* dropout, int max_steps, int window, float* d_frames, float* d_stop,
                        float* d_align, int32_t* d_nsteps, void* stream);

/* Parity aid (teacher forcing): the same loop, but the COMPLETE recurrent state is reloaded from d_states before every step and
 * the stop rule is ignored, so exactly n_steps steps run.  d_states [B][n_steps][b200tts_taco_state_floats(ctx, Tx_max)], one
 * record per step:  x[num_mels] | context[enc_dim] | c1 | h1 | c2 | h2 [lstm_units each] | mu | max_attention | pos_rec | 0 |
 * cumulated alignments[Tx_max] | alpha[Tx_max]   (the loop state of Architecture_wrappers.py:136-173 + attention.py:112-117).
 * Lets a test compare EVERY step of a long, numerically chaotic run against the oracle fed with the oracle's own state. */
int b200tts_taco_state_floats(const b200tts_taco* ctx, int Tx_max);
int b200tts_taco_decode_forced(b200tts_taco* ctx, const float* d_memory, const int32_t* d_lengths, int B, int Tx_max,
                               const b200tts_taco_dropout* dropout, int n_steps, int window, const float* d_states,
                               float* d_frames, float* d_stop, float* d_align, int32_t* d_nsteps, void* stream);

/* Run-once neighbours of the decoder loop (available when b200tts_taco_create also received the encoder / postnet
 * variables):
 *   b200tts_taco_encode   <- embedding lookup + EncoderConvolutions + EncoderRNN   tacotron.py:44-57, modules.py:145-217
 *   b200tts_taco_postnet  <- clip + Postnet + postnet_projection + residual + clip  tacotron.py:111-129, modules.py:345-376
 * d_ids [B][Tx_max] symbol ids (tacotron/utils/text.py:18-31), d_memory [B][Tx_max][enc_dim];
 * d_frames [B][max_steps][num_mels] raw decoder outputs, d_nsteps [B], d_mel [B][max_steps][num_mels] (rows >= nsteps untouched). */
int b200tts_taco_encode(b200tts_taco* ctx, const int32_t* d_ids, const int32_t* d_lengths, int B, int Tx_max, float* d_memory,
                        void* stream);
int b200tts_taco_postnet(b200tts_taco* ctx, const float* d_frames, const int32_t* d_nsteps, int B, int max_steps, float* d_mel,
                         void* stream);

/* The keep flags the PHILOX dropout mode draws: d_masks [B][steps][2][prenet_units]. */
int b200tts_taco_philox_masks(int device, uint64_t seed, uint64_t utterance_offset, int B, int steps, int prenet_units,
                              uint8_t* d_masks, void* stream);

/* Debug aid: mean SM cycles per CTA spent in {compute, barrier} of each of the 6 phases of the last grid-kernel
 * launch; only recorded when the environment variable B200TTS_GRID_PROF is set while generating. */
int b200tts_wavernn_debug_phase_cycles(b200tts_wavernn* ctx, double* out12);

#ifdef __cplusplus
}
#endif
#endif /* B200TTS_H_ */
