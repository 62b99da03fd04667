/* tcr_b200.h — C ABI of the B200-native TC-ResNet hot path (libtcr_b200.so).
 *
 * The reference (hyperconnect/TC-ResNet) has no FFI: its "plugin API" is Python-level and the
 * arithmetic runs inside TensorFlow 1.13's Session.run.  This header is the boundary a maintainer
 * binds with ctypes (see INTEGRATION.md); each entry point names the reference interface whose
 * arithmetic it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch / C++ types in signatures.
 *   - every function returns an int status (TCR_OK == 0); tcr_last_error() gives the message of the
 *     last failure on the calling thread.  Functions never throw and never exit.
 *   - the CALLER owns every tensor buffer (device pointers, fp32, row-major) and the stream;
 *     the library owns only the opaque handle and its private workspace.
 *   - one handle per (GPU, stream); a handle is not thread-safe, distinct handles are independent.
 *   - all activations are (N, T, C) row-major with C fastest (== the reference's NHWC [N,T,1,C]);
 *     conv weights are HWIO [k,1,C_in,C_out] exactly as TF stores them, so flat parameter buffers
 *     can be filled from / dumped to reference checkpoints by name (tcr_param_table).
 */
#ifndef TCR_B200_H_
#define TCR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TCR_ABI_VERSION 6

enum {
  TCR_OK = 0,
  TCR_ERR_INVALID = 1,      /* bad argument / unsupported configuration */
  TCR_ERR_CUDA = 2,         /* CUDA runtime or launch failure */
  TCR_ERR_UNSUPPORTED = 3,
  TCR_ERR_COMM = 4          /* NCCL failure or libnccl not loadable */
};

enum { TCR_MODEL_TCRESNET8 = 8, TCR_MODEL_TCRESNET14 = 14 };
enum { TCR_FEATURE_MFCC = 0, TCR_FEATURE_LOG_MEL = 1 };
/* What `input` points at (the `input_is_features` argument / field):
 *   TCR_INPUT_WAV_F32   fp32 samples in [-1,1], the output of contrib_audio.decode_wav + augmentation
 *                       (datasets/audio_data_wrapper.py:57-112);
 *   TCR_INPUT_FEATURES  precomputed features [n,T,F];
 *   TCR_INPUT_WAV_PCM16 int16 PCM samples as stored in the wav files; the kernel applies decode_wav's 1/32768 scaling
 *                       (exact in fp32), so the result is bit-identical to TCR_INPUT_WAV_F32 on the decoded samples.
 *                       Halves the host->device bytes of an un-augmented (evaluation / inference) batch. */
enum { TCR_INPUT_WAV_F32 = 0, TCR_INPUT_FEATURES = 1, TCR_INPUT_WAV_PCM16 = 2 };

typedef struct tcr_handle tcr_handle;
typedef void* tcr_stream;   /* cudaStream_t */

/* Everything that fixes shapes.  Mirrors the flags the reference threads through `args`:
 * datasets/audio_data_wrapper.py:61-110 (sample_rate, clip_duration_ms, window_size_ms,
 * window_stride_ms, num_mel_bins, num_mfccs, lower/upper_edge_hertz), factory/base.py:13-35
 * (num_classes, preprocess_method), factory/audio_nets.py:366-370 (width_multiplier,
 * dropout_keep_prob), audio_nets/tc_resnet.py:102-123 (BN decay 0.997, eps 0.001). */
typedef struct tcr_config {
  int32_t model;                  /* TCR_MODEL_TCRESNET8 | TCR_MODEL_TCRESNET14 (audio_nets/tc_resnet.py:57,65) */
  float   width_multiplier;       /* channels = int(c * width_multiplier); every count must be a multiple of 4 */
  int32_t num_classes;            /* 12 */
  int32_t sample_rate;            /* 16000 */
  int32_t clip_samples;           /* int(sample_rate * clip_duration_ms / 1000) = 16000 */
  int32_t window_size_samples;    /* int(sample_rate * window_size_ms / 1000): 640 (T=49) or 480 (T=98) */
  int32_t window_stride_samples;  /* 320 or 160 */
  int32_t num_mel_bins;           /* 64 */
  int32_t num_mfccs;              /* 40 */
  float   lower_edge_hertz;       /* 80 */
  float   upper_edge_hertz;       /* 7600 */
  int32_t feature_kind;           /* TCR_FEATURE_MFCC (power + DCT) | TCR_FEATURE_LOG_MEL (magnitude, no DCT) */
  int32_t max_batch;              /* workspace is sized for this many utterances per call */
  float   bn_decay;               /* 0.997 */
  float   bn_epsilon;             /* 0.001 */
  float   dropout_keep_prob;      /* 0.5 (1.0 disables dropout) */
  float   label_smoothing;        /* 0.0 */
  int32_t device;                 /* CUDA device ordinal */
} tcr_config;

typedef struct tcr_info {
  int32_t abi_version;
  int32_t frames;          /* T  = 1 + (clip - window) / stride */
  int32_t features;        /* F  = num_mfccs or num_mel_bins */
  int32_t fft_length;      /* next pow2 >= window */
  int32_t num_conv_layers; /* conv0 + per block (down?) + 2 */
  int32_t num_blocks;
  int32_t last_channels;
  int32_t last_frames;
  int64_t num_trainable;   /* floats in the flat `params`, `slots`, `grads` buffers */
  int64_t num_moving;      /* floats in the flat BN moving-statistics buffer */
  int64_t forward_flops_per_utt;   /* 2 FLOP per MAC, network only */
  int64_t workspace_bytes;
} tcr_info;

enum { TCR_KIND_WEIGHT = 0, TCR_KIND_BETA = 1, TCR_KIND_GAMMA = 2, TCR_KIND_MOVING_MEAN = 3, TCR_KIND_MOVING_VAR = 4 };

/* One row per TF variable.  `name` is the reference's variable name (e.g.
 * "TCResNet8/block0/conv0_0/BatchNorm/gamma"); trainables come first in
 * tf.trainable_variables() order (offsets into params/slots/grads), then the moving statistics
 * (offsets into the moving buffer).  Replaces the by-name access of common/model_loader.py:87-165
 * and the injection hook helper/trainer.py:145-154. */
typedef struct tcr_param_desc {
  char    name[96];
  int32_t kind;
  int32_t rank;
  int32_t shape[4];
  int64_t offset;
  int64_t numel;
} tcr_param_desc;

struct tcr_augment_clip;
/* Arguments of one training step == one `session.run(train_op)` of helper/trainer.py:312-321. */
typedef struct tcr_step_args {
  const float* input;        /* wav [n, clip_samples] in [-1,1], features [n,T,F], or (cast) int16 PCM: see TCR_INPUT_* */
  int32_t      input_is_features;   /* TCR_INPUT_WAV_F32 | TCR_INPUT_FEATURES | TCR_INPUT_WAV_PCM16 */
  const float* onehot;       /* [n, num_classes] fp32 (datasets/audio_data_wrapper.py:113-118) */
  int32_t      n;            /* utterances on THIS rank */
  float*       params;       /* flat trainables, updated in place */
  float*       slots;        /* flat momentum accumulators (`<var>/Momentum`), updated in place */
  float*       moving;       /* flat BN moving mean/variance, updated in place */
  float        learning_rate;
  float        momentum;     /* 0.9 */
  float        weight_decay; /* 0.001 */
  uint64_t     dropout_seed; /* counter-based RNG seed; ignored when dropout_mask != NULL or keep_prob == 1 */
  const float* dropout_mask; /* optional injected {0,1} mask [n, last_channels] (parity runs) */
  float*       losses;       /* optional device [2]: total_loss, model_loss (factory/audio_nets.py:161-183) */
  float*       logits;       /* optional device [n, num_classes] */
  float*       probs;        /* optional device [n, num_classes] softmax (output/softmax) */
  float*       grads;        /* optional device [num_trainable]: gradient of total_loss actually applied */
  int32_t      apply_update; /* 1: optimizer update (+ EMA) + BN moving update; 0: gradients only */
  /* Optional device input stage in front of the front-end (TCR_INPUT_WAV_PCM16 only, see tcr_augment_pcm16): when `clips` is not
   * NULL, `input` holds the wav files' int16 samples [n, pcm_stride] and the step first decodes / shifts / mixes / clips them
   * into an internal fp32 buffer.  Zero-initialise these fields when the stage is not used. */
  const struct tcr_augment_clip* clips;   /* [n]: device memory (tcr_train_step) / pinned host memory (tcr_train_step_host) */
  const float* background;   /* device: concatenated background recordings, may be NULL */
  int64_t      pcm_stride;   /* int16 samples per row of `input`; 0 = clip_samples; at most 2 * clip_samples */
  /* 1: the caller promises that `input` (and `clips`) are final when the call is made, i.e. no work queued on `stream` writes
   * them.  The front-end (input stage + MFCC) of this step then runs on the library's own low-priority stream into one of two
   * feature buffers and overlaps the tail of the previous step (weight-gradient tail, update, the cross-GPU arrival barrier);
   * the rest of the step waits for it on `stream`.  0: everything is ordered on `stream` (the default; zero-initialise).
   * tcr_train_step_host sets it itself: its inputs arrive on the library's copy stream. */
  int32_t      input_resident;
  /* Update rule (ABI v6; helper/trainer.py:171-197 build_optimizer).  A zero-initialised tail is today's momentum step.
   *   TCR_OPT_MOMENTUM  tf.train.MomentumOptimizer: slots = `<var>/Momentum`; `momentum` 0 is GradientDescentOptimizer.
   *   TCR_OPT_ADAM      tf.train.AdamOptimizer: slots = m (`<var>/Adam`, init 0), slots2 = v (`<var>/Adam_1`, init 0),
   *                     opt_scalars = device [2] {beta1_power, beta2_power} (init beta1, beta2).  Per element, in fp32:
   *                     alpha = lr*sqrt(1-beta2_power)/(1-beta1_power); m += (g-m)*(1-beta1); v += (g^2-v)*(1-beta2);
   *                     w -= m*alpha/(sqrt(v)+epsilon).  The powers are multiplied by beta1 / beta2 once per applied step,
   *                     inside the update launch (the caller owns the buffer, so CUDA-graph replays advance it as well).
   *   TCR_OPT_RMSPROP   tf.train.RMSPropOptimizer, not centered: slots = ms (`<var>/RMSProp`, init ONES), slots2 = mom
   *                     (`<var>/RMSProp_1`, init 0): ms += (g^2-ms)*(1-rms_decay); mom = mom*momentum + g*lr/sqrt(ms+epsilon);
   *                     w -= mom.
   * g is the gradient `grads` reports: weight decay included (L2 in the loss, not AdamW), averaged over ranks.
   * ema != NULL: tf.train.ExponentialMovingAverage(ema_decay).apply(trainables) after the update (helper/trainer.py:213-217):
   * shadow -= (shadow - w) * (1 - ema_decay), on the updated weights, fixed decay; the shadow (`<var>/ExponentialMovingAverage`)
   * starts as a copy of the initial weights.  apply_update == 0 changes none of this state. */
  int32_t      optimizer;    /* TCR_OPT_* */
  float*       slots2;       /* flat [num_trainable]: Adam v / RMSProp mom; NULL for momentum */
  float*       opt_scalars;  /* device [2]: Adam beta1_power, beta2_power; NULL otherwise */
  float        beta1;        /* 0.9 */
  float        beta2;        /* 0.999 */
  float        epsilon;      /* Adam 1e-8, RMSProp 1e-10 */
  float        rms_decay;    /* 0.9 */
  float*       ema;          /* flat [num_trainable] EMA shadows, or NULL: no EMA */
  float        ema_decay;    /* 0.999 */
} tcr_step_args;
enum { TCR_OPT_MOMENTUM = 0, TCR_OPT_ADAM = 1, TCR_OPT_RMSPROP = 2 };

int         tcr_abi_version(void);
const char* tcr_last_error(void);

/* Fills *cfg with the BASELINE shape: TCResNet8-1.0, 16 kHz 1 s clips, 40 ms / 20 ms windows (T=49). */
int tcr_config_default(tcr_config* cfg);

/* Builds the layer plan, constant tables (Hann window, FFT twiddles, banded mel weights, DCT) and
 * the device workspace.  Replaces graph construction in AudioNetModel.build
 * (factory/audio_nets.py:41-60) and tc_resnet (audio_nets/tc_resnet.py:6-54). */
int tcr_create(const tcr_config* cfg, tcr_handle** out);
int tcr_destroy(tcr_handle* h);
int tcr_get_info(const tcr_handle* h, tcr_info* out);
int tcr_param_table(const tcr_handle* h, const tcr_param_desc** descs, int32_t* count);

/* Xavier-uniform weights, gamma=1, beta=0, moving mean/var = 0/1, slots = 0
 * (TCResNet_arg_scope, audio_nets/tc_resnet.py:102-123).  Host-side RNG (not TF's), written with
 * cudaMemcpyAsync on `stream`.  Any of params/slots/moving may be NULL. */
int tcr_init_variables(tcr_handle* h, float* params, float* slots, float* moving, uint64_t seed, tcr_stream stream);

/* Front-end only: wav [n, clip_samples] -> features [n, T, F].
 * Replaces MFCCPreprocessor._preprocess / LogMelSpectrogramPreprocessor._preprocess
 * (datasets/preprocessors.py:64-96, 162-170, 183-194). */
int tcr_mfcc_forward(tcr_handle* h, const float* wav, float* features, int32_t n, tcr_stream stream);
/* Same front-end on int16 PCM samples [n, clip_samples] (decode_wav's 1/32768 scaling fused into the framing). */
int tcr_mfcc_forward_pcm16(tcr_handle* h, const int16_t* pcm, float* features, int32_t n, tcr_stream stream);

/* The per-clip input stage in front of the front-end, on the device (SURVEY.md 8f "next" row 1): decode_wav scaling, crop /
 * zero-pad to clip_samples, silent clips, time shift with zero fill, background mix and clip to [-1,1]
 * (datasets/augmentation_factory.py:30-211 as called from datasets/audio_data_wrapper.py:37-58).  The host makes the random
 * draws and passes them per clip, so the output is bit-identical to the host stage for the same draws.
 *   pcm        device int16 [n, pcm_stride]: the wav files' samples (row i holds clips[i].length valid samples)
 *   clips      device [n] tcr_augment_clip
 *   background device float: the background recordings concatenated (NULL: no mixing); bg_offset indexes into it
 *   wav_out    device float [n, clip_samples], what tcr_mfcc_forward / tcr_train_step take as TCR_INPUT_WAV_F32 */
typedef struct tcr_augment_clip {
  int32_t length;      /* valid int16 samples of the clip's row (longer clips are cropped, shorter zero-padded) */
  int32_t shift;       /* _shift_audio: out[i] = in[i - shift], zero outside; 0 for anchored_slice_or_pad */
  int32_t silent;      /* 1: the "" filename of a synthesised silent sample: zeros before the background mix */
  float   bg_volume;   /* 0 when the background is not mixed in (probability 1 - background_frequency, or evaluation) */
  int64_t bg_offset;   /* start of the random crop inside `background` (recording start + crop offset); < 0: none */
} tcr_augment_clip;
int tcr_augment_pcm16(tcr_handle* h, const int16_t* pcm, int64_t pcm_stride, const tcr_augment_clip* clips,
                      const float* background, float* wav_out, int32_t n, tcr_stream stream);
/* Length (floats) of the background bank the `background` pointers refer to: a clip whose crop [bg_offset, bg_offset + clip_samples)
 * does not fit is not mixed (instead of reading past the bank).  0 (default): offsets are trusted.  The host stage pads
 * recordings shorter than a clip, as augmentation_factory.py:60-75 does. */
int tcr_set_background_samples(tcr_handle* h, int64_t samples);

/* Forward pass.  is_training == 0: evaluate_audio.py path (BN moving statistics, dropout identity;
 * helper/base.py:52-125).  is_training == 1: the training graph's forward (batch statistics, dropout)
 * as run by the trainer's in-loop evaluation (helper/trainer.py:436-460); `moving` is not updated.
 * onehot/losses may be NULL; when both are given losses[0..1] = total_loss, model_loss. */
int tcr_forward(tcr_handle* h, const float* input, int32_t input_is_features, const float* params,
                const float* moving, int32_t n, int32_t is_training, uint64_t dropout_seed,
                const float* dropout_mask, const float* onehot, float weight_decay,
                float* logits, float* probs, float* losses, tcr_stream stream);

/* The evaluation consumer behind the forward pass, on the device (SURVEY.md 8f row 3): reduces one batch of scores and
 * one-hot labels to the integers every count-based metric of the reference is a function of, instead of shipping
 * [n, classes] arrays to the host per batch (helper/base.py:52-143, metrics/parser.py:135-147; accuracy, top-5, precision,
 * recall, F1, classification report: metrics/ops/non_tensor_ops.py:64-142, :146-295, :346-).
 *   scores  device [n, classes]: logits or softmax outputs of tcr_forward (arg-max and ranks are the same for both)
 *   onehot  device [n, classes]
 *   counts  device int64 [classes*classes + 2], ACCUMULATED (zero it before the first batch):
 *           [y*classes + p] confusion matrix (true row, predicted column; first maximum wins like np.argmax),
 *           [classes*classes] utterances whose true class is among the `topk` best scores, [classes*classes + 1] utterances */
int tcr_eval_accumulate(tcr_handle* h, const float* scores, const float* onehot, int32_t n, int32_t topk, int64_t* counts,
                        tcr_stream stream);

/* Forward + backward + optimizer update (momentum / Adam / RMSProp, optional EMA; see tcr_step_args::optimizer) + BN
 * moving-average update (helper/trainer.py:171-222, slim.learning.create_train_op).  With a communicator attached
 * (tcr_comm_init) gradients are averaged over ranks with one ncclAllReduce before the update. */
int tcr_train_step(tcr_handle* h, const tcr_step_args* args, tcr_stream stream);

/* The same step fed from PINNED HOST memory (the feed_dict / tf.data side of session.run(train_op): helper/trainer.py:312-321,
 * datasets/data_wrapper_base.py:100-108).  `a->input` and `a->onehot` are host pointers (cudaHostAlloc / pin_memory);
 * `a->losses` is ignored.  The batch is copied H2D on a private copy stream into one of 3 staging slots, the step runs on
 * `stream` behind it and its two losses are copied back; the call does not wait for the step it submits.  It returns,
 * in losses_out[0..1] and *losses_step, the losses of the step submitted `lag` calls earlier (*losses_step = -1 while
 * fewer than lag+1 steps are outstanding).  lag in [0,2]: 0 = synchronous, 1 = copy/compute overlap, 2 = also keeps
 * kernel launches ahead of the GPU.  The host buffers of a call may be reused once the call `lag`+1 later has
 * returned (or after tcr_host_flush).  tcr_host_flush returns the oldest outstanding losses, *losses_step = -1 when none. */
int tcr_train_step_host(tcr_handle* h, const tcr_step_args* a, int32_t lag, tcr_stream stream, float* losses_out,
                        int64_t* losses_step);
int tcr_host_flush(tcr_handle* h, float* losses_out, int64_t* losses_step);

/* Debug / parity inspection: device pointer of a named workspace tensor after the last call, e.g.
 * "features", "y:conv0", "y:block0/conv0_0", "out:block1", "g:block0/down", "grads".
 * Returns TCR_ERR_INVALID for unknown names. */
int tcr_workspace_tensor(tcr_handle* h, const char* name, float** ptr, int64_t* numel);

/* Data-parallel plumbing (no reference counterpart: const.py:7 hard-wires one device).  The unique id
 * (128 bytes, ncclUniqueId) is created on rank 0 and distributed by the host (torch.distributed). */
int tcr_comm_unique_id(void* id128);
int tcr_comm_init(tcr_handle* h, const void* id128, int32_t rank, int32_t world_size);
/* Parity-test flag (SURVEY.md 8(e)): BatchNorm batch statistics (forward) and BatchNorm-backward sums over the GLOBAL batch of all
 * ranks = the reference's single-device batch of world * n.  One NCCL all-reduce of 2*C floats per BN layer, forward and backward;
 * the step then runs on the per-layer kernels.  Not a production path: the default is local (per-replica) statistics.  No
 * reference counterpart (single device: const.py:7). */
int tcr_comm_set_sync_bn(tcr_handle* h, int32_t enable);

/* Peer-memory gradient exchange over NVLink / NVSwitch (optional, same node, world_size <= 8): every rank exports two CUDA IPC
 * handles (128 bytes: its double-buffered flat gradient and its arrival flags), the host gathers all ranks' handles (rank-major,
 * world_size x 128 bytes) and every rank attaches them.  From then on the update kernel of tcr_train_step announces its gradient
 * in every peer's flag array, waits for all ranks' flags and sums the ranks' gradients itself (fixed rank order: replicas stay
 * bit-identical) — compute and collective in ONE kernel, no ncclAllReduce launch in the step. */
int tcr_comm_p2p_export(tcr_handle* h, void* handles128);
int tcr_comm_p2p_attach(tcr_handle* h, const void* all_handles, int32_t rank, int32_t world_size);
/* Back to ncclAllReduce (e.g. when some rank could not map a peer): unmaps the peers and frees the exported buffers. */
int tcr_comm_p2p_detach(tcr_handle* h);
int tcr_comm_destroy(tcr_handle* h);

/* Measured fp32 FMA peak of the device the handle lives on (TFLOP/s), used as the compute-roofline
 * denominator by bench.py.  Launches a register-resident FMA loop and times it with CUDA events. */
int tcr_measure_fp32_peak(tcr_handle* h, double* tflops, tcr_stream stream);

/* DS-CNN (Hello-Edge) forward pass, inference mode: the reference's 2-D-conv comparison model
 * (audio_nets/ds_cnn.py:20-118; factory/audio_nets.py DSCNN{S,M,L}Model.build_inference; BASELINE.json config 5).
 * features [n, height, width] (== [N,H,W,1]); params = one flat fp32 buffer laid out by tcr_dscnn_param_table
 * (TF variable names "DSCNN/conv_1/weights", ".../batch_norm/moving_mean", "DSCNN/fc1/biases", ...).
 * size: 'S' or 'M' ('L' builds its table but its 276-channel head is not supported yet). */
typedef struct tcr_dscnn tcr_dscnn;
typedef struct tcr_dscnn_config {
  int32_t size;          /* 'S' | 'M' | 'L' */
  int32_t height;        /* frames, 49 */
  int32_t width;         /* coefficients, 40 (10 in the reference's DS-CNN recipes) */
  int32_t num_classes;   /* 12 */
  int32_t max_batch;
  int32_t device;
} tcr_dscnn_config;
int tcr_dscnn_create(const tcr_dscnn_config* cfg, tcr_dscnn** out);
int tcr_dscnn_destroy(tcr_dscnn* d);
int tcr_dscnn_param_table(const tcr_dscnn* d, const tcr_param_desc** descs, int32_t* count, int64_t* num_params,
                          int64_t* forward_flops_per_utt);
int tcr_dscnn_forward(tcr_dscnn* d, const float* features, const float* params, int32_t n, float* logits, float* probs,
                      tcr_stream stream);

/* Process-wide launch accounting (no reference counterpart; the reference only logs wall-clock per
 * session.run, helper/trainer.py:312-321).  tcr_launch_count: kernels launched by this library so far.
 * tcr_profile_enable(1) brackets every subsequent launch with CUDA events on its stream (adds overhead:
 * use a separate pass, not the timed region); tcr_profile_read synchronises and returns one row per
 * kernel name ("mfcc", "fwd:block0/conv0_0", "dx:...", "dw:...", "head", "grad_finalize", "update"). */
typedef struct tcr_kernel_stat {
  char    name[64];
  double  total_ms;
  int64_t launches;
} tcr_kernel_stat;
int tcr_profile_enable(int enable);
int tcr_profile_read(const tcr_kernel_stat** stats, int32_t* count);
int tcr_launch_count(uint64_t* launches);

#ifdef __cplusplus
}
#endif
#endif  /* TCR_B200_H_ */
