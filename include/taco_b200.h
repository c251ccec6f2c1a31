/*
 * taco_b200.h -- C ABI of the B200-native Tacotron synthesis forward path.
 *
 * The reference (Jim-Song/tacotron_multispeaker) is pure Python on TensorFlow
 * 1.x and has no FFI of its own; the boundary it offers for this path is the
 * Python contract
 *     Tacotron.initialize(inputs, input_lengths, mel_targets, linear_targets,
 *                         identities, id_num)          models/tacotron.py:18
 *     Synthesizer.load / Synthesizer.synthesize       synthesizer.py:14,37
 * whose body is one tf.Session.run (synthesizer.py:47).  This header is what a
 * binding for that body links against: each entry point below names the
 * reference lines it replaces.  INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *  - plain C, no torch / CUDA types in signatures; `stream` is a cudaStream_t
 *    passed as void* (NULL = legacy default stream).
 *  - every data pointer is a DEVICE pointer unless the name ends in `_host`.
 *  - all work is enqueued on the caller's stream; the only host syncs are the
 *    ones documented (`steps_out_host` read-back, workspace growth).
 *  - return value: 0 = TACO_OK, negative = error; taco_last_error() gives text.
 *  - one handle per GPU; a handle is not thread-safe.
 *  - tensors are dense row-major float32 / int32 with the reference's layouts:
 *      inputs [N,T_in] i32, input_lengths [N] i32, identities [N] i32,
 *      mel_targets [N,T_tgt,num_mels], mel_outputs [N,max_steps*r,num_mels],
 *      linear_outputs [N,max_steps*r,num_freq], alignments [N,T_in,max_steps]
 *    where max_steps = taco_max_steps(...).  Only the first `steps` decoder
 *    steps (steps*r frames) of each utterance are written.
 */
#ifndef TACO_B200_H_
#define TACO_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct taco_handle taco_handle;

/* Subset of reference hparams.py:5-53 that the forward path reads. */
typedef struct taco_hparams {
  int32_t num_mels;                /* hparams.py:11  (80)   */
  int32_t num_freq;                /* hparams.py:12  (1025) */
  int32_t outputs_per_step;        /* hparams.py:22  r      */
  int32_t max_iters;               /* hparams.py:34         */
  int32_t embedding_text_channels; /* hparams.py:39  (256)  */
  int32_t embedding_id_channels;   /* hparams.py:40  (64)   */
  int32_t num_symbols;             /* len(symbols2), models/tacotron.py:40 (7352) */
  int32_t id_num;                  /* rows of embedding_id; <=1 = single speaker (tacotron.py:48) */
} taco_hparams;

enum {
  TACO_OK = 0,
  TACO_ERR_INVALID = -1,        /* bad argument / shape                         */
  TACO_ERR_CUDA = -2,           /* a CUDA runtime call failed                   */
  TACO_ERR_MISSING_WEIGHT = -3, /* finalize: a variable was never set           */
  TACO_ERR_STATE = -4,          /* call order (e.g. forward before finalize)    */
  TACO_ERR_OOB_ID = -5,         /* symbol / speaker id outside its table        */
  TACO_ERR_UNSUPPORTED = -6     /* device is not sm_100 / shape beyond limits   */
};

enum { TACO_BN_MOVING = 0, TACO_BN_BATCH = 1 };   /* tf.layers.batch_normalization(training=) */
enum { TACO_ACT_NONE = 0, TACO_ACT_RELU = 1, TACO_ACT_SIGMOID = 2, TACO_ACT_TANH = 3 };
enum { TACO_CBHG_ENCODER = 0, TACO_CBHG_POST = 1 };

/* ---- lifetime ----------------------------------------------------------- */
/* Replaces create_model()+Tacotron.__init__ (models/__init__.py:4-8,
 * models/tacotron.py:14-15).  Fails with TACO_ERR_UNSUPPORTED when `device`
 * is not a compute-capability-10.x GPU: there is no CPU fallback. */
int taco_create(const taco_hparams* hp, int device, taco_handle** out);
int taco_destroy(taco_handle* h);
const char* taco_last_error(const taco_handle* h);
const char* taco_version(void);

/* ---- weights ------------------------------------------------------------ */
/* Replaces Saver.restore (synthesizer.py:33-34): one call per variable, named
 * as in the TF checkpoint with or without the "model/inference/" prefix
 * (SURVEY.md Appendix A).  `data_host` is HOST float32, copied immediately. */
int taco_set_weight(taco_handle* h, const char* tf_name, const float* data_host,
                    const int64_t* shape, int ndim);
/* Packs the variables into kernel layouts (BN folded to scale/shift, GRU
 * kernels split into input/recurrent parts, decoder matrices sliced per CTA of
 * the decode cluster) and uploads them.  Must be called once after all
 * taco_set_weight calls and again after any later taco_set_weight. */
int taco_finalize_weights(taco_handle* h);
/* Number of variables the path expects / name of the i-th one. */
int taco_num_weights(const taco_handle* h);
const char* taco_weight_name(const taco_handle* h, int i);

/* ---- shapes ------------------------------------------------------------- */
/* Decoder steps the loop can take: min(max_iters, T_tgt / r) when teacher
 * forcing (helpers.py:48-55,73), else max_iters (tacotron.py:94). */
int taco_max_steps(const taco_handle* h, int teacher_force, int T_tgt);

/* ---- the whole path: body of Tacotron.initialize (tacotron.py:35-104) ---- */
/* spk may be NULL (single-speaker branch, tacotron.py:56-58); mel_targets may
 * be NULL unless teacher_force.  bn_mode / teacher_force are separate because
 * the reference ties both to `linear_targets is not None` (tacotron.py:36) and
 * the host layer decides.  linear_out / align_out may be NULL to skip the
 * post-net / the alignment stack.  Writes the step count to *steps_out_host
 * (one stream sync). */
int taco_forward(taco_handle* h, const int32_t* ids, const int32_t* lengths, const int32_t* spk,
                 const float* mel_targets, int N, int T_in, int T_tgt, int bn_mode,
                 int teacher_force, float* mel_out, float* linear_out, float* align_out,
                 int32_t* steps_out_host, void* stream);

/* Same call with HOST buffers (pinned or pageable): copies inputs to the
 * device, runs taco_forward, copies the outputs back and synchronises.  This
 * is the shape of session.run(feed_dict) at synthesizer.py:42-47. */
int taco_forward_host(taco_handle* h, const int32_t* ids_host, const int32_t* lengths_host,
                      const int32_t* spk_host, const float* mel_targets_host, int N, int T_in,
                      int T_tgt, int bn_mode, int teacher_force, float* mel_out_host,
                      float* linear_out_host, float* align_out_host, int32_t* steps_out_host,
                      void* stream);

/* The same call in two halves, for callers that keep several batches in flight
 * (one handle + stream each): _begin ENQUEUES the input copies, the forward and
 * the output copies and returns without waiting for anything -- a free-running
 * decode is enqueued for max_iters steps and its step count is read at the end
 * (only an early stop, i.e. an exactly-zero frame, makes _end redo the post-net
 * on the shorter length); _wait blocks until the decoder loop of that forward
 * (TACO_STAGE_DECODER) or its last kernel (TACO_STAGE_COMPUTE) has finished --
 * the post-net resp. the output copies may still be running -- so that a caller
 * can start another handle's forward while this one's post-net fills the SMs
 * the next decoder leaves free and its 144 MB of D2H traffic drains; _end
 * waits for the copies and returns the step count.  The
 * host buffers must stay valid until _end returns.  taco_forward_host == _begin
 * followed by _end.  _wait and _end spin by default; with TACO_BLOCKING_SYNC=1 in the
 * environment at taco_create they sleep on blocking-sync events (for hosts with more
 * waiting threads than cores). */
int taco_forward_host_begin(taco_handle* h, const int32_t* ids_host, const int32_t* lengths_host,
                            const int32_t* spk_host, const float* mel_targets_host, int N,
                            int T_in, int T_tgt, int bn_mode, int teacher_force,
                            float* mel_out_host, float* linear_out_host, float* align_out_host,
                            void* stream);
enum { TACO_STAGE_DECODER = 0, TACO_STAGE_COMPUTE = 1 };
int taco_forward_host_wait(taco_handle* h, int stage);
int taco_forward_host_end(taco_handle* h, int32_t* steps_out_host, void* stream);

/* ---- stage-level entry points (unit parity against the oracle) ----------- */
/* tacotron.py:46-55: out [N,T_in,E(+E_id)].  OOB ids write a zero row and make
 * the call return TACO_ERR_OOB_ID at the next taco_check_ids(). */
int taco_embed(taco_handle* h, const int32_t* ids, const int32_t* spk, int N, int T_in,
               float* out, void* stream);
int taco_check_ids(taco_handle* h, void* stream); /* syncs; 0 or TACO_ERR_OOB_ID */
/* tacotron.py:46-63: embeddings -> prenet -> encoder CBHG.  memory_out [N,T_in,256]. */
int taco_encoder(taco_handle* h, const int32_t* ids, const int32_t* lengths, const int32_t* spk,
                 int N, int T_in, int bn_mode, float* memory_out, void* stream);
/* tacotron.py:66-97,104: attention decoder loop.  dec_out [N,max_steps,num_mels*r]
 * (== mel_outputs [N,max_steps*r,num_mels]), align_out [N,T_in,max_steps] or NULL. */
int taco_decode(taco_handle* h, const float* memory, int N, int T_in, const float* mel_targets,
                int T_tgt, int teacher_force, float* dec_out, float* align_out,
                int32_t* steps_out_host, void* stream);
/* modules.py:35-74 on arbitrary input: which = TACO_CBHG_ENCODER ([N,T,128] in)
 * or TACO_CBHG_POST ([N,T,num_mels] in); lengths may be NULL; out [N,T,256].
 * x_batch_stride / out_batch_stride are in floats (0 = dense).  x must be 16-byte aligned and its batch stride a
 * multiple of 4 floats (TACO_ERR_INVALID otherwise); likewise mel in taco_postnet, memory in taco_decode, x in
 * taco_bigru, x and kernel in taco_conv1d. */
int taco_cbhg(taco_handle* h, int which, const float* x, const int32_t* lengths, int N, int T,
              int bn_mode, int64_t x_batch_stride, float* out, void* stream);
/* tacotron.py:100-101: post CBHG + dense(num_freq).  mel [N,T,num_mels] with
 * batch stride mel_batch_stride floats, linear_out likewise. */
int taco_postnet(taco_handle* h, const float* mel, int N, int T, int bn_mode,
                 int64_t mel_batch_stride, float* linear_out, int64_t linear_batch_stride,
                 void* stream);
/* modules.py:68-74 alone: x [N,T,128] -> out [N,T,256]. */
int taco_bigru(taco_handle* h, int which, const float* x, const int32_t* lengths, int N, int T,
               float* out, void* stream);
/* tf.layers.conv1d(padding='same') + bias + activation on caller-supplied
 * device weights (modules.py:95-100; k=1 is tf.layers.dense).  x [N,T,Cin],
 * kernel [k,Cin,Cout], bias [Cout] or NULL, out [N,T,Cout]. */
int taco_conv1d(taco_handle* h, const float* x, int N, int T, int Cin, const float* kernel,
                const float* bias, int k, int Cout, int act, float* out, void* stream);

/* The two helper operators inside cbhg() that have no stage of their own, for unit parity:
 * tf.layers.max_pooling1d(pool_size=2, strides=1, padding='same') (modules.py:45-49) applied to scale[c] * x + shift[c]
 * (the folded batch-norm affine of the conv bank; NULL scale / shift = identity): x, out [N,T,C], C % 4 == 0; */
int taco_maxpool_affine(taco_handle* h, const float* x, int N, int T, int C, const float* scale,
                        const float* shift, float* out, void* stream);
/* and the training-mode statistics of tf.layers.batch_normalization (modules.py:101, is_training): biased moments of x [N,T,C]
 * over (N,T), folded with gamma / beta / epsilon 1e-3 into scale_out[c], shift_out[c] so that BN(x) = scale x + shift. C <= 2048. */
int taco_bn_batch_stats(taco_handle* h, const float* x, int N, int T, int C, const float* gamma,
                        const float* beta, float* scale_out, float* shift_out, void* stream);

/* ---- the dense / conv GEMM and the fused highway layers alone (unit tests of the kernels) ----------------------------- */
/* One conv1d('same') / dense layer with the whole epilogue of the forward's GEMMs:
 *   out[n, t, col_off + o] = act(sum_{j, c} x[n, t + j - (taps-1)/2, c] w[j, c, o] + bias[o]) * scale[o] + shift[o] + res[n, t, o]
 * (rows outside [0, T) read as zero).  bank > 1: `bank` convolutions of Cout channels side by side, conv ci with ci + 1 taps,
 * its outputs at columns col_off + ci Cout (the CBHG conv bank, modules.py:39-42).
 * Parameters are HOST float32 in the reference layouts, copied per call. */
typedef struct taco_gemm_desc {
  /* A operand: device fp32 x[n x_bs + t ldx + c], or (x_hi, x_lo) already split into bf16 hi / lo [N][T][Cp] with
   * Cp = Cin rounded up to 64 (what out_hi / out_lo of a previous call wrote); x is then not read */
  const float* x; int64_t x_bs; int32_t ldx;
  const void* x_hi; const void* x_lo;
  int32_t N, T, Cin, taps, bank, Cout;
  const float* w_host;      /* [taps, Cin, Cout]; bank: the kernels [ci + 1, Cin, Cout], ci = 0 .. bank-1, back to back */
  const float* bias_host;   /* [Cout] (bank: [bank Cout]) or NULL */
  const float* scale_host; const float* shift_host;   /* affine after the activation ([Cout], bank: [bank Cout]) or NULL */
  const float* res; int64_t res_bs; int32_t ldres;    /* device residual, or NULL */
  int32_t act;              /* TACO_ACT_* */
  float* out; int64_t out_bs; int32_t ldo, col_off;   /* device; NULL when only the bf16 copy is wanted */
  void* out_hi; void* out_lo; int32_t out_cp;         /* optional bf16 hi / lo copy of the result [N][T][out_cp], channels
                                                         Cout .. out_cp-1 zero (out_cp % 64 == 0; no bank) */
} taco_gemm_desc;
/* How the tensor-core kernel runs a GEMM: */
typedef struct taco_gemm_plan {
  int32_t valid;         /* 0: the arguments are refused */
  int32_t tiles;         /* 128 x 128 output tiles (all convs of a bank) */
  int32_t ctas;
  int32_t persistent;    /* 1: a CTA walks a list of tiles; 0: one tile per CTA */
  int32_t long_k;        /* the heaviest conv has >= 24 k-blocks of 64 inputs */
  int32_t stages;        /* 64 KB operand stages in shared memory */
  int32_t epi_warps;     /* 4 or 8 */
  int32_t acc_cols;      /* tensor-memory columns: 256 = two accumulators alternating across tiles, 128 = one */
  int32_t vec_epi;       /* 1: 128-bit epilogue loads / stores; 0: scalar (rows not 16-byte aligned) */
  int32_t variant;       /* compiled epilogue: 0 any (run time), 1 bias, 2 relu, 3 relu + affine, 4 affine + residual */
  int32_t smem_bytes;
} taco_gemm_plan;
/* The plan the tensor-core GEMM `d` gets on a device with `sms` SMs.  Reads the shape, the flags and only whether each
 * pointer is NULL and 16-byte aligned (the parameters count as aligned: the library stores them so).  No device needed.
 * TACO_ERR_INVALID (plan->valid = 0) when the launch would be refused. */
int taco_umma_plan(const taco_gemm_desc* d, int sms, taco_gemm_plan* plan);
/* Runs `d` on the tensor-core kernel in the handle's gemm mode (1 / 2: three / one bf16 products per k-step); writes the
 * plan it used to *plan (NULL allowed). */
int taco_gemm_unit(taco_handle* h, const taco_gemm_desc* d, taco_gemm_plan* plan, void* stream);
/* The fused highway layers of a CBHG: `layers` (1..4) times y = relu(x W_H + b_H) T + x (1 - T), T = sigmoid(x W_T + b_T),
 * on x [rows][128] (device, dense).  W_H / W_T: HOST [layers][128][128], b_H / b_T: HOST [layers][128].  out [rows][128]
 * and / or the bf16 hi / lo copy out_hi / out_lo [rows][128] (device, NULL to skip).  Three bf16 products per k-step in
 * gemm mode 1, one in mode 2. */
int taco_highway4_unit(taco_handle* h, const float* x, int64_t rows, int layers, const float* w_h_host,
                       const float* b_h_host, const float* w_t_host, const float* b_t_host, float* out, void* out_hi,
                       void* out_lo, void* stream);
/* The BiGRU recurrence of modules.py:68-74 alone, on caller-supplied hoisted projections and recurrent kernels.
 * impl 0: the fp32 FFMA kernel (bigru.cu), 1: the tensor-core kernel (bigru_mma.cu); independent of TACO_BIGRU and
 * of the gemm mode.  xproj [N,T,768] device, 16-byte aligned: [fw gates 256 | fw cand 128 | bw gates 256 | bw cand 128]
 * with the input biases included; lengths device int32 [N] or NULL; ug_host [2][128][256], uc_host [2][128][128]:
 * the recurrent halves (rows 128..255) of each direction's gates / candidate kernel; out [N,T,256] device, 16-byte
 * aligned.  TACO_ERR_INVALID for a bad impl, N <= 0, T <= 0, a NULL pointer or a misaligned xproj / out. */
int taco_bigru_unit(taco_handle* h, int impl, const float* xproj, const int32_t* lengths, int N, int T,
                    const float* ug_host, const float* uc_host, float* out, void* stream);

/* ---- vocoder: the step right after the path (SURVEY.md 8f rank 2) ----------- */
/* Fields of reference hparams.py:13-18,35-36 that util/audio.py reads. */
typedef struct taco_audio_params {
  int32_t sample_rate;        /* hparams.py:13 (20000) */
  int32_t griffin_lim_iters;  /* hparams.py:35 (100)   */
  double frame_length_ms;     /* hparams.py:14 (50)    */
  double frame_shift_ms;      /* hparams.py:15 (12.5)  */
  double preemphasis;         /* hparams.py:16 (0.97); 0 skips the inverse pre-emphasis */
  double min_level_db;        /* hparams.py:17 (-100)  */
  double ref_level_db;        /* hparams.py:18 (20)    */
  double power;               /* hparams.py:36 (1.5)   */
} taco_audio_params;
/* Samples per utterance that taco_griffin_lim writes for T frames: (T-1)*hop + win with
 * hop = int(frame_shift_ms/1000*sample_rate), win = int(frame_length_ms/1000*sample_rate)
 * (util/audio.py:114-118; tf.contrib.signal.inverse_stft's overlap_and_add). < 0 on bad arguments. */
int64_t taco_wav_length(const taco_audio_params* ap, int T);
/* audio.inv_spectrogram_tensorflow(linear_outputs) followed by audio.inv_preemphasis
 * (synthesizer.py:27,50; util/audio.py:23-24,39-46,78-91,105-112) for a batch: linear [N,T,num_freq]
 * (batch stride linear_batch_stride floats, 0 = dense) -> wav_out [N, taco_wav_length(ap,T)] float32.
 * Needs num_freq == 1025 (n_fft 2048) and win <= 2048; TACO_ERR_UNSUPPORTED otherwise.  Does not need weights. */
int taco_griffin_lim(taco_handle* h, const taco_audio_params* ap, const float* linear, int N, int T,
                     int64_t linear_batch_stride, float* wav_out, void* stream);

/* ---- analysis: waveform -> normalised spectrogram targets ------------------ */
/* Frames util/audio.py spectrogram / melspectrogram give an utterance of L samples: 1 + L / hop
 * (librosa.stft with center=True).  < 0 on bad arguments.  No device needed. */
int64_t taco_spectrogram_frames(const taco_audio_params* ap, int64_t L);
/* util/audio.py spectrogram(y) and melspectrogram(y) for a batch, in the [T, F] layout the model consumes (the
 * reference returns [F, T]): preemphasis (before padding) -> librosa 0.5.1 stft(n_fft 2048, hop, win, center=True,
 * reflect padding, periodic Hann centred in the frame) -> |D| -> 20 log10(max(1e-5, .)) - ref_level_db -> _normalize,
 * and the same on the mel filter bank librosa.filters.mel(sample_rate, 2048, num_mels) applied to |D|.
 * wav [N, L] dense; lengths_host [N] (HOST, each in [1, L]) or NULL (all L).  linear_out [N, T_out, num_freq] and
 * mel_out [N, T_out, num_mels], either may be NULL; rows t >= 1 + lengths[n] / hop are written as 0.0 (the targets'
 * padding).  Needs no weights.  TACO_ERR_INVALID: a length outside [1, L], or T_out < the longest utterance's frames.
 * TACO_ERR_UNSUPPORTED: num_freq != 1025, win > 2048, or N * T_out * 1025 >= 2^31.  Uses ap->preemphasis,
 * min_level_db and ref_level_db; griffin_lim_iters and power are not read. */
int taco_spectrogram(taco_handle* h, const taco_audio_params* ap, const float* wav, const int32_t* lengths_host, int N,
                     int64_t L, int T_out, float* linear_out, float* mel_out, void* stream);

/* ---- resampling: librosa 0.5.1 core.resample / core.load -------------------- */
/* Samples librosa.core.resample(y, sr_orig, sr_new, fix=True) returns for L input samples: ceil(L * (double)sr_new /
 * sr_orig), as numpy computes it.  < 0 on bad arguments.  No device needed. */
int64_t taco_resample_length(int64_t L, int32_t sr_orig, int32_t sr_new);
/* Where resampy 0.1.5's resample_f reads the filter for outputs t0 .. t0+count-1: n = int(reg) of the double time register
 * advanced by 1/ratio per output, and the table offset and interpolation factor of the left (frac = scale (reg - n)) and
 * right (scale - frac) wings, eta rounded to float.  The replay taco_resample uses.  TACO_ERR_INVALID on rates <= 0 or
 * t0 + count > 2^24.  Host only. */
int taco_resample_positions(int32_t sr_orig, int32_t sr_new, int64_t t0, int64_t count, int32_t* n, int32_t* offset_l,
                            float* eta_l, int32_t* offset_r, float* eta_r);
/* librosa.core.resample(x, sr_orig, sr_new, res_type='kaiser_best', fix=True) for a batch: resampy's band-limited
 * interpolation (kaiser_best: 64 zero crossings, 512 table entries per crossing, index step truncated to
 * int(min(1, ratio) 512), the accumulated time register) then fix_length.  x [N, L] dense float32 on the device;
 * lengths_host [N] (HOST, each in [1, L]) or NULL (all L).  y [N, L_out]: row n gets ceil(len * ratio) samples, of which
 * [int(len * ratio), ceil) are 0.0, and 0.0 up to L_out.  Equal rates copy the input.  Needs no weights.
 * TACO_ERR_INVALID: a rate <= 0, a length outside [1, L], or L_out < the longest output.  TACO_ERR_UNSUPPORTED:
 * N * L_out >= 2^31, sr_orig > 8 sr_new, or more than 2^24 filter outputs in a row. */
int taco_resample(taco_handle* h, int32_t sr_orig, int32_t sr_new, const float* x, const int32_t* lengths_host, int N,
                  int64_t L, float* y, int64_t L_out, void* stream);

/* ---- durations: per-symbol frame counts from a teacher-forced alignment ---------- */
/* Glow-TTS's monotonic alignment search (monotonic_align.maximum_path: recurrence, band, ties stay) in float64 over
 * align [N, T_in, steps] (device, dense, as taco_forward / taco_decode write it).  Utterance n has len = text_lengths_host[n]
 * symbols and F = frames_host[n] target frames (HOST int32), so Y = ceil(F / r) decoder steps (r = hparams
 * outputs_per_step).  Score s[y][x] = log(max((double)a[n, x, y], 2^-149)); cells max(0, len + y - Y) <= x <= min(len - 1,
 * y); Q[0][0] = s[0][0], Q[y][x] = s[y][x] + max(Q[y-1][x] (-inf if x == y), Q[y-1][x-1] (-inf if x == 0)); the
 * backtrack starts at len - 1 on step Y - 1 and moves to x - 1 after step y when x != 0 and (x == y or Q[y-1][x] <
 * Q[y-1][x-1]).  Step y covers min(r, F - y r) frames; durations_out [N, T_in] int32 (device) gets each symbol's frames
 * (sum F, each >= 1) and 0 for x >= len.  Rows x >= len and columns y >= Y are not read.  Deterministic (no atomics).
 * Needs no weights.  TACO_ERR_INVALID: a NULL pointer, N <= 0, steps <= 0, a length outside [1, T_in], frames outside
 * [1, steps r], or ceil(frames / r) < len (no monotonic path).  TACO_ERR_UNSUPPORTED: T_in > 512 or steps > 65536. */
int taco_durations(taco_handle* h, const float* align, int N, int T_in, int steps, const int32_t* text_lengths_host,
                   const int32_t* frames_host, int32_t* durations_out, void* stream);

/* ---- arithmetic mode of the dense layers ----------------------------------- */
/* The reference computes in fp32.  1 (default) = tcgen05 tensor cores with every operand
 * split into bf16 hi+lo and three products per k-step (fp32-class accuracy, meets the 1e-3
 * parity bound); 2 = plain bf16 operands with fp32 accumulation in the dense layers AND in
 * the decoder loop's mat-vecs (one product per k-step instead of three; separately stated
 * tolerance 5e-2, tests/test_gpu_parity.py).  Any other mode: TACO_ERR_INVALID.
 * The BiGRU recurrences always run in fp32. */
enum { TACO_GEMM_BF16X3 = 1, TACO_GEMM_BF16 = 2 };
int taco_set_gemm_mode(taco_handle* h, int mode);

/* ---- introspection for bench / tests ------------------------------------- */
/* Kernel launches issued by this handle since creation. */
int64_t taco_launch_count(const taco_handle* h);
/* Decoder launch geometry chosen at finalize: CTAs per cluster, samples per
 * cluster used for batch N. */
int taco_decoder_geometry(const taco_handle* h, int N, int* cluster_size, int* samples_per_cluster,
                          int* num_clusters);
/* How the default decoder (16-CTA clusters, mma.sync) runs a batch of N utterances with T_in input positions on a device
 * where max_clusters of its clusters are co-resident (7 on a B200).  No device needed. */
typedef struct taco_decoder_plan_t {
  int32_t valid;         /* 0: the decoder refuses the shape (T_in outside 1..512, N < 1) */
  int32_t clusters;      /* as taco_set_decoder_clusters(h, 0) picks them */
  int32_t s_max;         /* utterances in the largest cluster */
  int32_t att_res;       /* where the attention operands (exp(2 key) rows, memory columns) live: 3 shared memory,
                            4 tensor memory, 1 keys only / 2 memory only / 0 neither (re-read from global memory) */
  int32_t ring_kb;       /* weight-ring depth per background warp (1 KB chunk-tiles; batches of <= 2 per cluster may
                            deepen it at launch to hold a whole step) */
  int32_t smem_bytes;    /* dynamic shared memory per CTA */
} taco_decoder_plan_t;
int taco_decoder_plan(int N, int T_in, int max_clusters, taco_decoder_plan_t* plan);
/* Decoder geometry: 0 (default) picks the number of 16-CTA clusters (taco_decoder_plan; batch 32: 4 clusters of 8
 * utterances on 64 SMs); n > 0 uses n clusters of up to 8 utterances each. */
int taco_set_decoder_clusters(taco_handle* h, int n);
/* Device time (ms, CUDA events on `stream`) of the stages of the last
 * taco_forward when profiling is on: [0]=encoder [1]=decoder stage (memory
 * layer + loop + step count) [2]=postnet [3]=the decoder loop kernel alone. */
int taco_set_profiling(taco_handle* h, int on);
/* The forward (taco_forward, taco_forward_host*) is ~49 dependent kernel launches; the reference runs its graph with one
 * session.run (synthesizer.py:47).  When the same call (same device pointers, shapes and modes) arrives twice in a row on a
 * non-default stream, the launches are captured into a CUDA graph and replayed from then on.  On by default
 * (TACO_GRAPHS=0 in the environment, or on = 0 here, keeps plain launches). */
int taco_set_cuda_graphs(taco_handle* h, int on);
int taco_last_stage_ms(const taco_handle* h, float* ms4_host);

#ifdef __cplusplus
}
#endif
#endif /* TACO_B200_H_ */
