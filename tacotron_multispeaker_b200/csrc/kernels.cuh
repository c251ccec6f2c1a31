// Launcher interfaces of the CUDA kernels (one .cu per kernel family).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/taco_b200.h"
#include "decoder_cw.h"

namespace taco {

// ---- K1: embedding gather + speaker concat (gather.cu) --------------------
// out[n,t,:] = [ table[ids[n,t]] (E) | spk_table[spk[n]] (Es) ]; Es = 0 when spk == nullptr.
// Out-of-range ids write zeros and set *oob_flag (bit0 symbol, bit1 speaker).
void launch_gather_concat(const int32_t* ids, const int32_t* spk, const float* table, int V, int E,
                          const float* spk_table, int S, int Es, int N, int T, float* out,
                          int* oob_flag, cudaStream_t st);

// ---- conv1d-as-GEMM on tcgen05 tensor cores (conv_umma.cu) -------------------
// out[n,t,col_off+o] = epi( sum_{j<taps, c<Cin} x[n, t+j-pl, c] * w[j, c, o] ),  pl=(taps-1)/2,
// rows outside [0,T) read as zero (tf 'same' padding); taps=1 is a dense layer.  epi: act(. + bias), then the
// per-channel affine scale / shift, then the residual res (each optional).  bf16 operands staged by TMA, fp32
// accumulate in TMEM.
// a_hi/a_lo: activations split into bf16 hi+lo, dense [N][T][Cp] (Cp % 64 == 0, zero padded);
// b_hi/b_lo: W^T split likewise, [b_rows][Kld] with Kld = taps*Cp (K contiguous).
// nsplit = 3: hi*hi + hi*lo + lo*hi (fp32-class accuracy); nsplit = 1: plain bf16 (lo unused).
// bank > 1: `bank` convolutions of Cout channels each in one launch (grid.z); conv ci has ci+1
// taps, weight rows [ci*Cout, (ci+1)*Cout), bias/scale/shift offset ci*Cout, output column
// offset col_off + ci*Cout  (the CBHG conv bank, reference modules.py:39-42).
struct ConvUmma {
  const void* a_hi; const void* a_lo; int N, T, Cp;
  int Cin;                                  // real input channels (<= Cp; 0 = Cp): trailing all-zero k-steps are skipped
  const void* b_hi; const void* b_lo; int b_rows, Kld;
  int taps, bank, Cout, nsplit;
  const float* bias; const float* scale; const float* shift;
  const float* res; int64_t res_bs; int ldres;
  float* out; int64_t out_bs; int ldo; int col_off;   // out may be null when only the bf16 copy below is wanted
  int act;
  // optional: the result also (or only) as the bf16 hi / lo operand of the GEMM that consumes it, dense [N][T][out_cp] with the
  // channels Cout .. out_cp-1 written as zeros (out_cp % 64 == 0); 16-byte aligned rows, no bank, col_off 0
  void* out_hi = nullptr; void* out_lo = nullptr; int out_cp = 0;
};
// The launch shape of a ConvUmma on `sms` SMs (include/taco_b200.h, taco_gemm_plan); valid == 0: the launch is refused.
taco_gemm_plan umma_plan(const ConvUmma& c, int sms);
cudaError_t launch_conv_umma(const ConvUmma& c, cudaStream_t st, taco_gemm_plan* plan_out = nullptr);
// The highway layers of a CBHG (reference modules.py:63-64, 79-89) in one launch: x, out [rows][128] fp32 dense; w_hi = the layers'
// W^T hi / lo matrices [layer][hi|lo][256][128] bf16 (contiguous, columns interleaved (H_c, T_c)); bias[l] = [256] interleaved.
// out_hi / out_lo (nullable): bf16 hi / lo copy of the result for the GEMM that follows.
cudaError_t launch_highway4(const float* x, float* out, void* out_hi, void* out_lo, const void* w_hi, const float* const* bias,
                            int layers, long long rows, int nsplit, cudaStream_t st);
// x [N,T,C] fp32 (batch stride x_bs, row stride ldx) -> hi/lo bf16 [N][T][Cp], zero padded channels.
void launch_split_bf16(const float* x, int64_t x_bs, int ldx, int N, int T, int C, int Cp, void* hi, void* lo,
                       cudaStream_t st);
// w fp32 [taps*Cin][ldw] -> W^T hi/lo bf16 rows [row0, row0+Cout) of a [*, Kld] matrix, tap j at columns j*Cp.
void launch_pack_wt(const float* w, int ldw, int taps, int Cin, int Cout, int Cp, int Kld, int row0, void* hi,
                    void* lo, cudaStream_t st);

// ---- elementwise / statistics (elementwise.cu) -----------------------------
// Per-channel batch statistics over all (n,t) rows -> scale/shift of
// tf.layers.batch_normalization(training=True): biased variance, eps.
// acc: [2*C] doubles of scratch (zeroed inside).
void launch_bn_batch_stats(const float* x, int64_t x_bs, int ldx, int col_off, int N, int T, int C,
                           const float* gamma, const float* beta, float eps, double* acc,
                           float* scale_out, float* shift_out, cudaStream_t st);
// y[n,t,c] = max(a(x[n,t,c]), a(x[n,t+1,c])) with a = per-channel affine (or identity when
// scale == nullptr); last row passes through (max_pooling1d(2,1,'same')).
void launch_affine_maxpool_split(const float* x, void* hi, void* lo, int N, int T, int C, const float* scale,
                                 const float* shift, cudaStream_t st);
void launch_affine_maxpool(const float* x, float* y, int N, int T, int C, const float* scale,
                           const float* shift, cudaStream_t st);
// x[n,t,c] = x*scale[c] + shift[c] (+ res[n,t,c]) in place.
void launch_affine_inplace(float* x, int64_t x_bs, int ldx, int N, int T, int C, const float* scale,
                           const float* shift, const float* res, int64_t res_bs, int ldres,
                           cudaStream_t st);
// Decoder epilogue: number of steps taken by dynamic_decode given dec_out [N,max_steps,D].
void launch_find_steps(const float* dec_out, int N, int max_steps, int D, int* first_fin /*[N]*/,
                       int* steps_out /*[1]*/, cudaStream_t st);

// ---- K6b: bidirectional GRU recurrence (bigru.cu) ---------------------------
// xproj [N,T,768] = x*[Wg_fw|Wc_fw|Wg_bw|Wc_bw] + biases (hoisted input projection);
// ug [2][128][256], uc [2][128][128] recurrent kernels; lengths nullable; out [N,T,256] (+bs).
// Tensor-core variant (bigru_mma.cu): eight utterances per CTA, recurrent weights in tensor memory.  `frag` is the
// fragment stream built by bigru_mma_pack (bigru_mma_frag_words() 32-bit words per CBHG).
size_t bigru_mma_frag_words();
void bigru_mma_pack(const float* ug, const float* uc, uint32_t* dst);
cudaError_t launch_bigru_mma(const float* xproj, const void* frag, const int32_t* lengths, int N, int T, float* out,
                             int64_t out_bs, cudaStream_t st);
void launch_bigru(const float* xproj, const float* ug, const float* uc, const int32_t* lengths,
                  int N, int T, float* out, int64_t out_bs, cudaStream_t st);

// ---- K7: attention decoder (decoder.cu) --------------------------------------
struct DecoderWeights {   // all device pointers; *_s are per-CTA column slices [CS][K][Mc]
  int CS;                 // CTAs per cluster the slices were cut for
  int M;                  // num_mels
  int Dout, McO;          // num_mels*r and its per-CTA padded slice width
  const float *p1_s, *p1_b;     // prenet dense_1 [M+256 -> 256]
  const float *p2_s, *p2_b;     // prenet dense_2 [256 -> 128]
  const float *ga_s, *ga_b;     // attention GRU gates [384 -> (r|u) slice], bias permuted likewise
  const float *cxa_s, *cha_s, *ca_b;  // candidate: x-part [128->256], h-part [256->256], bias
  const float *qp_s;            // [256 -> (Wq | Wproj[:256])] slices
  const float *att_v;           // [256]
  const float *pc_s, *pc_b;     // Wproj[256:] [256 -> 256], bias
  const float *g1_s, *g1_b, *cx1_s, *ch1_s, *c1_b;   // decoder GRU 1
  const float *g2_s, *g2_b, *cx2_s, *ch2_s, *c2_b;   // decoder GRU 2
  const float *o_s, *o_b;       // output projection [256 -> McO*CS], bias padded
};
struct DecoderArgs {
  const float* memory;   // [N,T_in,256]
  const float* keys;     // [N,T_in,256] = memory * W_mem
  const float* targets;  // [N,T_tgt,M] or null (free running)
  int N, T_in, T_tgt, r, steps, max_steps;
  int att_res;           // keys/memory slices resident in shared memory, or (decoder_cw, cw::ATT_TMEM) in tensor memory (set by the launcher)
  int s_max;             // decoder_cw: largest number of samples per cluster in this launch (set by the launcher)
  float* dec_out;        // [N,max_steps,Dout]
  float* align_out;      // [N,T_in,max_steps] or null
  long long* trace;      // developer aid: per-phase clock stamps of one CTA (TACO_DEC_TRACE), or null
  int trace_cta;         // which CTA writes them (TACO_DEC_TRACE_CTA, default 0)
  int trace_warp;        // decoder_cw: background warp whose items are stamped (TACO_DEC_TRACE_WARP, default 8)
};
// v6 (decoder_cw.cu): cluster of 16, critical warp group + background groups, 11 exchanges per step (layout: decoder_cw.h).
// bf16_only: one product per chunk-tile (W_hi x_hi) instead of the fp32-class three (taco_set_gemm_mode(2)).
cudaError_t launch_decoder_cw(const cw::Weights& w, const DecoderArgs& a, int nclusters, cudaStream_t st, bool bf16_only = false);
size_t decoder_cw_smem_bytes(int s_max, int T_in, int att_res, int ring_kb);
// Host only: where the attention operands of a launch with <= s_max utterances per cluster live (att_res: 3 shared memory,
// cw::ATT_TMEM tensor memory, 1 / 2 / 0 partly or not resident) and the weight-ring depth; false if nothing fits.
bool decoder_cw_plan(int s_max, int T_in, int* att_res, int* ring_kb, size_t* smem);
int decoder_cw_max_clusters();

// S = samples per cluster (1,2,4,8).  Returns cudaError of the launch.
cudaError_t launch_decoder(const DecoderWeights& w, const DecoderArgs& a, int S, cudaStream_t st);
// Largest cluster size (16 or 8) the device can co-schedule for the decoder kernel.
int decoder_pick_cluster_size();
size_t decoder_smem_bytes(int S, int T_in, int M, int CS, bool att_res);
int decoder_max_clusters(int CS);

// Griffin-Lim vocoder (griffin_lim.cu): util/audio.py:39-46,78-91,105-112 + inv_preemphasis (:23-24) on the device.
struct GriffinLimArgs {
  const float* linear;   // [N][T][n_fft/2+1] normalised spectrogram (the post-net output), batch stride linear_bs floats
  int64_t linear_bs;
  int N, T, n_fft, win, hop, iters;
  float min_level_db, ref_level_db, power, preemphasis;
  float* wav;            // [N][(T-1)*hop + win]
};
size_t griffin_lim_ws_bytes(int N, int T, int win);
cudaError_t launch_griffin_lim(const GriffinLimArgs& a, void* ws, cudaStream_t st, int* launches);

// Spectrogram analysis (spectrogram.cu): util/audio.py spectrogram / melspectrogram (librosa 0.5.1 stft + filters.mel) on
// the device.  tw / window: the twiddles (GL_N / 4 + 1 float2) and periodic Hann window that launch_fft_tables writes.
// band: [num_mels][3] ints (first bin, bin count, offset into band_w) of the mel filter bank, band_w its fp32 weights.
struct SpectrogramArgs {
  const float* wav;      // [N][L]
  long long L;
  const int* lengths;    // [N] device, or null (all L)
  int N, T_out, win, hop, num_mels;
  float preemphasis;
  double min_level_db, ref_level_db;
  const float2* tw; const float* window;
  const int* band; const float* band_w;
  float* linear;         // [N][T_out][1025] or null
  float* mel;            // [N][T_out][num_mels] or null
};
void launch_fft_tables(float2* tw, float* win, int win_len, cudaStream_t st);
cudaError_t launch_spectrogram(const SpectrogramArgs& a, cudaStream_t st);

// Resampling (resample.cu): librosa 0.5.1 core.resample with resampy's kaiser_best filter.  pos[t] for t < n_pos: where
// output t reads the filter (the host's replay of resampy's time register); rows [RS_ROWS][taps]: (win, delta) of the
// filter at offset o + i index_step.  span: the longest input window a CTA of RS_T outputs stages (samples).
constexpr int RS_T = 128, RS_U = 16, RS_BLK = 32, RS_ROWS = 513;
struct ResamplePos { int n, off_l, off_r; float eta_l, eta_r; };
struct ResampleArgs {
  const float* x;        // [N][L]
  long long L;
  int N;
  const int* lengths;    // device [2N]: input samples per row, then the outputs the filter computes (int(len ratio))
  const ResamplePos* pos; long long n_pos;
  const float2* rows; int taps, span;
  float* y;              // [N][L_out]
  long long L_out;
  bool copy;             // equal rates: y = x, zero past each length
};
size_t resample_smem_bytes(int span);
cudaError_t launch_resample(const ResampleArgs& a, cudaStream_t st);

// Per-symbol durations (durations.cu): Glow-TTS's monotonic alignment search over teacher-forced attention, float64
// scores.  One CTA per utterance, one thread per symbol (blockDim = T_in rounded up to 32); alignment tiles of
// DUR_TILE steps staged in shared memory.  bits: one backpointer bit per (utterance, step, symbol).
constexpr int DUR_MAX_T_IN = 512, DUR_MAX_STEPS = 65536, DUR_TILE = 32;
struct DurationsArgs {
  const float* align;    // [N][T_in][steps]
  int N, T_in, steps, r;
  const int* lengths;    // device [2N]: text lengths, then target frame counts
  uint32_t* bits;        // [N][y_max][T_in rounded up to 32 / 32] words
  int y_max;             // the longest utterance's decoder steps, ceil(frames / r)
  int32_t* out;          // [N][T_in] frames per symbol, 0 past the text length
};
size_t durations_bits_bytes(int N, int T_in, int y_max);
cudaError_t launch_durations(const DurationsArgs& a, cudaStream_t st);

}  // namespace taco
