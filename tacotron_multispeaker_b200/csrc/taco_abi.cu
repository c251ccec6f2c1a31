// C ABI of the B200 Tacotron forward path (include/taco_b200.h): handle,
// variable store keyed by TF checkpoint names, packing into kernel layouts,
// and the launch sequence that replaces Tacotron.initialize's graph
// (reference models/tacotron.py:35-104) + Session.run (synthesizer.py:47).
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <map>
#include <string>
#include <vector>

#include "../../include/taco_b200.h"
#include "kernels.cuh"

using namespace taco;

namespace {

constexpr float kBnEps = 1e-3f;   // tf.layers.batch_normalization default
constexpr int DH = 256, DP = 128;

const char* kATT =
    "decoder/output_projection_wrapper/multi_rnn_cell/cell_0/output_projection_wrapper/"
    "concat_output_and_attention_wrapper/attention_wrapper/";
const char* kMRC = "decoder/output_projection_wrapper/multi_rnn_cell/";
const char* kPrefix = "model/inference/";

struct HostVar {
  std::vector<int64_t> shape;
  std::vector<float> data;
  bool set = false;
};

// One GEMM-shaped weight: fp32 [taps*Cin][ldw] for the FFMA path and W^T split into bf16 hi/lo
// ([b_rows][Kld], K contiguous) for the tcgen05 path.  A bank holds its convolutions back to back: conv ci has ci+1 taps,
// its fp32 rows [(ci+1)*Cin][ldw] start at row Cin*ci*(ci+1)/2 and its W^T rows are [ci*Cout, (ci+1)*Cout).
struct GemmW {
  size_t off = 0;                      // float offset of the fp32 weights in the staging arena, until w points at the upload
  const float* w = nullptr; int ldw = 0;
  uint16_t* b_hi = nullptr; uint16_t* b_lo = nullptr;
  int taps = 1, Cin = 0, Cout = 0, Cp = 0, Kld = 0, b_rows = 0, bank = 1;
  int member_taps(int ci) const { return bank > 1 ? ci + 1 : taps; }
  const float* member_w(int ci) const { return w + (size_t)ci * (ci + 1) / 2 * Cin * ldw; }
  // the fp32 weights in `arena` as uploaded; W^T hi at bt, lo right after it
  void place(const float* arena, uint16_t* bt) { w = arena + off; b_hi = bt; b_lo = bt + (size_t)b_rows * Kld; }
};
GemmW make_gemmw(size_t off, int ldw, int taps, int Cin, int Cout, int bank = 1) {
  GemmW g;
  g.off = off; g.ldw = ldw; g.taps = taps; g.Cin = Cin; g.Cout = Cout; g.bank = bank;
  g.Cp = (Cin + 63) & ~63;
  g.Kld = taps * g.Cp;
  g.b_rows = bank > 1 ? bank * Cout : Cout;
  return g;
}

struct CbhgDev {   // offsets (floats) into the device weight arena
  int K = 0, Cin = 0, P1 = 0, P2 = 0;
  size_t bank_scale = 0, bank_shift = 0, bank_gamma = 0, bank_beta = 0;
  size_t p1_b = 0, p1_scale = 0, p1_shift = 0, p1_gamma = 0, p1_beta = 0;
  size_t p2_b = 0, p2_scale = 0, p2_shift = 0, p2_gamma = 0, p2_beta = 0;
  size_t dense_b = 0;
  size_t hw_b[4] = {0, 0, 0, 0};
  size_t gru_bx = 0, gru_ug = 0, gru_uc = 0, gru_frag = 0;   // gru_frag: MMA fragment stream (bigru_mma.cu)
  size_t bank_bias = 0;                // biases of the K bank convolutions back to back
  GemmW g_bank, g_p1, g_p2, g_dense, g_hw[4], g_xproj;
};

struct Arena {   // host staging of the packed weights
  std::vector<float> buf;
  size_t alloc(size_t n) {
    size_t off = (buf.size() + 63) & ~size_t(63);
    buf.resize(off + n, 0.0f);
    return off;
  }
};

}  // namespace

struct taco_handle {
  taco_hparams hp;
  int device = 0;
  std::string err;
  std::vector<std::string> names;             // expected variables (short names)
  std::map<std::string, HostVar> vars;
  bool finalized = false;
  // packed weights
  float* dW = nullptr;
  size_t emb = 0, emb_id = 0, pre1_b = 0, pre2_b = 0, lin_b = 0;
  int emb_dim = 0;
  GemmW g_pre1, g_pre2, g_mem, g_lin;
  uint16_t* dB = nullptr;              // bf16 arena: W^T hi/lo for the tensor-core path
  int gemm_mode = 1;                   // 0 = fp32 FFMA, 1 = bf16x3 tcgen05 (fp32-class), 2 = bf16 tcgen05
  CbhgDev enc, post;
  DecoderWeights dec[2];               // slices cut for clusters of 8 ([0]) and 16 ([1]) CTAs
  int max_clusters[2] = {0, 0};        // co-resident clusters of each size on this device
  int force_cs = 0;
  int max_clusters_mma = 0;            // co-resident clusters of 16 of the default decoder
  cw::Weights decw;                    // critical-warp kernel (decoder_cw.cu): the default decoder
  int use_cw = 0;
  // workspace
  char* ws = nullptr;
  size_t ws_bytes = 0;
  char* stg = nullptr;                 // device staging of taco_forward_host (grow-only)
  size_t stg_bytes = 0;
  int* d_ints = nullptr;      // [0]=oob flag, [1]=steps, [2..]=first_fin[N]
  int d_ints_n = 0;
  int* h_pinned = nullptr;    // [0]=oob, [1]=steps   (mapped pinned memory: kernels write it directly)
  int* d_pinned = nullptr;    // device address of h_pinned
  int dec_clusters = 0;       // taco_set_decoder_clusters: 0 = pick for latency, n = use n clusters (throughput mode)
  int pending_steps = 0;      // step count of the forward started by taco_forward_host_begin
  // Free-running decodes almost always run max_iters steps (the stop condition is an exact-zero frame), so the forward
  // does not wait for the count in the middle: the post-net is enqueued for max_steps and the count is read from mapped
  // pinned memory at the end.  Only if it came out smaller is the post-net redone on the right length.
  struct Spec {
    bool active = false;
    int N = 0, T_in = 0, max_steps = 0, bn_mode = 0;
    float *d_mel = nullptr, *d_lin = nullptr, *lin_host = nullptr;
    size_t lin_bytes = 0;
  } spec;
  int64_t launches = 0;
  // CUDA graph of the forward's ~49 launches: captured the second time the same call (pointers, shapes, modes) arrives on a
  // non-default stream, replayed afterwards (one graph per handle)
  struct FwdKey {
    const void *ids, *len, *spk, *tgt, *mel, *lin, *al, *ws, *ints;
    void* stream;
    int N, T_in, T_tgt, bn, tf, gemm_mode, dec_clusters, defer;
    bool operator==(const FwdKey& o) const { return memcmp(this, &o, sizeof(FwdKey)) == 0; }
  };
  struct FwdGraph { FwdKey key; bool have_key = false; cudaGraphExec_t exec = nullptr; int64_t launches = 0; } fwd_graph;
  bool graphs_on = true;
  bool dev_env = false;   // TACO_DEV=1 at taco_create: the per-call developer switches below are read from the environment; otherwise no getenv on the forward path
  // the vocoder's ~105 launches per call likewise (key: arguments, workspace, stream)
  struct GlKey { GriffinLimArgs a; const void* ws; void* stream; };
  struct GlGraph { GlKey key; bool have_key = false; cudaGraphExec_t exec = nullptr; int launches = 0; } gl_graph;
  // taco_spectrogram's tables (twiddles, analysis window, mel band table) in an allocation of their own, so that a workspace
  // regrow does not drop them; rebuilt when (sample_rate, win) changes.  `host` is the source of the last upload.
  struct SpecTables {
    char* dev = nullptr; size_t bytes = 0;
    int sample_rate = 0, win = 0;
    std::vector<char> host;
  } spec_tab;
  // taco_resample's filter rows and replayed positions in an allocation of their own: [RS_ROWS][taps] float2 rows, then
  // n_pos ResamplePos; rebuilt when the rate pair changes or a call needs more positions.  span: the longest window a CTA
  // stages over those positions.
  struct ResTables {
    char* dev = nullptr; size_t bytes = 0;
    int sr_orig = 0, sr_new = 0, taps = 0, span = 0;
    int64_t n_pos = -1;
  } res_tab;
  bool launch_failed = false;        // a kernel launcher returned an error (sticky until check_launch reports it)
  bool profiling = false;
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // [4],[5] bracket the decoder kernel
  cudaEvent_t ev_compute = nullptr;   // taco_forward_host_begin: last kernel enqueued, output copies not yet
  cudaEvent_t ev_decoder = nullptr;   // ... and the end of the decoder loop (the post-net follows)
  cudaEvent_t ev_end = nullptr;       // blocking mode: end of the output copies
  bool blocking = false;              // TACO_BLOCKING_SYNC=1: host waits sleep instead of spinning (many lanes per core)
  float stage_ms[4] = {0, 0, 0, 0};
};

namespace {

int fail(taco_handle* h, int code, const std::string& msg) {
  if (h) h->err = msg;
  return code;
}
// The GEMM operand split (split_bf16_kernel), the FFMA conv and the decoder read activations with 16-byte vector loads at
// x + n*x_bs + t*ldx + c: the stage entry points refuse pointers and strides that would misalign them.
bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
bool rows16(const void* p, int64_t x_bs, int64_t ldx) { return al16(p) && x_bs % 4 == 0 && ldx % 4 == 0; }

#define CUDA_OK(h, expr)                                                                   \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess)                                                                 \
      return fail(h, TACO_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));   \
  } while (0)

void add_conv_names(std::vector<std::string>& n, const std::string& s) {
  n.push_back(s + "/conv1d/kernel");
  n.push_back(s + "/conv1d/bias");
  n.push_back(s + "/batch_normalization/gamma");
  n.push_back(s + "/batch_normalization/beta");
  n.push_back(s + "/batch_normalization/moving_mean");
  n.push_back(s + "/batch_normalization/moving_variance");
}
void add_cbhg_names(std::vector<std::string>& n, const std::string& s, int K, bool has_dense) {
  for (int k = 1; k <= K; ++k) add_conv_names(n, s + "/conv_bank/conv1d_" + std::to_string(k));
  add_conv_names(n, s + "/proj_1");
  add_conv_names(n, s + "/proj_2");
  if (has_dense) { n.push_back(s + "/dense/kernel"); n.push_back(s + "/dense/bias"); }
  for (int i = 1; i <= 4; ++i)
    for (const char* g : {"H", "T"}) {
      n.push_back(s + "/highway_" + std::to_string(i) + "/" + g + "/kernel");
      n.push_back(s + "/highway_" + std::to_string(i) + "/" + g + "/bias");
    }
  for (const char* d : {"fw", "bw"})
    for (const char* g : {"gates", "candidate"}) {
      n.push_back(s + "/bidirectional_rnn/" + d + "/gru_cell/" + g + "/kernel");
      n.push_back(s + "/bidirectional_rnn/" + d + "/gru_cell/" + g + "/bias");
    }
}

// Same inventory as tacotron_multispeaker_b200/weights.py:weight_specs (SURVEY Appendix A).
std::vector<std::string> expected_names(const taco_hparams& hp) {
  std::vector<std::string> n;
  const std::string att = kATT, dpw = att + "decoder_prenet_wrapper/", mrc = kMRC;
  n.push_back("embedding");
  if (hp.id_num > 1) n.push_back("embedding_id");
  for (const char* d : {"dense_1", "dense_2"}) {
    n.push_back(std::string("prenet/") + d + "/kernel");
    n.push_back(std::string("prenet/") + d + "/bias");
  }
  add_cbhg_names(n, "encoder_cbhg", 16, false);
  n.push_back("memory_layer/kernel");
  n.push_back("decoder/output_projection_wrapper/kernel");
  n.push_back("decoder/output_projection_wrapper/bias");
  n.push_back(mrc + "cell_0/output_projection_wrapper/kernel");
  n.push_back(mrc + "cell_0/output_projection_wrapper/bias");
  for (const char* d : {"dense_1", "dense_2"}) {
    n.push_back(dpw + "decoder_prenet/" + d + "/kernel");
    n.push_back(dpw + "decoder_prenet/" + d + "/bias");
  }
  for (const char* g : {"gates", "candidate"}) {
    n.push_back(dpw + "gru_cell/" + g + "/kernel");
    n.push_back(dpw + "gru_cell/" + g + "/bias");
  }
  n.push_back(att + "bahdanau_attention/query_layer/kernel");
  n.push_back(att + "bahdanau_attention/attention_v");
  for (int c = 1; c <= 2; ++c)
    for (const char* g : {"gates", "candidate"}) {
      n.push_back(mrc + "cell_" + std::to_string(c) + "/gru_cell/" + g + "/kernel");
      n.push_back(mrc + "cell_" + std::to_string(c) + "/gru_cell/" + g + "/bias");
    }
  add_cbhg_names(n, "post_cbhg", 8, hp.num_mels != 128);
  n.push_back("dense/kernel");
  n.push_back("dense/bias");
  return n;
}

const HostVar* getv(taco_handle* h, const std::string& name, std::initializer_list<int64_t> shape,
                    std::string* err) {
  auto it = h->vars.find(name);
  if (it == h->vars.end() || !it->second.set) {
    *err = std::string("missing variable ") + kPrefix + name;
    return nullptr;
  }
  const HostVar& v = it->second;
  if (v.shape.size() != shape.size() || !std::equal(shape.begin(), shape.end(), v.shape.begin())) {
    std::string s = "[";
    for (auto d : v.shape) s += std::to_string(d) + ",";
    std::string e = "[";
    for (auto d : shape) e += std::to_string(d) + ",";
    *err = std::string("variable ") + kPrefix + name + " has shape " + s + "] expected " + e + "]";
    return nullptr;
  }
  return &v;
}

#define GETV(var, name, ...)                                            \
  const HostVar* var = getv(h, name, {__VA_ARGS__}, &err);              \
  if (!var) return false;

// Copy a [rows, cols] matrix into the arena with leading dimension ld (zero padded).
size_t put_matrix(Arena& A, const float* src, int rows, int cols, int ld) {
  size_t off = A.alloc((size_t)rows * ld);
  for (int r = 0; r < rows; ++r) memcpy(&A.buf[off + (size_t)r * ld], src + (size_t)r * cols, sizeof(float) * cols);
  return off;
}
size_t put_vec(Arena& A, const float* src, int n) {
  size_t off = A.alloc(n);
  memcpy(&A.buf[off], src, sizeof(float) * n);
  return off;
}

// One highway layer (modules.py:79-89) as ONE GEMM: W_H, W_T [128][128] -> [128][256] with columns interleaved (H_c, T_c),
// biases likewise [256] (the epilogues and highway4_kernel read the gate pair of channel c from columns 2c, 2c + 1).
// Returns the offset of the weights.
size_t put_highway(Arena& A, const float* wh, const float* bh, const float* wt, const float* bt, size_t& b_off) {
  const size_t w_off = A.alloc(128 * 256);
  b_off = A.alloc(256);
  for (int r = 0; r < 128; ++r)
    for (int c = 0; c < 128; ++c) {
      A.buf[w_off + (size_t)r * 256 + 2 * c] = wh[(size_t)r * 128 + c];
      A.buf[w_off + (size_t)r * 256 + 2 * c + 1] = wt[(size_t)r * 128 + c];
    }
  for (int c = 0; c < 128; ++c) {
    A.buf[b_off + 2 * c] = bh[c];
    A.buf[b_off + 2 * c + 1] = bt[c];
  }
  return w_off;
}

// W^T of a GEMM as bf16 hi / lo at g.b_hi / g.b_lo, from its fp32 weights at g.w: one pack launch per bank member
void pack_gemmw(const GemmW& g, cudaStream_t st) {
  for (int ci = 0; ci < g.bank; ++ci)
    launch_pack_wt(g.member_w(ci), g.ldw, g.member_taps(ci), g.Cin, g.Cout, g.Cp, g.Kld, ci * g.Cout, g.b_hi, g.b_lo, st);
}

// conv1d() of the reference: kernel/bias + BN.  Emits weights, bias and the four
// BN-derived vectors at given column offset of pre-allocated vectors.
bool pack_bn(taco_handle* h, const std::string& scope, int C, float* scale, float* shift, float* gamma,
             float* beta, std::string& err) {
  const std::string bn = scope + "/batch_normalization/";
  GETV(g, bn + "gamma", C);
  GETV(b, bn + "beta", C);
  GETV(mm, bn + "moving_mean", C);
  GETV(mv, bn + "moving_variance", C);
  for (int c = 0; c < C; ++c) {
    const float sc = g->data[c] / sqrtf(mv->data[c] + kBnEps);
    scale[c] = sc;
    shift[c] = b->data[c] - mm->data[c] * sc;
    gamma[c] = g->data[c];
    beta[c] = b->data[c];
  }
  return true;
}

bool pack_cbhg(taco_handle* h, Arena& A, const std::string& s, int K, int Cin, int P1, int P2, CbhgDev& D,
               std::string& err) {
  D.K = K; D.Cin = Cin; D.P1 = P1; D.P2 = P2;
  const int BC = K * 128;
  D.bank_scale = A.alloc(BC); D.bank_shift = A.alloc(BC); D.bank_gamma = A.alloc(BC); D.bank_beta = A.alloc(BC);
  D.bank_bias = A.alloc(BC);
  D.g_bank = make_gemmw(A.alloc((size_t)K * (K + 1) / 2 * Cin * 128), 128, K, Cin, 128, K);
  for (int k = 1; k <= K; ++k) {
    const std::string sc = s + "/conv_bank/conv1d_" + std::to_string(k);
    GETV(w, sc + "/conv1d/kernel", k, Cin, 128);
    GETV(b, sc + "/conv1d/bias", 128);
    memcpy(&A.buf[D.g_bank.off + (size_t)(k - 1) * k / 2 * Cin * 128], w->data.data(), sizeof(float) * k * Cin * 128);
    const int o = (k - 1) * 128;
    memcpy(&A.buf[D.bank_bias + o], b->data.data(), sizeof(float) * 128);
    if (!pack_bn(h, sc, 128, &A.buf[D.bank_scale + o], &A.buf[D.bank_shift + o], &A.buf[D.bank_gamma + o],
                 &A.buf[D.bank_beta + o], err))
      return false;
  }
  {
    GETV(w, s + "/proj_1/conv1d/kernel", 3, BC, P1);
    GETV(b, s + "/proj_1/conv1d/bias", P1);
    D.g_p1 = make_gemmw(put_matrix(A, w->data.data(), 3 * BC, P1, P1), P1, 3, BC, P1);
    D.p1_b = put_vec(A, b->data.data(), P1);
    D.p1_scale = A.alloc(P1); D.p1_shift = A.alloc(P1); D.p1_gamma = A.alloc(P1); D.p1_beta = A.alloc(P1);
    if (!pack_bn(h, s + "/proj_1", P1, &A.buf[D.p1_scale], &A.buf[D.p1_shift], &A.buf[D.p1_gamma],
                 &A.buf[D.p1_beta], err))
      return false;
  }
  {
    GETV(w, s + "/proj_2/conv1d/kernel", 3, P1, P2);
    GETV(b, s + "/proj_2/conv1d/bias", P2);
    D.g_p2 = make_gemmw(put_matrix(A, w->data.data(), 3 * P1, P2, P2), P2, 3, P1, P2);
    D.p2_b = put_vec(A, b->data.data(), P2);
    D.p2_scale = A.alloc(P2); D.p2_shift = A.alloc(P2); D.p2_gamma = A.alloc(P2); D.p2_beta = A.alloc(P2);
    if (!pack_bn(h, s + "/proj_2", P2, &A.buf[D.p2_scale], &A.buf[D.p2_shift], &A.buf[D.p2_gamma],
                 &A.buf[D.p2_beta], err))
      return false;
  }
  if (P2 != 128) {   // reference modules.py:59-60
    GETV(w, s + "/dense/kernel", P2, 128);
    GETV(b, s + "/dense/bias", 128);
    D.g_dense = make_gemmw(put_matrix(A, w->data.data(), P2, 128, 128), 128, 1, P2, 128);
    D.dense_b = put_vec(A, b->data.data(), 128);
  }
  for (int i = 0; i < 4; ++i) {
    const std::string hs = s + "/highway_" + std::to_string(i + 1);
    GETV(wh, hs + "/H/kernel", 128, 128);
    GETV(bh, hs + "/H/bias", 128);
    GETV(wt, hs + "/T/kernel", 128, 128);
    GETV(bt, hs + "/T/bias", 128);
    D.g_hw[i] = make_gemmw(put_highway(A, wh->data.data(), bh->data.data(), wt->data.data(), bt->data.data(), D.hw_b[i]),
                           256, 1, 128, 256);
  }
  // BiGRU: gates/kernel [256,256] rows = [x(128); h(128)], candidate/kernel [256,128] likewise.
  const size_t gru_wx = A.alloc(128 * 768);
  D.gru_bx = A.alloc(768);
  D.gru_ug = A.alloc(2 * 128 * 256); D.gru_uc = A.alloc(2 * 128 * 128);
  int d = 0;
  for (const char* dn : {"fw", "bw"}) {
    const std::string gs = s + "/bidirectional_rnn/" + dn + "/gru_cell";
    GETV(wg, gs + "/gates/kernel", 256, 256);
    GETV(bg, gs + "/gates/bias", 256);
    GETV(wc, gs + "/candidate/kernel", 256, 128);
    GETV(bc, gs + "/candidate/bias", 128);
    for (int r = 0; r < 128; ++r) {
      memcpy(&A.buf[gru_wx + (size_t)r * 768 + d * 384], &wg->data[(size_t)r * 256], sizeof(float) * 256);
      memcpy(&A.buf[gru_wx + (size_t)r * 768 + d * 384 + 256], &wc->data[(size_t)r * 128], sizeof(float) * 128);
      memcpy(&A.buf[D.gru_ug + ((size_t)d * 128 + r) * 256], &wg->data[(size_t)(128 + r) * 256], sizeof(float) * 256);
      memcpy(&A.buf[D.gru_uc + ((size_t)d * 128 + r) * 128], &wc->data[(size_t)(128 + r) * 128], sizeof(float) * 128);
    }
    memcpy(&A.buf[D.gru_bx + d * 384], bg->data.data(), sizeof(float) * 256);
    memcpy(&A.buf[D.gru_bx + d * 384 + 256], bc->data.data(), sizeof(float) * 128);
    ++d;
  }
  D.gru_frag = A.alloc(bigru_mma_frag_words());
  bigru_mma_pack(&A.buf[D.gru_ug], &A.buf[D.gru_uc], reinterpret_cast<uint32_t*>(&A.buf[D.gru_frag]));
  D.g_xproj = make_gemmw(gru_wx, 768, 1, 128, 768);
  return true;
}

// Cut src[rows r0..r0+K) x given column lists] into CS per-CTA slices [CS][K][Mc].
// colmap(q, c) -> source column (or -1 for zero padding).
template <class F>
size_t put_slices(Arena& A, const float* src, int ld, int r0, int K, int CS, int Mc, F colmap) {
  size_t off = A.alloc((size_t)CS * K * Mc);
  for (int q = 0; q < CS; ++q)
    for (int k = 0; k < K; ++k)
      for (int c = 0; c < Mc; ++c) {
        const int sc = colmap(q, c);
        A.buf[off + ((size_t)q * K + k) * Mc + c] = sc < 0 ? 0.0f : src[(size_t)(r0 + k) * ld + sc];
      }
  return off;
}

struct DecOff {   // arena offsets of the decoder slices
  size_t p1_s, p1_b, p2_s, p2_b, ga_s, ga_b, cxa_s, cha_s, ca_b, qp_s, att_v, pc_s, pc_b;
  size_t g1_s, g1_b, cx1_s, ch1_s, c1_b, g2_s, g2_b, cx2_s, ch2_s, c2_b, o_s, o_b;
};

bool pack_decoder(taco_handle* h, Arena& A, int CS, DecOff& O, int& McO, std::string& err) {
  const int M = h->hp.num_mels, r = h->hp.outputs_per_step, Dout = M * r;
  const int Hc = DH / CS, Pc = DP / CS;
  McO = (CS == 16) ? 32 : 64;
  const std::string att = kATT, dpw = att + "decoder_prenet_wrapper/", mrc = kMRC;
  auto plain = [](int Mc) { return [Mc](int q, int c) { return q * Mc + c; }; };
  // gate columns: slice q = [r-cols q*Hc.. | u-cols 256+q*Hc..]  (TF GRUCell: r first, u second)
  auto gatecols = [Hc](int q, int c) { return c < Hc ? q * Hc + c : DH + q * Hc + (c - Hc); };
  {
    GETV(w1, dpw + "decoder_prenet/dense_1/kernel", M + DH, 256);
    GETV(b1, dpw + "decoder_prenet/dense_1/bias", 256);
    GETV(w2, dpw + "decoder_prenet/dense_2/kernel", 256, 128);
    GETV(b2, dpw + "decoder_prenet/dense_2/bias", 128);
    O.p1_s = put_slices(A, w1->data.data(), 256, 0, M + DH, CS, Hc, plain(Hc));
    O.p1_b = put_vec(A, b1->data.data(), 256);
    O.p2_s = put_slices(A, w2->data.data(), 128, 0, 256, CS, Pc, plain(Pc));
    O.p2_b = put_vec(A, b2->data.data(), 128);
  }
  auto pack_gru = [&](const std::string& scope, int Kx, size_t& g_s, size_t& g_b, size_t& cx_s, size_t& ch_s,
                      size_t& c_b) -> bool {
    GETV(wg, scope + "/gates/kernel", Kx + DH, 2 * DH);
    GETV(bg, scope + "/gates/bias", 2 * DH);
    GETV(wc, scope + "/candidate/kernel", Kx + DH, DH);
    GETV(bc, scope + "/candidate/bias", DH);
    g_s = put_slices(A, wg->data.data(), 2 * DH, 0, Kx + DH, CS, 2 * Hc, gatecols);
    g_b = A.alloc(2 * DH);
    for (int q = 0; q < CS; ++q)
      for (int c = 0; c < 2 * Hc; ++c) A.buf[g_b + q * 2 * Hc + c] = bg->data[gatecols(q, c)];
    cx_s = put_slices(A, wc->data.data(), DH, 0, Kx, CS, Hc, plain(Hc));
    ch_s = put_slices(A, wc->data.data(), DH, Kx, DH, CS, Hc, plain(Hc));
    c_b = put_vec(A, bc->data.data(), DH);
    return true;
  };
  if (!pack_gru(dpw + "gru_cell", DP, O.ga_s, O.ga_b, O.cxa_s, O.cha_s, O.ca_b)) return false;
  if (!pack_gru(mrc + "cell_1/gru_cell", DH, O.g1_s, O.g1_b, O.cx1_s, O.ch1_s, O.c1_b)) return false;
  if (!pack_gru(mrc + "cell_2/gru_cell", DH, O.g2_s, O.g2_b, O.cx2_s, O.ch2_s, O.c2_b)) return false;
  {
    GETV(wq, att + "bahdanau_attention/query_layer/kernel", 256, 256);
    GETV(v, att + "bahdanau_attention/attention_v", 256);
    GETV(wp, mrc + "cell_0/output_projection_wrapper/kernel", 512, 256);
    GETV(bp, mrc + "cell_0/output_projection_wrapper/bias", 256);
    // [Wq slice | Wproj[:256] slice] side by side: [CS][256][2*Hc]
    O.qp_s = A.alloc((size_t)CS * DH * 2 * Hc);
    for (int q = 0; q < CS; ++q)
      for (int k = 0; k < DH; ++k)
        for (int c = 0; c < Hc; ++c) {
          A.buf[O.qp_s + ((size_t)q * DH + k) * 2 * Hc + c] = wq->data[(size_t)k * 256 + q * Hc + c];
          A.buf[O.qp_s + ((size_t)q * DH + k) * 2 * Hc + Hc + c] = wp->data[(size_t)k * 256 + q * Hc + c];
        }
    O.att_v = put_vec(A, v->data.data(), 256);
    O.pc_s = put_slices(A, wp->data.data(), 256, 256, DH, CS, Hc, plain(Hc));
    O.pc_b = put_vec(A, bp->data.data(), 256);
  }
  {
    GETV(wo, "decoder/output_projection_wrapper/kernel", 256, Dout);
    GETV(bo, "decoder/output_projection_wrapper/bias", Dout);
    O.o_s = put_slices(A, wo->data.data(), Dout, 0, DH, CS, McO,
                       [McO, Dout](int q, int c) { int col = q * McO + c; return col < Dout ? col : -1; });
    O.o_b = A.alloc(CS * McO);
    memcpy(&A.buf[O.o_b], bo->data.data(), sizeof(float) * Dout);
  }
  return true;
}

// bf16 split helpers of the packers
inline uint16_t bf16_rn(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);   // NaN
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
inline float bf16_f(uint16_t b) { uint32_t u = (uint32_t)b << 16; float f; memcpy(&f, &u, 4); return f; }

#include "decoder_cw_pack.inc"

// ---- workspace ---------------------------------------------------------------
struct Bump {
  char* base; size_t cap, off = 0; bool overflow = false;
  Bump(char* b, size_t c) : base(b), cap(c) {}
  template <class T> T* take(size_t n) {
    off = (off + 255) & ~size_t(255);
    size_t bytes = n * sizeof(T);
    T* p = reinterpret_cast<T*>(base + off);
    off += bytes;
    if (off > cap) overflow = true;
    return p;
  }
};

size_t cbhg_ws_floats(int K, int P1, int P2, int64_t rows) {
  // bank + pooled + p1 + p2 + dense + 2 highway + xproj, plus slack for alignment
  return (size_t)rows * ((size_t)3 * K * 128 + P1 + P2 + 128 + 256 + 768 + 256) + 32768;   // + bf16 hi/lo staging (wide + narrow)
}

int ensure_ws(taco_handle* h, size_t bytes) {
  if (bytes <= h->ws_bytes) return TACO_OK;
  if (h->ws) { cudaDeviceSynchronize(); cudaFree(h->ws); h->ws = nullptr; h->ws_bytes = 0; }
  bytes += bytes / 8;
  CUDA_OK(h, cudaMalloc(&h->ws, bytes));
  h->ws_bytes = bytes;
  return TACO_OK;
}
int ensure_ints(taco_handle* h, int n) {
  if (n <= h->d_ints_n) return TACO_OK;
  if (h->d_ints) { cudaDeviceSynchronize(); cudaFree(h->d_ints); h->d_ints = nullptr; }
  CUDA_OK(h, cudaMalloc(&h->d_ints, sizeof(int) * n));
  CUDA_OK(h, cudaMemset(h->d_ints, 0, sizeof(int) * n));
  h->d_ints_n = n;
  return TACO_OK;
}

struct Ctx {
  taco_handle* h;
  cudaStream_t st;
  const float* W(size_t off) const { return h->dW + off; }
};

// A launcher returned e: the first such error of a call stays in h->err, and check_launch returns it at the end of the call.
void launch_error(taco_handle* h, cudaError_t e, const char* what) {
  if (e == cudaSuccess) return;
  if (!h->launch_failed) h->err = std::string(what) + ": " + cudaGetErrorString(e);
  h->launch_failed = true;
}

// bf16 hi/lo staging of a GEMM's activation operand (tcgen05 path)
struct BfScratch { void* hi = nullptr; void* lo = nullptr; };
BfScratch take_bf(Bump& ws, int64_t rows, int maxCp) {
  BfScratch s;
  s.hi = ws.take<uint16_t>((size_t)rows * maxCp);
  s.lo = ws.take<uint16_t>((size_t)rows * maxCp);
  return s;
}

// A operand [N][T][Cin] of a GEMM: fp32 x[n*x_bs + t*ldx + c], split into bf ahead of a tensor-core launch; or, presplit,
// already in bf as the hi / lo operand (written by the producer's epilogue), and x is not read.
struct GemmIn { const float* x; int64_t x_bs; int ldx; BfScratch bf; bool presplit = false; };
// Epilogue: act(acc + bias), then the per-channel affine, then the residual; EPI_HIGHWAY reads res as the carry input.
// A bank's convolution ci reads bias / scale / shift at ci*Cout.
struct GemmEpi {
  int act = TACO_ACT_NONE;
  const float* bias = nullptr; const float* scale = nullptr; const float* shift = nullptr;
  const float* res = nullptr; int64_t res_bs = 0; int ldres = 0;
  int epi = EPI_PLAIN;
};
// Results: fp32 out[n*out_bs + t*ldo + col_off + c], not written when out is null; on the tensor cores, optionally also the
// hi / lo operand [N][T][copy_cp] of the GEMM that consumes the result, so that no split pass runs in between.
struct GemmOut {
  float* out; int64_t out_bs; int ldo; int col_off = 0;
  const BfScratch* copy = nullptr; int copy_cp = 0;
};

// The tensor-core launch of one GEMM site; a is the split A operand.
ConvUmma make_umma(const GemmW& g, int N, int T, const BfScratch& a, const GemmEpi& ep, const GemmOut& o, int nsplit) {
  ConvUmma u;
  u.a_hi = a.hi; u.a_lo = a.lo; u.N = N; u.T = T; u.Cp = g.Cp; u.Cin = g.Cin;
  u.b_hi = g.b_hi; u.b_lo = g.b_lo; u.b_rows = g.b_rows; u.Kld = g.Kld;
  u.taps = g.taps; u.bank = g.bank; u.Cout = g.Cout; u.nsplit = nsplit;
  u.bias = ep.bias; u.scale = ep.scale; u.shift = ep.shift; u.res = ep.res; u.res_bs = ep.res_bs; u.ldres = ep.ldres;
  u.out = o.out; u.out_bs = o.out_bs; u.ldo = o.ldo; u.col_off = o.col_off; u.act = ep.act; u.epi = ep.epi;
  if (o.copy) { u.out_hi = o.copy->hi; u.out_lo = o.copy->lo; u.out_cp = o.copy_cp; }
  return u;
}

// One conv1d / dense site in the handle's gemm mode: the fp32 FFMA kernel (mode 0, one launch per bank member), or the split
// pass unless the operand is presplit, then the tensor-core kernel (mode 1: three bf16 products, mode 2: one).  *plan (if
// given) receives the tensor-core launch's plan.  A failed launch is also recorded as the call's sticky launch error.
cudaError_t run_gemm(Ctx& c, const GemmW& g, int N, int T, const GemmIn& in, const GemmEpi& ep, const GemmOut& o,
                     taco_gemm_plan* plan = nullptr) {
  taco_handle* h = c.h;
  if (h->gemm_mode == 0) {
    for (int ci = 0; ci < g.bank; ++ci) {
      const int m = ci * g.Cout;
      ConvGemm p;
      p.x = in.x; p.x_bs = in.x_bs; p.ldx = in.ldx; p.N = N; p.T = T; p.Cin = g.Cin; p.k = g.member_taps(ci);
      p.w = g.member_w(ci); p.ldw = g.ldw;
      p.bias = ep.bias ? ep.bias + m : nullptr; p.scale = ep.scale ? ep.scale + m : nullptr; p.shift = ep.shift ? ep.shift + m : nullptr;
      p.res = ep.res; p.res_bs = ep.res_bs; p.ldres = ep.ldres;
      p.out = o.out; p.out_bs = o.out_bs; p.ldo = o.ldo; p.col_off = o.col_off + m; p.Cout = g.Cout; p.act = ep.act; p.epi = ep.epi;
      launch_conv_gemm(p, c.st);
    }
    h->launches += g.bank;
    return cudaSuccess;
  }
  if (!in.presplit) launch_split_bf16(in.x, in.x_bs, in.ldx, N, T, g.Cin, g.Cp, in.bf.hi, in.bf.lo, c.st);
  const cudaError_t e = launch_conv_umma(make_umma(g, N, T, in.bf, ep, o, h->gemm_mode == 2 ? 1 : 3), c.st, plan);
  launch_error(h, e, "conv_umma launch");
  h->launches += in.presplit ? 1 : 2;
  return e;
}

// BiGRU recurrence: the fp32 FFMA kernel (1 utterance per CTA, weights in registers; default) or, TACO_BIGRU=mma, the
// tensor-core kernel (8 utterances per CTA, weights in tensor memory: 8 CTAs instead of 64 for a batch of 32, but
// 1.8 us instead of 0.8 us per step as it stands -- its epilogues and the tensor pipe do not overlap yet).
void run_bigru(Ctx& c, const CbhgDev& D, const float* xproj, const int32_t* lengths, int N, int T, float* out, int64_t out_bs) {
  const char* impl = c.h->dev_env ? getenv("TACO_BIGRU") : nullptr;   // developer switch (TACO_DEV=1): the parity tests run both
  const bool use_mma = impl && std::string(impl) == "mma";
  if (use_mma) {
    launch_error(c.h, launch_bigru_mma(xproj, c.W(D.gru_frag), lengths, N, T, out, out_bs, c.st), "bigru_mma launch");
  } else {
    launch_bigru(xproj, c.W(D.gru_ug), c.W(D.gru_uc), lengths, N, T, out, out_bs, c.st);
  }
  c.h->launches += 1;
}

// reference cbhg() (models/modules.py:35-74).  x: [N,T,Cin] with batch stride x_bs; out [N,T,256] dense.
// x_split (tensor-core path): x already as the conv bank's hi/lo operand [N][T][g_bank.Cp] (written by the producer's epilogue)
void run_cbhg(Ctx& c, const CbhgDev& D, Bump& ws, const float* x, int64_t x_bs, const int32_t* lengths, int N,
              int T, int bn_mode, float* out, const BfScratch* x_split = nullptr) {
  const int K = D.K, BC = K * 128, Cin = D.Cin;
  const int64_t rows = (int64_t)N * T;
  float* bank = ws.take<float>(rows * BC);
  float* pooled = ws.take<float>(rows * BC);
  float* p1 = ws.take<float>(rows * D.P1);
  float* p2 = ws.take<float>(rows * D.P2);
  float* hwa = ws.take<float>(rows * 128);
  float* hwb = ws.take<float>(rows * 128);
  float* xproj = ws.take<float>(rows * 768);
  float* bnv = ws.take<float>(2 * 2048);          // batch-mode scale | shift
  double* bnacc = ws.take<double>(2 * 2048);
  BfScratch sc, sc2;                 // sc: operands as wide as the bank output; sc2: the narrow ones in between (<= 256 channels)
  if (c.h->gemm_mode != 0) { sc = take_bf(ws, rows, BC); sc2 = take_bf(ws, rows, 256); }
  if (ws.overflow) return;
  const bool batch = bn_mode == TACO_BN_BATCH;
  // Producer-side operand split (tensor-core path, moving statistics): a GEMM whose result is only (or also) the A operand of
  // the next GEMM writes it as bf16 hi/lo from its own epilogue -- proj_1 -> proj_2, proj_2 -> dense -- instead of an fp32 round
  // trip through split_bf16_kernel.  Batch statistics need the fp32 tensors (moments, in-place affine): the split passes stay.
  const bool chain = c.h->gemm_mode != 0 && !batch;
  // conv bank: K convolutions written side by side (tf.concat, modules.py:39-42)
  run_gemm(c, D.g_bank, N, T, {x, x_bs, Cin, x_split != nullptr ? *x_split : sc, x_split != nullptr},
           {TACO_ACT_RELU, c.W(D.bank_bias), batch ? nullptr : c.W(D.bank_scale), batch ? nullptr : c.W(D.bank_shift)},
           {bank, (int64_t)T * BC, BC});
  // max-pool (+ batch-mode BN affine); on the tcgen05 path its output goes straight into the GEMM operand format
  const bool fuse_split = c.h->gemm_mode != 0 && D.g_p1.Cp == BC;
  if (batch) {
    launch_bn_batch_stats(bank, (int64_t)T * BC, BC, 0, N, T, BC, c.W(D.bank_gamma), c.W(D.bank_beta), kBnEps,
                          bnacc, bnv, bnv + 2048, c.st);
    c.h->launches += 2;
  }
  if (fuse_split) launch_affine_maxpool_split(bank, sc.hi, sc.lo, N, T, BC, batch ? bnv : nullptr, batch ? bnv + 2048 : nullptr, c.st);
  else launch_affine_maxpool(bank, pooled, N, T, BC, batch ? bnv : nullptr, batch ? bnv + 2048 : nullptr, c.st);
  c.h->launches += 1;
  // proj_1: conv k=3 + ReLU + BN
  run_gemm(c, D.g_p1, N, T, {pooled, (int64_t)T * BC, BC, sc, fuse_split},
           {TACO_ACT_RELU, c.W(D.p1_b), batch ? nullptr : c.W(D.p1_scale), batch ? nullptr : c.W(D.p1_shift)},
           {chain ? nullptr : p1, (int64_t)T * D.P1, D.P1, 0, chain ? &sc2 : nullptr, D.g_p2.Cp});   // proj_1's output feeds proj_2 only
  if (batch) {
    launch_bn_batch_stats(p1, (int64_t)T * D.P1, D.P1, 0, N, T, D.P1, c.W(D.p1_gamma), c.W(D.p1_beta), kBnEps,
                          bnacc, bnv, bnv + 2048, c.st);
    launch_affine_inplace(p1, (int64_t)T * D.P1, D.P1, N, T, D.P1, bnv, bnv + 2048, nullptr, 0, 0, c.st);
    c.h->launches += 3;
  }
  // proj_2: conv k=3 + BN (no activation) + residual (modules.py:53,56)
  const bool p2_to_dense = chain && D.P2 != 128;   // post-net: proj_2's output feeds the 80 -> 128 dense only
  run_gemm(c, D.g_p2, N, T, {p1, (int64_t)T * D.P1, D.P1, chain ? sc2 : sc, chain},
           {TACO_ACT_NONE, c.W(D.p2_b), batch ? nullptr : c.W(D.p2_scale), batch ? nullptr : c.W(D.p2_shift), batch ? nullptr : x,
            x_bs, Cin},
           {p2_to_dense ? nullptr : p2, (int64_t)T * D.P2, D.P2, 0, p2_to_dense ? &sc : nullptr, D.g_dense.Cp});
  if (batch) {
    launch_bn_batch_stats(p2, (int64_t)T * D.P2, D.P2, 0, N, T, D.P2, c.W(D.p2_gamma), c.W(D.p2_beta), kBnEps,
                          bnacc, bnv, bnv + 2048, c.st);
    launch_affine_inplace(p2, (int64_t)T * D.P2, D.P2, N, T, D.P2, bnv, bnv + 2048, x, x_bs, Cin, c.st);
    c.h->launches += 3;
  }
  const float* hin = p2;
  if (D.P2 != 128) {   // modules.py:59-60
    run_gemm(c, D.g_dense, N, T, {p2, (int64_t)T * D.P2, D.P2, sc, p2_to_dense}, {TACO_ACT_NONE, c.W(D.dense_b)},
             {hwb, (int64_t)T * 128, 128});
    hin = hwb;
  }
  // 4 highway layers (modules.py:63-64): one fused launch on the tensor-core path (the activation stays in registers, the result
  // comes out as the hi / lo operand of the GRU input projection), four GEMM launches in gemm mode 0
  const bool hw_fused = c.h->gemm_mode != 0;
  if (hw_fused) {
    const float* hb[4] = {c.W(D.hw_b[0]), c.W(D.hw_b[1]), c.W(D.hw_b[2]), c.W(D.hw_b[3])};
    launch_error(c.h, launch_highway4(hin, nullptr, sc.hi, sc.lo, D.g_hw[0].b_hi, hb, 4, rows, c.h->gemm_mode == 2 ? 1 : 3, c.st),
                 "highway4 launch");
    c.h->launches += 1;
  } else {
    float* bufs[2] = {hwa, hwb};
    int cur = 0;   // first output goes to hwa (hin is p2 or hwb)
    for (int i = 0; i < 4; ++i) {
      float* o = bufs[cur];
      run_gemm(c, D.g_hw[i], N, T, {hin, (int64_t)T * 128, 128, sc},
               {TACO_ACT_NONE, c.W(D.hw_b[i]), nullptr, nullptr, hin, (int64_t)T * 128, 128, EPI_HIGHWAY}, {o, (int64_t)T * 128, 128});
      hin = o;
      cur ^= 1;
    }
  }
  // hoisted GRU input projection for both directions, then the recurrence
  run_gemm(c, D.g_xproj, N, T, {hin, (int64_t)T * 128, 128, sc, hw_fused}, {TACO_ACT_NONE, c.W(D.gru_bx)},
           {xproj, (int64_t)T * 768, 768});
  run_bigru(c, D, xproj, lengths, N, T, out, (int64_t)T * 256);
}

// Decoder launch geometry: (cluster size, samples per cluster).  A cluster streams the whole
// decoder weight set once per step, so fewer/larger clusters save L2 bandwidth while more
// clusters shorten the per-sample work; clusters beyond the co-resident maximum run as extra
// waves.  Per-wave step times (us) measured on B200 (tools/dec_sweep.py, round 1).
// Clusters for the mma.sync decoder (decoder_cw.cu), <= 8 utterances each, maxc of them co-resident.  Every cluster count from
// ceil(N / 8) up is costed as waves x t(S), with t the step time of a cluster of S utterances; among the counts within
// CW_PICK_MARGIN of the cheapest, the fewest clusters win: a cluster holds 16 SMs for the whole decode, so fewer clusters leave
// more of the GPU to the other work in flight.  The margin is 20 %: batch 32 as 4 clusters of 8 decodes 18 % slower than as
// 7 clusters of 5 (11.03 vs 9.38 us/step) but takes 33 % fewer SM-microseconds per step, which is what several batches in
// flight share (+15 % mel frames/s with four in flight).  Small batches pay the same way: batch 4 runs as one cluster of 4.
constexpr float CW_PICK_MARGIN = 0.20f;
// t(S), us per free-running step, S = 1..8: decoder_cw_kernel with four clusters of S utterances at T_in 100 (attention
// operands on chip at every S), tools/dec_sweep.py on a B200 at a 1000 W power limit.
constexpr float CW_STEP_US[8] = {7.60f, 8.21f, 8.86f, 9.11f, 9.38f, 10.45f, 10.78f, 11.03f};
int pick_cw_clusters(int N, int maxc) {
  maxc = std::max(1, maxc);
  const int lo = (N + 7) / 8;
  float best = 1e30f;
  std::vector<float> cost;
  for (int ncl = lo; ncl <= N; ++ncl) {
    const int S = (N + ncl - 1) / ncl;
    cost.push_back((float)((ncl + maxc - 1) / maxc) * CW_STEP_US[S - 1]);
    best = std::min(best, cost.back());
    if (S == 1) break;
  }
  for (size_t i = 0; i < cost.size(); ++i)
    if (cost[i] <= best * (1.0f + CW_PICK_MARGIN)) return lo + (int)i;
  return lo;
}
int pick_mma_clusters(const taco_handle* h, int N) {
  if (h->dec_clusters > 0) return std::min(N, std::max(h->dec_clusters, (N + 7) / 8));
  const char* en = h->dev_env ? getenv("TACO_DEC_NCL") : nullptr;
  if (en && atoi(en) > 0) return std::min(N, std::max(atoi(en), (N + 7) / 8));
  const char* es = h->dev_env ? getenv("TACO_DEC_S") : nullptr;   // samples per cluster (tests sweep it; TACO_DEV=1)
  if (es && atoi(es) > 0) return (N + std::min(atoi(es), 8) - 1) / std::min(atoi(es), 8);
  return pick_cw_clusters(N, h->max_clusters_mma);
}

void pick_geometry(const taco_handle* h, int N, int* cs_out, int* s_out) {
  static const float t_wave[2][4] = {{12.3f, 15.6f, 20.2f, 35.2f},    // CS = 8 : S = 1,2,4,8
                                     {11.2f, 12.7f, 15.5f, 25.6f}};   // CS = 16
  const char* es = h->dev_env ? getenv("TACO_DEC_S") : nullptr;
  const int force_s = es ? atoi(es) : 0;
  float best = 1e30f;
  int bcs = 16, bs = 8;
  for (int ci = 0; ci < 2; ++ci) {
    const int cs = ci ? 16 : 8;
    if (h->force_cs && h->force_cs != cs) continue;
    if (h->max_clusters[ci] < 1) continue;
    for (int si = 0; si < 4; ++si) {
      const int S = 1 << si;
      if (force_s && force_s != S) continue;
      const int clusters = (N + S - 1) / S;
      const int waves = (clusters + h->max_clusters[ci] - 1) / h->max_clusters[ci];
      const float t = waves * t_wave[ci][si];
      if (t < best - 1e-3f) { best = t; bcs = cs; bs = S; }
    }
  }
  *cs_out = bcs;
  *s_out = bs;
}

int check_launch(taco_handle* h, const char* what) {
  if (h->launch_failed) {   // a launcher already consumed the CUDA error: report it instead of returning TACO_OK with garbage outputs
    h->launch_failed = false;
    cudaGetLastError();
    return TACO_ERR_CUDA;   // h->err was set where the launch failed
  }
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(h, TACO_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
  }
  return TACO_OK;
}

int do_encoder(taco_handle* h, Bump& ws, const int32_t* ids, const int32_t* lengths, const int32_t* spk, int N,
               int T_in, int bn_mode, float* memory_out, cudaStream_t st) {
  Ctx c{h, st};
  const taco_hparams& hp = h->hp;
  const bool multi = spk != nullptr && hp.id_num > 1;
  const int E = hp.embedding_text_channels, Es = multi ? hp.embedding_id_channels : 0;
  const int64_t rows = (int64_t)N * T_in;
  float* emb = ws.take<float>(rows * (E + Es));
  float* a1 = ws.take<float>(rows * 256);
  float* a2 = ws.take<float>(rows * 128);
  BfScratch sc, sc2;
  if (h->gemm_mode != 0) { sc = take_bf(ws, rows, 512); sc2 = take_bf(ws, rows, 512); }
  if (ws.overflow) return fail(h, TACO_ERR_INVALID, "workspace overflow (encoder)");
  launch_gather_concat(ids, multi ? spk : nullptr, c.W(h->emb), hp.num_symbols, E, multi ? c.W(h->emb_id) : nullptr,
                       hp.id_num, Es, N, T_in, emb, h->d_ints, st);
  h->launches += 1;
  // encoder prenet (modules.py:5-12; dropout is the identity, SURVEY §0)
  // prenet: dense_1's output feeds dense_2 only, dense_2's feeds the conv bank (as its operand) and proj_2 (as the fp32 residual)
  const bool chain = h->gemm_mode != 0;
  run_gemm(c, h->g_pre1, N, T_in, {emb, (int64_t)T_in * (E + Es), E + Es, sc}, {TACO_ACT_RELU, c.W(h->pre1_b)},
           {chain ? nullptr : a1, (int64_t)T_in * 256, 256, 0, chain ? &sc2 : nullptr, h->g_pre2.Cp});
  run_gemm(c, h->g_pre2, N, T_in, {a1, (int64_t)T_in * 256, 256, chain ? sc2 : sc, chain}, {TACO_ACT_RELU, c.W(h->pre2_b)},
           {a2, (int64_t)T_in * 128, 128, 0, chain ? &sc : nullptr, h->enc.g_bank.Cp});
  run_cbhg(c, h->enc, ws, a2, (int64_t)T_in * 128, lengths, N, T_in, bn_mode, memory_out, chain ? &sc : nullptr);
  if (ws.overflow) return fail(h, TACO_ERR_INVALID, "workspace overflow (encoder cbhg)");
  return check_launch(h, "encoder");
}

size_t encoder_ws_bytes(const taco_handle* h, int N, int T_in) {
  const int64_t rows = (int64_t)N * T_in;
  return sizeof(float) * ((size_t)rows * (h->emb_dim + 256 + 128 + 512 + 512) + cbhg_ws_floats(16, 128, 128, rows)) + 65536;
}
size_t postnet_ws_bytes(const taco_handle* h, int N, int T) {
  const int64_t rows = (int64_t)N * T;
  return sizeof(float) * ((size_t)rows * 512 + cbhg_ws_floats(8, 256, h->hp.num_mels, rows)) + 65536;
}

// defer_count: do not wait for the step count (optimistic max_steps; the caller reads it after its own synchronisation).
// count_later: do not even launch the step-count kernels here: the caller enqueues them (count_steps) after the post-net, which
// does not depend on them, so that they leave the critical path of the forward.
int count_steps(taco_handle* h, const float* dec_out, int N, int max_steps, cudaStream_t st) {
  int rc = ensure_ints(h, 2 + N);
  if (rc) return rc;
  // The step count goes straight into mapped pinned memory: a D2H copy here would queue on the copy engine behind
  // another handle's 144 MB output transfer and stall this forward in the middle (batches in flight on other streams).
  launch_find_steps(dec_out, N, max_steps, h->hp.num_mels * h->hp.outputs_per_step, h->d_ints + 2, h->d_pinned + 1, st);
  h->launches += 3;
  return TACO_OK;
}

int do_decode(taco_handle* h, Bump& ws, const float* memory, int N, int T_in, const float* mel_targets, int T_tgt,
              int teacher_force, float* dec_out, float* align_out, int32_t* steps_out_host, cudaStream_t st,
              bool defer_count = false, bool count_later = false) {
  Ctx c{h, st};
  const taco_hparams& hp = h->hp;
  if (T_in > 512) return fail(h, TACO_ERR_UNSUPPORTED, "T_in > 512 not supported by the decoder kernel");
  if (teacher_force && mel_targets == nullptr) return fail(h, TACO_ERR_INVALID, "teacher_force needs mel_targets");
  const int max_steps = taco_max_steps(h, teacher_force, T_tgt);
  if (max_steps <= 0) return fail(h, TACO_ERR_INVALID, "no decoder steps (T_tgt < r?)");
  float* keys = ws.take<float>((size_t)N * T_in * 256);
  BfScratch sc;
  if (h->gemm_mode != 0) sc = take_bf(ws, (int64_t)N * T_in, 256);
  if (ws.overflow) return fail(h, TACO_ERR_INVALID, "workspace overflow (decoder)");
  // BahdanauAttention memory_layer (no bias), once per utterance (tacotron.py:68)
  run_gemm(c, h->g_mem, N, T_in, {memory, (int64_t)T_in * 256, 256, sc}, {TACO_ACT_NONE}, {keys, (int64_t)T_in * 256, 256});
  DecoderArgs a;
  a.memory = memory; a.keys = keys; a.targets = teacher_force ? mel_targets : nullptr;
  a.N = N; a.T_in = T_in; a.T_tgt = T_tgt; a.r = hp.outputs_per_step; a.steps = max_steps; a.max_steps = max_steps;
  a.dec_out = dec_out; a.align_out = align_out; a.att_res = 0; a.s_max = 0; a.trace = nullptr; a.trace_cta = 0; a.trace_warp = 8;
  const char* trace_path = h->dev_env ? getenv("TACO_DEC_TRACE") : nullptr;   // developer aid (TACO_DEV=1): per-phase clock stamps of one CTA
  long long* d_trace = nullptr;
  if (trace_path) {
    cudaMalloc(&d_trace, 512 * sizeof(long long));
    cudaMemsetAsync(d_trace, 0, 512 * sizeof(long long), st);
    a.trace = d_trace;
    if (const char* tc = getenv("TACO_DEC_TRACE_CTA")) a.trace_cta = atoi(tc);
    if (const char* tw = getenv("TACO_DEC_TRACE_WARP")) a.trace_warp = atoi(tw);
  }
  int CS = 16, S = 8;
  pick_geometry(h, N, &CS, &S);
  if (h->dev_env && getenv("TACO_DEBUG"))
    fprintf(stderr, "[taco] decode N=%d T_in=%d steps=%d CS=%d S=%d kernel=%s max_clusters(8)=%d (16)=%d\n", N, T_in,
            max_steps, CS, S, h->use_cw ? "cw" : "v2", h->max_clusters[0], h->max_clusters[1]);
  if (h->profiling) cudaEventRecord(h->ev[4], st);
  const bool fits8 = (N + pick_mma_clusters(h, N) - 1) / pick_mma_clusters(h, N) <= 8;
  const bool use_cw = h->use_cw && fits8;
  cudaError_t e = use_cw ? launch_decoder_cw(h->decw, a, pick_mma_clusters(h, N), st, /*bf16_only=*/h->gemm_mode == 2)
                         : launch_decoder(h->dec[CS == 16 ? 1 : 0], a, S, st);
  if (h->profiling) cudaEventRecord(h->ev[5], st);
  if (e != cudaSuccess) return fail(h, TACO_ERR_CUDA, std::string("decoder launch: ") + cudaGetErrorString(e));
  h->launches += 1;
  if (d_trace) {
    long long ht[512];
    cudaStreamSynchronize(st);
    cudaMemcpy(ht, d_trace, sizeof(ht), cudaMemcpyDeviceToHost);
    cudaFree(d_trace);
    if (FILE* f = fopen(trace_path, "w")) {
      fprintf(f, "# N=%d T_in=%d CS=%d S=%d\n", N, T_in, CS, S);
      for (int i = 0; i < 512; ++i) fprintf(f, "%d %lld\n", i, ht[i]);
      fclose(f);
    }
  }
  int steps = max_steps;
  if (!teacher_force) {
    if (!count_later) {
      int rc = count_steps(h, dec_out, N, max_steps, st);
      if (rc) return rc;
    }
    if (!defer_count) {
      CUDA_OK(h, cudaStreamSynchronize(st));
      steps = *(volatile int*)(h->h_pinned + 1);
    }   // else: optimistic max_steps; the caller reads h_pinned[1] after its own synchronisation
  }
  if (steps_out_host) *steps_out_host = steps;
  return check_launch(h, "decoder");
}

int do_postnet(taco_handle* h, Bump& ws, const float* mel, int N, int T, int bn_mode, int64_t mel_bs,
               float* linear_out, int64_t lin_bs, cudaStream_t st) {
  Ctx c{h, st};
  const taco_hparams& hp = h->hp;
  float* post = ws.take<float>((size_t)N * T * 256);
  BfScratch sc;
  if (h->gemm_mode != 0) sc = take_bf(ws, (int64_t)N * T, 256);
  if (ws.overflow) return fail(h, TACO_ERR_INVALID, "workspace overflow (postnet)");
  run_cbhg(c, h->post, ws, mel, mel_bs, nullptr, N, T, bn_mode, post);
  if (ws.overflow) return fail(h, TACO_ERR_INVALID, "workspace overflow (postnet cbhg)");
  // linear_outputs = tf.layers.dense(post_outputs, num_freq)  (tacotron.py:101)
  run_gemm(c, h->g_lin, N, T, {post, (int64_t)T * 256, 256, sc}, {TACO_ACT_NONE, c.W(h->lin_b)}, {linear_out, lin_bs, hp.num_freq});
  return check_launch(h, "postnet");
}

// The weight of a unit GEMM (its fp32 weights staged at offset 0, ldw = Cout rounded up to 4).  For a bank, taps = bank: the
// heaviest conv and the width of the weight rows.
GemmW unit_gemmw(const taco_gemm_desc& d) {
  const int bank = d.bank > 1 ? d.bank : 1;
  return make_gemmw(0, (d.Cout + 3) & ~3, bank > 1 ? bank : d.taps, d.Cin, d.Cout, bank);
}
// Its epilogue and outputs, with the parameters at the given device pointers
GemmEpi unit_epi(const taco_gemm_desc& d, const float* bias, const float* scale, const float* shift) {
  return {d.act, bias, scale, shift, d.res, d.res_bs, d.ldres, d.epi};
}
GemmOut unit_out(const taco_gemm_desc& d, const BfScratch& copy) { return {d.out, d.out_bs, d.ldo, d.col_off, &copy, d.out_cp}; }

}  // namespace

// =============================== C ABI ========================================
extern "C" {

const char* taco_version(void) { return "taco_b200 0.1 (sm_100a)"; }

int taco_create(const taco_hparams* hp, int device, taco_handle** out) {
  if (!hp || !out) return TACO_ERR_INVALID;
  *out = nullptr;
  if (hp->num_mels <= 0 || hp->num_mels > 128 || hp->num_mels % 4 || hp->outputs_per_step <= 0 ||
      hp->num_mels * hp->outputs_per_step > 512 || hp->max_iters <= 0 || hp->num_freq <= 0 ||
      hp->embedding_text_channels <= 0 || hp->embedding_text_channels % 4 || hp->embedding_id_channels % 4 ||
      hp->num_symbols <= 0)
    return TACO_ERR_INVALID;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
    cudaGetLastError();
    return TACO_ERR_UNSUPPORTED;   // no GPU: this library has no CPU path
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return TACO_ERR_CUDA;
  if (prop.major != 10) return TACO_ERR_UNSUPPORTED;   // kernels are built for sm_100a only
  if (cudaSetDevice(device) != cudaSuccess) return TACO_ERR_CUDA;
  taco_handle* h = new taco_handle();
  h->hp = *hp;
  h->device = device;
  h->names = expected_names(*hp);
  h->emb_dim = hp->embedding_text_channels + (hp->id_num > 1 ? hp->embedding_id_channels : 0);
  if (cudaHostAlloc(&h->h_pinned, sizeof(int) * 4, cudaHostAllocMapped) != cudaSuccess ||
      cudaHostGetDevicePointer(&h->d_pinned, h->h_pinned, 0) != cudaSuccess) { delete h; return TACO_ERR_CUDA; }
  for (int i = 0; i < 6; ++i) cudaEventCreate(&h->ev[i]);
  {
    // The pipelined host API has one waiting thread per batch in flight.  With more waiting threads than host cores
    // (8 ranks x 6 lanes on a 16-core box) spinning waits starve the threads that enqueue work: TACO_BLOCKING_SYNC=1
    // makes taco_forward_host_wait / _end sleep on blocking-sync events instead.
    const char* bs = getenv("TACO_BLOCKING_SYNC");
    h->blocking = bs && atoi(bs) != 0;
    const char* gr = getenv("TACO_GRAPHS");
    h->graphs_on = !(gr && atoi(gr) == 0);
    const char* dv = getenv("TACO_DEV");
    h->dev_env = dv && atoi(dv) != 0;
    const unsigned flags = cudaEventDisableTiming | (h->blocking ? cudaEventBlockingSync : 0u);
    cudaEventCreateWithFlags(&h->ev_compute, flags);
    cudaEventCreateWithFlags(&h->ev_decoder, flags);
    cudaEventCreateWithFlags(&h->ev_end, flags);
  }
  if (ensure_ints(h, 2 + 1024) != TACO_OK) { taco_destroy(h); return TACO_ERR_CUDA; }
  *out = h;
  return TACO_OK;
}

int taco_destroy(taco_handle* h) {
  if (!h) return TACO_OK;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  if (h->fwd_graph.exec) cudaGraphExecDestroy(h->fwd_graph.exec);
  if (h->gl_graph.exec) cudaGraphExecDestroy(h->gl_graph.exec);
  if (h->dW) cudaFree(h->dW);
  if (h->dB) cudaFree(h->dB);
  if (h->ws) cudaFree(h->ws);
  if (h->stg) cudaFree(h->stg);
  if (h->d_ints) cudaFree(h->d_ints);
  if (h->spec_tab.dev) cudaFree(h->spec_tab.dev);
  if (h->res_tab.dev) cudaFree(h->res_tab.dev);
  if (h->h_pinned) cudaFreeHost(h->h_pinned);
  for (int i = 0; i < 6; ++i) if (h->ev[i]) cudaEventDestroy(h->ev[i]);
  if (h->ev_compute) cudaEventDestroy(h->ev_compute);
  if (h->ev_decoder) cudaEventDestroy(h->ev_decoder);
  if (h->ev_end) cudaEventDestroy(h->ev_end);
  delete h;
  return TACO_OK;
}

const char* taco_last_error(const taco_handle* h) { return h ? h->err.c_str() : "null handle"; }

int taco_num_weights(const taco_handle* h) { return h ? (int)h->names.size() : 0; }
const char* taco_weight_name(const taco_handle* h, int i) {
  if (!h || i < 0 || i >= (int)h->names.size()) return nullptr;
  return h->names[i].c_str();
}

int taco_set_weight(taco_handle* h, const char* tf_name, const float* data_host, const int64_t* shape, int ndim) {
  if (!h || !tf_name || !data_host || !shape || ndim < 1 || ndim > 4) return fail(h, TACO_ERR_INVALID, "bad argument");
  std::string name = tf_name;
  const size_t pl = strlen(kPrefix);
  if (name.compare(0, pl, kPrefix) == 0) name = name.substr(pl);
  bool known = false;
  for (const auto& n : h->names) if (n == name) { known = true; break; }
  if (!known) return fail(h, TACO_ERR_INVALID, "unknown variable: " + std::string(tf_name));
  HostVar& v = h->vars[name];
  v.shape.assign(shape, shape + ndim);
  size_t n = 1;
  for (int i = 0; i < ndim; ++i) { if (shape[i] <= 0) return fail(h, TACO_ERR_INVALID, "bad shape"); n *= (size_t)shape[i]; }
  v.data.assign(data_host, data_host + n);
  v.set = true;
  h->finalized = false;
  return TACO_OK;
}

int taco_finalize_weights(taco_handle* h) {
  if (h && h->fwd_graph.exec) { cudaGraphExecDestroy(h->fwd_graph.exec); h->fwd_graph.exec = nullptr; }
  if (h) h->fwd_graph.have_key = false;
  if (!h) return TACO_ERR_INVALID;
  CUDA_OK(h, cudaSetDevice(h->device));
  const taco_hparams& hp = h->hp;
  std::string err;
  Arena A;
  auto bad = [&](int code) { return fail(h, code, err); };
  auto build = [&]() -> bool {
    GETV(emb, "embedding", hp.num_symbols, hp.embedding_text_channels);
    h->emb = put_vec(A, emb->data.data(), (int)emb->data.size());
    if (hp.id_num > 1) {
      GETV(eid, "embedding_id", hp.id_num, hp.embedding_id_channels);
      h->emb_id = put_vec(A, eid->data.data(), (int)eid->data.size());
    }
    GETV(w1, "prenet/dense_1/kernel", h->emb_dim, 256);
    GETV(b1, "prenet/dense_1/bias", 256);
    GETV(w2, "prenet/dense_2/kernel", 256, 128);
    GETV(b2, "prenet/dense_2/bias", 128);
    h->g_pre1 = make_gemmw(put_matrix(A, w1->data.data(), h->emb_dim, 256, 256), 256, 1, h->emb_dim, 256);
    h->pre1_b = put_vec(A, b1->data.data(), 256);
    h->g_pre2 = make_gemmw(put_matrix(A, w2->data.data(), 256, 128, 128), 128, 1, 256, 128);
    h->pre2_b = put_vec(A, b2->data.data(), 128);
    if (!pack_cbhg(h, A, "encoder_cbhg", 16, 128, 128, 128, h->enc, err)) return false;
    GETV(mw, "memory_layer/kernel", 256, 256);
    h->g_mem = make_gemmw(put_matrix(A, mw->data.data(), 256, 256, 256), 256, 1, 256, 256);
    if (!pack_cbhg(h, A, "post_cbhg", 8, hp.num_mels, 256, hp.num_mels, h->post, err)) return false;
    GETV(lw, "dense/kernel", 256, hp.num_freq);
    GETV(lb, "dense/bias", hp.num_freq);
    const int lin_ld = (hp.num_freq + 3) & ~3;
    h->g_lin = make_gemmw(put_matrix(A, lw->data.data(), 256, hp.num_freq, lin_ld), lin_ld, 1, 256, hp.num_freq);
    h->lin_b = put_vec(A, lb->data.data(), hp.num_freq);
    return true;
  };
  if (!build()) return bad(err.rfind("missing", 0) == 0 ? TACO_ERR_MISSING_WEIGHT : TACO_ERR_INVALID);
  // decoder weight slices for both cluster sizes; the launch picks per batch size (pick_geometry)
  const char* env = getenv("TACO_DEC_CS");
  h->force_cs = env ? atoi(env) : 0;
  if (h->force_cs != 8 && h->force_cs != 16) h->force_cs = 0;
  h->max_clusters[0] = decoder_max_clusters(8);
  h->max_clusters[1] = decoder_max_clusters(16);
  if (h->max_clusters[0] < 1 && h->max_clusters[1] < 1)
    return fail(h, TACO_ERR_UNSUPPORTED, "decoder cluster cannot be scheduled on this device");
  DecOff O[2];
  int McO[2] = {0, 0};
  for (int ci = 0; ci < 2; ++ci)
    if (!pack_decoder(h, A, ci ? 16 : 8, O[ci], McO[ci], err))
      return bad(err.rfind("missing", 0) == 0 ? TACO_ERR_MISSING_WEIGHT : TACO_ERR_INVALID);
  const bool mma_ok = hp.num_mels % 16 == 0 && hp.num_mels <= 128;   // decoder_cw: num_mels and num_mels*r multiples of the 16-column tile
  CwOff O6;
  if (mma_ok && !pack_decoder_cw(h, A, O6, h->decw, err))
    return bad(err.rfind("missing", 0) == 0 ? TACO_ERR_MISSING_WEIGHT : TACO_ERR_INVALID);
  if (h->dW) { cudaDeviceSynchronize(); cudaFree(h->dW); h->dW = nullptr; }
  CUDA_OK(h, cudaMalloc(&h->dW, sizeof(float) * A.buf.size()));
  CUDA_OK(h, cudaMemcpy(h->dW, A.buf.data(), sizeof(float) * A.buf.size(), cudaMemcpyHostToDevice));
  {   // bf16 W^T hi/lo copies for the tcgen05 GEMMs, packed on the device from the fp32 arena
    std::vector<GemmW*> gs = {&h->g_pre1, &h->g_pre2, &h->g_mem, &h->g_lin};
    for (CbhgDev* D : {&h->enc, &h->post}) {
      gs.push_back(&D->g_bank); gs.push_back(&D->g_p1); gs.push_back(&D->g_p2);
      if (D->P2 != 128) gs.push_back(&D->g_dense);
      // the four highway layers back to back, [layer][hi|lo][256][128] (2 * 256 * 128 elements each, a multiple of 128): the
      // layout launch_highway4 reads from g_hw[0].b_hi
      for (int i = 0; i < 4; ++i) gs.push_back(&D->g_hw[i]);
      gs.push_back(&D->g_xproj);
    }
    auto bt_elems = [](const GemmW* g) { return ((size_t)2 * g->b_rows * g->Kld + 127) & ~size_t(127); };
    size_t nb = 0;
    for (GemmW* g : gs) nb += bt_elems(g);
    if (h->dB) { cudaDeviceSynchronize(); cudaFree(h->dB); h->dB = nullptr; }
    CUDA_OK(h, cudaMalloc(&h->dB, sizeof(uint16_t) * nb));
    CUDA_OK(h, cudaMemset(h->dB, 0, sizeof(uint16_t) * nb));
    uint16_t* bt = h->dB;
    for (GemmW* g : gs) {
      g->place(h->dW, bt);
      bt += bt_elems(g);
      pack_gemmw(*g, 0);
    }
    CUDA_OK(h, cudaDeviceSynchronize());
    const char* gm = getenv("TACO_GEMM");
    if (gm) h->gemm_mode = !strcmp(gm, "ffma") ? 0 : (!strcmp(gm, "bf16") ? 2 : 1);
  }
  const float* B = h->dW;
  {
    const char* ei = getenv("TACO_DEC_IMPL");   // "cw" (default) | "v2": developer switch to the fp32 FFMA decoder
    // "cw" (default): decoder_cw.cu
    for (int lay = 0; lay < 2; ++lay) { h->decw.tmem_img[lay] = B + O6.tmem[lay]; h->decw.ring[lay] = B + O6.ring[lay]; }
    h->decw.bias = B + O6.bias; h->decw.att_v = B + O6.att_v;
    h->use_cw = mma_ok && decoder_cw_max_clusters() >= 1 && !(ei && strcmp(ei, "cw") != 0);
    h->max_clusters_mma = h->use_cw ? decoder_cw_max_clusters() : 0;
  }
  for (int ci = 0; ci < 2; ++ci) {
    DecoderWeights& d = h->dec[ci];
    const DecOff& o = O[ci];
    d.CS = ci ? 16 : 8; d.M = hp.num_mels; d.Dout = hp.num_mels * hp.outputs_per_step; d.McO = McO[ci];
    d.p1_s = B + o.p1_s; d.p1_b = B + o.p1_b; d.p2_s = B + o.p2_s; d.p2_b = B + o.p2_b;
    d.ga_s = B + o.ga_s; d.ga_b = B + o.ga_b; d.cxa_s = B + o.cxa_s; d.cha_s = B + o.cha_s; d.ca_b = B + o.ca_b;
    d.qp_s = B + o.qp_s; d.att_v = B + o.att_v; d.pc_s = B + o.pc_s; d.pc_b = B + o.pc_b;
    d.g1_s = B + o.g1_s; d.g1_b = B + o.g1_b; d.cx1_s = B + o.cx1_s; d.ch1_s = B + o.ch1_s; d.c1_b = B + o.c1_b;
    d.g2_s = B + o.g2_s; d.g2_b = B + o.g2_b; d.cx2_s = B + o.cx2_s; d.ch2_s = B + o.ch2_s; d.c2_b = B + o.c2_b;
    d.o_s = B + o.o_s; d.o_b = B + o.o_b;
  }
  h->finalized = true;
  return TACO_OK;
}

int taco_max_steps(const taco_handle* h, int teacher_force, int T_tgt) {
  if (!h) return 0;
  if (!teacher_force) return h->hp.max_iters;
  const int r = h->hp.outputs_per_step;
  // TacoTrainingHelper feeds targets[:, r-1::r], i.e. floor(T_tgt / r) frames (helpers.py:48-55)
  const int n = T_tgt / r;
  return n < h->hp.max_iters ? n : h->hp.max_iters;
}

#define REQUIRE_READY(h)                                                          \
  if (!h) return TACO_ERR_INVALID;                                                \
  if (!h->finalized) return fail(h, TACO_ERR_STATE, "weights not finalized");     \
  CUDA_OK(h, cudaSetDevice(h->device));

int taco_embed(taco_handle* h, const int32_t* ids, const int32_t* spk, int N, int T_in, float* out, void* stream) {
  REQUIRE_READY(h);
  if (!ids || !out || N <= 0 || T_in <= 0) return fail(h, TACO_ERR_INVALID, "bad argument");
  const taco_hparams& hp = h->hp;
  const bool multi = spk != nullptr && hp.id_num > 1;
  launch_gather_concat(ids, multi ? spk : nullptr, h->dW + h->emb, hp.num_symbols, hp.embedding_text_channels,
                       multi ? h->dW + h->emb_id : nullptr, hp.id_num, multi ? hp.embedding_id_channels : 0, N, T_in,
                       out, h->d_ints, (cudaStream_t)stream);
  h->launches += 1;
  return check_launch(h, "embed");
}

int taco_check_ids(taco_handle* h, void* stream) {
  REQUIRE_READY(h);
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_OK(h, cudaMemcpyAsync(h->h_pinned, h->d_ints, sizeof(int), cudaMemcpyDeviceToHost, st));
  CUDA_OK(h, cudaMemsetAsync(h->d_ints, 0, sizeof(int), st));
  CUDA_OK(h, cudaStreamSynchronize(st));
  if (h->h_pinned[0] & 1) return fail(h, TACO_ERR_OOB_ID, "symbol id outside the embedding table");
  if (h->h_pinned[0] & 2) return fail(h, TACO_ERR_OOB_ID, "speaker id outside the embedding_id table");
  return TACO_OK;
}

int taco_encoder(taco_handle* h, const int32_t* ids, const int32_t* lengths, const int32_t* spk, int N, int T_in,
                 int bn_mode, float* memory_out, void* stream) {
  REQUIRE_READY(h);
  if (!ids || !memory_out || N <= 0 || T_in <= 0) return fail(h, TACO_ERR_INVALID, "bad argument");
  int rc = ensure_ws(h, encoder_ws_bytes(h, N, T_in));
  if (rc) return rc;
  Bump ws(h->ws, h->ws_bytes);
  return do_encoder(h, ws, ids, lengths, spk, N, T_in, bn_mode, memory_out, (cudaStream_t)stream);
}

int taco_decode(taco_handle* h, const float* memory, int N, int T_in, const float* mel_targets, int T_tgt,
                int teacher_force, float* dec_out, float* align_out, int32_t* steps_out_host, void* stream) {
  REQUIRE_READY(h);
  if (!memory || !dec_out || N <= 0 || T_in <= 0) return fail(h, TACO_ERR_INVALID, "bad argument");
  if (!al16(memory)) return fail(h, TACO_ERR_INVALID, "memory must be 16-byte aligned");
  int rc = ensure_ws(h, sizeof(float) * (size_t)N * T_in * 512 + 65536);
  if (rc) return rc;
  Bump ws(h->ws, h->ws_bytes);
  return do_decode(h, ws, memory, N, T_in, mel_targets, T_tgt, teacher_force, dec_out, align_out, steps_out_host,
                   (cudaStream_t)stream);
}

int taco_cbhg(taco_handle* h, int which, const float* x, const int32_t* lengths, int N, int T, int bn_mode,
              int64_t x_batch_stride, float* out, void* stream) {
  REQUIRE_READY(h);
  if (!x || !out || N <= 0 || T <= 0) return fail(h, TACO_ERR_INVALID, "bad argument");
  const CbhgDev& D = which == TACO_CBHG_ENCODER ? h->enc : h->post;
  if (x_batch_stride == 0) x_batch_stride = (int64_t)T * D.Cin;
  if (!rows16(x, x_batch_stride, D.Cin))
    return fail(h, TACO_ERR_INVALID, "x must be 16-byte aligned, with a batch stride and a width that are multiples of 4 floats");
  int rc = ensure_ws(h, sizeof(float) * cbhg_ws_floats(D.K, D.P1, D.P2, (int64_t)N * T) + 65536);
  if (rc) return rc;
  Bump ws(h->ws, h->ws_bytes);
  Ctx c{h, (cudaStream_t)stream};
  run_cbhg(c, D, ws, x, x_batch_stride, lengths, N, T, bn_mode, out);
  if (ws.overflow) return fail(h, TACO_ERR_INVALID, "workspace overflow (cbhg)");
  return check_launch(h, "cbhg");
}

int taco_postnet(taco_handle* h, const float* mel, int N, int T, int bn_mode, int64_t mel_batch_stride,
                 float* linear_out, int64_t linear_batch_stride, void* stream) {
  REQUIRE_READY(h);
  if (!mel || !linear_out || N <= 0 || T <= 0) return fail(h, TACO_ERR_INVALID, "bad argument");
  if (mel_batch_stride == 0) mel_batch_stride = (int64_t)T * h->hp.num_mels;
  if (!rows16(mel, mel_batch_stride, h->hp.num_mels))
    return fail(h, TACO_ERR_INVALID, "mel must be 16-byte aligned, with a batch stride and a width that are multiples of 4 floats");
  if (linear_batch_stride == 0) linear_batch_stride = (int64_t)T * h->hp.num_freq;
  int rc = ensure_ws(h, postnet_ws_bytes(h, N, T));
  if (rc) return rc;
  Bump ws(h->ws, h->ws_bytes);
  return do_postnet(h, ws, mel, N, T, bn_mode, mel_batch_stride, linear_out, linear_batch_stride,
                    (cudaStream_t)stream);
}

int taco_bigru(taco_handle* h, int which, const float* x, const int32_t* lengths, int N, int T, float* out,
               void* stream) {
  REQUIRE_READY(h);
  if (!x || !out || N <= 0 || T <= 0) return fail(h, TACO_ERR_INVALID, "bad argument");
  if (!al16(x)) return fail(h, TACO_ERR_INVALID, "x must be 16-byte aligned");
  const CbhgDev& D = which == TACO_CBHG_ENCODER ? h->enc : h->post;
  int rc = ensure_ws(h, sizeof(float) * (size_t)N * T * 1024 + 65536);
  if (rc) return rc;
  Bump ws(h->ws, h->ws_bytes);
  Ctx c{h, (cudaStream_t)stream};
  float* xproj = ws.take<float>((size_t)N * T * 768);
  BfScratch sc;
  if (h->gemm_mode != 0) sc = take_bf(ws, (int64_t)N * T, 128);
  run_gemm(c, D.g_xproj, N, T, {x, (int64_t)T * 128, 128, sc}, {TACO_ACT_NONE, c.W(D.gru_bx)}, {xproj, (int64_t)T * 768, 768});
  run_bigru(c, D, xproj, lengths, N, T, out, (int64_t)T * 256);
  return check_launch(h, "bigru");
}

int taco_conv1d(taco_handle* h, const float* x, int N, int T, int Cin, const float* kernel, const float* bias, int k,
                int Cout, int act, float* out, void* stream) {
  if (!h) return TACO_ERR_INVALID;
  CUDA_OK(h, cudaSetDevice(h->device));
  if (!x || !kernel || !out || N <= 0 || T <= 0 || Cin <= 0 || Cin % 4 || k <= 0 || Cout <= 0)
    return fail(h, TACO_ERR_INVALID, "bad argument (Cin must be a multiple of 4)");
  if (!al16(x) || !al16(kernel)) return fail(h, TACO_ERR_INVALID, "x and kernel must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  Ctx c{h, st};
  GemmIn in{x, (int64_t)T * Cin, Cin, {}};
  GemmW g;
  if (h->gemm_mode != 0) {   // tensor-core path: pack W^T hi/lo and split x on the device, then one UMMA launch
    g = make_gemmw(0, Cout, k, Cin, Cout);
    const size_t nb = (size_t)g.b_rows * g.Kld, na = (size_t)N * T * g.Cp;
    int rc = ensure_ws(h, sizeof(uint16_t) * 2 * (nb + na) + 65536);
    if (rc) return rc;
    Bump ws(h->ws, h->ws_bytes);
    g.w = kernel;
    g.b_hi = ws.take<uint16_t>(nb);
    g.b_lo = ws.take<uint16_t>(nb);
    in.bf = take_bf(ws, (int64_t)N * T, g.Cp);
    pack_gemmw(g, st);
    h->launches += 1;
  } else {
    g = make_gemmw(0, (Cout + 3) & ~3, k, Cin, Cout);
    g.w = kernel;
    if (g.ldw != Cout) {   // pad the leading dimension for 128-bit weight loads
      int rc = ensure_ws(h, sizeof(float) * (size_t)k * Cin * g.ldw + 65536);
      if (rc) return rc;
      CUDA_OK(h, cudaMemsetAsync(h->ws, 0, sizeof(float) * (size_t)k * Cin * g.ldw, st));
      CUDA_OK(h, cudaMemcpy2DAsync(h->ws, sizeof(float) * g.ldw, kernel, sizeof(float) * Cout, sizeof(float) * Cout,
                                   (size_t)k * Cin, cudaMemcpyDeviceToDevice, st));
      g.w = reinterpret_cast<const float*>(h->ws);
    }
  }
  run_gemm(c, g, N, T, in, {act, bias}, {out, (int64_t)T * Cout, Cout});
  return check_launch(h, "conv1d");
}

// ---- unit entry points for the two helper kernels of the CBHG that have no stage of their own --------------------------------
int taco_maxpool_affine(taco_handle* h, const float* x, int N, int T, int C, const float* scale, const float* shift, float* out,
                        void* stream) {
  REQUIRE_READY(h);
  if (!x || !out || N <= 0 || T <= 0 || C <= 0 || (C & 3) || ((scale == nullptr) != (shift == nullptr)))
    return fail(h, TACO_ERR_INVALID, "bad argument");
  launch_affine_maxpool(x, out, N, T, C, scale, shift, (cudaStream_t)stream);
  h->launches += 1;
  return check_launch(h, "maxpool_affine");
}

int taco_bn_batch_stats(taco_handle* h, const float* x, int N, int T, int C, const float* gamma, const float* beta,
                        float* scale_out, float* shift_out, void* stream) {
  REQUIRE_READY(h);
  if (!x || !gamma || !beta || !scale_out || !shift_out || N <= 0 || T <= 0 || C <= 0 || C > 2048)
    return fail(h, TACO_ERR_INVALID, "bad argument");
  int rc = ensure_ws(h, sizeof(double) * 2 * 2048 + 256);
  if (rc) return rc;
  launch_bn_batch_stats(x, (int64_t)T * C, C, 0, N, T, C, gamma, beta, kBnEps, reinterpret_cast<double*>(h->ws), scale_out, shift_out,
                        (cudaStream_t)stream);
  h->launches += 2;
  return check_launch(h, "bn_batch_stats");
}

// ---- the GEMM and the fused highway kernel alone ------------------------------------------------------------------------------
int taco_umma_plan(const taco_gemm_desc* d, int sms, taco_gemm_plan* plan) {
  if (!plan) return TACO_ERR_INVALID;
  memset(plan, 0, sizeof(*plan));
  if (!d) return TACO_ERR_INVALID;
  alignas(16) static const float param[4] = {0.f, 0.f, 0.f, 0.f};   // stands for the parameters the library stores aligned
  const BfScratch copy{d->out_hi, d->out_lo};
  *plan = umma_plan(make_umma(unit_gemmw(*d), d->N, d->T, {},
                              unit_epi(*d, d->bias_host ? param : nullptr, d->scale_host ? param : nullptr, d->shift_host ? param : nullptr),
                              unit_out(*d, copy), 3),
                    sms);
  return plan->valid ? TACO_OK : TACO_ERR_INVALID;
}

int taco_gemm_unit(taco_handle* h, const taco_gemm_desc* d, taco_gemm_plan* plan, void* stream) {
  if (!h) return TACO_ERR_INVALID;
  CUDA_OK(h, cudaSetDevice(h->device));
  if (plan) memset(plan, 0, sizeof(*plan));
  if (!d || d->N <= 0 || d->T <= 0 || d->Cin <= 0 || d->Cout <= 0 || d->bank < 1 || (d->bank == 1 && d->taps < 1) || !d->w_host ||
      (d->epi != TACO_EPI_PLAIN && d->epi != TACO_EPI_HIGHWAY) || ((d->scale_host == nullptr) != (d->shift_host == nullptr)))
    return fail(h, TACO_ERR_INVALID, "bad argument");
  const bool hw = d->epi == TACO_EPI_HIGHWAY, bank = d->bank > 1, presplit = d->x_hi != nullptr;
  if (hw && (d->Cin != 128 || d->Cout != 256 || bank || d->taps != 1 || !d->w2_host || !d->bias_host || !d->bias2_host || !d->res ||
             d->scale_host))
    return fail(h, TACO_ERR_INVALID, "highway: 128 -> 256 interleaved (H, T) columns, one tap, W_T, b_H, b_T and the carry input");
  if (presplit ? d->x_lo == nullptr : (d->x == nullptr || !rows16(d->x, d->x_bs, d->ldx)))
    return fail(h, TACO_ERR_INVALID, "x: 16-byte aligned rows with strides that are multiples of 4 floats, or both halves of a split operand");
  const int gm = h->gemm_mode;
  if (gm == 0 && (presplit || d->out_hi != nullptr || d->out == nullptr))
    return fail(h, TACO_ERR_INVALID, "gemm mode 0 (FFMA) reads and writes fp32 only");
  const int nparam = bank ? d->bank * d->Cout : d->Cout;
  GemmW g = unit_gemmw(*d);
  // parameters: staged on the host as taco_finalize_weights stages them, then one copy to the device
  Arena A;
  size_t b_off = 0, sc_off = 0, sh_off = 0;
  if (hw) g.off = put_highway(A, d->w_host, d->bias_host, d->w2_host, d->bias2_host, b_off);
  else g.off = put_matrix(A, d->w_host, (bank ? d->bank * (d->bank + 1) / 2 : d->taps) * d->Cin, d->Cout, g.ldw);
  if (!hw && d->bias_host) b_off = put_vec(A, d->bias_host, nparam);
  if (d->scale_host) { sc_off = put_vec(A, d->scale_host, nparam); sh_off = put_vec(A, d->shift_host, nparam); }
  const size_t nbt = gm ? (size_t)2 * g.b_rows * g.Kld : 0, na = gm && !presplit ? (size_t)2 * d->N * d->T * g.Cp : 0;
  int rc = ensure_ws(h, sizeof(float) * A.buf.size() + sizeof(uint16_t) * (nbt + na) + 65536);
  if (rc) return rc;
  Bump ws(h->ws, h->ws_bytes);
  float* dP = ws.take<float>(A.buf.size());
  uint16_t* bt = ws.take<uint16_t>(nbt);
  BfScratch sc;
  if (na) sc = take_bf(ws, (int64_t)d->N * d->T, g.Cp);
  if (ws.overflow) return fail(h, TACO_ERR_INVALID, "workspace overflow (gemm unit)");
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_OK(h, cudaMemcpyAsync(dP, A.buf.data(), sizeof(float) * A.buf.size(), cudaMemcpyHostToDevice, st));
  const float* bias = d->bias_host ? dP + b_off : nullptr;
  const float* scale = d->scale_host ? dP + sc_off : nullptr;
  const float* shift = d->scale_host ? dP + sh_off : nullptr;
  g.place(dP, bt);
  if (gm) {
    pack_gemmw(g, st);
    h->launches += g.bank;
  }
  if (presplit) sc = {const_cast<void*>(d->x_hi), const_cast<void*>(d->x_lo)};
  const BfScratch copy{d->out_hi, d->out_lo};
  Ctx c{h, st};
  taco_gemm_plan q = {};
  const cudaError_t e = run_gemm(c, g, d->N, d->T, {d->x, d->x_bs, d->ldx, sc, presplit}, unit_epi(*d, bias, scale, shift),
                                 unit_out(*d, copy), &q);
  if (plan) *plan = q;
  rc = check_launch(h, "gemm unit");
  return e != cudaSuccess && !q.valid ? TACO_ERR_INVALID : rc;   // a refused plan is an invalid argument
}

int taco_highway4_unit(taco_handle* h, const float* x, int64_t rows, int layers, const float* w_h_host, const float* b_h_host,
                       const float* w_t_host, const float* b_t_host, float* out, void* out_hi, void* out_lo, void* stream) {
  if (!h) return TACO_ERR_INVALID;
  CUDA_OK(h, cudaSetDevice(h->device));
  if (!x || rows <= 0 || rows > 0x7fffffffLL || layers < 1 || layers > 4 || !w_h_host || !b_h_host || !w_t_host || !b_t_host ||
      (out == nullptr && out_hi == nullptr) || ((out_hi == nullptr) != (out_lo == nullptr)))
    return fail(h, TACO_ERR_INVALID, "bad argument");
  if (!al16(x) || !al16(out) || !al16(out_hi) || !al16(out_lo)) return fail(h, TACO_ERR_INVALID, "x and the outputs must be 16-byte aligned");
  if (h->gemm_mode == 0) return fail(h, TACO_ERR_UNSUPPORTED, "the fused highway kernel runs on the tensor cores only (gemm mode 1 or 2)");
  Arena A;
  size_t w_off[4], b_off[4];
  for (int l = 0; l < layers; ++l)
    w_off[l] = put_highway(A, w_h_host + (size_t)l * 128 * 128, b_h_host + (size_t)l * 128, w_t_host + (size_t)l * 128 * 128,
                           b_t_host + (size_t)l * 128, b_off[l]);
  GemmW g = make_gemmw(0, 256, 1, 128, 256);
  const size_t per_layer = (size_t)2 * g.b_rows * g.Kld;   // [hi|lo][256][128]: the layout launch_highway4 reads, layer after layer
  int rc = ensure_ws(h, sizeof(float) * A.buf.size() + sizeof(uint16_t) * per_layer * layers + 65536);
  if (rc) return rc;
  Bump ws(h->ws, h->ws_bytes);
  float* dP = ws.take<float>(A.buf.size());
  uint16_t* bt = ws.take<uint16_t>(per_layer * layers);
  if (ws.overflow) return fail(h, TACO_ERR_INVALID, "workspace overflow (highway4 unit)");
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_OK(h, cudaMemcpyAsync(dP, A.buf.data(), sizeof(float) * A.buf.size(), cudaMemcpyHostToDevice, st));
  const float* hb[4] = {nullptr, nullptr, nullptr, nullptr};
  for (int l = 0; l < layers; ++l) {
    g.off = w_off[l];
    g.place(dP, bt + per_layer * l);
    pack_gemmw(g, st);
    hb[l] = dP + b_off[l];
  }
  cudaError_t e = launch_highway4(x, out, out_hi, out_lo, bt, hb, layers, rows, h->gemm_mode == 2 ? 1 : 3, st);
  if (e != cudaSuccess) return fail(h, TACO_ERR_CUDA, std::string("highway4 launch: ") + cudaGetErrorString(e));
  h->launches += layers + 1;
  return check_launch(h, "highway4 unit");
}

int taco_bigru_unit(taco_handle* h, int impl, const float* xproj, const int32_t* lengths, int N, int T, const float* ug_host,
                    const float* uc_host, float* out, void* stream) {
  if (!h) return TACO_ERR_INVALID;
  CUDA_OK(h, cudaSetDevice(h->device));
  if ((impl != 0 && impl != 1) || !xproj || !ug_host || !uc_host || !out || N <= 0 || T <= 0)
    return fail(h, TACO_ERR_INVALID, "bad argument");
  if (!al16(xproj) || !al16(out)) return fail(h, TACO_ERR_INVALID, "xproj and out must be 16-byte aligned");
  // the recurrent kernels (and for impl 1 their fragment stream), staged on the host as pack_cbhg stages them
  Arena A;
  const size_t ug = A.alloc(2 * 128 * 256), uc = A.alloc(2 * 128 * 128);
  memcpy(&A.buf[ug], ug_host, sizeof(float) * 2 * 128 * 256);
  memcpy(&A.buf[uc], uc_host, sizeof(float) * 2 * 128 * 128);
  size_t frag = 0;
  if (impl == 1) {
    frag = A.alloc(bigru_mma_frag_words());
    bigru_mma_pack(&A.buf[ug], &A.buf[uc], reinterpret_cast<uint32_t*>(&A.buf[frag]));
  }
  int rc = ensure_ws(h, sizeof(float) * A.buf.size() + 65536);
  if (rc) return rc;
  Bump ws(h->ws, h->ws_bytes);
  float* dP = ws.take<float>(A.buf.size());
  if (ws.overflow) return fail(h, TACO_ERR_INVALID, "workspace overflow (bigru unit)");
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_OK(h, cudaMemcpyAsync(dP, A.buf.data(), sizeof(float) * A.buf.size(), cudaMemcpyHostToDevice, st));
  const int64_t out_bs = (int64_t)T * 256;
  if (impl == 1) {
    cudaError_t e = launch_bigru_mma(xproj, dP + frag, lengths, N, T, out, out_bs, st);
    if (e != cudaSuccess) return fail(h, TACO_ERR_CUDA, std::string("bigru_mma launch: ") + cudaGetErrorString(e));
  } else {
    launch_bigru(xproj, dP + ug, dP + uc, lengths, N, T, out, out_bs, st);
  }
  h->launches += 1;
  return check_launch(h, "bigru unit");
}

// Post-net again on the true length after an early stop (the all-zero frame case): rare, synchronous.
static int redo_postnet(taco_handle* h, int N, int T_in, int max_steps, int steps, int bn_mode, const float* mel,
                        float* linear_out, cudaStream_t st) {
  const taco_hparams& hp = h->hp;
  const int r = hp.outputs_per_step, maxT = max_steps * r;
  Bump ws(h->ws, h->ws_bytes);
  ws.take<float>((size_t)N * T_in * 256);   // same carve-up as the forward: encoder memory first
  int rc = do_postnet(h, ws, mel, N, steps * r, bn_mode, (int64_t)maxT * hp.num_mels, linear_out,
                      (int64_t)maxT * hp.num_freq, st);
  if (rc) return rc;
  CUDA_OK(h, cudaStreamSynchronize(st));
  return TACO_OK;
}

// defer_final: do not synchronise at all (taco_forward_host_begin); the caller finishes with finish_spec().
static int forward_impl(taco_handle* h, const int32_t* ids, const int32_t* lengths, const int32_t* spk,
                        const float* mel_targets, int N, int T_in, int T_tgt, int bn_mode, int teacher_force, float* mel_out,
                        float* linear_out, float* align_out, int32_t* steps_out_host, void* stream, bool defer_final) {
  REQUIRE_READY(h);
  if (!ids || !mel_out || N <= 0 || T_in <= 0) return fail(h, TACO_ERR_INVALID, "bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const taco_hparams& hp = h->hp;
  const int r = hp.outputs_per_step, M = hp.num_mels;
  const int max_steps = taco_max_steps(h, teacher_force, T_tgt);
  if (max_steps <= 0) return fail(h, TACO_ERR_INVALID, "no decoder steps");
  const int maxT = max_steps * r;
  size_t need = encoder_ws_bytes(h, N, T_in) + sizeof(float) * (size_t)N * T_in * 768 + 65536;
  const size_t need_post = postnet_ws_bytes(h, N, maxT) + sizeof(float) * (size_t)N * T_in * 768 + 65536;
  if (linear_out && need_post > need) need = need_post;
  int rc = ensure_ws(h, need);
  if (rc) return rc;
  rc = ensure_ints(h, 2 + N);
  if (rc) return rc;
  // ---- CUDA graph: replay / capture / plain enqueue ----
  taco_handle::FwdKey key;
  memset(&key, 0, sizeof(key));
  key.ids = ids; key.len = lengths; key.spk = spk; key.tgt = mel_targets; key.mel = mel_out; key.lin = linear_out; key.al = align_out;
  key.ws = h->ws; key.ints = h->d_ints; key.stream = stream;
  key.N = N; key.T_in = T_in; key.T_tgt = T_tgt; key.bn = bn_mode; key.tf = teacher_force; key.gemm_mode = h->gemm_mode;
  key.dec_clusters = h->dec_clusters; key.defer = defer_final ? 1 : 0;
  const bool graph_ok = h->graphs_on && !h->profiling && st != nullptr && st != cudaStreamLegacy && st != cudaStreamPerThread &&
                        !(h->dev_env && (getenv("TACO_DEC_TRACE") != nullptr || getenv("TACO_DEBUG") != nullptr));
  auto& G = h->fwd_graph;
  bool capture = false, replayed = false;
  if (!graph_ok || !G.have_key || !(G.key == key)) {
    if (G.exec) { cudaGraphExecDestroy(G.exec); G.exec = nullptr; }
    G.have_key = graph_ok;
    G.key = key;
  } else if (G.exec) {
    const cudaError_t ge = cudaGraphLaunch(G.exec, st);
    if (ge != cudaSuccess) return fail(h, TACO_ERR_CUDA, std::string("graph launch: ") + cudaGetErrorString(ge));
    h->launches += G.launches;
    replayed = true;
  } else {
    capture = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
    if (!capture) cudaGetLastError();
  }
  int steps = max_steps;
  const int64_t launches0 = h->launches;
  auto enqueue = [&]() -> int {
    Bump ws(h->ws, h->ws_bytes);
    float* memory = ws.take<float>((size_t)N * T_in * 256);
    const size_t mark = ws.off;
    if (h->profiling) cudaEventRecord(h->ev[0], st);
    int rc2 = do_encoder(h, ws, ids, lengths, spk, N, T_in, bn_mode, memory, st);
    if (rc2) return rc2;
    if (h->profiling) cudaEventRecord(h->ev[1], st);
    ws.off = mark;   // encoder scratch is dead; stream order keeps reuse safe
    rc2 = do_decode(h, ws, memory, N, T_in, mel_targets, T_tgt, teacher_force, mel_out, align_out, &steps, st,
                    /*defer_count=*/true, /*count_later=*/true);
    if (rc2) return rc2;
    if (h->profiling) cudaEventRecord(h->ev[2], st);
    if (defer_final) {
      if (capture) cudaEventRecordWithFlags(h->ev_decoder, st, cudaEventRecordExternal);
      else cudaEventRecord(h->ev_decoder, st);
    }
    if (linear_out) {
      ws.off = mark;
      rc2 = do_postnet(h, ws, mel_out, N, steps * r, bn_mode, (int64_t)maxT * M, linear_out,
                       (int64_t)maxT * hp.num_freq, st);
      if (rc2) return rc2;
    }
    if (!teacher_force) {               // dynamic_decode's step count (exact-zero frames): off the critical path, after the post-net
      rc2 = count_steps(h, mel_out, N, max_steps, st);
      if (rc2) return rc2;
    }
    return TACO_OK;
  };
  if (!replayed) {
    rc = enqueue();
    if (capture) {
      cudaGraph_t graph = nullptr;
      const cudaError_t ce = cudaStreamEndCapture(st, &graph);
      if (rc == TACO_OK && ce == cudaSuccess && graph != nullptr) {
        cudaError_t ie = cudaGraphInstantiate(&G.exec, graph, 0);
        if (ie == cudaSuccess) ie = cudaGraphLaunch(G.exec, st);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) {
          if (G.exec) { cudaGraphExecDestroy(G.exec); G.exec = nullptr; }
          G.have_key = false;
          return fail(h, TACO_ERR_CUDA, std::string("graph instantiate / launch: ") + cudaGetErrorString(ie));
        }
        G.launches = h->launches - launches0;
      } else {
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        G.have_key = false;
        if (rc == TACO_OK) return fail(h, TACO_ERR_CUDA, std::string("graph capture: ") + cudaGetErrorString(ce));
      }
    }
    if (rc) return rc;
  }
  if (steps_out_host) *steps_out_host = steps;
  if (h->profiling) cudaEventRecord(h->ev[3], st);
  h->spec.active = false;
  if (!teacher_force) {
    if (defer_final) {
      h->spec.active = true;
      h->spec.N = N; h->spec.T_in = T_in; h->spec.max_steps = max_steps; h->spec.bn_mode = bn_mode;
      h->spec.d_mel = mel_out; h->spec.d_lin = linear_out;
    } else {
      CUDA_OK(h, cudaStreamSynchronize(st));
      steps = *(volatile int*)(h->h_pinned + 1);
      if (steps != max_steps && linear_out) {
        rc = redo_postnet(h, N, T_in, max_steps, steps, bn_mode, mel_out, linear_out, st);
        if (rc) return rc;
      }
      if (steps_out_host) *steps_out_host = steps;
    }
  }
  if (h->profiling && !defer_final) {
    cudaEventSynchronize(h->ev[3]);
    for (int i = 0; i < 3; ++i) cudaEventElapsedTime(&h->stage_ms[i], h->ev[i], h->ev[i + 1]);
    cudaEventElapsedTime(&h->stage_ms[3], h->ev[4], h->ev[5]);
  }
  return TACO_OK;
}

int taco_forward(taco_handle* h, const int32_t* ids, const int32_t* lengths, const int32_t* spk,
                 const float* mel_targets, int N, int T_in, int T_tgt, int bn_mode, int teacher_force, float* mel_out,
                 float* linear_out, float* align_out, int32_t* steps_out_host, void* stream) {
  return forward_impl(h, ids, lengths, spk, mel_targets, N, T_in, T_tgt, bn_mode, teacher_force, mel_out, linear_out,
                      align_out, steps_out_host, stream, /*defer_final=*/false);
}

int taco_forward_host_begin(taco_handle* h, const int32_t* ids_host, const int32_t* lengths_host, const int32_t* spk_host,
                            const float* mel_targets_host, int N, int T_in, int T_tgt, int bn_mode, int teacher_force,
                            float* mel_out_host, float* linear_out_host, float* align_out_host, void* stream) {
  REQUIRE_READY(h);
  h->pending_steps = 0;
  if (!ids_host || !mel_out_host || N <= 0 || T_in <= 0) return fail(h, TACO_ERR_INVALID, "bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const taco_hparams& hp = h->hp;
  const int max_steps = taco_max_steps(h, teacher_force, T_tgt);
  if (max_steps <= 0) return fail(h, TACO_ERR_INVALID, "no decoder steps");
  const int maxT = max_steps * hp.outputs_per_step;
  // device staging lives in a private allocation so that taco_forward may regrow its workspace
  const size_t n_ids = (size_t)N * T_in, n_tgt = teacher_force ? (size_t)N * T_tgt * hp.num_mels : 0;
  const size_t n_mel = (size_t)N * maxT * hp.num_mels, n_lin = linear_out_host ? (size_t)N * maxT * hp.num_freq : 0;
  const size_t n_al = align_out_host ? (size_t)N * T_in * max_steps : 0;
  size_t bytes = 256 * 8 + sizeof(int32_t) * (n_ids + 2 * (size_t)N) + sizeof(float) * (n_tgt + n_mel + n_lin + n_al);
  if (bytes > h->stg_bytes) {
    if (h->stg) { cudaDeviceSynchronize(); cudaFree(h->stg); h->stg = nullptr; h->stg_bytes = 0; }
    CUDA_OK(h, cudaMalloc(&h->stg, bytes));
    h->stg_bytes = bytes;
  }
  Bump b(h->stg, h->stg_bytes);
  int32_t* d_ids = b.take<int32_t>(n_ids);
  int32_t* d_len = b.take<int32_t>(N);
  int32_t* d_spk = b.take<int32_t>(N);
  float* d_tgt = n_tgt ? b.take<float>(n_tgt) : nullptr;
  float* d_mel = b.take<float>(n_mel);
  float* d_lin = n_lin ? b.take<float>(n_lin) : nullptr;
  float* d_al = n_al ? b.take<float>(n_al) : nullptr;
  int rc = TACO_OK;
  auto cp = [&](void* d, const void* s, size_t n, cudaMemcpyKind k) {
    if (rc == TACO_OK && cudaMemcpyAsync(d, s, n, k, st) != cudaSuccess) rc = fail(h, TACO_ERR_CUDA, "memcpy failed");
  };
  cp(d_ids, ids_host, sizeof(int32_t) * n_ids, cudaMemcpyHostToDevice);
  if (lengths_host) cp(d_len, lengths_host, sizeof(int32_t) * N, cudaMemcpyHostToDevice);
  if (spk_host) cp(d_spk, spk_host, sizeof(int32_t) * N, cudaMemcpyHostToDevice);
  if (n_tgt) cp(d_tgt, mel_targets_host, sizeof(float) * n_tgt, cudaMemcpyHostToDevice);
  int steps = 0;
  if (rc == TACO_OK)
    rc = forward_impl(h, d_ids, lengths_host ? d_len : nullptr, spk_host ? d_spk : nullptr, d_tgt, N, T_in, T_tgt,
                      bn_mode, teacher_force, d_mel, d_lin, d_al, &steps, stream, /*defer_final=*/true);
  if (rc == TACO_OK) {
    cudaEventRecord(h->ev_compute, st);
    cp(mel_out_host, d_mel, sizeof(float) * n_mel, cudaMemcpyDeviceToHost);
    if (n_lin) cp(linear_out_host, d_lin, sizeof(float) * n_lin, cudaMemcpyDeviceToHost);
    if (n_al) cp(align_out_host, d_al, sizeof(float) * n_al, cudaMemcpyDeviceToHost);
  }
  h->pending_steps = steps;
  h->spec.lin_host = linear_out_host;
  h->spec.lin_bytes = sizeof(float) * n_lin;
  return rc;   // nothing was waited for: kernels and output copies are in flight on `stream` (taco_forward_host_end)
}

int taco_forward_host_wait(taco_handle* h, int stage) {
  REQUIRE_READY(h);
  if (stage != TACO_STAGE_DECODER && stage != TACO_STAGE_COMPUTE) return fail(h, TACO_ERR_INVALID, "bad stage");
  const cudaError_t e = cudaEventSynchronize(stage == TACO_STAGE_DECODER ? h->ev_decoder : h->ev_compute);
  if (e != cudaSuccess) return fail(h, TACO_ERR_CUDA, std::string("event sync: ") + cudaGetErrorString(e));
  return TACO_OK;
}

int taco_forward_host_end(taco_handle* h, int32_t* steps_out_host, void* stream) {
  REQUIRE_READY(h);
  cudaError_t e;
  if (h->blocking) {
    e = cudaEventRecord(h->ev_end, (cudaStream_t)stream);
    if (e == cudaSuccess) e = cudaEventSynchronize(h->ev_end);
  } else {
    e = cudaStreamSynchronize((cudaStream_t)stream);
  }
  if (e != cudaSuccess) return fail(h, TACO_ERR_CUDA, std::string("sync: ") + cudaGetErrorString(e));
  if (h->spec.active) {   // free-running forward enqueued with the optimistic step count
    h->spec.active = false;
    const int steps = *(volatile int*)(h->h_pinned + 1);
    if (steps != h->spec.max_steps && h->spec.d_lin) {
      int rc2 = redo_postnet(h, h->spec.N, h->spec.T_in, h->spec.max_steps, steps, h->spec.bn_mode, h->spec.d_mel,
                             h->spec.d_lin, (cudaStream_t)stream);
      if (rc2) return rc2;
      if (cudaMemcpy(h->spec.lin_host, h->spec.d_lin, h->spec.lin_bytes, cudaMemcpyDeviceToHost) != cudaSuccess)
        return fail(h, TACO_ERR_CUDA, "memcpy failed");
    }
    h->pending_steps = steps;
    if (h->profiling) {
      for (int i = 0; i < 3; ++i) cudaEventElapsedTime(&h->stage_ms[i], h->ev[i], h->ev[i + 1]);
      cudaEventElapsedTime(&h->stage_ms[3], h->ev[4], h->ev[5]);
    }
  }
  const int rc = taco_check_ids(h, stream);
  if (steps_out_host) *steps_out_host = h->pending_steps;
  return rc;
}

int taco_forward_host(taco_handle* h, const int32_t* ids_host, const int32_t* lengths_host, const int32_t* spk_host,
                      const float* mel_targets_host, int N, int T_in, int T_tgt, int bn_mode, int teacher_force,
                      float* mel_out_host, float* linear_out_host, float* align_out_host, int32_t* steps_out_host,
                      void* stream) {
  const int rc = taco_forward_host_begin(h, ids_host, lengths_host, spk_host, mel_targets_host, N, T_in, T_tgt, bn_mode,
                                         teacher_force, mel_out_host, linear_out_host, align_out_host, stream);
  if (rc != TACO_OK) {
    if (h) cudaStreamSynchronize((cudaStream_t)stream);
    return rc;
  }
  return taco_forward_host_end(h, steps_out_host, stream);
}

static bool audio_geometry(const taco_audio_params* ap, int* hop, int* win) {
  if (!ap || ap->sample_rate <= 0) return false;
  *hop = (int)(ap->frame_shift_ms / 1000.0 * ap->sample_rate);    // util/audio.py:116
  *win = (int)(ap->frame_length_ms / 1000.0 * ap->sample_rate);   // util/audio.py:117
  return *hop >= 1 && *win >= 1;
}

int64_t taco_wav_length(const taco_audio_params* ap, int T) {
  int hop = 0, win = 0;
  if (T < 1 || !audio_geometry(ap, &hop, &win)) return -1;
  return (int64_t)(T - 1) * hop + win;
}

int taco_griffin_lim(taco_handle* h, const taco_audio_params* ap, const float* linear, int N, int T,
                     int64_t linear_batch_stride, float* wav_out, void* stream) {
  if (!h) return TACO_ERR_INVALID;
  CUDA_OK(h, cudaSetDevice(h->device));
  int hop = 0, win = 0;
  if (!linear || !wav_out || N <= 0 || T <= 0 || !audio_geometry(ap, &hop, &win) || ap->griffin_lim_iters < 0)
    return fail(h, TACO_ERR_INVALID, "bad argument");
  const int n_fft = (h->hp.num_freq - 1) * 2;                     // util/audio.py:115
  if (n_fft != 2048 || win > n_fft) return fail(h, TACO_ERR_UNSUPPORTED, "griffin_lim: n_fft must be 2048 and win <= n_fft");
  if ((int64_t)N * T > 0x7fffffff / 1025) return fail(h, TACO_ERR_UNSUPPORTED, "griffin_lim: too many frames for one call");
  int rc = ensure_ws(h, griffin_lim_ws_bytes(N, T, win));
  if (rc) return rc;
  GriffinLimArgs a;
  a.linear = linear;
  a.linear_bs = linear_batch_stride ? linear_batch_stride : (int64_t)T * h->hp.num_freq;
  a.N = N; a.T = T; a.n_fft = n_fft; a.win = win; a.hop = hop; a.iters = ap->griffin_lim_iters;
  a.min_level_db = (float)ap->min_level_db; a.ref_level_db = (float)ap->ref_level_db;
  a.power = (float)ap->power; a.preemphasis = (float)ap->preemphasis;
  a.wav = wav_out;
  int launches = 0;
  cudaStream_t st = (cudaStream_t)stream;
  taco_handle::GlKey key;
  memset(&key, 0, sizeof(key));
  key.a.linear = a.linear; key.a.linear_bs = a.linear_bs; key.a.N = a.N; key.a.T = a.T; key.a.n_fft = a.n_fft; key.a.win = a.win;
  key.a.hop = a.hop; key.a.iters = a.iters; key.a.min_level_db = a.min_level_db; key.a.ref_level_db = a.ref_level_db;
  key.a.power = a.power; key.a.preemphasis = a.preemphasis; key.a.wav = a.wav;
  key.ws = h->ws; key.stream = stream;
  const bool graph_ok = h->graphs_on && st != nullptr && st != cudaStreamLegacy && st != cudaStreamPerThread;
  auto& G = h->gl_graph;
  bool capture = false;
  if (!graph_ok || !G.have_key || memcmp(&G.key, &key, sizeof(key)) != 0) {
    if (G.exec) { cudaGraphExecDestroy(G.exec); G.exec = nullptr; }
    G.have_key = graph_ok;
    G.key = key;
  } else if (G.exec) {                     // third and later identical calls: one graph launch instead of ~105 kernel launches
    CUDA_OK(h, cudaGraphLaunch(G.exec, st));
    h->launches += G.launches;
    return TACO_OK;
  } else {
    capture = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
    if (!capture) cudaGetLastError();
  }
  const cudaError_t le = launch_griffin_lim(a, h->ws, st, &launches);
  if (capture) {
    cudaGraph_t graph = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(st, &graph);
    cudaError_t ie = (le == cudaSuccess && ce == cudaSuccess && graph) ? cudaGraphInstantiate(&G.exec, graph, 0) : cudaErrorUnknown;
    if (graph) cudaGraphDestroy(graph);
    if (ie == cudaSuccess) ie = cudaGraphLaunch(G.exec, st);
    if (ie != cudaSuccess) {               // capture not possible here: plain launches from now on for this key
      cudaGetLastError();
      if (G.exec) { cudaGraphExecDestroy(G.exec); G.exec = nullptr; }
      G.have_key = false;
      launches = 0;
      CUDA_OK(h, launch_griffin_lim(a, h->ws, st, &launches));
    } else {
      G.launches = launches;
    }
  } else {
    CUDA_OK(h, le);
  }
  h->launches += launches;
  return check_launch(h, "griffin_lim");
}

// librosa 0.5.1 filters.mel(sr, n_fft, n_mels) with fmin 0, fmax sr / 2, htk=False (the Slaney scale: linear below 1 kHz
// at 200/3 Hz per mel, log step ln(6.4) / 27 above), in double: the triangle of band i over linspace(0, sr/2, n_fft/2 + 1)
// is max(0, min((f - f_i) / (f_{i+1} - f_i), (f_{i+2} - f) / (f_{i+2} - f_{i+1}))) * 2 / (f_{i+2} - f_i).  Stored sparse:
// band[3 i ..] = (first bin, bin count, offset into w) of the bins where the triangle is positive.
static void mel_band_table(int sr, int n_fft, int num_mels, std::vector<int>& band, std::vector<float>& w) {
  const double f_sp = 200.0 / 3.0, min_log_hz = 1000.0, min_log_mel = min_log_hz / f_sp, logstep = log(6.4) / 27.0;
  auto hz_to_mel = [&](double f) { return f >= min_log_hz ? min_log_mel + log(f / min_log_hz) / logstep : f / f_sp; };
  auto mel_to_hz = [&](double m) { return m >= min_log_mel ? min_log_hz * exp(logstep * (m - min_log_mel)) : f_sp * m; };
  const int bins = n_fft / 2 + 1, npts = num_mels + 2;
  const double f_max = sr / 2.0, mmax = hz_to_mel(f_max);
  std::vector<double> mf(npts);
  for (int i = 0; i < npts; ++i) mf[i] = mel_to_hz(i == npts - 1 ? mmax : i * (mmax / (npts - 1)));   // np.linspace
  band.assign(3 * (size_t)num_mels, 0);
  w.clear();
  for (int i = 0; i < num_mels; ++i) {
    const double enorm = 2.0 / (mf[i + 2] - mf[i]);
    band[3 * i + 2] = (int)w.size();
    for (int k = 0; k < bins; ++k) {
      const double f = k == bins - 1 ? f_max : k * (f_max / (bins - 1));   // np.linspace(0, sr / 2, bins)
      const double v = fmax(0.0, fmin((f - mf[i]) / (mf[i + 1] - mf[i]), (mf[i + 2] - f) / (mf[i + 2] - mf[i + 1])));
      if (v > 0.0) {
        if (band[3 * i + 1] == 0) band[3 * i] = k;
        band[3 * i + 1] = k - band[3 * i] + 1;
        w.resize(band[3 * i + 2] + band[3 * i + 1], 0.0f);
        w.back() = (float)(v * enorm);
      }
    }
  }
}

// byte offsets in h->spec_tab.dev: twiddles (513 float2) | window (up to 2048 floats) | band [num_mels][3] | band weights
struct SpecLayout { size_t win, band, w; };
static SpecLayout spec_layout(int num_mels) {
  auto a256 = [](size_t x) { return (x + 255) & ~size_t(255); };
  SpecLayout o;
  o.win = a256(513 * sizeof(float2));
  o.band = o.win + a256(2048 * sizeof(float));
  o.w = o.band + a256(3 * (size_t)num_mels * sizeof(int));
  return o;
}

// (re)builds h->spec_tab when the sample rate or the window length changes
static int ensure_spec_tables(taco_handle* h, int sr, int win, cudaStream_t st) {
  auto& S = h->spec_tab;
  if (S.dev && S.sample_rate == sr && S.win == win) return TACO_OK;
  std::vector<int> band;
  std::vector<float> bw;
  mel_band_table(sr, 2048, h->hp.num_mels, band, bw);
  const SpecLayout o = spec_layout(h->hp.num_mels);
  const size_t o_win = o.win, o_band = o.band, o_w = o.w, bytes = o_w + bw.size() * sizeof(float) + 256;
  if (S.dev) cudaDeviceSynchronize();   // work on other streams may still read the old tables
  if (bytes > S.bytes) {
    if (S.dev) { cudaFree(S.dev); S.dev = nullptr; S.bytes = 0; }
    CUDA_OK(h, cudaMalloc(&S.dev, bytes));
    S.bytes = bytes;
  }
  S.sample_rate = 0;
  S.host.assign(bytes - o_band, 0);
  memcpy(S.host.data(), band.data(), band.size() * sizeof(int));
  memcpy(S.host.data() + (o_w - o_band), bw.data(), bw.size() * sizeof(float));
  CUDA_OK(h, cudaMemcpyAsync(S.dev + o_band, S.host.data(), S.host.size(), cudaMemcpyHostToDevice, st));
  launch_fft_tables(reinterpret_cast<float2*>(S.dev), reinterpret_cast<float*>(S.dev + o_win), win, st);
  h->launches += 1;
  CUDA_OK(h, cudaPeekAtLastError());
  S.sample_rate = sr;
  S.win = win;
  return TACO_OK;
}

int64_t taco_spectrogram_frames(const taco_audio_params* ap, int64_t L) {
  int hop = 0, win = 0;
  if (L < 1 || !audio_geometry(ap, &hop, &win)) return -1;
  return 1 + L / hop;
}

int taco_spectrogram(taco_handle* h, const taco_audio_params* ap, const float* wav, const int32_t* lengths_host, int N,
                     int64_t L, int T_out, float* linear_out, float* mel_out, void* stream) {
  if (!h) return TACO_ERR_INVALID;
  CUDA_OK(h, cudaSetDevice(h->device));
  int hop = 0, win = 0;
  if (!wav || N <= 0 || L <= 0 || T_out <= 0 || !audio_geometry(ap, &hop, &win))
    return fail(h, TACO_ERR_INVALID, "spectrogram: bad argument");
  int64_t max_frames = 0;
  for (int n = 0; n < N; ++n) {
    const int64_t len = lengths_host ? lengths_host[n] : L;
    if (len < 1 || len > L) return fail(h, TACO_ERR_INVALID, "spectrogram: a length outside [1, L]");
    if (1 + len / hop > max_frames) max_frames = 1 + len / hop;
  }
  if (T_out < max_frames) return fail(h, TACO_ERR_INVALID, "spectrogram: T_out is shorter than the longest utterance's frames");
  const int n_fft = (h->hp.num_freq - 1) * 2;
  if (n_fft != 2048 || win > n_fft) return fail(h, TACO_ERR_UNSUPPORTED, "spectrogram: n_fft must be 2048 and win <= n_fft");
  if ((int64_t)N * T_out * 1025 >= ((int64_t)1 << 31)) return fail(h, TACO_ERR_UNSUPPORTED, "spectrogram: too many frames for one call");
  if (!linear_out && !mel_out) return TACO_OK;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = ensure_spec_tables(h, ap->sample_rate, win, st);
  if (rc) return rc;
  int* d_len = nullptr;
  if (lengths_host) {
    rc = ensure_ws(h, sizeof(int32_t) * (size_t)N + 256);
    if (rc) return rc;
    d_len = reinterpret_cast<int*>(h->ws);
    CUDA_OK(h, cudaMemcpyAsync(d_len, lengths_host, sizeof(int32_t) * (size_t)N, cudaMemcpyHostToDevice, st));
  }
  const char* base = h->spec_tab.dev;
  const SpecLayout o = spec_layout(h->hp.num_mels);
  SpectrogramArgs a;
  a.wav = wav; a.L = L; a.lengths = d_len;
  a.N = N; a.T_out = T_out; a.win = win; a.hop = hop; a.num_mels = h->hp.num_mels;
  a.preemphasis = (float)ap->preemphasis; a.min_level_db = ap->min_level_db; a.ref_level_db = ap->ref_level_db;
  a.tw = reinterpret_cast<const float2*>(base); a.window = reinterpret_cast<const float*>(base + o.win);
  a.band = reinterpret_cast<const int*>(base + o.band); a.band_w = reinterpret_cast<const float*>(base + o.w);
  a.linear = linear_out; a.mel = mel_out;
  CUDA_OK(h, launch_spectrogram(a, st));
  h->launches += 1;
  return check_launch(h, "spectrogram");
}

// ---- resampling: librosa 0.5.1 core.resample / resampy 0.1.5 kaiser_best ----------------------------------------------
static constexpr int kResZeros = 64, kResTable = 512;                   // num_zeros, 2^precision
static constexpr int kResNwin = kResZeros * kResTable + 1;              // 32 769 entries
static constexpr double kResBeta = 14.769656459379492, kResRolloff = 0.9475937167399596;
static constexpr int64_t kResMaxOutputs = (int64_t)1 << 24;            // cap on the replayed positions (20 B each)

static double res_ratio(int32_t sr_orig, int32_t sr_new) { return (double)sr_new / (double)sr_orig; }
static int res_index_step(double ratio) { return (int)(std::min(1.0, ratio) * kResTable); }

// resampy's resample_f register, replayed exactly: a double advanced by 1 / ratio per output (never t / ratio).  Output t
// takes n = int(reg), frac = scale (reg - n); offset / eta of the left wing from frac * 512, of the right wing from
// (scale - frac) * 512.  Kept free of contractions so that it matches the float64 replay of the tests bit for bit.
__attribute__((optimize("fp-contract=off")))
static void res_replay(int32_t sr_orig, int32_t sr_new, int64_t t0, int64_t count, int32_t* n, int32_t* off_l, float* eta_l,
                       int32_t* off_r, float* eta_r) {
  const double ratio = res_ratio(sr_orig, sr_new), scale = std::min(1.0, ratio), inc = 1.0 / ratio;
  double reg = 0.0;
  for (int64_t t = 0; t < t0 + count; reg += inc, ++t) {
    if (t < t0) continue;
    const int64_t k = t - t0;
    const int32_t nn = (int32_t)reg;
    double frac = scale * (reg - nn);
    double index_frac = frac * kResTable;
    const int32_t ol = (int32_t)index_frac;
    const double el = index_frac - ol;
    frac = scale - frac;
    index_frac = frac * kResTable;
    const int32_t orr = (int32_t)index_frac;
    n[k] = nn; off_l[k] = ol; eta_l[k] = (float)el; off_r[k] = orr; eta_r[k] = (float)(index_frac - orr);
  }
}

// kaiser_best's half window (resampy sinc_window: kaiser(2n+1, beta)[n:] * rolloff * sinc(rolloff * linspace(0, 64, n+1)))
// times ratio when downsampling, and its forward difference (last entry 0), laid out as rows[o][i] = (win, delta) at
// o + i index_step for i < (nwin - o) / index_step, zero after.
static void res_rows(double ratio, int taps, std::vector<float2>& rows) {
  std::vector<double> win(kResNwin), delta(kResNwin, 0.0);
  const double n = kResNwin - 1, i0b = std::cyl_bessel_i(0.0, kResBeta);
  for (int m = 0; m < kResNwin; ++m) {
    const double r = m / n, taper = std::cyl_bessel_i(0.0, kResBeta * sqrt(std::max(0.0, 1.0 - r * r))) / i0b;
    const double x = kResRolloff * (m * ((double)kResZeros / n)), s = m == 0 ? 1.0 : sin(M_PI * x) / (M_PI * x);
    win[m] = taper * (kResRolloff * s);
    if (ratio < 1) win[m] *= ratio;
  }
  for (int m = 0; m + 1 < kResNwin; ++m) delta[m] = win[m + 1] - win[m];
  const int step = res_index_step(ratio);
  rows.assign((size_t)RS_ROWS * taps, make_float2(0.0f, 0.0f));
  for (int o = 0; o < RS_ROWS; ++o)
    for (int i = 0; i < (kResNwin - o) / step && i < taps; ++i)
      rows[(size_t)o * taps + i] = make_float2((float)win[o + i * step], (float)delta[o + i * step]);
}

// (re)builds h->res_tab when the rate pair changes or more than the cached positions are needed
static int ensure_res_tables(taco_handle* h, int32_t sr_orig, int32_t sr_new, int64_t n_pos, cudaStream_t st) {
  auto& R = h->res_tab;
  if (R.dev && R.sr_orig == sr_orig && R.sr_new == sr_new && R.n_pos >= n_pos) return TACO_OK;
  const double ratio = res_ratio(sr_orig, sr_new);
  const int taps = kResNwin / res_index_step(ratio);
  std::vector<float2> rows;
  res_rows(ratio, taps, rows);
  std::vector<int32_t> n(n_pos), ol(n_pos), orr(n_pos);
  std::vector<float> el(n_pos), er(n_pos);
  res_replay(sr_orig, sr_new, 0, n_pos, n.data(), ol.data(), el.data(), orr.data(), er.data());
  std::vector<ResamplePos> pos(n_pos);
  int span = 1;
  for (int64_t t = 0; t < n_pos; ++t) {
    pos[t] = ResamplePos{n[t], ol[t], orr[t], el[t], er[t]};
    if (t % RS_T == 0) {
      const int64_t tl = std::min(t + RS_T, n_pos) - 1;
      span = std::max<int64_t>(span, n[tl] - n[t] + 2 * (int64_t)taps);
    }
  }
  const size_t rows_bytes = ((rows.size() * sizeof(float2)) + 255) & ~size_t(255);
  const size_t bytes = rows_bytes + pos.size() * sizeof(ResamplePos);
  if (R.dev) cudaDeviceSynchronize();   // work on other streams may still read the old tables
  R.n_pos = -1;
  if (bytes > R.bytes) {
    if (R.dev) { cudaFree(R.dev); R.dev = nullptr; R.bytes = 0; }
    CUDA_OK(h, cudaMalloc(&R.dev, bytes));
    R.bytes = bytes;
  }
  CUDA_OK(h, cudaMemcpyAsync(R.dev, rows.data(), rows.size() * sizeof(float2), cudaMemcpyHostToDevice, st));
  if (n_pos)
    CUDA_OK(h, cudaMemcpyAsync(R.dev + rows_bytes, pos.data(), pos.size() * sizeof(ResamplePos), cudaMemcpyHostToDevice, st));
  CUDA_OK(h, cudaStreamSynchronize(st));   // the host vectors are the copies' sources
  R.sr_orig = sr_orig; R.sr_new = sr_new; R.taps = taps; R.span = span; R.n_pos = n_pos;
  return TACO_OK;
}

int64_t taco_resample_length(int64_t L, int32_t sr_orig, int32_t sr_new) {
  if (L < 1 || sr_orig <= 0 || sr_new <= 0) return -1;
  return (int64_t)ceil((double)L * res_ratio(sr_orig, sr_new));
}

int taco_resample_positions(int32_t sr_orig, int32_t sr_new, int64_t t0, int64_t count, int32_t* n, int32_t* offset_l,
                            float* eta_l, int32_t* offset_r, float* eta_r) {
  if (sr_orig <= 0 || sr_new <= 0 || t0 < 0 || count < 0 || t0 + count > kResMaxOutputs) return TACO_ERR_INVALID;
  if (count && (!n || !offset_l || !eta_l || !offset_r || !eta_r)) return TACO_ERR_INVALID;
  res_replay(sr_orig, sr_new, t0, count, n, offset_l, eta_l, offset_r, eta_r);
  return TACO_OK;
}

int taco_resample(taco_handle* h, int32_t sr_orig, int32_t sr_new, const float* x, const int32_t* lengths_host, int N,
                  int64_t L, float* y, int64_t L_out, void* stream) {
  if (!h) return TACO_ERR_INVALID;
  CUDA_OK(h, cudaSetDevice(h->device));
  if (!x || !y || N <= 0 || L <= 0 || L_out <= 0 || sr_orig <= 0 || sr_new <= 0)
    return fail(h, TACO_ERR_INVALID, "resample: bad argument");
  const double ratio = res_ratio(sr_orig, sr_new);
  const bool copy = sr_orig == sr_new;
  std::vector<int32_t> len(2 * (size_t)N);
  int64_t longest = 0, n_pos = 0;
  for (int i = 0; i < N; ++i) {
    const int64_t li = lengths_host ? lengths_host[i] : L;
    if (li < 1 || li > L) return fail(h, TACO_ERR_INVALID, "resample: a length outside [1, L]");
    const int64_t computed = copy ? li : (int64_t)((double)li * ratio);   // resampy: int(L ratio) filter outputs
    len[i] = (int32_t)li;
    len[N + i] = (int32_t)std::min<int64_t>(computed, INT32_MAX);
    longest = std::max(longest, taco_resample_length(li, sr_orig, sr_new));
    n_pos = std::max(n_pos, computed);
  }
  if (L_out < longest) return fail(h, TACO_ERR_INVALID, "resample: L_out is shorter than the longest output");
  if ((int64_t)N * L_out >= ((int64_t)1 << 31)) return fail(h, TACO_ERR_UNSUPPORTED, "resample: N * L_out >= 2^31");
  if (!copy && (int64_t)sr_orig > 8 * (int64_t)sr_new)   // the staged window of a CTA grows with the factor (130 KB at 8x)
    return fail(h, TACO_ERR_UNSUPPORTED, "resample: downsampling by more than 8x");
  if (!copy && n_pos > kResMaxOutputs) return fail(h, TACO_ERR_UNSUPPORTED, "resample: more than 2^24 outputs per row");
  cudaStream_t st = (cudaStream_t)stream;
  if (!copy) {
    const int rc = ensure_res_tables(h, sr_orig, sr_new, n_pos, st);
    if (rc) return rc;
  }
  int rc = ensure_ws(h, len.size() * sizeof(int32_t) + 256);
  if (rc) return rc;
  int* d_len = reinterpret_cast<int*>(h->ws);
  CUDA_OK(h, cudaMemcpyAsync(d_len, len.data(), len.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  ResampleArgs a;
  a.x = x; a.L = L; a.N = N; a.lengths = d_len;
  a.pos = nullptr; a.n_pos = 0; a.rows = nullptr; a.taps = 0; a.span = 0;
  a.y = y; a.L_out = L_out; a.copy = copy;
  if (!copy) {
    const auto& R = h->res_tab;
    const size_t rows_bytes = (((size_t)RS_ROWS * R.taps * sizeof(float2)) + 255) & ~size_t(255);
    a.rows = reinterpret_cast<const float2*>(R.dev);
    a.pos = reinterpret_cast<const ResamplePos*>(R.dev + rows_bytes);
    a.n_pos = n_pos; a.taps = R.taps; a.span = R.span;
  }
  CUDA_OK(h, launch_resample(a, st));
  h->launches += 1;
  return check_launch(h, "resample");
}

int64_t taco_launch_count(const taco_handle* h) { return h ? h->launches : 0; }

int taco_decoder_geometry(const taco_handle* h, int N, int* cluster_size, int* samples_per_cluster, int* num_clusters) {
  if (!h || !h->finalized) return TACO_ERR_STATE;
  int CS = 16, S = 8;
  pick_geometry(h, N, &CS, &S);
  int ncl = (N + S - 1) / S;
  if (h->use_cw && N > 0) {
    ncl = pick_mma_clusters(h, N);
    CS = 16;
    S = (N + ncl - 1) / ncl;
  }
  if (cluster_size) *cluster_size = CS;
  if (samples_per_cluster) *samples_per_cluster = S;
  if (num_clusters) *num_clusters = ncl;
  return TACO_OK;
}

int taco_set_gemm_mode(taco_handle* h, int mode) {
  if (!h || mode < 0 || mode > 2) return TACO_ERR_INVALID;
  h->gemm_mode = mode;
  return TACO_OK;
}

int taco_decoder_plan(int N, int T_in, int max_clusters, taco_decoder_plan_t* plan) {
  if (!plan) return TACO_ERR_INVALID;
  memset(plan, 0, sizeof(*plan));
  if (N < 1 || T_in < 1 || T_in > 512 || max_clusters < 1) return TACO_ERR_INVALID;
  const int ncl = pick_cw_clusters(N, max_clusters), S = (N + ncl - 1) / ncl;
  int att_res = 0, ring_kb = 0;
  size_t smem = 0;
  if (!decoder_cw_plan(S, T_in, &att_res, &ring_kb, &smem)) return TACO_ERR_INVALID;
  plan->valid = 1; plan->clusters = ncl; plan->s_max = S; plan->att_res = att_res; plan->ring_kb = ring_kb;
  plan->smem_bytes = (int32_t)smem;
  return TACO_OK;
}

int taco_set_decoder_clusters(taco_handle* h, int n) {
  if (!h || n < 0) return TACO_ERR_INVALID;
  h->dec_clusters = n;
  return TACO_OK;
}

int taco_set_cuda_graphs(taco_handle* h, int on) {
  if (!h) return TACO_ERR_INVALID;
  h->graphs_on = on != 0;
  if (!h->graphs_on && h->fwd_graph.exec) { cudaGraphExecDestroy(h->fwd_graph.exec); h->fwd_graph.exec = nullptr; }
  if (!h->graphs_on && h->gl_graph.exec) { cudaGraphExecDestroy(h->gl_graph.exec); h->gl_graph.exec = nullptr; }
  h->fwd_graph.have_key = false;
  h->gl_graph.have_key = false;
  return TACO_OK;
}

int taco_set_profiling(taco_handle* h, int on) {
  if (!h) return TACO_ERR_INVALID;
  h->profiling = on != 0;
  return TACO_OK;
}
int taco_last_stage_ms(const taco_handle* h, float* ms4_host) {
  if (!h || !ms4_host) return TACO_ERR_INVALID;
  for (int i = 0; i < 4; ++i) ms4_host[i] = h->stage_ms[i];
  return TACO_OK;
}

}  // extern "C"
