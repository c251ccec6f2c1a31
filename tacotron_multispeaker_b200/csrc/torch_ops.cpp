// TORCH_LIBRARY(taco_b200, ...): the C ABI of include/taco_b200.h as PyTorch custom operators.
//
// north_star / SURVEY.md 8(b) ask for the hot path "behind the reference's own plugin/operator API"; the reference has no
// FFI (pure Python on TensorFlow 1.x: models/tacotron.py:18, synthesizer.py:47), so a maintainer moving it to PyTorch would
// call these ops where the TF graph ran.  The operators are THIN: they check tensor dtype / device / contiguity, allocate
// the outputs and pass raw device pointers plus the current CUDA stream to libtaco_b200.so.  No compute is done by torch.
//
//   handle = engine.handle   (int64: the taco_handle* created by taco_create / loaded by taco_set_weight + finalize)
//   taco_b200::forward(handle, ids, lengths, spk?, mel_targets?, teacher_force, bn_mode, num_mels, num_freq, r, want_linear, want_alignments)
//       -> (mel [N,steps*r,M], linear [N,steps*r,F] | empty, alignments [N,T_in,steps] | empty, steps)
//   taco_b200::encoder(handle, ids, lengths, spk?, bn_mode) -> memory [N,T_in,256]
//   taco_b200::decode(handle, memory, mel_targets?, teacher_force) -> (decoder_out [N,steps,M*r], alignments, steps)
//   taco_b200::postnet(handle, mel, bn_mode) -> linear [N,T,F]
//   taco_b200::griffin_lim(handle, linear, iters, sample_rate, frame_shift_ms, frame_length_ms, ...) -> wav [N,L]
//   taco_b200::spectrogram(handle, wav, lengths?, T_out?, sample_rate, frame_shift_ms, frame_length_ms, ...)
//       -> (linear [N,T_out,num_freq], mel [N,T_out,num_mels])
//   taco_b200::resample(handle, wav, lengths?, orig_sr, target_sr) -> y [N, L_out] (L_out: the longest ceil(len ratio))
//   taco_b200::durations(handle, align, text_lengths, frames) -> int32 [N, T_in] frames per symbol
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/library.h>
#include <torch/types.h>

#include <algorithm>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/taco_b200.h"

namespace {

taco_handle* H(int64_t h) {
  TORCH_CHECK(h != 0, "taco_b200: null handle");
  return reinterpret_cast<taco_handle*>(static_cast<intptr_t>(h));
}
void ck(taco_handle* h, int rc, const char* what) {
  TORCH_CHECK(rc == TACO_OK, "taco_b200::", what, " failed (", rc, "): ", taco_last_error(h));
}
const at::Tensor& dev_i32(const at::Tensor& t, const char* name) {
  TORCH_CHECK(t.is_cuda() && t.scalar_type() == at::kInt && t.is_contiguous(), "taco_b200: ", name, " must be a contiguous int32 CUDA tensor");
  return t;
}
const at::Tensor& dev_f32(const at::Tensor& t, const char* name) {
  TORCH_CHECK(t.is_cuda() && t.scalar_type() == at::kFloat && t.is_contiguous(), "taco_b200: ", name, " must be a contiguous float32 CUDA tensor");
  return t;
}
void* stream_of(const at::Tensor& t) { return at::cuda::getCurrentCUDAStream(t.get_device()).stream(); }

std::tuple<at::Tensor, at::Tensor, at::Tensor, int64_t> forward(int64_t handle, const at::Tensor& ids, const at::Tensor& lengths,
                                                                 const c10::optional<at::Tensor>& spk,
                                                                 const c10::optional<at::Tensor>& mel_targets, bool teacher_force,
                                                                 int64_t bn_mode, int64_t num_mels, int64_t num_freq,
                                                                 int64_t outputs_per_step, bool want_linear, bool want_alignments) {
  taco_handle* h = H(handle);
  dev_i32(ids, "ids"); dev_i32(lengths, "lengths");
  TORCH_CHECK(ids.dim() == 2 && lengths.dim() == 1 && lengths.size(0) == ids.size(0), "taco_b200::forward: ids [N,T_in], lengths [N]");
  c10::cuda::CUDAGuard guard(ids.device());
  const int N = (int)ids.size(0), T_in = (int)ids.size(1);
  const int32_t* spk_p = nullptr;
  if (spk.has_value() && spk->defined()) {
    dev_i32(*spk, "identities");
    TORCH_CHECK(spk->dim() == 1 && spk->size(0) == N, "taco_b200::forward: identities [N]");
    spk_p = spk->data_ptr<int32_t>();
  }
  const float* tg_p = nullptr;
  int T_tgt = 0;
  if (teacher_force) {
    TORCH_CHECK(mel_targets.has_value() && mel_targets->defined(), "taco_b200::forward: teacher_force needs mel_targets");
    dev_f32(*mel_targets, "mel_targets");
    TORCH_CHECK(mel_targets->dim() == 3 && mel_targets->size(0) == N && mel_targets->size(2) == num_mels, "taco_b200::forward: mel_targets [N,T_tgt,num_mels]");
    tg_p = mel_targets->data_ptr<float>();
    T_tgt = (int)mel_targets->size(1);
  }
  const int ms = taco_max_steps(h, teacher_force ? 1 : 0, T_tgt);
  TORCH_CHECK(ms > 0, "taco_b200::forward: no decoder steps");
  const int64_t maxT = (int64_t)ms * outputs_per_step;
  auto opt = ids.options().dtype(at::kFloat);
  at::Tensor mel = at::zeros({N, maxT, num_mels}, opt);
  at::Tensor lin = want_linear ? at::zeros({N, maxT, num_freq}, opt) : at::empty({0}, opt);
  at::Tensor al = want_alignments ? at::zeros({N, T_in, ms}, opt) : at::empty({0}, opt);
  int32_t steps = 0;
  ck(h, taco_forward(h, ids.data_ptr<int32_t>(), lengths.data_ptr<int32_t>(), spk_p, tg_p, N, T_in, T_tgt, (int)bn_mode,
                     teacher_force ? 1 : 0, mel.data_ptr<float>(), want_linear ? lin.data_ptr<float>() : nullptr,
                     want_alignments ? al.data_ptr<float>() : nullptr, &steps, stream_of(ids)),
     "forward");
  const int64_t T = (int64_t)steps * outputs_per_step;
  return std::make_tuple(mel.narrow(1, 0, T), want_linear ? lin.narrow(1, 0, T) : lin, want_alignments ? al.narrow(2, 0, steps) : al,
                         (int64_t)steps);
}

at::Tensor encoder(int64_t handle, const at::Tensor& ids, const at::Tensor& lengths, const c10::optional<at::Tensor>& spk, int64_t bn_mode) {
  taco_handle* h = H(handle);
  dev_i32(ids, "ids"); dev_i32(lengths, "lengths");
  TORCH_CHECK(ids.dim() == 2 && lengths.dim() == 1 && lengths.size(0) == ids.size(0), "taco_b200::encoder: ids [N,T_in], lengths [N]");
  c10::cuda::CUDAGuard guard(ids.device());
  const int N = (int)ids.size(0), T_in = (int)ids.size(1);
  const int32_t* spk_p = nullptr;
  if (spk.has_value() && spk->defined()) { dev_i32(*spk, "identities"); spk_p = spk->data_ptr<int32_t>(); }
  at::Tensor memory = at::empty({N, T_in, 256}, ids.options().dtype(at::kFloat));
  ck(h, taco_encoder(h, ids.data_ptr<int32_t>(), lengths.data_ptr<int32_t>(), spk_p, N, T_in, (int)bn_mode, memory.data_ptr<float>(), stream_of(ids)), "encoder");
  return memory;
}

std::tuple<at::Tensor, at::Tensor, int64_t> decode(int64_t handle, const at::Tensor& memory, const c10::optional<at::Tensor>& mel_targets,
                                                   bool teacher_force, int64_t num_mels, int64_t outputs_per_step) {
  taco_handle* h = H(handle);
  dev_f32(memory, "memory");
  TORCH_CHECK(memory.dim() == 3 && memory.size(2) == 256, "taco_b200::decode: memory [N,T_in,256]");
  c10::cuda::CUDAGuard guard(memory.device());
  const int N = (int)memory.size(0), T_in = (int)memory.size(1);
  const float* tg_p = nullptr;
  int T_tgt = 0;
  if (teacher_force) {
    TORCH_CHECK(mel_targets.has_value() && mel_targets->defined(), "taco_b200::decode: teacher_force needs mel_targets");
    dev_f32(*mel_targets, "mel_targets");
    tg_p = mel_targets->data_ptr<float>();
    T_tgt = (int)mel_targets->size(1);
  }
  const int ms = taco_max_steps(h, teacher_force ? 1 : 0, T_tgt);
  TORCH_CHECK(ms > 0, "taco_b200::decode: no decoder steps");
  at::Tensor dec = at::zeros({N, ms, num_mels * outputs_per_step}, memory.options());
  at::Tensor al = at::zeros({N, T_in, ms}, memory.options());
  int32_t steps = 0;
  ck(h, taco_decode(h, memory.data_ptr<float>(), N, T_in, tg_p, T_tgt, teacher_force ? 1 : 0, dec.data_ptr<float>(), al.data_ptr<float>(), &steps,
                    stream_of(memory)),
     "decode");
  return std::make_tuple(dec.narrow(1, 0, steps), al.narrow(2, 0, steps), (int64_t)steps);
}

at::Tensor postnet(int64_t handle, const at::Tensor& mel, int64_t bn_mode, int64_t num_freq) {
  taco_handle* h = H(handle);
  dev_f32(mel, "mel");
  TORCH_CHECK(mel.dim() == 3, "taco_b200::postnet: mel [N,T,num_mels]");
  c10::cuda::CUDAGuard guard(mel.device());
  const int N = (int)mel.size(0), T = (int)mel.size(1);
  at::Tensor lin = at::empty({N, T, num_freq}, mel.options());
  ck(h, taco_postnet(h, mel.data_ptr<float>(), N, T, (int)bn_mode, (int64_t)T * mel.size(2), lin.data_ptr<float>(), (int64_t)T * num_freq, stream_of(mel)),
     "postnet");
  return lin;
}

at::Tensor griffin_lim(int64_t handle, const at::Tensor& linear, int64_t iters, int64_t sample_rate, double frame_shift_ms, double frame_length_ms,
                       double min_level_db, double ref_level_db, double power, double preemphasis) {
  taco_handle* h = H(handle);
  dev_f32(linear, "linear");
  TORCH_CHECK(linear.dim() == 3, "taco_b200::griffin_lim: linear [N,T,num_freq]");
  c10::cuda::CUDAGuard guard(linear.device());
  taco_audio_params ap;
  ap.sample_rate = (int32_t)sample_rate;
  ap.griffin_lim_iters = (int32_t)iters;
  ap.frame_length_ms = frame_length_ms;
  ap.frame_shift_ms = frame_shift_ms;
  ap.preemphasis = preemphasis;
  ap.min_level_db = min_level_db;
  ap.ref_level_db = ref_level_db;
  ap.power = power;
  const int N = (int)linear.size(0), T = (int)linear.size(1);
  const int64_t L = taco_wav_length(&ap, T);
  TORCH_CHECK(L > 0, "taco_b200::griffin_lim: bad audio parameters");
  at::Tensor wav = at::empty({N, L}, linear.options());
  ck(h, taco_griffin_lim(h, &ap, linear.data_ptr<float>(), N, T, 0, wav.data_ptr<float>(), stream_of(linear)), "griffin_lim");
  return wav;
}

// wav [N, L] on the device; lengths (host integers, each in [1, L]) or None = all L; T_out None = the longest utterance's frames
std::tuple<at::Tensor, at::Tensor> spectrogram(int64_t handle, const at::Tensor& wav, at::OptionalIntArrayRef lengths,
                                               c10::optional<int64_t> T_out, int64_t sample_rate, double frame_shift_ms,
                                               double frame_length_ms, double min_level_db, double ref_level_db,
                                               double preemphasis, int64_t num_mels, int64_t num_freq) {
  taco_handle* h = H(handle);
  dev_f32(wav, "wav");
  TORCH_CHECK(wav.dim() == 2, "taco_b200::spectrogram: wav [N,L]");
  c10::cuda::CUDAGuard guard(wav.device());
  taco_audio_params ap{};
  ap.sample_rate = (int32_t)sample_rate;
  ap.frame_length_ms = frame_length_ms;
  ap.frame_shift_ms = frame_shift_ms;
  ap.preemphasis = preemphasis;
  ap.min_level_db = min_level_db;
  ap.ref_level_db = ref_level_db;
  const int N = (int)wav.size(0);
  const int64_t L = wav.size(1);
  std::vector<int32_t> len;
  int64_t T = 0;
  if (lengths.has_value()) {
    TORCH_CHECK((int64_t)lengths->size() == N, "taco_b200::spectrogram: lengths [N]");
    for (int64_t v : *lengths) {
      TORCH_CHECK(v >= 1 && v <= L, "taco_b200::spectrogram: lengths must be in [1, L]");
      len.push_back((int32_t)v);
      T = std::max<int64_t>(T, taco_spectrogram_frames(&ap, v));
    }
  } else {
    T = taco_spectrogram_frames(&ap, L);
  }
  TORCH_CHECK(T > 0, "taco_b200::spectrogram: bad audio parameters");
  if (T_out.has_value()) T = *T_out;
  at::Tensor lin = at::empty({N, T, num_freq}, wav.options());
  at::Tensor mel = at::empty({N, T, num_mels}, wav.options());
  ck(h, taco_spectrogram(h, &ap, wav.data_ptr<float>(), lengths.has_value() ? len.data() : nullptr, N, L, (int)T,
                         lin.data_ptr<float>(), mel.data_ptr<float>(), stream_of(wav)),
     "spectrogram");
  return std::make_tuple(lin, mel);
}

// wav [N, L] on the device; lengths (host integers, each in [1, L]) or None = all L
at::Tensor resample(int64_t handle, const at::Tensor& wav, at::OptionalIntArrayRef lengths, int64_t orig_sr, int64_t target_sr) {
  taco_handle* h = H(handle);
  dev_f32(wav, "wav");
  TORCH_CHECK(wav.dim() == 2, "taco_b200::resample: wav [N,L]");
  c10::cuda::CUDAGuard guard(wav.device());
  const int N = (int)wav.size(0);
  const int64_t L = wav.size(1);
  std::vector<int32_t> len;
  int64_t L_out = 0;
  if (lengths.has_value()) {
    TORCH_CHECK((int64_t)lengths->size() == N, "taco_b200::resample: lengths [N]");
    for (int64_t v : *lengths) {
      TORCH_CHECK(v >= 1 && v <= L, "taco_b200::resample: lengths must be in [1, L]");
      len.push_back((int32_t)v);
      L_out = std::max<int64_t>(L_out, taco_resample_length(v, (int32_t)orig_sr, (int32_t)target_sr));
    }
  } else {
    L_out = taco_resample_length(L, (int32_t)orig_sr, (int32_t)target_sr);
  }
  TORCH_CHECK(L_out > 0, "taco_b200::resample: bad sample rates");
  at::Tensor y = at::empty({N, L_out}, wav.options());
  ck(h, taco_resample(h, (int32_t)orig_sr, (int32_t)target_sr, wav.data_ptr<float>(), lengths.has_value() ? len.data() : nullptr,
                      N, L, y.data_ptr<float>(), L_out, stream_of(wav)),
     "resample");
  return y;
}

// align [N, T_in, steps] on the device; text_lengths / frames host integers [N]
at::Tensor durations(int64_t handle, const at::Tensor& align, at::IntArrayRef text_lengths, at::IntArrayRef frames) {
  taco_handle* h = H(handle);
  dev_f32(align, "align");
  TORCH_CHECK(align.dim() == 3, "taco_b200::durations: align [N,T_in,steps]");
  c10::cuda::CUDAGuard guard(align.device());
  const int64_t N = align.size(0), T_in = align.size(1), steps = align.size(2);
  TORCH_CHECK((int64_t)text_lengths.size() == N && (int64_t)frames.size() == N, "taco_b200::durations: text_lengths [N], frames [N]");
  std::vector<int32_t> len, fr;
  for (int64_t v : text_lengths) {
    TORCH_CHECK(v >= 1 && v <= T_in, "taco_b200::durations: text_lengths must be in [1, T_in]");
    len.push_back((int32_t)v);
  }
  for (int64_t v : frames) {
    TORCH_CHECK(v >= 1 && v <= INT32_MAX, "taco_b200::durations: frames must be >= 1");
    fr.push_back((int32_t)v);
  }
  at::Tensor out = at::empty({N, T_in}, align.options().dtype(at::kInt));
  ck(h, taco_durations(h, align.data_ptr<float>(), (int)N, (int)T_in, (int)steps, len.data(), fr.data(), out.data_ptr<int32_t>(),
                       stream_of(align)),
     "durations");
  return out;
}

}  // namespace

TORCH_LIBRARY(taco_b200, m) {
  m.def("forward(int handle, Tensor ids, Tensor lengths, Tensor? identities, Tensor? mel_targets, bool teacher_force, int bn_mode, "
        "int num_mels, int num_freq, int outputs_per_step, bool want_linear=True, bool want_alignments=True) -> (Tensor, Tensor, Tensor, int)");
  m.def("encoder(int handle, Tensor ids, Tensor lengths, Tensor? identities, int bn_mode) -> Tensor");
  m.def("decode(int handle, Tensor memory, Tensor? mel_targets, bool teacher_force, int num_mels, int outputs_per_step) -> (Tensor, Tensor, int)");
  m.def("postnet(int handle, Tensor mel, int bn_mode, int num_freq) -> Tensor");
  m.def("griffin_lim(int handle, Tensor linear, int iters, int sample_rate, float frame_shift_ms, float frame_length_ms, float min_level_db, "
        "float ref_level_db, float power, float preemphasis) -> Tensor");
  m.def("spectrogram(int handle, Tensor wav, int[]? lengths, int? T_out, int sample_rate, float frame_shift_ms, float frame_length_ms, "
        "float min_level_db, float ref_level_db, float preemphasis, int num_mels, int num_freq) -> (Tensor, Tensor)");
  m.def("resample(int handle, Tensor wav, int[]? lengths, int orig_sr, int target_sr) -> Tensor");
  m.def("durations(int handle, Tensor align, int[] text_lengths, int[] frames) -> Tensor");
}
TORCH_LIBRARY_IMPL(taco_b200, CUDA, m) {
  m.impl("forward", &forward);
  m.impl("encoder", &encoder);
  m.impl("decode", &decode);
  m.impl("postnet", &postnet);
  m.impl("griffin_lim", &griffin_lim);
  m.impl("spectrogram", &spectrogram);
  m.impl("resample", &resample);
  m.impl("durations", &durations);
}
