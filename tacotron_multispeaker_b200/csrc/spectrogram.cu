// Spectrogram analysis of the reference's audio module (util/audio.py spectrogram / melspectrogram: preemphasis ->
// librosa.stft -> |D| -> _amp_to_db -> _normalize, and _linear_to_mel with librosa.filters.mel) for a batch of
// waveforms on the device.
//
// One launch: a CTA owns one frame of one utterance and does
//   reflect-padded, pre-emphasised, windowed samples -> 2048-point FFT in shared memory (fft2048.cuh, the forward
//   transform of the Griffin-Lim kernel) -> |X| of the 1025 bins in shared memory -> the normalised dB row of the linear
//   spectrogram (coalesced) and the mel bands reduced from a sparse band table.
//
// librosa 0.5.1 conventions restated (stft with center=True, pad_mode reflect; filters.mel with the Slaney scale and
// the 2 / (f[i+2] - f[i]) band scaling): the signal is pre-emphasised BEFORE padding, padded by n_fft/2 on each side
// with np.pad(mode='reflect') (the even periodic extension of period 2 (L-1) when the pad is longer than the signal;
// for L = 1 the sample repeated), and frame t covers the padded samples [t hop, t hop + n_fft) with the periodic Hann
// window of `win` points centred in them (lpad = (n_fft - win) / 2).  Only |D| is used and |DFT| does not change under a
// circular shift, so the `win` windowed samples sit at positions 0 .. win-1 of the transform, as in gl_iter_kernel.
#include <cuda_runtime.h>
#include <stdint.h>

#include "fft2048.cuh"
#include "kernels.cuh"

namespace taco {
namespace {

// pre-emphasised sample p[j] = y[j] - a y[j-1] (p[0] = y[0]) at the reflect-padded position j of an utterance of L samples
__device__ __forceinline__ float pre_at(const float* __restrict__ y, long long j, long long L, float a) {
  if (j < 0 || j >= L) {
    if (L == 1) {
      j = 0;
    } else {
      const long long P = 2 * (L - 1);
      j %= P;
      if (j < 0) j += P;
      if (j >= L) j = P - j;
    }
  }
  const float v = __ldg(y + j);
  return j > 0 ? fmaf(-a, __ldg(y + j - 1), v) : v;
}

// clip((20 log10(max(1e-5, x)) - ref_level_db - min_level_db) / -min_level_db, 0, 1) as log2 x * c1 + c0
__device__ __forceinline__ float norm_db(float x, float c1, float c0) {
  return fminf(fmaxf(fmaf(log2f(fmaxf(1e-5f, x)), c1, c0), 0.0f), 1.0f);
}

__global__ void __launch_bounds__(GL_NT)
spec_frame_kernel(const float* __restrict__ wav, long long L, const int* __restrict__ lengths, int T_out, int win, int hop,
                  float preemph, float c1, float c0, const float2* __restrict__ tw, const float* __restrict__ win_g,
                  const int* __restrict__ band, const float* __restrict__ band_w, int num_mels,
                  float* __restrict__ lin_out, float* __restrict__ mel_out) {
  __shared__ float2 d[GL_DSIZE];
  __shared__ float mag[GL_BINS];
  const int tid = threadIdx.x;
  const int frame = blockIdx.x, n = frame / T_out, t = frame - n * T_out;
  const long long Li = lengths ? lengths[n] : L;
  float* lrow = lin_out ? lin_out + (size_t)frame * GL_BINS : nullptr;
  float* mrow = mel_out ? mel_out + (size_t)frame * num_mels : nullptr;
  if (t >= 1 + Li / hop) {   // the zero padding of the batch's targets
    if (lrow)
      for (int f = tid; f < GL_BINS; f += GL_NT) lrow[f] = 0.0f;
    if (mrow)
      for (int b = tid; b < num_mels; b += GL_NT) mrow[b] = 0.0f;
    return;
  }
  const float* y = wav + (size_t)n * L;
  const long long j0 = (long long)t * hop - GL_N / 2 + (GL_N - win) / 2;   // original index of windowed sample 0
  float2 xin[GL_M / GL_NT];
#pragma unroll
  for (int j = 0; j < GL_M / GL_NT; ++j) {
    const int i = 2 * (tid + GL_NT * j);
    float2 x = make_float2(0.0f, 0.0f);
    if (i < win) x.x = pre_at(y, j0 + i, Li, preemph) * __ldg(win_g + i);
    if (i + 1 < win) x.y = pre_at(y, j0 + i + 1, Li, preemph) * __ldg(win_g + i + 1);
    xin[j] = x;
  }
  dif_pass<3, 7, false>(d, tw, tid, xin); __syncthreads();
  dif_pass<3, 4>(d, tw, tid); __syncthreads();
  dif_pass<4, 0>(d, tw, tid);
  __syncthreads();
  constexpr int NPAIR = (GL_M / 2 + GL_NT) / GL_NT;   // bin pairs (k, M - k), k = tid + 128 j <= 512
#pragma unroll
  for (int j = 0; j < NPAIR; ++j) {
    const int k = tid + GL_NT * j;
    if (k <= GL_M / 2) {
      const int km = GL_M - k;
      const int pk = PD((int)(__brev((unsigned)k) >> 22)), pm = PD((int)(__brev((unsigned)(km & (GL_M - 1))) >> 22));
      const float2 w = __ldg(tw + k);
      const float2 zk = d[pk], zm = d[pm];
      // E = (Z[k] + conj Z[M-k]) / 2, O = (Z[k] - conj Z[M-k]) / 2i;  X[k] = E + W^k O,  X[M-k] = conj(E - W^k O)
      const float2 e = make_float2(0.5f * (zk.x + zm.x), 0.5f * (zk.y - zm.y));
      const float2 o = make_float2(0.5f * (zk.y + zm.y), -0.5f * (zk.x - zm.x));
      const float2 tt = cmul(w, o);
      const float ax = e.x + tt.x, ay = e.y + tt.y, bx = e.x - tt.x, by = e.y - tt.y;
      mag[k] = sqrtf(fmaf(ax, ax, ay * ay));
      mag[km] = sqrtf(fmaf(bx, bx, by * by));
    }
  }
  __syncthreads();
  if (lrow)
    for (int f = tid; f < GL_BINS; f += GL_NT) lrow[f] = norm_db(mag[f], c1, c0);
  if (mrow)
    for (int b = tid; b < num_mels; b += GL_NT) {
      const int first = __ldg(band + 3 * b), cnt = __ldg(band + 3 * b + 1), off = __ldg(band + 3 * b + 2);
      float acc = 0.0f;
      for (int q = 0; q < cnt; ++q) acc = fmaf(__ldg(band_w + off + q), mag[first + q], acc);
      mrow[b] = norm_db(acc, c1, c0);
    }
}

}  // namespace

void launch_fft_tables(float2* tw, float* win, int win_len, cudaStream_t st) {
  gl_tables_kernel<<<(GL_N + 255) / 256, 256, 0, st>>>(tw, win, win_len);
}

cudaError_t launch_spectrogram(const SpectrogramArgs& a, cudaStream_t st) {
  if (a.win < 1 || a.win > GL_N || a.hop < 1 || a.N < 1 || a.T_out < 1 || a.L < 1 || a.num_mels < 0)
    return cudaErrorInvalidValue;
  // dB / -min_level_db = log2(x) * 20 log10(2) / -min_level_db;  offset (-ref_level_db - min_level_db) / -min_level_db
  const double c1 = 20.0 * 0.30102999566398120 / -a.min_level_db, c0 = (-a.ref_level_db - a.min_level_db) / -a.min_level_db;
  spec_frame_kernel<<<(unsigned)((size_t)a.N * a.T_out), GL_NT, 0, st>>>(
      a.wav, a.L, a.lengths, a.T_out, a.win, a.hop, a.preemphasis, (float)c1, (float)c0, a.tw, a.window, a.band, a.band_w,
      a.num_mels, a.linear, a.mel);
  return cudaGetLastError();
}

}  // namespace taco
