// Band-limited resampling of a batch of waveforms: librosa 0.5.1 core.resample (res_type 'kaiser_best', fix=True), which
// is resampy 0.1.5's resample_f followed by fix_length.
//
// resampy's output t reads the filter at positions that depend only on t (a double time register advanced by 1 / ratio per
// output), so the host replays the register once per rate pair and hands the kernel, per t, (n, offset_l, eta_l, offset_r,
// eta_r) (ResamplePos).  A tap's weight is linear in eta, win[o] + eta delta[o], so a wing is A.x + eta D.x with A and D
// the row `offset` of a re-laid-out table: rows[o][i] = (win[o + i index_step], delta[o + i index_step]), zero past the
// row's (nwin - o) / index_step taps.  Samples outside [0, len) contribute nothing: the staged window is zero there.
//
// One CTA: RS_T consecutive outputs (one per thread) x RS_U utterances.  The CTA stages the input window its outputs read
// (positions n_first - taps + 1 .. n_last + taps) for its utterances in shared memory, four utterances per 16-byte word and
// one plane per four utterances (so that a quarter warp's loads at different samples spread over all banks), then every
// thread runs both wings over all `taps` of its rows with the RS_U utterances in registers: per tap one 8-byte weight load
// (L1: a CTA touches a handful of rows), RS_U / 4 16-byte shared loads of x and 2 RS_U FFMA.  Partial sums of RS_BLK taps
// keep the fp32 error well under the test bound.  What bounds it: the loads -- 32 lanes read x at ~32 different samples
// (at least 4 shared-memory wavefronts per 16-byte load, more on bank conflicts) and their rows at a handful of
// different L1 lines, against 8 issue cycles of a warp's 32 FFMA per tap.
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>

#include "kernels.cuh"

namespace taco {
namespace {

__device__ __forceinline__ void fma4(float* acc, float w, const float4& x) {
  acc[0] = fmaf(w, x.x, acc[0]); acc[1] = fmaf(w, x.y, acc[1]); acc[2] = fmaf(w, x.z, acc[2]); acc[3] = fmaf(w, x.w, acc[3]);
}

// y[u] += sum_i row[i].x x(base + DIR i, u) + eta sum_i row[i].y x(base + DIR i, u);  x(s, u) = xs[u / 4][s].(u % 4)
template <int DIR>
__device__ __forceinline__ void wing(const float4* xs, int J, int base, const float2* __restrict__ row, int taps, float eta,
                                     float (&y)[RS_U]) {
  float a[RS_U], d[RS_U];
#pragma unroll
  for (int u = 0; u < RS_U; ++u) a[u] = d[u] = 0.0f;
  for (int i0 = 0; i0 < taps; i0 += RS_BLK) {
    float pa[RS_U], pd[RS_U];
#pragma unroll
    for (int u = 0; u < RS_U; ++u) pa[u] = pd[u] = 0.0f;
    const int i1 = min(taps, i0 + RS_BLK);
#pragma unroll 4
    for (int i = i0; i < i1; ++i) {
      const float2 w = __ldg(row + i);
      const float4* xp = xs + base + DIR * i;
#pragma unroll
      for (int q = 0; q < RS_U / 4; ++q) {
        const float4 xq = xp[q * J];
        fma4(pa + 4 * q, w.x, xq);
        fma4(pd + 4 * q, w.y, xq);
      }
    }
#pragma unroll
    for (int u = 0; u < RS_U; ++u) { a[u] += pa[u]; d[u] += pd[u]; }
  }
#pragma unroll
  for (int u = 0; u < RS_U; ++u) y[u] += fmaf(eta, d[u], a[u]);
}

__global__ void __launch_bounds__(RS_T) resample_kernel(const ResampleArgs a) {
  extern __shared__ float4 xs[];   // [RS_U / 4][window]: four utterances per 16-byte word, one plane per four
  const int tid = threadIdx.x;
  const long long t0 = (long long)blockIdx.x * RS_T, t = t0 + tid;
  const int u0 = blockIdx.y * RS_U, nu = min(RS_U, a.N - u0);
  float y[RS_U];
#pragma unroll
  for (int u = 0; u < RS_U; ++u) y[u] = 0.0f;
  __shared__ int s_len[RS_U];
  if (tid < RS_U) s_len[tid] = tid < nu ? a.lengths[u0 + tid] : 0;
  __syncthreads();
  if (t0 < a.n_pos) {   // uniform over the CTA
    const long long tl = min(t0 + RS_T, a.n_pos) - 1;
    const int jlo = a.pos[t0].n - (a.taps - 1);
    const int J = a.pos[tl].n + a.taps + 1 - jlo;   // <= a.span
    for (int k = tid; k < RS_U * J; k += RS_T) {   // coalesced along each utterance's samples
      const int u = k / J, jj = k - u * J;
      const long long j = (long long)jlo + jj;
      float v = 0.0f;
      if (j >= 0 && j < s_len[u]) v = __ldg(a.x + (size_t)(u0 + u) * a.L + j);
      reinterpret_cast<float*>(xs + (u >> 2) * J + jj)[u & 3] = v;
    }
    __syncthreads();
    if (t < a.n_pos) {
      const ResamplePos p = a.pos[t];
      wing<-1>(xs, J, p.n - jlo, a.rows + (size_t)p.off_l * a.taps, a.taps, p.eta_l, y);
      wing<1>(xs, J, p.n + 1 - jlo, a.rows + (size_t)p.off_r * a.taps, a.taps, p.eta_r, y);
    }
  }
  if (t < a.L_out)
#pragma unroll
    for (int u = 0; u < RS_U; ++u)
      if (u < nu) a.y[(size_t)(u0 + u) * a.L_out + t] = t < a.lengths[a.N + u0 + u] ? y[u] : 0.0f;
}

// equal rates: librosa returns the input unchanged
__global__ void resample_copy_kernel(const ResampleArgs a) {
  const long long total = (long long)a.N * a.L_out;
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
    const long long n = k / a.L_out, t = k - n * a.L_out;
    a.y[k] = t < a.lengths[n] ? __ldg(a.x + n * a.L + t) : 0.0f;
  }
}

}  // namespace

size_t resample_smem_bytes(int span) { return (size_t)span * RS_U * sizeof(float); }

cudaError_t launch_resample(const ResampleArgs& a, cudaStream_t st) {
  if (a.N < 1 || a.L < 1 || a.L_out < 1 || !a.x || !a.y || !a.lengths) return cudaErrorInvalidValue;
  if (a.copy) {
    const long long total = (long long)a.N * a.L_out;
    const unsigned blocks = (unsigned)std::min<long long>((total + 255) / 256, 148LL * 16);
    resample_copy_kernel<<<blocks, 256, 0, st>>>(a);
    return cudaGetLastError();
  }
  if (a.taps < 1 || a.span < 1 || (a.n_pos > 0 && (!a.pos || !a.rows))) return cudaErrorInvalidValue;
  const size_t smem = resample_smem_bytes(a.span);
  if (smem > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(resample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  const dim3 grid((unsigned)((a.L_out + RS_T - 1) / RS_T), (unsigned)((a.N + RS_U - 1) / RS_U));
  resample_kernel<<<grid, RS_T, smem, st>>>(a);
  return cudaGetLastError();
}

}  // namespace taco
