// Griffin-Lim vocoder of the reference's synthesis graph (util/audio.py:39-46 inv_spectrogram_tensorflow,
// :78-91 _griffin_lim_tensorflow, :105-112 tf.contrib.signal.stft / inverse_stft, synthesizer.py:27,50) for a
// whole batch of linear spectrograms on the device.
//
// One Griffin-Lim iteration is ONE launch: a CTA owns one frame of one utterance and does
//   overlap-add of the previous iteration's windowed inverse frames (the signal is never materialised)
//   -> analysis window -> 2048-point FFT in shared memory -> est / max(1e-8, |est|) * S
//   -> inverse FFT in shared memory -> synthesis window -> its inverse frame for the next iteration.
// The forward transform is decimation in frequency (natural order in, bit-reversed out), the phase step works on
// the bit-reversed positions, and the inverse is decimation in time (bit-reversed in, natural out): no reordering
// pass.  The real 2048-point transforms are 1024-point complex ones on even/odd packed samples; three or four
// radix-2 stages are done in registers per shared-memory round trip (8 or 16 elements per thread, passes of
// 3 + 3 + 4 stages), so a transform is three round trips, all of them bank-conflict free (one pad per 16 elements).
//
// TF conventions restated: frame(signal, win, hop, pad_end=False), periodic Hann of `win` points for analysis AND
// synthesis (inverse_stft's default window_fn, no window-sum normalisation), rfft/irfft of n_fft = 2 (num_freq - 1)
// points with the frame zero-padded at its end, irfft scaled by 1/n_fft and cut to `win` samples, overlap_and_add.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "fft2048.cuh"
#include "kernels.cuh"

namespace taco {
namespace {

// util/audio.py:42-43: S = db_to_amp(denormalize(x) + ref_level_db) ** power, as one exp2
__global__ void gl_mags_kernel(const float* __restrict__ lin, int64_t lin_bs, int T, int F, float scale_db,
                               float off_db, float expo, float* __restrict__ mags, int64_t total) {
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = idx / F;
    const int f = (int)(idx - row * F), n = (int)(row / T), t = (int)(row - (int64_t)n * T);
    float x = __ldg(lin + (int64_t)n * lin_bs + (int64_t)t * F + f);
    x = fminf(fmaxf(x, 0.0f), 1.0f);
    mags[idx] = exp2f(fmaf(x, scale_db, off_db) * expo);
  }
}

// the inverse: decimation in time, half-spans q, 2q, ..., (R/2) q, conjugate twiddles
template <int LOGR, int LOGQ>
__device__ __forceinline__ void dit_core(float2 (&v)[1 << LOGR], int lo, const float2* tw) {
  constexpr int R = 1 << LOGR, Q = 1 << LOGQ;
  static_assert(R <= 16, "constant twiddles go up to W_16");
  float2 wbs[LOGR];
  wbs[LOGR - 1] = make_float2(1.0f, 0.0f);
  if (LOGQ > 0) {
    wbs[LOGR - 1] = __ldg(tw + lo * (GL_N / (R * Q)));
#pragma unroll
    for (int s = LOGR - 2; s >= 0; --s) wbs[s] = cmul(wbs[s + 1], wbs[s + 1]);
  }
#pragma unroll
  for (int s = 0; s < LOGR; ++s) {
    const int hs = 1 << s;
#pragma unroll
    for (int m = 0; m < R; ++m) {
      if (m & hs) continue;
      float2 b = mul_w16<true>(v[m + hs], (m & (hs - 1)) * (8 / hs));
      if (LOGQ > 0) b = cmul_conj(b, wbs[s]);
      const float2 a = v[m];
      v[m] = cadd(a, b);
      v[m + hs] = csub(a, b);
    }
  }
}
template <int LOGR, int LOGQ, bool STORE = true>
__device__ __forceinline__ void dit_pass(float2* d, const float2* tw, int tid, float2* vout = nullptr) {
  constexpr int R = 1 << LOGR, Q = 1 << LOGQ;
  static_assert(GL_M / R <= GL_NT, "one group per thread");
  if (tid < GL_M / R) {   // GL_M / R <= GL_NT: at most one group per thread
    const int g = tid;
    const int lo = g & (Q - 1), base = ((g >> LOGQ) << (LOGR + LOGQ)) + lo;
    static_assert(Q >= 16 || R * Q <= 16, "padded stride");
    static_assert(Q == 128 || R * Q <= 128, "per-256 pad");
    constexpr int PS = Q >= 16 ? Q + Q / 16 : Q;
    float2* dp = d + PD(base);
    float2 v[R];
#pragma unroll
    for (int m = 0; m < R; ++m) v[m] = dp[m * PS + (Q == 128 ? (m >> 1) : 0)];
    dit_core<LOGR, LOGQ>(v, lo, tw);
#pragma unroll
    for (int m = 0; m < R; ++m) {
      if (STORE) dp[m * PS + (Q == 128 ? (m >> 1) : 0)] = v[m];
      else vout[m] = v[m];
    }
  }
}

// sum over the frames that cover sample m of utterance rows r[t][0..win)
__device__ __forceinline__ float ola_at(const float* __restrict__ r, int m, int T, int win, int hop) {
  const int num = m - win + hop;
  const int t_lo = num > 0 ? num / hop : 0;
  const int t_hi = min(T - 1, m / hop);
  float acc = 0.0f;
  for (int tp = t_lo; tp <= t_hi; ++tp) acc += __ldg(r + (size_t)tp * win + (m - tp * hop));
  return acc;
}
// samples i, i + 1 of frame t before the analysis window (i, win and hop even: both samples are covered by the same
// frames and every address is 8-byte aligned).  Frame t + dd holds them at offset i - dd hop; K = (win - 1) / hop
// frames overlap on each side.  KT >= 0: K known at compile time (all loads issued back to back).
template <int KT>
__device__ __forceinline__ float2 ola2_frame(const float* __restrict__ r, int t, int i, int T, int win, int hop, int K) {
  const float* p = r + (size_t)t * win + i;
  const int step = win - hop;
  float2 acc = make_float2(0.0f, 0.0f);
  if (KT >= 0) {
    float2 v[2 * (KT >= 0 ? KT : 0) + 1];
#pragma unroll
    for (int dd = -KT; dd <= KT; ++dd) {
      const bool ok = (unsigned)(i - dd * hop) < (unsigned)win && (unsigned)(t + dd) < (unsigned)T;
      v[dd + KT] = ok ? __ldg(reinterpret_cast<const float2*>(p + dd * step)) : make_float2(0.0f, 0.0f);
    }
#pragma unroll
    for (int dd = -KT; dd <= KT; ++dd) {
      const bool ok = (unsigned)(i - dd * hop) < (unsigned)win && (unsigned)(t + dd) < (unsigned)T;
      if (ok) { acc.x += v[dd + KT].x; acc.y += v[dd + KT].y; }
    }
  } else {
    for (int dd = -K; dd <= K; ++dd)
      if ((unsigned)(i - dd * hop) < (unsigned)win && (unsigned)(t + dd) < (unsigned)T) {
        const float2 v = __ldg(reinterpret_cast<const float2*>(p + dd * step));
        acc.x += v.x; acc.y += v.y;
      }
  }
  return acc;
}

// util/audio.py:88-89: mag * x / max(1e-8, |x|) = mag * x * rsqrt(max(1e-16, |x|^2)); MUFU.RSQ has no slow path for
// the tiny values of silent frames (sqrtf and the division do)
__device__ __forceinline__ float2 to_magnitude(float2 x, float mag) {
  const float s = mag * rsqrtf(fmaxf(1e-16f, fmaf(x.x, x.x, x.y * x.y)));
  return make_float2(x.x * s, x.y * s);
}

// One Griffin-Lim iteration for frame blockIdx.x (FIRST: the zero-phase start, util/audio.py:84-85).
// The real 2048-point transforms run as 1024-point complex ones on z[m] = x[2m] + i x[2m+1]; the phase step
// un-mixes the bin pair (k, 1024 - k), rescales both and mixes them again for the inverse.
// REF: win == 4 hop, both even (the reference's 1000 / 250): sample i of an interior frame is the sum of exactly
// four rows at constant distances; other geometries and the three frames at each end take the predicated loop.
// Twiddles (4 KB, L1 resident) and the frame's magnitudes are read straight from global memory: a thread needs two
// twiddles per transform and the magnitudes of its own five bin pairs, requested before the forward transform.
template <bool FIRST, bool REF>
__global__ void __launch_bounds__(GL_NT)
gl_iter_kernel(const float* __restrict__ mags, const float* __restrict__ r_prev, float* __restrict__ r_next,
               const float2* __restrict__ tw, const float* __restrict__ win_g, int T, int win, int hop) {
  __shared__ float2 d[GL_DSIZE];
  constexpr int NPAIR = (GL_M / 2 + GL_NT) / GL_NT;   // bin pairs (k, M - k), k = tid + 128 j <= 512
  const int tid = threadIdx.x;
  const int frame = blockIdx.x, n = frame / T, t = frame - n * T;
  const bool even = REF || ((win | hop) & 1) == 0;
  if (!FIRST) asm volatile("griddepcontrol.launch_dependents;");   // the next iteration may start to launch
  float mk[NPAIR], mkm[NPAIR];
  {
    const float* mrow = mags + (size_t)frame * GL_BINS;
#pragma unroll
    for (int j = 0; j < NPAIR; ++j) {
      const int k = tid + GL_NT * j;
      mk[j] = k <= GL_M / 2 ? __ldg(mrow + k) : 0.0f;
      mkm[j] = k <= GL_M / 2 ? __ldg(mrow + GL_M - k) : 0.0f;
    }
  }
  if (!FIRST) {
    // Iterations are launched with programmatic stream serialisation: this grid may become resident while the previous
    // iteration drains (its magnitudes are already requested above); nothing of the previous iteration is touched
    // before this point, and the previous grid's rows are complete and visible after it.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    float2 xin[GL_M / GL_NT];
    const float* r = r_prev + (size_t)n * T * win;
    if (REF && t >= 3 && t + 3 < T) {
      const float* pt = r + (size_t)t * win;
      const int step = win - hop;   // frame t + dd holds sample i at pt[i + dd step]
#pragma unroll
      for (int j = 0; j < GL_M / GL_NT; ++j) {
        const int i = 2 * (tid + GL_NT * j);
        float2 x = make_float2(0.0f, 0.0f);
        if (i < win) {
          const int a = (i >= hop) + (i >= 2 * hop) + (i >= 3 * hop);   // frames t + a - 3 .. t + a cover sample i
          const float* q = pt + i + (a - 3) * step;
          const float2 v0 = __ldg(reinterpret_cast<const float2*>(q));
          const float2 v1 = __ldg(reinterpret_cast<const float2*>(q + step));
          const float2 v2 = __ldg(reinterpret_cast<const float2*>(q + 2 * step));
          const float2 v3 = __ldg(reinterpret_cast<const float2*>(q + 3 * step));
          const float2 w = __ldg(reinterpret_cast<const float2*>(win_g + i));
          x.x = (((v0.x + v1.x) + v2.x) + v3.x) * w.x;
          x.y = (((v0.y + v1.y) + v2.y) + v3.y) * w.y;
        }
        xin[j] = x;
      }
    } else {
      const int K = (win - 1) / hop;
#pragma unroll
      for (int j = 0; j < GL_M / GL_NT; ++j) {
        const int i = 2 * (tid + GL_NT * j);
        float2 x = make_float2(0.0f, 0.0f);
        if (even) {
          if (i < win) {
            const float2 w = __ldg(reinterpret_cast<const float2*>(win_g + i));
            x = ola2_frame<-1>(r, t, i, T, win, hop, K);
            x.x *= w.x; x.y *= w.y;
          }
        } else {
          if (i < win) x.x = ola_at(r, t * hop + i, T, win, hop) * __ldg(win_g + i);
          if (i + 1 < win) x.y = ola_at(r, t * hop + i + 1, T, win, hop) * __ldg(win_g + i + 1);
        }
        xin[j] = x;
      }
    }
    // element tid + 128 j is input j of thread tid's group in the first pass: no shared-memory trip for the frame
    dif_pass<3, 7, false>(d, tw, tid, xin); __syncthreads();
    dif_pass<3, 4>(d, tw, tid); __syncthreads();
    dif_pass<4, 0>(d, tw, tid);
    __syncthreads();
  }
#pragma unroll
  for (int j = 0; j < NPAIR; ++j) {
    const int k = tid + GL_NT * j;
    if (k <= GL_M / 2) {
      const int km = GL_M - k;
      const int pk = PD((int)(__brev((unsigned)k) >> 22)), pm = PD((int)(__brev((unsigned)(km & (GL_M - 1))) >> 22));
      const float2 w = __ldg(tw + k);
      float2 yk, ym;
      if (FIRST) {
        yk = make_float2(mk[j], 0.0f);
        ym = make_float2(mkm[j], 0.0f);
      } else {
        const float2 zk = d[pk], zm = d[pm];
        // E = (Z[k] + conj Z[M-k]) / 2, O = (Z[k] - conj Z[M-k]) / 2i;  X[k] = E + W^k O,  X[M-k] = conj(E - W^k O)
        const float2 e = make_float2(0.5f * (zk.x + zm.x), 0.5f * (zk.y - zm.y));
        const float2 o = make_float2(0.5f * (zk.y + zm.y), -0.5f * (zk.x - zm.x));
        const float2 tt = cmul(w, o);
        yk = to_magnitude(make_float2(e.x + tt.x, e.y + tt.y), mk[j]);
        ym = to_magnitude(make_float2(e.x - tt.x, -(e.y - tt.y)), mkm[j]);
      }
      // Z'[k] = E' + i O' with E' = Y[k] + conj Y[M-k], O' = (Y[k] - conj Y[M-k]) conj(W^k)   (the 1/2 is in the final scale)
      const float2 ep = make_float2(yk.x + ym.x, yk.y - ym.y);
      const float2 op = cmul_conj(make_float2(yk.x - ym.x, yk.y + ym.y), w);
      d[pk] = make_float2(ep.x - op.y, ep.y + op.x);
      if (k != 0 && k != GL_M / 2) d[pm] = make_float2(ep.x + op.y, op.x - ep.y);
    }
  }
  __syncthreads();
  dit_pass<4, 0>(d, tw, tid); __syncthreads();
  dit_pass<3, 4>(d, tw, tid); __syncthreads();
  float2 zout[GL_M / GL_NT];   // ... and the last pass leaves element tid + 128 j in register j
  dit_pass<3, 7, false>(d, tw, tid, zout);
  float* o = r_next + (size_t)frame * win;
#pragma unroll
  for (int j = 0; j < GL_M / GL_NT; ++j) {
    const int i = 2 * (tid + GL_NT * j);
    const float2 z = zout[j];
    if (even) {
      if (i < win) {
        const float2 w = __ldg(reinterpret_cast<const float2*>(win_g + i));
        *reinterpret_cast<float2*>(o + i) = make_float2(z.x * (w.x * (1.0f / GL_N)), z.y * (w.y * (1.0f / GL_N)));
      }
    } else {
      if (i < win) o[i] = z.x * (__ldg(win_g + i) * (1.0f / GL_N));
      if (i + 1 < win) o[i + 1] = z.y * (__ldg(win_g + i + 1) * (1.0f / GL_N));
    }
  }
}

// overlap_and_add of the last inverse frames: y [N, L]
__global__ void gl_ola_kernel(const float* __restrict__ r, float* __restrict__ y, int T, int win, int hop, int L) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x, n = blockIdx.y;
  if (m < L) y[(size_t)n * L + m] = ola_at(r + (size_t)n * T * win, m, T, win, hop);
}

// util/audio.py:23-24 inv_preemphasis = lfilter([1], [1, -a]): y[i] = x[i] + a y[i-1], in place.  One CTA per
// utterance; warp w owns a contiguous segment and walks it 32 samples at a time (coalesced): a shuffle scan with the
// powers a, a^2, ..., a^16 gives the 32 outputs of a step, the last one carries into the next step.  The state at
// the end of each segment is chained over the 32 warps, and a second pass adds carry * a^(k+1) to the head of each
// segment until the factor has decayed by 1e-12 (a = 0.97: 900 samples; far below any rounding of the first pass).
__global__ void __launch_bounds__(1024) gl_deemph_kernel(float* __restrict__ y, int L, float a) {
  __shared__ float zend[32];
  __shared__ float carry[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* p = y + (size_t)blockIdx.x * L;
  const int seg = (((L + 31) / 32) + 31) & ~31;
  const int s = min(L, warp * seg), e = min(L, s + seg);
  const float a2 = a * a, a4 = a2 * a2, a8 = a4 * a4, a16 = a8 * a8, a32 = a16 * a16;
  float alp = a;                                   // a^(lane + 1)
  if (lane & 1) alp *= a;
  if (lane & 2) alp *= a2;
  if (lane & 4) alp *= a4;
  if (lane & 8) alp *= a8;
  if (lane & 16) alp *= a16;
  float c = 0.0f;
  float x = s + lane < e ? p[s + lane] : 0.0f;
  for (int i0 = s; i0 < e; i0 += 32) {
    const int i = i0 + lane;
    const float xn = i + 32 < e ? p[i + 32] : 0.0f;   // next step's sample, requested before the scan
    float v = x, t;
    t = __shfl_up_sync(0xffffffffu, v, 1);  if (lane >= 1) v = fmaf(a, t, v);
    t = __shfl_up_sync(0xffffffffu, v, 2);  if (lane >= 2) v = fmaf(a2, t, v);
    t = __shfl_up_sync(0xffffffffu, v, 4);  if (lane >= 4) v = fmaf(a4, t, v);
    t = __shfl_up_sync(0xffffffffu, v, 8);  if (lane >= 8) v = fmaf(a8, t, v);
    t = __shfl_up_sync(0xffffffffu, v, 16); if (lane >= 16) v = fmaf(a16, t, v);
    v = fmaf(alp, c, v);
    if (i < e) p[i] = v;
    c = __shfl_sync(0xffffffffu, v, 31);
    x = xn;
  }
  if (lane == 0) zend[warp] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    const float aseg = powf(a, (float)seg);
    float cc = 0.0f;
    for (int w = 0; w < 32; ++w) { carry[w] = cc; cc = fmaf(aseg, cc, zend[w]); }
  }
  __syncthreads();
  const float cw = carry[warp];
  if (cw != 0.0f) {
    float f = cw * alp;
    const float tiny = fabsf(cw) * 1e-12f;
    for (int i = s + lane; i < e && fabsf(f) >= tiny; i += 32) { p[i] += f; f *= a32; }
  }
}

}  // namespace

size_t griffin_lim_ws_bytes(int N, int T, int win) {
  const size_t frames = (size_t)N * T;
  return frames * GL_BINS * sizeof(float) + 2 * frames * win * sizeof(float) + GL_TW * sizeof(float2) +
         (size_t)win * sizeof(float) + 4096;
}

cudaError_t launch_griffin_lim(const GriffinLimArgs& a, void* ws, cudaStream_t st, int* launches) {
  if (a.n_fft != GL_N || a.win < 1 || a.win > GL_N || a.hop < 1 || a.N < 1 || a.T < 1 || a.iters < 0)
    return cudaErrorInvalidValue;
  const size_t frames = (size_t)a.N * a.T;
  char* p = static_cast<char*>(ws);
  auto take = [&](size_t bytes) { char* q = p; p += (bytes + 255) & ~size_t(255); return q; };
  float* mags = reinterpret_cast<float*>(take(frames * GL_BINS * sizeof(float)));
  float* r0 = reinterpret_cast<float*>(take(frames * a.win * sizeof(float)));
  float* r1 = reinterpret_cast<float*>(take(frames * a.win * sizeof(float)));
  float2* tw = reinterpret_cast<float2*>(take(GL_TW * sizeof(float2)));
  float* win = reinterpret_cast<float*>(take((size_t)a.win * sizeof(float)));
  gl_tables_kernel<<<(GL_N + 255) / 256, 256, 0, st>>>(tw, win, a.win);
  const int64_t total = (int64_t)frames * GL_BINS;
  // dB = clip(x, 0, 1) * (-min_level_db) + min_level_db + ref_level_db;  S^power = 10^(0.05 * power * dB)
  gl_mags_kernel<<<(unsigned)((total + 1023) / 1024 < 148 * 16 ? (total + 1023) / 1024 : 148 * 16), 256, 0, st>>>(
      a.linear, a.linear_bs, a.T, GL_BINS, -a.min_level_db, a.min_level_db + a.ref_level_db,
      0.05f * a.power * 3.3219280948873623f, mags, total);
  float *cur = r0, *nxt = r1;
  const bool ref = a.win == 4 * a.hop && ((a.win | a.hop) & 1) == 0;   // the reference's 1000 / 250
  if (ref) gl_iter_kernel<true, true><<<(unsigned)frames, GL_NT, 0, st>>>(mags, nullptr, cur, tw, win, a.T, a.win, a.hop);
  else gl_iter_kernel<true, false><<<(unsigned)frames, GL_NT, 0, st>>>(mags, nullptr, cur, tw, win, a.T, a.win, a.hop);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)frames);
  cfg.blockDim = dim3(GL_NT);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  const char* pdl = getenv("TACO_GL_PDL");      // programmatic dependent launch of the iterations (TACO_GL_PDL=0: off)
  cfg.numAttrs = (pdl && atoi(pdl) == 0) ? 0 : 1;   // batch 1 x 1000 frames: 1.43 -> 1.20 ms; batch 32: 19.8 -> 19.6 ms
  for (int it = 0; it < a.iters; ++it) {
    const float* rp = cur;
    cudaError_t e = ref ? cudaLaunchKernelEx(&cfg, gl_iter_kernel<false, true>, (const float*)mags, rp, nxt, (const float2*)tw,
                                             (const float*)win, a.T, a.win, a.hop)
                        : cudaLaunchKernelEx(&cfg, gl_iter_kernel<false, false>, (const float*)mags, rp, nxt, (const float2*)tw,
                                             (const float*)win, a.T, a.win, a.hop);
    if (e != cudaSuccess) return e;
    float* tmp = cur; cur = nxt; nxt = tmp;
  }
  const int L = (a.T - 1) * a.hop + a.win;
  gl_ola_kernel<<<dim3((L + 255) / 256, a.N), 256, 0, st>>>(cur, a.wav, a.T, a.win, a.hop, L);
  if (a.preemphasis != 0.0f) gl_deemph_kernel<<<a.N, 1024, 0, st>>>(a.wav, L, a.preemphasis);
  if (launches) *launches = 4 + a.iters + (a.preemphasis != 0.0f ? 1 : 0);
  return cudaGetLastError();
}

}  // namespace taco
