// The 2048-point real FFT of the Griffin-Lim vocoder (griffin_lim.cu) and of the spectrogram analysis (spectrogram.cu):
// packed-pair complex arithmetic, the padded shared-memory layout, the decimation-in-frequency passes and the table kernel.
// A real 2048-point transform is a 1024-point complex one on z[m] = x[2m] + i x[2m+1]; one CTA of GL_NT threads owns one
// transform.  Everything is in an unnamed namespace: each translation unit that includes this compiles its own copy.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace taco {
namespace {

constexpr int GL_N = 2048, GL_M = GL_N / 2, GL_BINS = GL_N / 2 + 1, GL_NT = 128;
constexpr int GL_TW = GL_N / 4 + 1;   // twiddles W_N^k the kernel touches: k <= N/4

// Complex arithmetic on the packed fp32 pair instructions of sm_100 (FADD2 / FMUL2 / FFMA2: one issue slot for both halves; the
// kernel is issue bound, IPC 3.1 of 4).  Products and sums are rounded exactly where the scalar forms rounded them, so results
// are bit-identical: a b = (a.x, a.x) (b.x, b.y) + (a.y, a.y) (-b.y, b.x), a conj(b) = (a.x, a.y) (b.x, b.x) + (a.y, a.x) (b.y, -b.y).
typedef unsigned long long u64;
__device__ __forceinline__ u64 pk(float x, float y) { u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(x), "f"(y)); return r; }
__device__ __forceinline__ float2 up(u64 v) { float2 o; asm("mov.b64 {%0, %1}, %2;" : "=f"(o.x), "=f"(o.y) : "l"(v)); return o; }
__device__ __forceinline__ float2 cadd(float2 a, float2 b) {
  u64 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(pk(a.x, a.y)), "l"(pk(b.x, b.y))); return up(r);
}
__device__ __forceinline__ float2 csub(float2 a, float2 b) {
  u64 r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(pk(a.x, a.y)), "l"(pk(b.x, b.y))); return up(r);
}
__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
  u64 t, r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(t) : "l"(pk(a.y, a.y)), "l"(pk(-b.y, b.x)));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(pk(a.x, a.x)), "l"(pk(b.x, b.y)), "l"(t));
  return up(r);
}
__device__ __forceinline__ float2 cmul_conj(float2 a, float2 b) {   // a * conj(b)
  u64 t, r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(t) : "l"(pk(a.y, a.x)), "l"(pk(b.y, -b.y)));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(pk(a.x, a.y)), "l"(pk(b.x, b.x)), "l"(t));
  return up(r);
}
// element i of the transform sits at PD(i): one pad per 16 elements makes every FFT pass bank-conflict free, one more
// per 256 spreads the bit-reversed positions of the phase step (stride 64) over the banks (3.9 -> 1.5 wavefronts)
__device__ __forceinline__ int PD(int i) { return i + (i >> 4) + (i >> 8); }
constexpr int GL_DSIZE = GL_M + GL_M / 16 + GL_M / 256;

// a * exp(-i pi j / 8) (CONJ: a * exp(+i pi j / 8)), j a compile-time constant after unrolling
template <bool CONJ>
__device__ __forceinline__ float2 mul_w16(float2 a, int j) {
  constexpr float C1 = 0.9238795325112867f, S1 = 0.3826834323650898f, H = 0.7071067811865476f;
  float c, s;
  switch (j) {
    case 0: return a;
    case 4: return CONJ ? make_float2(-a.y, a.x) : make_float2(a.y, -a.x);
    case 1: c = C1; s = S1; break;
    case 2: c = H; s = H; break;
    case 3: c = S1; s = C1; break;
    case 5: c = -S1; s = C1; break;
    case 6: c = -H; s = H; break;
    default: c = -C1; s = S1; break;
  }
  const float2 w = make_float2(c, -s);
  return CONJ ? cmul_conj(a, w) : cmul(a, w);
}

// twiddles exp(-2 pi i k / 2048), k <= 512, and the periodic Hann window, evaluated in double
__global__ void gl_tables_kernel(float2* tw, float* win, int win_len) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < GL_TW) {
    double s, c;
    sincospi(-2.0 * (double)i / (double)GL_N, &s, &c);
    tw[i] = make_float2((float)c, (float)s);
  }
  if (i < win_len) win[i] = (float)(0.5 - 0.5 * cospi(2.0 * (double)i / (double)win_len));
}

// LOGR radix-2 stages of the 1024-point transform, decimation in frequency, half-spans (R/2) q, ..., q (R = 2^LOGR,
// q = 2^LOGQ), in registers.  The twiddle of stage s for element lo + j q is W_{2 hs q}^{lo} * W_{2 hs}^{j}: one table
// read per group (squared from stage to stage) times a constant.
template <int LOGR, int LOGQ>
__device__ __forceinline__ void dif_core(float2 (&v)[1 << LOGR], int lo, const float2* tw) {
  constexpr int R = 1 << LOGR, Q = 1 << LOGQ;
  static_assert(R <= 16, "constant twiddles go up to W_16");
  float2 wb = make_float2(1.0f, 0.0f);
  if (LOGQ > 0) wb = __ldg(tw + lo * (GL_N / (R * Q)));
#pragma unroll
  for (int s = 0; s < LOGR; ++s) {
    const int hs = R >> (s + 1);
#pragma unroll
    for (int m = 0; m < R; ++m) {
      if (m & hs) continue;
      const float2 a = v[m], b = v[m + hs];
      v[m] = cadd(a, b);
      float2 t = mul_w16<false>(csub(a, b), (m & (hs - 1)) * (8 / hs));
      if (LOGQ > 0) t = cmul(t, wb);
      v[m + hs] = t;
    }
    if (LOGQ > 0) wb = cmul(wb, wb);
  }
}
template <int LOGR, int LOGQ, bool LOAD = true>
__device__ __forceinline__ void dif_pass(float2* d, const float2* tw, int tid, float2* vin = nullptr) {
  constexpr int R = 1 << LOGR, Q = 1 << LOGQ;
  static_assert(GL_M / R <= GL_NT, "one group per thread");
  if (tid < GL_M / R) {   // GL_M / R <= GL_NT: at most one group per thread
    const int g = tid;
    const int lo = g & (Q - 1), base = ((g >> LOGQ) << (LOGR + LOGQ)) + lo;
    // element m sits at PD(base + m q) = PD(base) + m PS + (m q >> 8): q is a multiple of 16, or base is and the group
    // fits in 16; the per-256 pad moves only for q = 128 (base < 128), otherwise a group stays inside one 256 block
    static_assert(Q >= 16 || R * Q <= 16, "padded stride");
    static_assert(Q == 128 || R * Q <= 128, "per-256 pad");
    constexpr int PS = Q >= 16 ? Q + Q / 16 : Q;
    float2* dp = d + PD(base);
    float2 v[R];
#pragma unroll
    for (int m = 0; m < R; ++m) v[m] = LOAD ? dp[m * PS + (Q == 128 ? (m >> 1) : 0)] : vin[m];
    dif_core<LOGR, LOGQ>(v, lo, tw);
#pragma unroll
    for (int m = 0; m < R; ++m) dp[m * PS + (Q == 128 ? (m >> 1) : 0)] = v[m];
  }
}

}  // namespace
}  // namespace taco
