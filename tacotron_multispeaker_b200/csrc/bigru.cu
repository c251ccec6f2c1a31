// K6b: recurrence of the CBHG bidirectional GRU as a persistent kernel.
//
// Replaces tf.nn.bidirectional_dynamic_rnn(GRUCell(128), GRUCell(128), x,
// sequence_length) at reference models/modules.py:68-74 (a tf.while_loop of
// T_in resp. T_out=1000 iterations per direction).  The input halves of the
// GRU kernels are hoisted into one dense GEMM (xproj, conv_umma.cu); what is
// left per step and direction is
//     [r|u] = sigmoid(xg_t + h U_g)      U_g [128,256]
//     c     = tanh  (xc_t + (r*h) U_c)   U_c [128,128]   (reset BEFORE matmul: TF GRUCell)
//     h'    = u*h + (1-u)*c
// One CTA owns (direction, NS samples) for the whole sequence: the gate kernel
// U_g and the candidate kernel U_c live in REGISTERS (64 + 32 per thread x 512
// threads) for all steps, h lives in shared memory, nothing
// crosses CTAs, and the hoisted projections stream in through a 4-deep
// cp.async ring.  What bounds a step is the shared-memory -> register path
// that broadcasts h to the threads (ncu: 45% short-scoreboard in the first
// version, where every thread read a 64-float slice of h): a thread therefore
// covers 8 gate / 4 candidate columns of an 8-float k-slice (8x less LDS
// traffic) and the 16 slices of a column group are summed inside a half warp
// by shuffles, so a step needs two block barriers.
#include "common.cuh"
#include "kernels.cuh"

namespace taco {

namespace {
constexpr int H = 128;        // GRU width
constexpr int XW = 768;       // xproj row: [fw gates 256 | fw cand 128 | bw gates 256 | bw cand 128]
constexpr int RING = 12;      // prefetch distance (steps) of the hoisted projections: covers the L2/HBM latency

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int Nw> __device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(Nw) : "memory");
}

// h and r*h are stored so that the 16 k-slices (8 floats each) a warp reads together are two
// contiguous 256 B runs: element k = 8*ks + 4*j + i sits at (j*16 + ks)*4 + i.
__device__ __forceinline__ int idx_k(int k) { return (((k >> 2) & 1) * 16 + (k >> 3)) * 4 + (k & 3); }

template <int NS>
__global__ void __launch_bounds__(512, 1)
bigru_kernel(const float* __restrict__ xproj, const float* __restrict__ ug,
             const float* __restrict__ uc, const int32_t* __restrict__ lengths, int N, int T,
             float* __restrict__ out, int64_t out_bs) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int dir = blockIdx.y;
  const int n0 = blockIdx.x * NS;

  extern __shared__ __align__(16) float sm[];
  float* hs = sm;                                    // [NS][128]  h        (idx_k layout)
  float* rh = hs + NS * H;                           // [NS][128]  r*h      (idx_k layout)
  float* us = rh + NS * H;                           // [NS][128]  update gate
  float* ring = us + NS * H;                         // [RING][NS][384] hoisted projections
  __shared__ int s_len[NS];

  // ---- recurrent weights -> registers.  The shared-memory -> register path (128 B/clk) is what
  // bounds a step, so a thread covers MANY columns of a SHORT k-slice: 8 gate columns x 8 k and
  // 4 candidate columns x 8 k (64 + 32 weights); the 16 k-slices of a column group sit in the 16
  // lanes of a half warp and are summed with shuffles.
  const int ks = lane & 15, cgp = warp * 2 + (lane >> 4);     // k-slice, column group (0..31)
  float wg[8][8], wc[4][8];
  {
    const float* Ug = ug + (size_t)dir * H * 2 * H;
    const float* Uc = uc + (size_t)dir * H * H;
#pragma unroll
    for (int kk = 0; kk < 8; ++kk) {
#pragma unroll
      for (int c = 0; c < 8; ++c) wg[c][kk] = __ldg(Ug + (ks * 8 + kk) * (2 * H) + cgp * 8 + c);
#pragma unroll
      for (int c = 0; c < 4; ++c) wc[c][kk] = __ldg(Uc + (ks * 8 + kk) * H + cgp * 4 + c);
    }
  }
  // column whose total this lane holds after the shuffle reductions
  const int gsel = ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
  const int gcol = cgp * 8 + gsel;                   // gate column (0..255): r for < 128, u otherwise
  const int csel = ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
  const int ccol = cgp * 4 + csel;                   // candidate column (0..127)

  if (tid < NS) {
    int L = 0;
    if (n0 + tid < N) {
      L = lengths ? lengths[n0 + tid] : T;
      L = max(0, min(L, T));
    }
    s_len[tid] = L;
  }
  for (int i = tid; i < NS * 3 * H; i += 512) hs[i] = 0.f;
  __syncthreads();
  int len[NS], maxlen = 0;
#pragma unroll
  for (int s = 0; s < NS; ++s) { len[s] = s_len[s]; maxlen = max(maxlen, len[s]); }

  // outputs are zero for t >= len (dynamic_rnn zero_output); this CTA's 128 columns.
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    if (n0 + s >= N) continue;
    float* o = out + (int64_t)(n0 + s) * out_bs + dir * H;
    for (int i = len[s] * H + tid; i < T * H; i += 512) o[(int64_t)(i >> 7) * (2 * H) + (i & 127)] = 0.f;
  }

  // cp.async producer: thread (s, q) copies float4 q of sample s' 384-float row.  Only the first 3 NS warps copy; the
  // others skip the address arithmetic altogether (warp-uniform branch), and the ring slot is a running counter.
  const int ps = tid / 96, pq = tid - ps * 96;
  const bool copier = warp < 3 * NS;
  const int pL = (copier && ps < NS) ? s_len[ps] : 0;
  const float* psrc = xproj + ((int64_t)(n0 + ps) * T + (dir == 0 ? 0 : pL - 1)) * XW + dir * (3 * H) + pq * 4;
  const int64_t pstep = dir == 0 ? XW : -XW;                     // forward walks up, backward starts at L-1 and walks down
  float* pdst = ring + (size_t)ps * (3 * H) + pq * 4;
  int islot = 0, istep = 0;                                       // next step to request and its ring slot
  auto issue = [&]() {
    if (copier) {
      if (istep < pL) cp_async16(pdst + (size_t)islot * NS * (3 * H), psrc + (int64_t)istep * pstep);
      cp_async_commit();
      ++istep;
      islot = islot + 1 == RING ? 0 : islot + 1;
    }
  };
#pragma unroll
  for (int p = 0; p < RING - 1; ++p) issue();
  if (copier) cp_async_wait<RING - 2>();     // step 0's projections have landed (this thread's part) ...
  __syncthreads();               // ... and are visible to every thread

  int rslot = 0;
  for (int step = 0; step < maxlen; ++step) {
    issue();
    if (copier) cp_async_wait<RING - 2>();   // this thread's part of step+1's projections has landed; the two
                                             // barriers below publish it before step+1 reads it
    const float* xr = ring + (size_t)rslot * NS * (3 * H);
    rslot = rslot + 1 == RING ? 0 : rslot + 1;

    // ---- gates: 8 columns x this lane's 8 k, then sum over the 16 k-slices ----
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      const float4 h0 = *reinterpret_cast<const float4*>(hs + s * H + ks * 4);
      const float4 h1 = *reinterpret_cast<const float4*>(hs + s * H + 64 + ks * 4);
      const float hv[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
      float a[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) a[c] = 0.f;
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
#pragma unroll
        for (int c = 0; c < 8; c += 2) ffma2(a[c], a[c + 1], hv[kk], hv[kk], wg[c][kk], wg[c + 1][kk]);
      }
      // recursive halving over lane bits 3,2,1 (8 -> 4 -> 2 -> 1 values), butterfly over bit 0
      {
        const bool up = (lane & 8) != 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float send = up ? a[i] : a[i + 4], keep = up ? a[i + 4] : a[i];
          a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
      }
      {
        const bool up = (lane & 4) != 0;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const float send = up ? a[i] : a[i + 2], keep = up ? a[i + 2] : a[i];
          a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
        }
      }
      {
        const bool up = (lane & 2) != 0;
        const float send = up ? a[0] : a[1], keep = up ? a[1] : a[0];
        a[0] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
      }
      float g = a[0] + __shfl_xor_sync(0xffffffffu, a[0], 1);
      if (!(lane & 1)) {
        g = sigmoid_f(xr[s * 3 * H + gcol] + g);
        if (gcol < H) rh[s * H + idx_k(gcol)] = g * hs[s * H + idx_k(gcol)];
        else us[s * H + gcol - H] = g;
      }
    }
    __syncthreads();             // r*h and u complete
    // ---- candidate: 4 columns x this lane's 8 k of r*h, then sum over the 16 k-slices ----
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      const float4 r0 = *reinterpret_cast<const float4*>(rh + s * H + ks * 4);
      const float4 r1 = *reinterpret_cast<const float4*>(rh + s * H + 64 + ks * 4);
      const float rv[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
      float a[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
        ffma2(a[0], a[1], rv[kk], rv[kk], wc[0][kk], wc[1][kk]);
        ffma2(a[2], a[3], rv[kk], rv[kk], wc[2][kk], wc[3][kk]);
      }
      {
        const bool up = (lane & 8) != 0;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const float send = up ? a[i] : a[i + 2], keep = up ? a[i + 2] : a[i];
          a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
      }
      {
        const bool up = (lane & 4) != 0;
        const float send = up ? a[0] : a[1], keep = up ? a[1] : a[0];
        a[0] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
      }
      float cs = a[0] + __shfl_xor_sync(0xffffffffu, a[0], 2);
      cs += __shfl_xor_sync(0xffffffffu, cs, 1);
      if (!(lane & 3) && step < len[s]) {
        const float c = tanh_f(xr[s * 3 * H + 2 * H + ccol] + cs);
        const float u = us[s * H + ccol], h = hs[s * H + idx_k(ccol)];
        const float hn = u * h + (1.0f - u) * c;
        hs[s * H + idx_k(ccol)] = hn;
        const int pos = dir == 0 ? step : len[s] - 1 - step;
        out[(int64_t)(n0 + s) * out_bs + (int64_t)pos * (2 * H) + dir * H + ccol] = hn;
      }
    }
    __syncthreads();             // new h complete before the next step's gate phase
  }
  if (copier) cp_async_wait<0>();
}

template <int NS>
constexpr size_t bigru_smem_bytes() {
  return sizeof(float) * (size_t)(NS * 3 * H + RING * NS * 3 * H);
}

}  // namespace

void launch_bigru(const float* xproj, const float* ug, const float* uc, const int32_t* lengths,
                  int N, int T, float* out, int64_t out_bs, cudaStream_t st) {
  if (N <= 0 || T <= 0) return;
  // Samples per CTA: keep 2*ceil(N/NS) CTAs within one wave of 148 SMs when possible.
  int NS = 1;
  while (NS < 4 && 2 * ((N + NS - 1) / NS) > 148) NS *= 2;
  dim3 grid((N + NS - 1) / NS, 2);
  static bool attr_done[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr_done[dev & 63]) {
    cudaFuncSetAttribute(bigru_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bigru_smem_bytes<1>());
    cudaFuncSetAttribute(bigru_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bigru_smem_bytes<2>());
    cudaFuncSetAttribute(bigru_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bigru_smem_bytes<4>());
    attr_done[dev & 63] = true;
  }
  if (NS == 1) bigru_kernel<1><<<grid, 512, bigru_smem_bytes<1>(), st>>>(xproj, ug, uc, lengths, N, T, out, out_bs);
  else if (NS == 2) bigru_kernel<2><<<grid, 512, bigru_smem_bytes<2>(), st>>>(xproj, ug, uc, lengths, N, T, out, out_bs);
  else bigru_kernel<4><<<grid, 512, bigru_smem_bytes<4>(), st>>>(xproj, ug, uc, lengths, N, T, out, out_bs);
}

}  // namespace taco
