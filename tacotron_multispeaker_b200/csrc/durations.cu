// Per-symbol durations from a teacher-forced attention alignment: the monotonic alignment search of Glow-TTS's
// monotonic_align.maximum_path (recurrence, band and tie rule), accumulated in float64, then frames per symbol.
//
// Utterance n has X text symbols, F target frames and Y = ceil(F / r) decoder steps.  Score s[y][x] = log(max((double)
// a[n][x][y], 2^-149)); cell (y, x) lies in the band max(0, X + y - Y) <= x <= min(X - 1, y); Q[0][0] = s[0][0] and
// Q[y][x] = s[y][x] + max(Q[y-1][x] (-inf when x == y), Q[y-1][x-1] (-inf when x == 0)).  The backtrack starts at X - 1
// on step Y - 1 and moves to x - 1 after step y when x != 0 and (x == y or Q[y-1][x] < Q[y-1][x-1]): a tie stays.
//
// One CTA per utterance, thread x owns symbol x and keeps Q[y][x] in a register.  The pass over y is sequential: per step
// a thread takes its left neighbour's Q[y-1] from a shuffle (lane 0 from shared memory, written by the previous warp's
// lane 31 one step earlier and double-buffered by step parity), so one CTA barrier per step suffices.  The decision bit
// of every (y, x) is taken in the same step (it compares the same two Q[y-1] values) and stored as one ballot word per
// warp and step in a global workspace.  Alignment columns are strided by `steps` floats, so the kernel stages tiles of
// X rows x DUR_TILE steps with coalesced row reads (cp.async, 4 bytes per lane, rows padded to DUR_TILE + 1 floats so
// that the per-thread column reads are free of bank conflicts), the next tile in flight while the current one is
// consumed; each thread computes the float64 logs of its own in-band cells of a tile into registers before the tile's
// sequential pass.  Warp 0 then walks the path back 32 steps at a time: its lanes load the two bit words of their step
// that the path can touch, and the walk reads them by shuffle, summing min(r, F - y r) frames per step into the symbol's
// duration.  Nothing outside rows < X and columns < Y of the alignment is read; no atomics.
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"
#include "kernels.cuh"

namespace taco {
namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kRow = DUR_TILE + 1;   // padded row of a staged tile (floats)

__device__ __forceinline__ void cp_async4(float* dst, const float* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait1() { asm volatile("cp.async.wait_group 1;\n" ::: "memory"); }

__global__ void __launch_bounds__(DUR_MAX_T_IN, 1) durations_kernel(const DurationsArgs a) {
  extern __shared__ float tiles[];   // [2][blockDim.x][kRow]
  __shared__ double edge[2][DUR_MAX_T_IN / 32];
  __shared__ int dur[DUR_MAX_T_IN];
  const int n = blockIdx.x, x = threadIdx.x, lane = x & 31, warp = x >> 5, W = blockDim.x >> 5;
  const int X = a.lengths[n], F = a.lengths[a.N + n], r = a.r;
  const int Y = (F + r - 1) / r;
  const float* an = a.align + (size_t)n * a.T_in * a.steps;
  uint32_t* bits = a.bits + (size_t)n * a.y_max * W;
  dur[x] = 0;
  if (lane == 0) edge[0][warp] = edge[1][warp] = -INFINITY;

  // tile k: steps [k DUR_TILE, (k + 1) DUR_TILE) of rows < X into buffer k & 1; warp w copies rows w, w + W, ...
  auto stage = [&](int k) {
    const int y = k * DUR_TILE + lane;
    float* dst = tiles + (size_t)(k & 1) * blockDim.x * kRow + lane;
    if (y < Y)
      for (int row = warp; row < X; row += W) cp_async4(dst + row * kRow, an + (size_t)row * a.steps + y);
    cp_async_commit();
  };

  const int ntiles = (Y + DUR_TILE - 1) / DUR_TILE;
  stage(0);
  double q = -INFINITY;   // Q[y - 1][x]
  int e = 0;              // edge buffer holding Q[y - 1] of the warps' last lanes
  for (int k = 0; k < ntiles; ++k) {
    // buffer (k + 1) & 1 was last read by the logs of tile k - 1, which every thread finished before that tile's barriers
    if (k + 1 < ntiles) stage(k + 1); else cp_async_commit();
    cp_async_wait1();
    __syncthreads();
    const int y0 = k * DUR_TILE;
    const float* src = tiles + (size_t)(k & 1) * blockDim.x * kRow + x * kRow;
    double s[DUR_TILE];
#pragma unroll
    for (int j = 0; j < DUR_TILE; ++j) {
      const int y = y0 + j;
      const bool band = x < X && y < Y && x >= X + y - Y && x <= y;
      s[j] = band ? log(fmax((double)src[j], 0x1p-149)) : 0.0;
    }
#pragma unroll
    for (int j = 0; j < DUR_TILE; ++j) {
      const int y = y0 + j;
      if (y >= Y) break;   // uniform over the CTA
      double ql = __shfl_up_sync(kFull, q, 1);
      if (lane == 0) ql = warp ? edge[e][warp - 1] : -INFINITY;
      double qn = -INFINITY;
      bool back = false;
      if (x < X && x >= X + y - Y && x <= y) {
        if (y == 0) {
          qn = s[j];
        } else {
          const double stay = x == y ? -INFINITY : q, adv = x == 0 ? -INFINITY : ql;
          back = x != 0 && (x == y || stay < adv);
          qn = s[j] + fmax(stay, adv);
        }
      }
      const uint32_t word = __ballot_sync(kFull, back);
      if (lane == 0) bits[(size_t)y * W + warp] = word;
      if (lane == 31) edge[e ^ 1][warp] = qn;
      q = qn;
      e ^= 1;
      __syncthreads();
    }
  }

  // the bits are visible to the CTA after the last barrier of the pass
  if (warp == 0) {
    int cx = X - 1, acc = 0;
    for (int yb = Y - 1; yb >= 0; yb -= 32) {
      // within these 32 steps the path stays in words w and w - 1 (it moves down by at most one symbol per step)
      const int w = cx >> 5, yl = yb - lane;
      uint32_t hi = 0, lo = 0;
      if (yl >= 0) {
        hi = bits[(size_t)yl * W + w];
        if (w > 0) lo = bits[(size_t)yl * W + w - 1];
      }
#pragma unroll
      for (int l = 0; l < 32; ++l) {
        const int y = yb - l;
        if (y < 0) break;   // uniform over the warp
        const uint32_t h = __shfl_sync(kFull, hi, l), lw = __shfl_sync(kFull, lo, l);
        acc += min(r, F - y * r);
        const uint32_t word = (cx >> 5) == w ? h : lw;
        if ((word >> (cx & 31)) & 1u) {
          if (lane == 0) dur[cx] = acc;
          acc = 0;
          --cx;
        }
      }
    }
    if (lane == 0) dur[cx] = acc;   // cx == 0 here
  }
  __syncthreads();
  if (x < a.T_in) a.out[(size_t)n * a.T_in + x] = dur[x];
}

int dur_threads(int T_in) { return (T_in + 31) / 32 * 32; }

}  // namespace

size_t durations_bits_bytes(int N, int T_in, int y_max) {
  return (size_t)N * y_max * (dur_threads(T_in) / 32) * sizeof(uint32_t);
}

cudaError_t launch_durations(const DurationsArgs& a, cudaStream_t st) {
  if (a.N < 1 || a.T_in < 1 || a.T_in > DUR_MAX_T_IN || a.steps < 1 || a.r < 1 || a.y_max < 1 || !a.align ||
      !a.lengths || !a.bits || !a.out)
    return cudaErrorInvalidValue;
  const int threads = dur_threads(a.T_in);
  const size_t smem = (size_t)2 * threads * kRow * sizeof(float);
  if (smem > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(durations_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  durations_kernel<<<a.N, threads, smem, st>>>(a);
  return cudaGetLastError();
}

}  // namespace taco
