// conv1d('same') / dense as a TMA-fed tcgen05 implicit GEMM (sm_100a).
//
// The dense and conv1d layers of the reference (models/modules.py:93-101, :10,
// :59-60, models/tacotron.py:68,101) on the 5th-generation tensor
// cores.  D[128 rows (n, t0..t0+127)] x [128 output channels] accumulates in
// TMEM (fp32) over k-blocks of 64 input channels per filter tap:
//
//   A tile  = activations x[n, t0 + j - pad_left + (0..127), c0..c0+63]  (bf16)
//             one 3-D TMA box per (tap j, channel block); rows outside [0,T)
//             are zero-filled by the TMA unit -- that IS the 'same' padding,
//             so no im2col buffer and no boundary code.
//   B tile  = W^T[out channel o0..o0+127][j*Cp + c0 .. +63]  (bf16, K-major)
//
// fp32 parity: the reference computes in fp32, so each operand is split into
// bf16 hi + bf16 lo (x = hi + lo to ~2^-17) and every k-step issues the three
// products hi*hi + hi*lo + lo*hi into the same fp32 TMEM accumulator (the
// dropped lo*lo term is ~2^-18 relative).  NSPLIT=1 is the plain bf16 mode.
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = MMA issuer (one
// elected thread), warps 2..5 = epilogue (TMEM -> registers -> smem transpose
// -> coalesced global stores, with bias / activation / folded BN /
// residual).  3-stage smem ring (64 KB per stage) with full/empty
// mbarriers; tcgen05.commit releases stages and signals the epilogue.
#include <cuda.h>
#include <cuda_bf16.h>

#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <unordered_map>

#include "common.cuh"
#include "kernels.cuh"

namespace taco {

namespace {
constexpr int BM = 128, BN = 128, BK = 64, MAX_STAGES = 3, NTHREADS_MAX = 320;   // 2 role warps + 4 or 8 epilogue warps
constexpr uint32_t TILE_BYTES = BM * BK * 2;            // 16 KB: one bf16 operand tile (A or B)
constexpr uint32_t STAGE_BYTES = 4 * TILE_BYTES;        // A_hi | A_lo | B_hi | B_lo
constexpr int EPI_LD = 36;                              // floats per staged row: 32 + 4 keeps 128-bit rows conflict free
constexpr uint32_t EPI_WARP_BYTES = 32 * EPI_LD * 4;    // per-warp 32 x 36 fp32 transpose staging (both epilogue paths)
// dynamic smem: 1024 (alignment slack) + stages * 64 KB + [transpose staging] + barriers
__host__ __device__ constexpr uint32_t smem_bytes(int stages, int epi_warps) {
  return 1024u + (uint32_t)stages * STAGE_BYTES + (uint32_t)epi_warps * EPI_WARP_BYTES + 256u;
}

struct UmmaArgs {
  int N, T, Cp;            // activation rows / padded channels (Cp % 64 == 0)
  int kvalid;              // input channels rounded up to 16: k-steps beyond them multiply zero padding and are skipped
  int taps, bank;          // bank > 1: conv index ci = bank-1-blockIdx.z has ci+1 taps
  int Cout;                // output channels per conv
  const float* bias; const float* scale; const float* shift;
  const float* res; long long res_bs; int ldres;
  float* out; long long out_bs; int ldo; int col_off;
  void* out_hi; void* out_lo; int out_cp;   // bf16 hi / lo copy of the result [N][T][out_cp] (null: none)
  int act;
  int stages;              // smem ring depth (1..3)
  int vec_epi;             // 1: rows are 16 B aligned -> direct 128-bit stores from the TMEM registers
  int nx, ny, ntiles;      // tile list: nx = N * ceil(T / 128) row tiles, ny column tiles, ntiles = nx * ny * bank
  int acc_cols;            // TMEM columns to allocate: 256 (two accumulators, persistent CTAs) or 128 (one tile per CTA)
  int epi_warps;           // 4 or 8 (block = 64 + 32 * epi_warps threads)
};

// ---- PTX wrappers -------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t mb, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mb), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t mb, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t mb) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(mb) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mb, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(mb), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t mb, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(mb), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t mb, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(mb), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, fp32 accumulate, issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t mb) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mb) : "memory");
}
// K-major, SWIZZLE_128B operand tile: rows are 128 B apart, 8-row groups 1024 B apart.
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFF) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}


// (a, b) -> packed bf16 hi pair (return) and lo pair.  One packed conversion (F2FP, FMA pipe) per pair instead of two scalar
// F2F on the XU pipe, which the sigmoids' EX2 / RCP already saturate (ncu: mio_throttle on the conversions).
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b, uint32_t& lo_out) {
  uint32_t hi;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(b), "f"(a));      // upper half <- first source
  const float ra = a - __uint_as_float(hi << 16), rb = b - __uint_as_float(hi & 0xffff0000u);
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(lo_out) : "f"(rb), "f"(ra));
  return hi;
}

// ---- epilogue -----------------------------------------------------------------------------------------------------
struct EpiTile {
  int n, tq, o0;           // utterance, first row of this warp's 32 rows, first column of the tile
  const float* bias; const float* scale; const float* shift;
  int col_off;
};
template <int ACT> __device__ __forceinline__ float act_t(float v, int act) {
  if (ACT == 0) return v;
  if (ACT == 1) return fmaxf(v, 0.0f);
  return apply_act(v, act);
}
__device__ __forceinline__ void stage_rows_f4(float* stg, int lane, const uint32_t (&v)[32]) {
#pragma unroll
  for (int g = 0; g < 8; ++g)
    *reinterpret_cast<float4*>(stg + lane * EPI_LD + 4 * g) =
        make_float4(__uint_as_float(v[4 * g]), __uint_as_float(v[4 * g + 1]), __uint_as_float(v[4 * g + 2]), __uint_as_float(v[4 * g + 3]));
}

// Vector path (rows 16 B aligned): a thread reads ONE ROW of the accumulator from TMEM (32 columns per load).  Storing from
// there would touch 32 different rows per instruction (32 half-used sectors); the chunk is transposed through a 32 x 36
// shared-memory tile instead, so that a store instruction covers 4 rows x 128 contiguous bytes and the residual is read the
// same way.  Bias / activation / BN affine / residual run after the transpose.
template <int ACT, bool SC, bool RES>
__device__ __forceinline__ void epi_plain_vec(const UmmaArgs& p, const EpiTile& e, float* stg, uint32_t acc, int ch_lo, int ch_hi, int lane) {
  const int rsub = lane >> 3, c4 = lane & 7;                              // after the transpose: row 4 i + rsub, columns 4 c4 .. 4 c4 + 3
#pragma unroll 1
  for (int ch = ch_lo; ch < ch_hi; ++ch) {
    const int cbase = e.o0 + ch * 32;
    if (cbase >= p.Cout && !(p.out_hi != nullptr && cbase < p.out_cp)) break;   // warp-uniform (padding channels of the bf16 copy are zero-filled)
    uint32_t v[32];
    tmem_ld32(acc + (uint32_t)(ch * 32), v);
    stage_rows_f4(stg, lane, v);
    __syncwarp();
    const int col = cbase + 4 * c4;
    const bool cok = col < p.Cout;                                        // Cout % 4 == 0 on this path
    float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f), sc4 = make_float4(1.f, 1.f, 1.f, 1.f), sh4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (cok) {
      if (e.bias) b4 = ldg_f4(e.bias + col);
      if (SC && e.scale) { sc4 = ldg_f4(e.scale + col); sh4 = ldg_f4(e.shift + col); }
    }
    float* orow = p.out != nullptr ? p.out + (long long)e.n * p.out_bs + (long long)(e.tq + rsub) * p.ldo + e.col_off + col : nullptr;
    const bool has_res = RES && p.res != nullptr;
    const float* rrow = has_res ? p.res + (long long)e.n * p.res_bs + (long long)(e.tq + rsub) * p.ldres + col : nullptr;
    const int rows_left = p.T - e.tq - rsub;                              // row 4 i + rsub is valid iff 4 i < rows_left
    // bf16 hi / lo copy for the consuming GEMM: row (n T + t) of [N][T][out_cp], zeros in the padding channels
    const bool bf_out = p.out_hi != nullptr && col < p.out_cp;
    uint16_t* hrow = nullptr; uint16_t* lrow = nullptr;
    if (bf_out) {
      const long long r0 = ((long long)e.n * p.T + e.tq + rsub) * p.out_cp + col;
      hrow = reinterpret_cast<uint16_t*>(p.out_hi) + r0;
      lrow = reinterpret_cast<uint16_t*>(p.out_lo) + r0;
    }
#pragma unroll
    for (int i0 = 0; i0 < 8; i0 += 4) {                                  // four rows per thread at a time: residuals requested up front
      float4 r4[4];
      if (RES) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          r4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (has_res && cok && 4 * (i0 + i) < rows_left) r4[i] = ldg_f4(rrow + (4 * (i0 + i)) * p.ldres);
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float4 x = *reinterpret_cast<const float4*>(stg + (4 * (i0 + i) + rsub) * EPI_LD + 4 * c4);
        x.x = act_t<ACT>(x.x + b4.x, p.act); x.y = act_t<ACT>(x.y + b4.y, p.act);
        x.z = act_t<ACT>(x.z + b4.z, p.act); x.w = act_t<ACT>(x.w + b4.w, p.act);
        if (SC) { x.x = fmaf(x.x, sc4.x, sh4.x); x.y = fmaf(x.y, sc4.y, sh4.y); x.z = fmaf(x.z, sc4.z, sh4.z); x.w = fmaf(x.w, sc4.w, sh4.w); }
        if (4 * (i0 + i) < rows_left) {
          if (RES) { x.x += r4[i].x; x.y += r4[i].y; x.z += r4[i].z; x.w += r4[i].w; }
          if (cok && orow != nullptr) *reinterpret_cast<float4*>(orow + (4 * (i0 + i)) * p.ldo) = x;
          if (bf_out) {
            if (!cok) x = make_float4(0.f, 0.f, 0.f, 0.f);
            uint2 h2, l2;
            h2.x = pack_bf16x2(x.x, x.y, l2.x); h2.y = pack_bf16x2(x.z, x.w, l2.y);
            *reinterpret_cast<uint2*>(hrow + (4 * (i0 + i)) * p.out_cp) = h2;
            *reinterpret_cast<uint2*>(lrow + (4 * (i0 + i)) * p.out_cp) = l2;
          }
        }
      }
    }
    __syncwarp();
  }
}

// Scalar path (rows not 16 B aligned, e.g. the 1025-wide linear output): the chunk is staged with a pitch of 33 floats (scalar
// stores of a row-per-lane tile are then conflict free), lane = column afterwards: one store instruction writes 128 contiguous
// bytes of one output row.
template <int ACT, bool SC, bool RES>
__device__ __forceinline__ void epi_plain_scalar(const UmmaArgs& p, const EpiTile& e, float* stg, uint32_t acc, int ch_lo, int ch_hi, int lane) {
  constexpr int LD = 33;
#pragma unroll 1
  for (int ch = ch_lo; ch < ch_hi; ++ch) {
    const int cbase = e.o0 + ch * 32;
    if (cbase >= p.Cout) break;                                           // warp-uniform
    uint32_t v[32];
    tmem_ld32(acc + (uint32_t)(ch * 32), v);
#pragma unroll
    for (int c = 0; c < 32; ++c) stg[lane * LD + c] = __uint_as_float(v[c]);
    __syncwarp();
    const int col = cbase + lane;
    const bool cok = col < p.Cout;
    float b = 0.f, sc = 1.f, sh = 0.f;
    if (cok) {
      if (e.bias) b = __ldg(e.bias + col);
      if (SC && e.scale) { sc = __ldg(e.scale + col); sh = __ldg(e.shift + col); }
    }
    const int nrows = min(32, p.T - e.tq);                                // warp-uniform
    float* optr = p.out + (long long)e.n * p.out_bs + (long long)e.tq * p.ldo + e.col_off + col;
    const bool has_res = RES && p.res != nullptr;
    const float* rptr = has_res ? p.res + (long long)e.n * p.res_bs + (long long)e.tq * p.ldres + col : nullptr;
    const float* sp = stg + lane;
    const int ldo = p.ldo, ldres = p.ldres;
    if (nrows == 32) {                                                    // full tile: no row predicates, row pointers advance by ldo
#pragma unroll
      for (int r0 = 0; r0 < 32; r0 += 8) {
        float x[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          x[r] = act_t<ACT>(sp[(r0 + r) * LD] + b, p.act);
          if (SC) x[r] = fmaf(x[r], sc, sh);
        }
        if (cok) {
          if (has_res) {
#pragma unroll
            for (int r = 0; r < 8; ++r) { x[r] += __ldg(rptr); rptr += ldres; }
          }
#pragma unroll
          for (int r = 0; r < 8; ++r) { *optr = x[r]; optr += ldo; }
        }
      }
    } else if (cok) {
      for (int r = 0; r < nrows; ++r) {
        float x = act_t<ACT>(sp[r * LD] + b, p.act);
        if (SC) x = fmaf(x, sc, sh);
        if (has_res) { x += __ldg(rptr); rptr += ldres; }
        *optr = x;
        optr += ldo;
      }
    }
    __syncwarp();
  }
}

template <int NSPLIT, int EV>
__global__ void __launch_bounds__(NTHREADS_MAX, 2)
conv_umma_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
                 const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo,
                 const UmmaArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const int STAGES = p.stages;
  const uint32_t epi_bytes = (uint32_t)p.epi_warps * EPI_WARP_BYTES;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;       // SWIZZLE_128B tiles need 1024 B alignment
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  float* epi = reinterpret_cast<float*>(smem_al + STAGES * STAGE_BYTES);
  const uint32_t bar0 = smem_base + STAGES * STAGE_BYTES + epi_bytes;    // full[S], empty[S], tmem_full[2], tmem_empty[2], tmem ptr
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (MAX_STAGES + s); };
  auto tfull_bar = [&](int b) { return bar0 + 8u * (2 * MAX_STAGES + b); };
  auto tempty_bar = [&](int b) { return bar0 + 8u * (2 * MAX_STAGES + 2 + b); };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem_al + STAGES * STAGE_BYTES + epi_bytes + 8 * (2 * MAX_STAGES + 4));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tps = (p.T + BM - 1) / BM;
  const int kcb = p.Cp / BK;
  // Persistent CTA: tiles blockIdx.x, blockIdx.x + gridDim.x, ... in the order (conv of the bank, heavy first; column
  // tile; row tile fastest, so that the CTAs working at the same time share their weight tiles in L2).  The TMA, MMA and
  // epilogue roles each walk the same list; the accumulator alternates between two 128-column TMEM buffers, so the
  // epilogue of tile i overlaps the loads and MMAs of tile i+1.
  struct Tile { int n, t0, o0, ci, taps, pl, nkb, brow0; };
  auto decode = [&](int L) {
    Tile q;
    const int x = L % p.nx, r = L / p.nx, y = r % p.ny, z = r / p.ny;   // row tile fastest: neighbours share the weight tile
    q.n = x / tps; q.t0 = (x - q.n * tps) * BM; q.o0 = y * BN;
    q.ci = p.bank > 1 ? p.bank - 1 - z : 0;                               // heavy convs first
    q.taps = p.bank > 1 ? q.ci + 1 : p.taps;
    q.pl = (q.taps - 1) >> 1;
    q.nkb = q.taps * kcb;
    q.brow0 = q.ci * p.Cout + q.o0;
    return q;
  };

  if (threadIdx.x == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA_hi)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB_hi)) : "memory");
    if (NSPLIT > 1) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA_lo)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB_lo)) : "memory");
    }
    for (int s = 0; s < MAX_STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(tfull_bar(b), 1); mbar_init(tempty_bar(b), (uint32_t)p.epi_warps); }   // every epilogue warp releases a buffer
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {   // TMEM: two 128-column fp32 accumulators, allocated (and later freed) by this warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"((uint32_t)p.acc_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int it = 0;                                                         // k-block counter over all tiles of this CTA
      for (int L = blockIdx.x; L < p.ntiles; L += gridDim.x) {
        const Tile q = decode(L);
        for (int kb = 0; kb < q.nkb; ++kb, ++it) {
          const int s = it % STAGES;
          mbar_wait(empty_bar(s), ((it / STAGES) & 1) ^ 1);
          const uint32_t st = smem_base + s * STAGE_BYTES;
          mbar_expect_tx(full_bar(s), NSPLIT > 1 ? STAGE_BYTES : 2 * TILE_BYTES);
          const int j = kb / kcb, c0 = (kb - j * kcb) * BK;
          const int tt = q.t0 + j - q.pl;                                 // may be < 0 or run past T: zero fill
          tma_load_3d(st, &tmA_hi, full_bar(s), c0, tt, q.n);
          tma_load_2d(st + 2 * TILE_BYTES, &tmB_hi, full_bar(s), j * p.Cp + c0, q.brow0);
          if (NSPLIT > 1) {
            tma_load_3d(st + TILE_BYTES, &tmA_lo, full_bar(s), c0, tt, q.n);
            tma_load_2d(st + 3 * TILE_BYTES, &tmB_lo, full_bar(s), j * p.Cp + c0, q.brow0);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      // kind::f16: C=F32 (bit4), A=BF16 (bit7), B=BF16 (bit10), both K-major, N>>3 at bit17, M>>4 at bit24
      constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
      int it = 0, i = 0;
      for (int L = blockIdx.x; L < p.ntiles; L += gridDim.x, ++i) {
        const Tile q = decode(L);
        const int b = i & 1;
        mbar_wait(tempty_bar(b), ((i >> 1) & 1) ^ 1);                     // the epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t acc = tmem_base + (uint32_t)(b * BN);
        for (int kb = 0; kb < q.nkb; ++kb, ++it) {
          const int s = it % STAGES;
          mbar_wait(full_bar(s), (it / STAGES) & 1);
          tc_fence_after();
          const uint32_t st = smem_base + s * STAGE_BYTES;
          const uint64_t a_hi = umma_desc(st), a_lo = umma_desc(st + TILE_BYTES);
          const uint64_t b_hi = umma_desc(st + 2 * TILE_BYTES), b_lo = umma_desc(st + 3 * TILE_BYTES);
          const int nk = min(BK / 16, (p.kvalid - (kb % kcb) * BK + 15) >> 4);   // e.g. 80 channels: 4 + 1 k-steps per tap, not 8
#pragma unroll
          for (int kk = 0; kk < BK / 16; ++kk) {
            if (kk >= nk) break;
            const uint64_t adv = (uint64_t)(kk * 32 >> 4);                // 16 bf16 = 32 B along K inside the swizzle row
            umma_bf16(acc, a_hi + adv, b_hi + adv, idesc, (kb | kk) != 0);
            if (NSPLIT > 1) {
              umma_bf16(acc, a_hi + adv, b_lo + adv, idesc, 1u);
              umma_bf16(acc, a_lo + adv, b_hi + adv, idesc, 1u);
            }
          }
          umma_commit(empty_bar(s));                                      // stage free once these MMAs have read it
        }
        umma_commit(tfull_bar(b));                                        // accumulator complete
      }
    }
  } else {
    // ===================== epilogue (warps 2 .. 2 + EW - 1) =====================
    // A warp may read the TMEM lane quarter (warp & 3); with eight epilogue warps two warps share a quarter and split the
    // four 32-column chunks of a tile between them.  The per-element work is compiled for the launch's (activation, BN
    // affine, residual) combination: a run-time switch inside the loops cost ~30 instructions per stored row.
    const int quarter = warp & 3;                                         // TMEM lanes this warp may read
    const int half = (warp - 2) >> 2;                                     // 0 (warps 2..5) or 1 (warps 6..9)
    const int ch_lo = p.epi_warps == 8 ? 2 * half : 0, ch_hi = p.epi_warps == 8 ? 2 * half + 2 : BN / 32;
    float* stg = epi + (warp - 2) * 32 * EPI_LD;
    int i = 0;
    for (int L = blockIdx.x; L < p.ntiles; L += gridDim.x, ++i) {
      const Tile q = decode(L);
      const int ab = i & 1;
      const uint32_t acc = tmem_base + (uint32_t)(ab * BN) + ((uint32_t)(quarter * 32) << 16);
      mbar_wait(tfull_bar(ab), (i >> 1) & 1);
      tc_fence_after();
      EpiTile e;
      e.n = q.n; e.tq = q.t0 + quarter * 32; e.o0 = q.o0;
      e.bias = p.bias ? p.bias + q.ci * p.Cout : nullptr;
      e.scale = p.scale ? p.scale + q.ci * p.Cout : nullptr;
      e.shift = p.shift ? p.shift + q.ci * p.Cout : nullptr;
      e.col_off = p.col_off + q.ci * p.Cout;
      // EV: the launch's epilogue variant, compiled in (0 = any combination, decided at run time)
      constexpr int A = EV == 0 ? 2 : ((EV == 2 || EV == 3) ? 1 : 0);
      constexpr bool S = EV == 0 || EV == 3 || EV == 4, R = EV == 0 || EV == 4;
      if (p.vec_epi) epi_plain_vec<A, S, R>(p, e, stg, acc, ch_lo, ch_hi, lane);
      else epi_plain_scalar<A, S, R>(p, e, stg, acc, ch_lo, ch_hi, lane);
      // this warp has read its lanes of the accumulator: hand the buffer back to the MMA issuer
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(ab));
    }   // tile loop
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.acc_cols) : "memory");
  }
}

// ---- the four highway layers of a CBHG in ONE kernel (reference models/modules.py:63-64, 79-89) -------------------------
// highwaynet x 4 on [rows, 128]: y = relu(x W_H + b_H) T + x (1 - T), T = sigmoid(x W_T + b_T), four times.  As four
// conv_umma launches (+ four hi/lo split passes) the 16 MB activation made eight HBM / L2 round trips and every launch paid its
// own pipeline fill (25.7 us each for 2.1 GF).  Here a CTA owns 128 rows for all layers: the activation lives in the epilogue
// threads' REGISTERS (one row x 32 channels per thread, four threads per row), is re-written as bf16 hi / lo operand tiles in
// shared memory (128-byte swizzle, K-major: what TMA would have produced) for the next layer's tcgen05.mma, and only the weights
// (128 KB per layer, hi + lo, L2 resident) stream in by TMA -- prefetched during the previous layer's epilogue.
struct Hw4Args {
  const float* x; float* out;          // [rows][128] fp32, dense (out nullable: only the bf16 copy is wanted)
  void* out_hi; void* out_lo;          // optional bf16 hi / lo copy of the result [rows][128] (operand of the next GEMM), or null
  const float* bias[4];                // per layer [256], interleaved (b_H[c], b_T[c])
  int rows, layers, ntiles;
};
constexpr uint32_t HW_A_BYTES = 4 * TILE_BYTES;                  // A_hi kb0 | A_hi kb1 | A_lo kb0 | A_lo kb1   (64 KB)
constexpr uint32_t HW_BSTAGE = 4 * TILE_BYTES;                   // per k-block: B_hi (256 x 64, 32 KB) | B_lo (32 KB)
constexpr uint32_t HW_SMEM = 1024u + HW_A_BYTES + 2 * HW_BSTAGE + 256u + 4 * 256 * 4;   // + the four layers' biases
constexpr int HW_THREADS = 64 + 16 * 32;                       // TMA warp, MMA warp, sixteen epilogue warps

template <int NSPLIT>
__global__ void __launch_bounds__(HW_THREADS, 1)
highway4_kernel(const __grid_constant__ CUtensorMap tmB, const Hw4Args p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t a_base = smem_base, b_base = smem_base + HW_A_BYTES;
  const uint32_t bar0 = b_base + 2 * HW_BSTAGE;                    // b_full[2], b_empty[2], a_ready, acc_full, tmem slot
  auto b_full = [&](int kb) { return bar0 + 8u * kb; };
  auto b_empty = [&](int kb) { return bar0 + 16u + 8u * kb; };
  const uint32_t a_ready = bar0 + 32u;
  auto acc_full = [&](int half) { return bar0 + 40u + 8u * half; };   // accumulator columns 128 half .. 128 half + 127 complete
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem_al + HW_A_BYTES + 2 * HW_BSTAGE + 56);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* bias_s = reinterpret_cast<float*>(smem_al + HW_A_BYTES + 2 * HW_BSTAGE + 256);   // [4 layers][256] (b_H, b_T) interleaved
  for (int i = threadIdx.x; i < p.layers * 256; i += HW_THREADS) bias_s[i] = __ldg(p.bias[i >> 8] + (i & 255));

  if (threadIdx.x == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB)) : "memory");
    for (int kb = 0; kb < 2; ++kb) { mbar_init(b_full(kb), 1); mbar_init(b_empty(kb), 1); }
    mbar_init(a_ready, HW_THREADS - 64);                              // every epilogue thread arrives
    mbar_init(acc_full(0), 1); mbar_init(acc_full(1), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32((const void*)tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer: the layer's W^T (hi, lo), one k-block of 64 inputs per stage =====================
    if (lane == 0) {
      int n = 0;
      for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x)
        for (int l = 0; l < p.layers; ++l, ++n)
          for (int kb = 0; kb < 2; ++kb) {
            mbar_wait(b_empty(kb), (n & 1) ^ 1);
            const uint32_t st = b_base + kb * HW_BSTAGE;
            mbar_expect_tx(b_full(kb), NSPLIT > 1 ? HW_BSTAGE : HW_BSTAGE / 2);
            tma_load_3d(st, &tmB, b_full(kb), kb * BK, 0, 2 * l);
            if (NSPLIT > 1) tma_load_3d(st + 2 * TILE_BYTES, &tmB, b_full(kb), kb * BK, 0, 2 * l + 1);
          }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer: D[128 x 256] = A[128 x 128] W[128 x 256], three products per k-step =====================
    if (lane == 0) {
      // The 256 accumulator columns are produced as two halves of 128 (channels 0-63, then 64-127), each with its own commit: the
      // epilogue warps of the first half run while the tensor core works on the second.
      constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
      int n = 0;
      for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x)
        for (int l = 0; l < p.layers; ++l, ++n) {
          mbar_wait(a_ready, n & 1);                                  // operand tiles written, accumulator drained
          tc_fence_after();
          for (int half = 0; half < 2; ++half) {
            for (int kb = 0; kb < 2; ++kb) {
              if (half == 0) { mbar_wait(b_full(kb), n & 1); tc_fence_after(); }
              const uint64_t a_hi = umma_desc(a_base + kb * TILE_BYTES), a_lo = umma_desc(a_base + (2 + kb) * TILE_BYTES);
              const uint32_t brow = (uint32_t)half * 128u * 128u;      // weight rows 128 half ..: 128 rows x 128 bytes into the tile
              const uint64_t b_hi = umma_desc(b_base + kb * HW_BSTAGE + brow), b_lo = umma_desc(b_base + kb * HW_BSTAGE + 2 * TILE_BYTES + brow);
#pragma unroll
              for (int kk = 0; kk < BK / 16; ++kk) {
                const uint64_t adv = (uint64_t)(kk * 32 >> 4);
                umma_bf16(tmem_base + (uint32_t)half * 128u, a_hi + adv, b_hi + adv, idesc, (kb | kk) != 0);
                if (NSPLIT > 1) {
                  umma_bf16(tmem_base + (uint32_t)half * 128u, a_hi + adv, b_lo + adv, idesc, 1u);
                  umma_bf16(tmem_base + (uint32_t)half * 128u, a_lo + adv, b_hi + adv, idesc, 1u);
                }
              }
              if (half == 1) umma_commit(b_empty(kb));                // weights of this k-block consumed: the next layer's may land
            }
            umma_commit(acc_full(half));
          }
        }
    }
  } else {
    // ===================== epilogue warps 2..17: the activation in registers, gate math, operand tiles =====================
    // Sixteen warps (four per TMEM lane quarter, 32 channels each): the gate math is latency bound (EX2 -> RCP chains), four warps
    // per scheduler hide it better than two (8 warps x 64 channels: 55.7 us for the post-net's 250 tiles).
    const int quarter = warp & 3, part = (warp - 2) >> 2;             // TMEM lane quarter; channels 32 part .. 32 part + 31
    const int hf = part >> 1, j0 = (part & 1) * 4;                    // k-block of those channels, first 16-byte chunk inside its rows
    const int r = quarter * 32 + lane;                                // row of the tile = TMEM lane
    const uint32_t a_row = (uint32_t)((r >> 3) * 1024 + (r & 7) * 128);
    auto write_operands = [&](const float (&x)[32]) {
      const uint32_t hi_t = a_base + hf * TILE_BYTES + a_row, lo_t = a_base + (2 + hf) * TILE_BYTES + a_row;
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        const int j = j0 + jj;
        uint4 h4, l4;
        h4.x = pack_bf16x2(x[8 * jj + 0], x[8 * jj + 1], l4.x); h4.y = pack_bf16x2(x[8 * jj + 2], x[8 * jj + 3], l4.y);
        h4.z = pack_bf16x2(x[8 * jj + 4], x[8 * jj + 5], l4.z); h4.w = pack_bf16x2(x[8 * jj + 6], x[8 * jj + 7], l4.w);
        const uint32_t off = (uint32_t)((j ^ (r & 7)) << 4);          // 128-byte swizzle: 16-byte chunk j of row r sits at j ^ (r % 8)
        asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(hi_t + off), "r"(h4.x), "r"(h4.y), "r"(h4.z), "r"(h4.w) : "memory");
        asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(lo_t + off), "r"(l4.x), "r"(l4.y), "r"(l4.z), "r"(l4.w) : "memory");
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the tensor core's async proxy
      tc_fence_before();
      mbar_arrive(a_ready);
    };
    int n = 0;
    for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
      const long long row = (long long)tile * BM + r;
      const bool rok = row < p.rows;
      float x[32];
      {
        const float4* src = reinterpret_cast<const float4*>(p.x + row * 128 + part * 32);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 v4 = rok ? __ldg(src + i) : make_float4(0.f, 0.f, 0.f, 0.f);
          x[4 * i] = v4.x; x[4 * i + 1] = v4.y; x[4 * i + 2] = v4.z; x[4 * i + 3] = v4.w;
        }
      }
      write_operands(x);
      for (int l = 0; l < p.layers; ++l, ++n) {
        mbar_wait(acc_full(hf), n & 1);
        tc_fence_after();
        const float* bias = bias_s + l * 256 + part * 64;
#pragma unroll
        for (int ch = 0; ch < 2; ++ch) {
          uint32_t v[32];
          tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(part * 64 + ch * 32), v);
#pragma unroll
          for (int i = 0; i < 16; i += 2) {
            const float4 b4 = *reinterpret_cast<const float4*>(bias + ch * 32 + 2 * i);   // (b_H, b_T) of channels i, i + 1
            const float H0 = fmaxf(__uint_as_float(v[2 * i]) + b4.x, 0.f), T0 = sigmoid_f(__uint_as_float(v[2 * i + 1]) + b4.y);
            const float H1 = fmaxf(__uint_as_float(v[2 * i + 2]) + b4.z, 0.f), T1 = sigmoid_f(__uint_as_float(v[2 * i + 3]) + b4.w);
            x[ch * 16 + i] = fmaf(T0, H0 - x[ch * 16 + i], x[ch * 16 + i]);              // H T + x (1 - T)
            x[ch * 16 + i + 1] = fmaf(T1, H1 - x[ch * 16 + i + 1], x[ch * 16 + i + 1]);
          }
        }
        // The half-1 MMAs read both A k-blocks too and are not covered by acc_full(0): the hf = 0 warps wait for their commit
        // before overwriting k-block 0 (for the next layer, or the next tile at the top of the loop).  The gate math above has
        // already overlapped them.
        if (hf == 0) mbar_wait(acc_full(1), n & 1);
        if (l + 1 < p.layers) write_operands(x);                      // next layer's A operand (also releases the accumulator)
      }
      // results: fp32 rows (and, for the GEMM that follows, their bf16 hi / lo split)
      if (rok) {
        if (p.out != nullptr) {
          float4* dst = reinterpret_cast<float4*>(p.out + row * 128 + part * 32);
#pragma unroll
          for (int i = 0; i < 8; ++i) dst[i] = make_float4(x[4 * i], x[4 * i + 1], x[4 * i + 2], x[4 * i + 3]);
        }
        if (p.out_hi != nullptr) {
          uint4* dh = reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(p.out_hi) + row * 128 + part * 32);
          uint4* dl = reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(p.out_lo) + row * 128 + part * 32);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            uint4 h4, l4;
            h4.x = pack_bf16x2(x[8 * j + 0], x[8 * j + 1], l4.x); h4.y = pack_bf16x2(x[8 * j + 2], x[8 * j + 3], l4.y);
            h4.z = pack_bf16x2(x[8 * j + 4], x[8 * j + 5], l4.z); h4.w = pack_bf16x2(x[8 * j + 6], x[8 * j + 7], l4.w);
            dh[j] = h4; dl[j] = l4;
          }
        }
      }
      // the accumulator of this tile's last layer has been read: the first layer of the next tile may overwrite it (its
      // a_ready arrival comes from write_operands at the top of the loop, after tc_fence_before)
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem_base) : "memory");
  }
}

// fp32 -> bf16 hi + bf16 lo (x ~= hi + lo), channels zero-padded to Cp.
__global__ void __launch_bounds__(256)
split_bf16_kernel(const float* __restrict__ x, long long x_bs, int ldx, int N, int T, int C, int Cp,
                  __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  const int Cq = Cp >> 2;
  const long long total = (long long)N * T * Cq;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int q = (int)(i % Cq);
    const long long row = i / Cq;
    const int t = (int)(row % T), n = (int)(row / T);
    const int c = q * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c + 3 < C) v = ldg_f4(x + n * x_bs + (long long)t * ldx + c);
    else if (c < C) {
      const float* px = x + n * x_bs + (long long)t * ldx;
      v.x = px[c];
      if (c + 1 < C) v.y = px[c + 1];
      if (c + 2 < C) v.z = px[c + 2];
    }
    const __nv_bfloat16 h0 = __float2bfloat16_rn(v.x), h1 = __float2bfloat16_rn(v.y), h2 = __float2bfloat16_rn(v.z), h3 = __float2bfloat16_rn(v.w);
    const __nv_bfloat16 l0 = __float2bfloat16_rn(v.x - __bfloat162float(h0)), l1 = __float2bfloat16_rn(v.y - __bfloat162float(h1));
    const __nv_bfloat16 l2 = __float2bfloat16_rn(v.z - __bfloat162float(h2)), l3 = __float2bfloat16_rn(v.w - __bfloat162float(h3));
    __nv_bfloat162 hA, hB, lA, lB;
    hA.x = h0; hA.y = h1; hB.x = h2; hB.y = h3; lA.x = l0; lA.y = l1; lB.x = l2; lB.y = l3;
    uint2 ph, plo;
    ph.x = *reinterpret_cast<uint32_t*>(&hA); ph.y = *reinterpret_cast<uint32_t*>(&hB);
    plo.x = *reinterpret_cast<uint32_t*>(&lA); plo.y = *reinterpret_cast<uint32_t*>(&lB);
    reinterpret_cast<uint2*>(hi)[i] = ph;
    reinterpret_cast<uint2*>(lo)[i] = plo;
  }
}

__global__ void __launch_bounds__(256)
pack_wt_kernel(const float* __restrict__ w, int ldw, int taps, int Cin, int Cout, int Cp, int Kld, int row0,
               __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  const long long total = (long long)Cout * taps * Cp;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % Cp);
    const int j = (int)((i / Cp) % taps);
    const int o = (int)(i / ((long long)Cp * taps));
    const float v = c < Cin ? __ldg(w + (long long)(j * Cin + c) * ldw + o) : 0.f;
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    const long long dst = (long long)(row0 + o) * Kld + (long long)j * Cp + c;
    hi[dst] = h;
    lo[dst] = __float2bfloat16_rn(v - __bfloat162float(h));
  }
}

// ---- host: tensor maps ------------------------------------------------------------
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_tmapEncodeTiled get_encode() {
  static PFN_tmapEncodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_tmapEncodeTiled>(p);
  }
  return fn;
}
bool make_map(CUtensorMap* m, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
              const cuuint32_t* box) {
  PFN_tmapEncodeTiled enc = get_encode();
  if (!enc) return false;
  cuuint32_t es[3] = {1, 1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), dims, strides_bytes, box, es,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
}  // namespace

void launch_split_bf16(const float* x, int64_t x_bs, int ldx, int N, int T, int C, int Cp, void* hi, void* lo,
                       cudaStream_t st) {
  const long long total = (long long)N * T * (Cp / 4);
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks < 1) blocks = 1;
  split_bf16_kernel<<<blocks, 256, 0, st>>>(x, x_bs, ldx, N, T, C, Cp, reinterpret_cast<__nv_bfloat16*>(hi),
                                            reinterpret_cast<__nv_bfloat16*>(lo));
}

void launch_pack_wt(const float* w, int ldw, int taps, int Cin, int Cout, int Cp, int Kld, int row0, void* hi,
                    void* lo, cudaStream_t st) {
  const long long total = (long long)Cout * taps * Cp;
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks < 1) blocks = 1;
  pack_wt_kernel<<<blocks, 256, 0, st>>>(w, ldw, taps, Cin, Cout, Cp, Kld, row0, reinterpret_cast<__nv_bfloat16*>(hi),
                                         reinterpret_cast<__nv_bfloat16*>(lo));
}

// Tensor maps are pure functions of (base pointer, shape, box): encoded once and kept (the workspace and the weight arena
// are stable between forwards, so a forward re-uses its 84 maps instead of calling cuTensorMapEncodeTiled 84 times).
namespace {
struct MapKey {
  const void* base; uint64_t d0, d1, d2; uint32_t rank;
  bool operator==(const MapKey& o) const { return base == o.base && d0 == o.d0 && d1 == o.d1 && d2 == o.d2 && rank == o.rank; }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    uint64_t h = reinterpret_cast<uintptr_t>(k.base) * 0x9E3779B97F4A7C15ull;
    h ^= (k.d0 + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2));
    h ^= (k.d1 * 0xC2B2AE3D27D4EB4Full + (h << 6) + (h >> 2));
    h ^= (k.d2 * 0x165667B19E3779F9ull + k.rank + (h << 6) + (h >> 2));
    return (size_t)h;
  }
};
std::mutex g_map_mu;
std::unordered_map<MapKey, CUtensorMap, MapKeyHash> g_maps;

// A: activations [N][T][Cp] bf16, box {64 channels, 128 rows, 1 utterance};  B: W^T [rows][Kld] bf16, box {64, 128}
bool get_map_a(CUtensorMap* m, const void* base, int Cp, int T, int N) {
  const MapKey k{base, (uint64_t)Cp, (uint64_t)T, (uint64_t)N, 3u};
  std::lock_guard<std::mutex> lk(g_map_mu);
  auto it = g_maps.find(k);
  if (it != g_maps.end()) { *m = it->second; return true; }
  const cuuint64_t dims[3] = {(cuuint64_t)Cp, (cuuint64_t)T, (cuuint64_t)N};
  const cuuint64_t str[2] = {(cuuint64_t)Cp * 2, (cuuint64_t)T * Cp * 2};
  const cuuint32_t box[3] = {BK, BM, 1};
  if (!make_map(m, base, 3, dims, str, box)) return false;
  if (g_maps.size() > 8192) g_maps.clear();
  g_maps.emplace(k, *m);
  return true;
}
bool get_map_b(CUtensorMap* m, const void* base, int Kld, int rows) {
  const MapKey k{base, (uint64_t)Kld, (uint64_t)rows, 0u, 2u};
  std::lock_guard<std::mutex> lk(g_map_mu);
  auto it = g_maps.find(k);
  if (it != g_maps.end()) { *m = it->second; return true; }
  const cuuint64_t dims[2] = {(cuuint64_t)Kld, (cuuint64_t)rows};
  const cuuint64_t str[1] = {(cuuint64_t)Kld * 2};
  const cuuint32_t box[2] = {BK, BN};
  if (!make_map(m, base, 2, dims, str, box)) return false;
  if (g_maps.size() > 8192) g_maps.clear();
  g_maps.emplace(k, *m);
  return true;
}
int env_int(const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; }
}  // namespace

// Launch shapes (developer switches read once: TACO_UMMA_PERSISTENT = 0 / 1 forces, TACO_UMMA_EW, TACO_UMMA_STAGES_MAX, TACO_UMMA_CTAS):
//  * long K (>= 24 k-blocks: the 3 x 1024 -> 256 projection, the conv banks): bound by loads and MMAs.  Persistent CTAs, one per
//    SM, three 64 KB stages, two TMEM accumulators (the epilogue of tile i overlaps the main loop of tile i+1), 4 epilogue warps.
//  * short K with more than two tiles per SM (the 1025-wide linear output, the GRU input projections at full length): bound by the
//    epilogue.  Persistent as well, but with EIGHT epilogue warps and two stages.
//  * few tiles: one tile per CTA, eight epilogue warps, a shallow ring so that two CTAs share an SM.
// Reads only the shape, the flags and whether each pointer is null or 16-byte aligned: no device access.
taco_gemm_plan umma_plan(const ConvUmma& c, int sms) {
  taco_gemm_plan q;
  memset(&q, 0, sizeof(q));
  if (c.N <= 0 || c.T <= 0 || c.Cp <= 0 || c.Cp % BK || c.Kld % BK || c.taps <= 0 || c.Cout <= 0 || sms <= 0) return q;
  const int ny = (c.Cout + BN - 1) / BN;
  const long long ntiles = (long long)c.N * ((c.T + BM - 1) / BM) * ny * (c.bank > 1 ? c.bank : 1);
  if (ntiles > 0x7fffffffLL) return q;
  q.tiles = (int)ntiles;
  static const int force = env_int("TACO_UMMA_PERSISTENT", -1), ew_force = env_int("TACO_UMMA_EW", 0);
  static const int stage_cap = env_int("TACO_UMMA_STAGES_MAX", 0), cta_cap = env_int("TACO_UMMA_CTAS", 0);
  static const int stage_force = env_int("TACO_UMMA_STAGES", 0);
  const int nkb_max = c.taps * (c.Cp / BK);
  const bool long_k = nkb_max >= 24;
  const bool persistent = force >= 0 ? force != 0 : (long_k || q.tiles > 2 * sms);
  q.long_k = long_k; q.persistent = persistent;
  q.epi_warps = ew_force == 4 || ew_force == 8 ? ew_force : (long_k ? 4 : 8);
  if (persistent) q.stages = long_k ? MAX_STAGES : 2;
  else q.stages = nkb_max >= 3 ? 2 : 1;
  if (stage_force >= 1 && !long_k) q.stages = stage_force > MAX_STAGES ? MAX_STAGES : stage_force;
  if (stage_cap >= 1 && q.stages > stage_cap) q.stages = stage_cap;
  while (smem_bytes(q.stages, q.epi_warps) > 227u * 1024u && q.stages > 1) --q.stages;
  int nctas = persistent ? (cta_cap > 0 ? cta_cap : sms) : q.tiles;
  if (nctas > q.tiles) nctas = q.tiles;
  q.ctas = nctas;
  q.acc_cols = nctas < q.tiles ? 256 : 128;
  auto al4 = [](long long v) { return (v & 3) == 0; };
  q.vec_epi = (al4(c.ldo) && al4(c.col_off) && al4(c.out_bs) && al4(c.Cout) &&
               (c.out == nullptr || (reinterpret_cast<uintptr_t>(c.out) & 15) == 0) &&
               (c.res == nullptr || (al4(c.ldres) && al4(c.res_bs) && (reinterpret_cast<uintptr_t>(c.res) & 15) == 0)) &&
               (c.bias == nullptr || (reinterpret_cast<uintptr_t>(c.bias) & 15) == 0) &&
               (c.scale == nullptr || ((reinterpret_cast<uintptr_t>(c.scale) & 15) == 0 && (reinterpret_cast<uintptr_t>(c.shift) & 15) == 0)))
                  ? 1 : 0;
  q.smem_bytes = (int)smem_bytes(q.stages, q.epi_warps);
  // epilogue variant: the combinations the forward uses are compiled in, anything else takes the run-time variant 0
  if (c.act == 0 && !c.scale && !c.res) q.variant = 1;
  else if (c.act == 1 && !c.scale && !c.res) q.variant = 2;
  else if (c.act == 1 && c.scale && !c.res) q.variant = 3;
  else if (c.act == 0 && c.scale && c.res) q.variant = 4;
  // refusals
  if (c.out_hi != nullptr && (c.out_lo == nullptr || !q.vec_epi || c.bank > 1 || c.col_off != 0 || (c.out_cp & 63) ||
                              c.out_cp < c.Cout || c.out_cp > ny * BN))
    return q;
  if (c.out == nullptr && c.out_hi == nullptr) return q;
  if ((c.scale == nullptr) != (c.shift == nullptr)) return q;
  q.valid = 1;
  return q;
}

cudaError_t launch_conv_umma(const ConvUmma& c, cudaStream_t st, taco_gemm_plan* plan_out) {
  if (c.N <= 0 || c.T <= 0) return cudaSuccess;
  static int n_sm[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (n_sm[dev & 63] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    n_sm[dev & 63] = v;
  }
  const taco_gemm_plan q = umma_plan(c, n_sm[dev & 63]);
  if (plan_out) *plan_out = q;
  if (!q.valid) return cudaErrorInvalidValue;
  CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
  const bool split = c.nsplit > 1;
  if (!get_map_a(&ma_hi, c.a_hi, c.Cp, c.T, c.N) || !get_map_b(&mb_hi, c.b_hi, c.Kld, c.b_rows) ||
      !get_map_a(&ma_lo, split ? c.a_lo : c.a_hi, c.Cp, c.T, c.N) || !get_map_b(&mb_lo, split ? c.b_lo : c.b_hi, c.Kld, c.b_rows))
    return cudaErrorInvalidValue;
  UmmaArgs p;
  p.N = c.N; p.T = c.T; p.Cp = c.Cp; p.kvalid = c.Cin > 0 && c.Cin < c.Cp ? (c.Cin + 15) & ~15 : c.Cp; p.taps = c.taps; p.bank = c.bank; p.Cout = c.Cout;
  p.bias = c.bias; p.scale = c.scale; p.shift = c.shift; p.res = c.res; p.res_bs = c.res_bs; p.ldres = c.ldres;
  p.out = c.out; p.out_bs = c.out_bs; p.ldo = c.ldo; p.col_off = c.col_off; p.act = c.act;
  p.out_hi = c.out_hi; p.out_lo = c.out_lo; p.out_cp = c.out_cp;
  p.nx = c.N * ((c.T + BM - 1) / BM);
  p.ny = (c.Cout + BN - 1) / BN;
  p.ntiles = q.tiles;
  p.epi_warps = q.epi_warps; p.stages = q.stages; p.acc_cols = q.acc_cols; p.vec_epi = q.vec_epi;
  dim3 grid(q.ctas, 1, 1);
  using KernelFn = void (*)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const UmmaArgs);
  static const KernelFn kernels[2][5] = {
      {conv_umma_kernel<3, 0>, conv_umma_kernel<3, 1>, conv_umma_kernel<3, 2>, conv_umma_kernel<3, 3>, conv_umma_kernel<3, 4>},
      {conv_umma_kernel<1, 0>, conv_umma_kernel<1, 1>, conv_umma_kernel<1, 2>, conv_umma_kernel<1, 3>, conv_umma_kernel<1, 4>}};
  static bool attr_done[64] = {false};
  bool& attr_set = attr_done[dev & 63];
  if (!attr_set) {
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < 5; ++b) {
        cudaError_t e1 = cudaFuncSetAttribute(kernels[a][b], cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e1 != cudaSuccess) return e1;
      }
    attr_set = true;
  }
  const int nthreads = 64 + 32 * p.epi_warps;
  kernels[split ? 0 : 1][q.variant]<<<grid, nthreads, (uint32_t)q.smem_bytes, st>>>(ma_hi, ma_lo, mb_hi, mb_lo, p);
  return cudaGetLastError();
}

// Four (or fewer) highway layers in one launch.  w_hi: the layers' W^T hi / lo matrices, [layer][hi|lo][256][128] bf16, contiguous.
cudaError_t launch_highway4(const float* x, float* out, void* out_hi, void* out_lo, const void* w_hi, const float* const* bias,
                            int layers, long long rows, int nsplit, cudaStream_t st) {
  if (rows <= 0 || layers <= 0) return cudaSuccess;
  if (layers > 4 || rows > 0x7fffffffLL) return cudaErrorInvalidValue;
  CUtensorMap mb;
  {
    const MapKey k{w_hi, 128u, 256u, (uint64_t)(2 * layers), 33u};
    std::lock_guard<std::mutex> lk(g_map_mu);
    auto it = g_maps.find(k);
    if (it != g_maps.end()) mb = it->second;
    else {
      const cuuint64_t dims[3] = {128, 256, (cuuint64_t)(2 * layers)};
      const cuuint64_t str[2] = {128 * 2, 256 * 128 * 2};
      const cuuint32_t box[3] = {BK, 256, 1};
      if (!make_map(&mb, w_hi, 3, dims, str, box)) return cudaErrorInvalidValue;
      g_maps.emplace(k, mb);
    }
  }
  Hw4Args p;
  p.x = x; p.out = out; p.out_hi = out_hi; p.out_lo = out_lo;
  for (int i = 0; i < 4; ++i) p.bias[i] = bias[i < layers ? i : 0];
  p.rows = (int)rows; p.layers = layers; p.ntiles = (int)((rows + BM - 1) / BM);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
  static bool attr_done[64] = {false};
  if (!attr_done[dev & 63]) {
    cudaError_t e1 = cudaFuncSetAttribute(highway4_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)HW_SMEM);
    cudaError_t e2 = cudaFuncSetAttribute(highway4_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)HW_SMEM);
    if (e1 != cudaSuccess) return e1;
    if (e2 != cudaSuccess) return e2;
    attr_done[dev & 63] = true;
  }
  const int grid = p.ntiles < sms ? p.ntiles : sms;
  if (nsplit > 1) highway4_kernel<3><<<grid, HW_THREADS, HW_SMEM, st>>>(mb, p);
  else highway4_kernel<1><<<grid, HW_THREADS, HW_SMEM, st>>>(mb, p);
  return cudaGetLastError();
}

}  // namespace taco
