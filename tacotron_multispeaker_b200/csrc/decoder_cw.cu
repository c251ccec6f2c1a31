// K7 (v6): the attention decoder loop as one persistent cluster kernel with a CRITICAL warp group and BACKGROUND groups.
//
// Operator: tf.contrib.seq2seq.dynamic_decode(BasicDecoder(output_cell, helper, zero_state), maximum_iterations=max_iters) of
// reference models/tacotron.py:66-94 with DecoderPrenetWrapper / ConcatOutputAndAttentionWrapper (models/rnn_wrappers.py:22-24,
// 50-52), BahdanauAttention + AttentionWrapper (SURVEY Appendix B.2), two ResidualWrapper(GRUCell(256)), the 80*r output
// projection and TacoTestHelper / TacoTrainingHelper (models/helpers.py:26-38,68-77).
//
// Why this shape (measured on the v5 kernel, profiles/r2_decoder_*.md): a decoder step is a chain of dependent phases, each
// ending in an all-gather inside the cluster (~500-650 clk).  With all 16 warps of a CTA in lock step, every phase also paid
// late MMAs + a 512-thread barrier + a reduction + whatever "window work" the slowest warp carried (~700-1200 clk).  Here
//   * per phase only ONE 16-column tile is on the critical path (reset gates r, candidates, prenet, query); its late operand is
//     multiplied by the four critical warps (12-15, one per SM sub-partition, <= 4 chunk-tiles each, A fragments preloaded from
//     tensor memory), cross-reduced behind a 128-thread named barrier and pushed by the same warps;
//   * everything else -- products with operands that are complete earlier (recurrent states, previous context), the update
//     gates / candidate x-parts (needed one phase later), the 512->256 projection y0 and the 80r output projection -- runs in
//     the background groups A/B/C from a host-written item list and meets the critical group in partial-tile slots behind
//     bar.arrive / bar.sync pairs;
//   * two linear folds remove exchanges: the fed-back frame is never formed (W_o[:, -80:] W_1[:80] multiplies y2 = y0+h1'+h2'
//     directly; teacher forcing reads the target frame instead), and the 512->256 projection is folded into GRU-1's x-parts
//     (W_p W_g1x, W_p W_c1x), so a free-running step has 11 exchanges instead of 13;
//   * mat-vecs: mma.sync m16n8k16, bf16 hi/lo split operands, hi*hi + lo*hi + hi*lo in fp32 (fp32-class accuracy).
#include <cuda_bf16.h>
#include <stdlib.h>

#include "common.cuh"
#include "decoder_cw.h"
#include "kernels.cuh"

namespace taco {

namespace {
using namespace cw;

// ---- shared memory: fixed part, then the S-dependent buffers ---------------------------------------------------------
constexpr uint32_t OFF_MBAR = 0;                                   // N_MBAR x 8
constexpr uint32_t OFF_TMEM = OFF_MBAR + N_MBAR * 8;               // TMEM base address
constexpr uint32_t OFF_VB = OFF_TMEM + 4;                          // sum_k v_k - min(||v||_1, 40)
constexpr uint32_t OFF_INV = OFF_TMEM + 16;                        // 1 / softmax normaliser per sample [8]
constexpr uint32_t OFF_MX = OFF_INV + 32;                          // exact-softmax mode: row maximum per sample [8]
constexpr uint32_t OFF_BIAS = 256;
constexpr uint32_t OFF_VATT = OFF_BIAS + N_BIAS * 4;               // 1216
constexpr uint32_t OFF_STG = OFF_VATT + DHID * 4;                  // staged rows: warps 8..15, 2 samples x 64 B each
constexpr uint32_t OFF_Y0S = OFF_STG + 8 * 128;                    // this CTA's y0 tile, fp32 [8 samples][16 columns]
constexpr uint32_t OFF_REDS = OFF_Y0S + 8 * 16 * 4;                // partial softmax normalisers [16 warps][8]
constexpr uint32_t OFF_SLOTS = (OFF_REDS + NW * 8 * 4 + 127u) & ~127u;
constexpr uint32_t OFF_X = (OFF_SLOTS + N_SLOTS * SLOT_F * 4 + 127u) & ~127u;
static_assert(OFF_BIAS % 16 == 0 && OFF_VATT % 16 == 0 && OFF_STG % 16 == 0 && OFF_SLOTS % 16 == 0, "alignment");

struct Dyn { uint32_t pq, sc, stage, pn, ksl, msl, ring, total; };
__host__ __device__ inline Dyn make_dyn(int S, int T_in, int att_res, int ring_kb) {
  Dyn d;
  const uint32_t csb = (uint32_t)S * 64u;
  const uint32_t npq = (uint32_t)(T_in * S) / CS + 4;
  auto up = [](uint32_t v) { return (v + 127u) & ~127u; };
  d.pq = up(OFF_X + (uint32_t)X_CHUNKS * csb);                       // exp(2 * processed query) fp32 [chunk][n][16]
  d.sc = up(d.pq + 16 * csb);                                      // exp(score - B) (or the raw score)  [j][n]
  d.stage = up(d.sc + (uint32_t)T_in * S * 4 + 16u);               // this CTA's pairs
  d.pn = d.stage + ((npq * 4 + 15u) & ~15u);                       // sample index of this CTA's pairs (bytes)
  d.ksl = up(d.pn + npq);                                          // exp(2 * keys) rows of this CTA's pairs
  d.msl = up(d.ksl + ((att_res & 1) ? npq * DHID * 4 : 0u));       // memory columns of this CTA
  d.ring = up(d.msl + ((att_res & 2) ? (uint32_t)S * T_in * 64u : 0u));
  d.total = d.ring + 12u * (uint32_t)ring_kb * 1024u;
  return d;
}

// ---- PTX helpers -------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t mb, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mb), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t mb, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mb, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(mb), "r"(parity), "r"(0x989680u)
      : "memory");
}
__device__ __forceinline__ void st_async_v4(uint32_t raddr, uint4 v, uint32_t rmbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1,%2,%3,%4}, [%5];"
               ::"r"(raddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "r"(rmbar) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint32_t lds32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ float lds_f(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts_f(uint32_t addr, float v) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts_f4(uint32_t addr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ uint4 ldg_stream(const uint4* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.b32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ void cp_async16(uint32_t saddr, const void* g) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_pending(int pend) {   // warp-uniform, 0..7
  switch (pend) {
    case 0: asm volatile("cp.async.wait_group 0;" ::: "memory"); break;
    case 1: asm volatile("cp.async.wait_group 1;" ::: "memory"); break;
    case 2: asm volatile("cp.async.wait_group 2;" ::: "memory"); break;
    case 3: asm volatile("cp.async.wait_group 3;" ::: "memory"); break;
    case 4: asm volatile("cp.async.wait_group 4;" ::: "memory"); break;
    case 5: asm volatile("cp.async.wait_group 5;" ::: "memory"); break;
    case 6: asm volatile("cp.async.wait_group 6;" ::: "memory"); break;
    default: asm volatile("cp.async.wait_group 7;" ::: "memory"); break;
  }
}
// named barriers: the background groups arrive, the critical group (or a group among itself) syncs
__device__ __forceinline__ void nb_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void nb_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }

// tensor memory as a weight store: 32x32b.x8 = the eight 32-bit words (hi uint4, lo uint4) of one chunk-tile per lane
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint4& hi, uint4& lo) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(hi.x), "=r"(hi.y), "=r"(hi.z), "=r"(hi.w), "=r"(lo.x), "=r"(lo.y), "=r"(lo.z), "=r"(lo.w)
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint4& hi, const uint4& lo) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               :: "r"(taddr), "r"(hi.x), "r"(hi.y), "r"(hi.z), "r"(hi.w), "r"(lo.x), "r"(lo.y), "r"(lo.z), "r"(lo.w) : "memory");
}
// attention operands in tensor memory (layout TL_ATT): four 32-bit words per lane
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint4& v) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(taddr));
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint4& v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" :: "r"(taddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ float4 u2f(const uint4& v) {
  return make_float4(__uint_as_float(v.x), __uint_as_float(v.y), __uint_as_float(v.z), __uint_as_float(v.w));
}
__device__ __forceinline__ uint4 f2u(const float4& v) {
  return make_uint4(__float_as_uint(v.x), __float_as_uint(v.y), __float_as_uint(v.z), __float_as_uint(v.w));
}
__device__ __forceinline__ void reg_fence1(uint4& a) { asm volatile("" : "+r"(a.x), "+r"(a.y), "+r"(a.z), "+r"(a.w)); }
__device__ __forceinline__ void reg_fence(uint4& a, uint4& b) {
  asm volatile("" : "+r"(a.x), "+r"(a.y), "+r"(a.z), "+r"(a.w), "+r"(b.x), "+r"(b.y), "+r"(b.z), "+r"(b.w));
}

// D += A(16x16, row) * B(16x8, col), bf16 inputs, fp32 accumulate
__device__ __forceinline__ void mma16816(float (&d)[4], const uint4& a, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b0), "r"(b1));
}
// fp32 -> bf16 hi (round to nearest) + bf16 lo (remainder); packs two values per 32-bit word
__device__ __forceinline__ void split2(float v0, float v1, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat16 h0 = __float2bfloat16_rn(v0), h1 = __float2bfloat16_rn(v1);
  const __nv_bfloat16 l0 = __float2bfloat16_rn(v0 - __bfloat162float(h0));
  const __nv_bfloat16 l1 = __float2bfloat16_rn(v1 - __bfloat162float(h1));
  hi = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
  lo = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
}
// reducer thread (n, c) holds v = activation [n][16q + c]: split into bf16 hi/lo, pair with the neighbouring column (lane ^ 1)
// and write the two words of the pair into the staged row `stg_n` (MMA B-fragment order).  Executed by whole warps.
__device__ __forceinline__ void stage_x(uint32_t stg_n, int c, float v) {
  // packed conversions (F2FP on the FMA pipe) instead of two scalar F2F on the XU pipe: same round-to-nearest results
  uint32_t hp, lp;
  asm("cvt.rn.bf16x2.f32 %0, %1, %1;" : "=r"(hp) : "f"(v));
  const uint32_t hv = hp & 0xffffu;
  asm("cvt.rn.bf16x2.f32 %0, %1, %1;" : "=r"(lp) : "f"(v - __uint_as_float(hv << 16)));
  const uint32_t lv = lp & 0xffffu;
  const uint32_t hn = __shfl_xor_sync(0xffffffffu, hv, 1), ln = __shfl_xor_sync(0xffffffffu, lv, 1);
  if ((c & 1) == 0) {
    const uint32_t wa = stg_n + (uint32_t)((((c & 7) >> 1) * 4 + (c >> 3)) * 4);
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(wa), "r"(hv | (hn << 16)) : "memory");
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(wa + 8), "r"(lv | (ln << 16)) : "memory");
  }
}
// D fragment (row g / g+8 = tile column, col 2t / 2t+1 = sample) -> slot[sample][column]
__device__ __forceinline__ void store_tile(uint32_t slot, int g, int t, const float (&hh)[4], const float (&hl)[4], const float (&lh)[4]) {
  const uint32_t p = slot + (uint32_t)(((2 * t) * RS + g) * 4);
  sts_f(p, hh[0] + (hl[0] + lh[0]));
  sts_f(p + RS * 4, hh[1] + (hl[1] + lh[1]));
  sts_f(p + 32, hh[2] + (hl[2] + lh[2]));
  sts_f(p + RS * 4 + 32, hh[3] + (hl[3] + lh[3]));
}
__device__ __forceinline__ float sum4(uint32_t red_nc, int slot0) {   // element (n, c) summed over four consecutive slots
  const float a = lds_f(red_nc + (slot0 + 0) * SLOT_F * 4), b = lds_f(red_nc + (slot0 + 1) * SLOT_F * 4);
  const float c = lds_f(red_nc + (slot0 + 2) * SLOT_F * 4), d = lds_f(red_nc + (slot0 + 3) * SLOT_F * 4);
  return (a + b) + (c + d);
}

struct Args {
  const void* tmem_img;
  const void* ring;          // this mode's ring: [16 CTAs][12 warps][ring_stride] KB
  int ring_len[12];
  int ring_stride;
  const float* bias;         // [16 CTAs][N_BIAS]
  const float* att_v;
  int M, Dout;
  int exact_softmax;         // ||v||_1 > 40: exchange raw scores and subtract the row maximum (one more pass in the context phase)
  int ring_kb;               // ring depth per background warp
};

#define TRM(i) do { if (TRACE && a.trace != nullptr && step == 8 && blockIdx.x == a.trace_cta && tid == 12 * 32) a.trace[i] = clock64(); } while (0)
#define TRW(base) do { if (TRACE && a.trace != nullptr && step == 8 && blockIdx.x == a.trace_cta && lane == 0) a.trace[(base) + warp] = clock64(); } while (0)

// BF16: plain bf16 mode (taco_set_gemm_mode(2)): only W_hi * x_hi is multiplied (one MMA per chunk-tile instead of three);
// the lo halves of the packed weights and of the staged activations are carried but not used.  Stated tolerance: 5e-2.
// SMALL: launches whose clusters all hold <= 2 utterances run the attention phases on the critical group alone (compiled out otherwise)
template <bool TRACE, bool BF16, bool SMALL>
__global__ void __launch_bounds__(NT, 1)
decoder_cw_kernel(const __grid_constant__ Args w, const __grid_constant__ Program prog, const DecoderArgs a, const int nclusters) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int g = lane >> 2, t = lane & 3;
  const int q = (int)cluster_ctarank();
  const int cid = (int)cluster_id_x();
  const int base = a.N / nclusters, rem = a.N % nclusters;
  const int S = base + (cid < rem ? 1 : 0);
  const int n0 = cid * base + min(cid, rem);
  const int M = w.M, Dout = w.Dout, T_in = a.T_in;
  const bool res_k = (a.att_res & 1) != 0, res_m = (a.att_res & 2) != 0, att_tm = (a.att_res & ATT_TMEM) != 0;
  const bool exact = w.exact_softmax != 0;
  const Dyn L = make_dyn(S, T_in, a.att_res, w.ring_kb);
  const uint32_t sbase = smem_u32(smem_raw);
  const uint32_t csb = (uint32_t)S * 64u;
  const uint32_t mb0 = sbase + OFF_MBAR;
  const int NP = T_in * S, NQ = (NP + 3) >> 2;
  const int p0 = 4 * ((q * NQ) / CS), npq = min(NP, 4 * (((q + 1) * NQ) / CS)) - p0;
  const bool free_run = a.targets == nullptr;
  if (S == 0) { cluster_sync_all(); cluster_sync_all(); return; }
#define TRX(i) do { if (TRACE && a.trace != nullptr && blockIdx.x == a.trace_cta && tid == 12 * 32) a.trace[i] = clock64(); } while (0)
  TRX(24);

  // ---- prologue ------------------------------------------------------------------------------------------------------
  for (uint32_t i = OFF_TMEM + tid * 4; i < L.ring; i += NT * 4) *reinterpret_cast<uint32_t*>(smem_raw + i) = 0u;
  if (tid < N_MBAR) mbar_init(mb0 + tid * 8, 1);
  __syncthreads();
  if (tid < N_BIAS) reinterpret_cast<float*>(smem_raw + OFF_BIAS)[tid] = __ldg(w.bias + q * N_BIAS + tid);
  if (tid < DHID) reinterpret_cast<float*>(smem_raw + OFF_VATT)[tid] = __ldg(w.att_v + tid);
  if (res_k) {
    float* ksl = reinterpret_cast<float*>(smem_raw + L.ksl);
    for (int i = tid; i < npq * (DHID / 4); i += NT) {   // exp(2 key): tanh(k + p) = 1 - 2 / (1 + e^{2k} e^{2p})
      const int c4 = i % (DHID / 4), pp = i / (DHID / 4), p = p0 + pp, j = p / S, n = p - j * S;
      float4 k4 = ldg_f4(a.keys + ((size_t)(n0 + n) * T_in + j) * DHID + c4 * 4);
      k4.x = __expf(2.0f * fminf(fmaxf(k4.x, -30.f), 30.f)); k4.y = __expf(2.0f * fminf(fmaxf(k4.y, -30.f), 30.f));
      k4.z = __expf(2.0f * fminf(fmaxf(k4.z, -30.f), 30.f)); k4.w = __expf(2.0f * fminf(fmaxf(k4.w, -30.f), 30.f));
      *reinterpret_cast<float4*>(ksl + (size_t)pp * DHID + c4 * 4) = k4;
    }
  }
  if (res_m) {
    float* msl = reinterpret_cast<float*>(smem_raw + L.msl);
    for (int i = tid; i < S * T_in * 4; i += NT) {
      const int c4 = i & 3, r = i >> 2, s = r / T_in, j = r - s * T_in;
      *reinterpret_cast<float4*>(msl + ((size_t)j * S + s) * 16 + c4 * 4) =
          ldg_f4(a.memory + ((size_t)(n0 + s) * T_in + j) * DHID + q * 16 + c4 * 4);   // [j][n][16]
    }
  }
  {
    float vbound = 0.f, vsum = 0.f;   // B = min(||v||_1, 40) >= any score (|tanh| <= 1); sum_k v_k
#pragma unroll
    for (int i = 0; i < 8; ++i) { const float vv = __ldg(w.att_v + lane + 32 * i); vbound += fabsf(vv); vsum += vv; }
    vbound = fminf(warp_sum(vbound), 40.0f);
    vsum = warp_sum(vsum);
    if (tid == 0) sts_f(sbase + OFF_VB, exact ? vsum : vsum - vbound);
  }
  for (int pp = tid; pp < npq; pp += NT) smem_raw[L.pn + pp] = (unsigned char)((p0 + pp) % S);
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(sbase + OFF_TMEM) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = lds32(sbase + OFF_TMEM);
  const int gw = warp & 3;                                                    // index inside the group = SM sub-partition = TMEM lane quarter
  const uint32_t tq = tmem_base + ((uint32_t)(gw * 32) << 16);                 // this warp's lane quarter, column 0
  {   // fill the quarter: the four warps of a quarter take every fourth chunk-tile
    const uint4* img = reinterpret_cast<const uint4*>(w.tmem_img) + ((size_t)(q * 4 + gw) * TMEM_TILES) * 64 + lane;
    const int tiles = att_tm ? TMEM_ATT_TILES : TMEM_TILES;
    for (int i0 = (warp >> 2); i0 < tiles; i0 += 16) {
      uint4 hi[4], lo[4];
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (i0 + 4 * k < tiles) { hi[k] = ldg_stream(img + (size_t)(i0 + 4 * k) * 64); lo[k] = ldg_stream(img + (size_t)(i0 + 4 * k) * 64 + 32); }
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (i0 + 4 * k < tiles) tmem_st8(tq + (uint32_t)(i0 + 4 * k) * 8u, hi[k], lo[k]);
    }
    if (att_tm) {   // attention operands of this quarter (decoder_cw.h, TL_ATT), split over its four warps
      const uint32_t tk = tq + (uint32_t)TMEM_ATT_COL0, tm = tk + (uint32_t)att_key_cols(S, T_in);
      for (int m = warp >> 2; 8 * m + 2 * gw < npq; m += 4)   // pairs 8 m + 2 gw + e
        for (int e = 0; e < 2; ++e) {
          const int pp = 8 * m + 2 * gw + e;
          if (pp >= npq) break;
          const int p = p0 + pp, j = p / S, n = p - j * S;
          const float* krow = a.keys + ((size_t)(n0 + n) * T_in + j) * DHID + 4 * lane;
          float4 k0 = ldg_f4(krow), k1 = ldg_f4(krow + 128);
          k0.x = __expf(2.0f * fminf(fmaxf(k0.x, -30.f), 30.f)); k0.y = __expf(2.0f * fminf(fmaxf(k0.y, -30.f), 30.f));
          k0.z = __expf(2.0f * fminf(fmaxf(k0.z, -30.f), 30.f)); k0.w = __expf(2.0f * fminf(fmaxf(k0.w, -30.f), 30.f));
          k1.x = __expf(2.0f * fminf(fmaxf(k1.x, -30.f), 30.f)); k1.y = __expf(2.0f * fminf(fmaxf(k1.y, -30.f), 30.f));
          k1.z = __expf(2.0f * fminf(fmaxf(k1.z, -30.f), 30.f)); k1.w = __expf(2.0f * fminf(fmaxf(k1.w, -30.f), 30.f));
          tmem_st8(tk + (uint32_t)(2 * m + e) * 8u, f2u(k0), f2u(k1));
        }
      for (int jq = warp >> 2; 4 * jq + gw < T_in; jq += 4) {   // positions j = 4 jq + gw
        const int j = 4 * jq + gw;
        float4 m4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (g < S) m4 = ldg_f4(a.memory + ((size_t)(n0 + g) * T_in + j) * DHID + q * 16 + 4 * t);
        tmem_st4(tm + (uint32_t)jq * 4u, f2u(m4));
      }
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  if (tid == 12 * 32) {   // expected byte counts of step 0 (later steps: re-armed after each wait)
    const uint32_t blk = CS * (uint32_t)S * 64u;
    mbar_expect_tx(mb0 + MB_P1 * 8, blk);  mbar_expect_tx(mb0 + MB_P2 * 8, blk / 2); mbar_expect_tx(mb0 + MB_P3 * 8, blk);
    mbar_expect_tx(mb0 + MB_P4 * 8, blk);  mbar_expect_tx(mb0 + MB_P5 * 8, blk);     mbar_expect_tx(mb0 + MB_P6 * 8, (uint32_t)NQ * 16u);
    mbar_expect_tx(mb0 + MB_P7 * 8, blk);  mbar_expect_tx(mb0 + MB_P9 * 8, blk);     mbar_expect_tx(mb0 + MB_H1 * 8, blk);
    mbar_expect_tx(mb0 + MB_P10 * 8, blk); mbar_expect_tx(mb0 + MB_P11 * 8, blk);    mbar_expect_tx(mb0 + MB_P12 * 8, blk);
    mbar_expect_tx(mb0 + MB_H2 * 8, blk);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  cluster_sync_all();   // buffers zeroed, mbarriers initialised, tensor memory filled everywhere before anyone pushes
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  TRX(25);

  const uint32_t BLK = CS * csb;
  const uint32_t xl = sbase + OFF_X + (uint32_t)min(g, S - 1) * 64u + (uint32_t)t * 16u;   // lane part of a B-fragment address
  // reducer thread of warps 8..15: sample rn, column rc of this CTA's tile
  const int rn = 2 * gw + (lane >> 4), rc = lane & 15;
  const uint32_t red_nc = sbase + OFF_SLOTS + (uint32_t)(rn * RS + rc) * 4u;   // + slot * SLOT_F * 4
  const uint32_t bias_c = sbase + OFF_BIAS + rc * 4;
  const uint32_t stg_w = sbase + OFF_STG + (uint32_t)((warp & 7) * 128);
  const uint32_t stg_n = stg_w + (uint32_t)(lane >> 4) * 64u;
#define BIAS(tab) lds_f(bias_c + (tab) * 4)
#define XADDR(chunk) (xl + (uint32_t)(chunk) * csb)
  // push the two staged rows of this warp (samples 2gw, 2gw+1) to all 16 peers (or, `pair`, to the 8 peers of this CTA's parity)
  auto send_rows = [&](uint32_t dst, int bar, bool pair) {
    __syncwarp();
    const int wg = lane & 7, sn = 2 * gw + (wg >> 2);
    if (sn < S) {
      const uint32_t off = (uint32_t)sn * 64u + (uint32_t)(wg & 3) * 16u;
      const uint4 v = lds128(stg_w + (uint32_t)(wg >> 2) * 64u + (uint32_t)(wg & 3) * 16u);
#pragma unroll
      for (int it = 0; it < 4; ++it) {
        if (pair && it >= 2) break;
        const uint32_t k = (uint32_t)(it * 4 + (lane >> 3));
        const uint32_t peer = pair ? 2u * k + (uint32_t)(q & 1) : k;
        st_async_v4(mapa_u32(sbase + dst + off, peer), v, mapa_u32(mb0 + (uint32_t)bar * 8u, peer));
      }
    }
  };

  // ---- attention phases (all 16 warps) --------------------------------------------------------------------------------
  // P6: Bahdanau scores of this CTA's (position, sample) pairs: exp(v . tanh(keys + pq) - B)
  // v.tanh(k + p) = sum v - 2 sum_k v_k / (1 + e^{2k} e^{2p}); four elements share one MUFU.RCP (denominators clamped to 2^30).
  const int p6_wr = (warp + 4) & 15;                                         // pair slot of this warp: 12, 13, 14, 15, 0, 1, ...
  const int p6_na = (p0 + min(2 * p6_wr, max(npq - 1, 0))) % S, p6_nb = (p0 + min(2 * p6_wr + 1, max(npq - 1, 0))) % S;
  auto p6_compute = [&](int pair_stride) {
    const uint32_t pq_l = sbase + L.pq + (uint32_t)(lane >> 2) * csb + (uint32_t)(lane & 3) * 16u;
    const float4 v0 = lds_f4(sbase + OFF_VATT + lane * 16), v1 = lds_f4(sbase + OFF_VATT + 512 + lane * 16);
    constexpr float BIG = 1073741824.0f;   // 2^30
    auto quad = [&](const float4& k, const float4& e, const float4& v) -> float {
      const float da = fminf(fmaf(k.x, e.x, 1.0f), BIG), db = fminf(fmaf(k.y, e.y, 1.0f), BIG);
      const float dc = fminf(fmaf(k.z, e.z, 1.0f), BIG), dd = fminf(fmaf(k.w, e.w, 1.0f), BIG);
      const float ab = da * db, cd = dc * dd;
      const float nab = fmaf(v.x, db, v.y * da), ncd = fmaf(v.z, dd, v.w * dc);
      return fmaf(nab, cd, ncd * ab) * rcp_approx(ab * cd);
    };
    auto pair_q = [&](const float4& k0, const float4& k1, int n) -> float {
      const float4 e0 = lds_f4(pq_l + (uint32_t)n * 64u), e1 = lds_f4(pq_l + (uint32_t)n * 64u + 8 * csb);
      return quad(k0, e0, v0) + quad(k1, e1, v1);
    };
    // keys first (their address does not depend on the sample index), then the query of the pair's sample
    auto pair_sum = [&](int pl, int n) -> float {
      float4 k0, k1;
      if (res_k) {
        k0 = lds_f4(sbase + L.ksl + (uint32_t)pl * (DHID * 4) + lane * 16);
        k1 = lds_f4(sbase + L.ksl + (uint32_t)pl * (DHID * 4) + 512 + lane * 16);
      } else {
        const int j = (p0 + pl) / S;
        const float* krow = a.keys + ((size_t)(n0 + n) * T_in + j) * DHID + 4 * lane;
        k0 = ldg_f4(krow); k1 = ldg_f4(krow + 128);
        k0.x = __expf(2.0f * fminf(fmaxf(k0.x, -30.f), 30.f)); k0.y = __expf(2.0f * fminf(fmaxf(k0.y, -30.f), 30.f));
        k0.z = __expf(2.0f * fminf(fmaxf(k0.z, -30.f), 30.f)); k0.w = __expf(2.0f * fminf(fmaxf(k0.w, -30.f), 30.f));
        k1.x = __expf(2.0f * fminf(fmaxf(k1.x, -30.f), 30.f)); k1.y = __expf(2.0f * fminf(fmaxf(k1.y, -30.f), 30.f));
        k1.z = __expf(2.0f * fminf(fmaxf(k1.z, -30.f), 30.f)); k1.w = __expf(2.0f * fminf(fmaxf(k1.w, -30.f), 30.f));
      }
      return pair_q(k0, k1, n);
    };
    const float vb = lds_f(sbase + OFF_VB);
    // the critical warps (12..15) own the first pairs: with few utterances per cluster nobody waits for a background warp here
    for (int pp = 2 * p6_wr; pp < npq; pp += pair_stride) {
      const bool two = pp + 1 < npq, first = pp == 2 * p6_wr;
      const int na = first ? p6_na : (int)smem_raw[L.pn + pp], nb = first ? p6_nb : (int)smem_raw[L.pn + (two ? pp + 1 : pp)];
      float sa, sb;
      if (att_tm) {   // pp is even and (pp >> 1) & 3 == gw: both rows sit in this warp's lane quarter, side by side
        uint4 ka0, ka1, kb0, kb1;
        const uint32_t kc = tq + (uint32_t)TMEM_ATT_COL0 + (uint32_t)(pp >> 3) * 16u;
        tmem_ld8(kc, ka0, ka1);
        tmem_ld8(kc + (two ? 8u : 0u), kb0, kb1);
        tmem_wait_ld();
        reg_fence(ka0, ka1); reg_fence(kb0, kb1);
        sa = pair_q(u2f(ka0), u2f(ka1), na);
        sb = pair_q(u2f(kb0), u2f(kb1), nb);
      } else {
        sa = pair_sum(pp, na); sb = pair_sum(two ? pp + 1 : pp, nb);
      }
      const bool up = lane >= 16;
      float sv = (up ? sb : sa) + __shfl_xor_sync(0xffffffffu, up ? sa : sb, 16);
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) sv += __shfl_xor_sync(0xffffffffu, sv, o);
      const float sc = fmaf(-2.0f, sv, vb);                                  // score - B   (exact mode: the raw score)
      const float ex = exact ? sc : __expf(fmaxf(sc, -80.0f));
      if (lane == 0 || (lane == 16 && two)) sts_f(sbase + L.stage + (uint32_t)(up ? pp + 1 : pp) * 4u, ex);
    }
  };
  const uint32_t rmb0 = mapa_u32(mb0, (uint32_t)warp);                      // peer `warp`: its mbarriers ...
  const uint32_t rx = mapa_u32(sbase + lane * 16, (uint32_t)warp);          // ... and this lane's 16 bytes at offset 0
  auto p6_send = [&]() {   // warp p -> peer p: this CTA's pairs into sc[p0 ..], four per DSMEM transaction
    if (lane < ((npq + 3) >> 2)) st_async_v4(rx + L.sc + (uint32_t)p0 * 4u, lds128(sbase + L.stage + lane * 16), rmb0 + MB_P6 * 8);
  };
  // P7: partial context slice sum_j p_j memory[j][16q..16q+15] and partial normaliser; warp w takes positions j = w (mod 16),
  // lane (g, t): sample g, columns 4t..4t+3
  auto p7_compute = [&]() {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f), acc2 = make_float4(0.f, 0.f, 0.f, 0.f);
    float ssum = 0.f, ssum2 = 0.f, mx = 0.f;
    if (exact) {   // row maximum over all T_in positions of sample g (four lanes share a sample; idle lanes redo the last sample)
      const int gs = min(g, S - 1);
      mx = -3.0e38f;
      for (int j = t; j < T_in; j += 4) mx = fmaxf(mx, lds_f(sbase + L.sc + (uint32_t)(j * S + gs) * 4u));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
      if (warp == 12 && t == 0 && g < S) sts_f(sbase + OFF_MX + g * 4, mx);
    }
    if (att_tm) {
      // the resident loop below with the memory columns read from this warp's lane quarter: position j sits in quarter j & 3 =
      // warp & 3.  tcgen05.ld takes the whole warp, so lanes of absent samples (g >= S) run along with zero weights.
      const bool live = g < S;
      uint32_t pa = sbase + L.sc + (uint32_t)(warp * S + min(g, S - 1)) * 4u;
      const uint32_t dp = (uint32_t)NW * S * 4u;
      const uint32_t tm = tq + (uint32_t)(TMEM_ATT_COL0 + att_key_cols(S, T_in)) + (uint32_t)(warp >> 2) * 4u;
      for (int j = warp; j < T_in; j += 4 * NW) {
        float pv[4];
        uint4 mr[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint32_t o = j + i * NW < T_in ? (uint32_t)i : 0u;
          pv[i] = lds_f(pa + o * dp);
          tmem_ld4(tm + (uint32_t)(j >> 4) * 16u + o * 16u, mr[i]);
        }
        tmem_wait_ld();
        float4 mv[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          reg_fence1(mr[i]);
          mv[i] = u2f(mr[i]);
          if (exact) pv[i] = __expf(pv[i] - mx);
          if (j + i * NW >= T_in || !live) pv[i] = 0.f;
        }
        acc.x = fmaf(pv[0], mv[0].x, acc.x); acc.y = fmaf(pv[0], mv[0].y, acc.y); acc.z = fmaf(pv[0], mv[0].z, acc.z); acc.w = fmaf(pv[0], mv[0].w, acc.w);
        acc2.x = fmaf(pv[1], mv[1].x, acc2.x); acc2.y = fmaf(pv[1], mv[1].y, acc2.y); acc2.z = fmaf(pv[1], mv[1].z, acc2.z); acc2.w = fmaf(pv[1], mv[1].w, acc2.w);
        acc.x = fmaf(pv[2], mv[2].x, acc.x); acc.y = fmaf(pv[2], mv[2].y, acc.y); acc.z = fmaf(pv[2], mv[2].z, acc.z); acc.w = fmaf(pv[2], mv[2].w, acc.w);
        acc2.x = fmaf(pv[3], mv[3].x, acc2.x); acc2.y = fmaf(pv[3], mv[3].y, acc2.y); acc2.z = fmaf(pv[3], mv[3].z, acc2.z); acc2.w = fmaf(pv[3], mv[3].w, acc2.w);
        ssum += pv[0] + pv[2]; ssum2 += pv[1] + pv[3];
        pa += 4 * dp;
      }
      acc.x += acc2.x; acc.y += acc2.y; acc.z += acc2.z; acc.w += acc2.w;
      ssum += ssum2;
    } else if (g < S) {
      uint32_t pa = sbase + L.sc + (uint32_t)(warp * S + g) * 4u;
      const uint32_t dp = (uint32_t)NW * S * 4u;
      if (res_m) {
        uint32_t ma = sbase + L.msl + (uint32_t)((warp * S + g) * 16 + t * 4) * 4u;
        const uint32_t dm = (uint32_t)NW * S * 64u;
        // four positions per trip, all eight loads issued before the first FMA; positions past T_in re-read the trip's first
        // (valid) address and count as zero: no branches inside the loop
        for (int j = warp; j < T_in; j += 4 * NW) {
          float pv[4];
          float4 mv[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint32_t o = j + i * NW < T_in ? (uint32_t)i : 0u;
            pv[i] = lds_f(pa + o * dp);
            mv[i] = lds_f4(ma + o * dm);
          }
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            if (exact) pv[i] = __expf(pv[i] - mx);
            if (j + i * NW >= T_in) pv[i] = 0.f;
          }
          acc.x = fmaf(pv[0], mv[0].x, acc.x); acc.y = fmaf(pv[0], mv[0].y, acc.y); acc.z = fmaf(pv[0], mv[0].z, acc.z); acc.w = fmaf(pv[0], mv[0].w, acc.w);
          acc2.x = fmaf(pv[1], mv[1].x, acc2.x); acc2.y = fmaf(pv[1], mv[1].y, acc2.y); acc2.z = fmaf(pv[1], mv[1].z, acc2.z); acc2.w = fmaf(pv[1], mv[1].w, acc2.w);
          acc.x = fmaf(pv[2], mv[2].x, acc.x); acc.y = fmaf(pv[2], mv[2].y, acc.y); acc.z = fmaf(pv[2], mv[2].z, acc.z); acc.w = fmaf(pv[2], mv[2].w, acc.w);
          acc2.x = fmaf(pv[3], mv[3].x, acc2.x); acc2.y = fmaf(pv[3], mv[3].y, acc2.y); acc2.z = fmaf(pv[3], mv[3].z, acc2.z); acc2.w = fmaf(pv[3], mv[3].w, acc2.w);
          ssum += pv[0] + pv[2]; ssum2 += pv[1] + pv[3];
          pa += 4 * dp; ma += 4 * dm;
        }
      } else {
        for (int j = warp; j < T_in; j += NW) {
          float pv = lds_f(pa);
          if (exact) pv = __expf(pv - mx);
          const float4 m0 = ldg_f4(a.memory + ((size_t)(n0 + g) * T_in + j) * DHID + q * 16 + 4 * t);
          acc.x = fmaf(pv, m0.x, acc.x); acc.y = fmaf(pv, m0.y, acc.y); acc.z = fmaf(pv, m0.z, acc.z); acc.w = fmaf(pv, m0.w, acc.w);
          ssum += pv;
          pa += dp;
        }
      }
      acc.x += acc2.x; acc.y += acc2.y; acc.z += acc2.z; acc.w += acc2.w;
      ssum += ssum2;
    }
    sts_f4(sbase + OFF_SLOTS + (uint32_t)(SL_CTX + warp) * (SLOT_F * 4) + (uint32_t)(g * RS + t * 4) * 4u, acc);
    if (t == 0) sts_f(sbase + OFF_REDS + (uint32_t)(warp * 8 + g) * 4u, ssum);
  };

  // ---- attention on the critical group alone (S <= 2, operands resident, bounded-score softmax): batch-1 latency -----------
  // With one or two utterances per cluster the pairs of a CTA fit the four critical warps, and a 512-thread phase costs more in
  // barriers and late background warps than it saves: the background groups skip the attention phases altogether.
  const bool small_att = SMALL && S <= 2 && res_k && res_m && !exact;
  auto p6_send_crit = [&]() {   // critical warp gw -> peers 4 gw .. 4 gw + 3, eight 16-byte words per peer and trip
    const uint32_t peer = (uint32_t)(4 * gw + (lane >> 3));
    const uint32_t rsc = mapa_u32(sbase + L.sc + (uint32_t)p0 * 4u, peer), rmb = mapa_u32(mb0 + MB_P6 * 8, peer);
    for (int word = lane & 7; word < ((npq + 3) >> 2); word += 8)
      st_async_v4(rsc + (uint32_t)word * 16u, lds128(sbase + L.stage + (uint32_t)word * 16u), rmb);
  };
  // partial context of critical warp gw: positions j = gw + 4 (sub + nsub i); lane = (sub, sample, column quad t)
  auto p7_compute_crit = [&](uint32_t slot) {
    const int smp = S == 2 ? (g & 1) : 0, sub = S == 2 ? (g >> 1) : g, nsub = S == 2 ? 4 : 8;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f), acc2 = make_float4(0.f, 0.f, 0.f, 0.f);
    float ssum = 0.f, ssum2 = 0.f;
    const int j0 = gw + 4 * sub, dj = 4 * nsub;
    uint32_t pa = sbase + L.sc + (uint32_t)(j0 * S + smp) * 4u;
    uint32_t ma = sbase + L.msl + (uint32_t)((j0 * S + smp) * 16 + t * 4) * 4u;
    const uint32_t dp = (uint32_t)(dj * S) * 4u, dm = (uint32_t)(dj * S) * 64u;
    for (int j = j0; j < T_in; j += 2 * dj) {
      const bool two = j + dj < T_in;
      float pv0 = lds_f(pa), pv1 = lds_f(pa + (two ? dp : 0u));
      const float4 m0 = lds_f4(ma), m1 = lds_f4(ma + (two ? dm : 0u));
      if (!two) pv1 = 0.f;
      acc.x = fmaf(pv0, m0.x, acc.x); acc.y = fmaf(pv0, m0.y, acc.y); acc.z = fmaf(pv0, m0.z, acc.z); acc.w = fmaf(pv0, m0.w, acc.w);
      acc2.x = fmaf(pv1, m1.x, acc2.x); acc2.y = fmaf(pv1, m1.y, acc2.y); acc2.z = fmaf(pv1, m1.z, acc2.z); acc2.w = fmaf(pv1, m1.w, acc2.w);
      ssum += pv0; ssum2 += pv1;
      pa += 2 * dp; ma += 2 * dm;
    }
    acc.x += acc2.x; acc.y += acc2.y; acc.z += acc2.z; acc.w += acc2.w;
    ssum += ssum2;
    // sum over the position sub-slots: lane bits 2..4 (one utterance) or 3..4 (two)
    for (int o = 16; o >= (S == 2 ? 8 : 4); o >>= 1) {
      acc.x += __shfl_xor_sync(0xffffffffu, acc.x, o); acc.y += __shfl_xor_sync(0xffffffffu, acc.y, o);
      acc.z += __shfl_xor_sync(0xffffffffu, acc.z, o); acc.w += __shfl_xor_sync(0xffffffffu, acc.w, o);
      ssum += __shfl_xor_sync(0xffffffffu, ssum, o);
    }
    if (sub == 0) {
      sts_f4(slot + (uint32_t)(smp * RS + t * 4) * 4u, acc);
      if (t == 0) sts_f(sbase + OFF_REDS + (uint32_t)(gw * 8 + smp) * 4u, ssum);
    }
  };

  if (warp >= 12) {
    // =====================================================================================================================
    // CRITICAL GROUP
    // =====================================================================================================================
    uint4 wa[8];                                   // A fragments of the next late part: four chunk-tiles (hi, lo)
    float st_ha = 0.f, st_h1 = 0.f, st_h2 = 0.f, st_y1 = 0.f;   // recurrent state (and y1) of element (rn, rc), fp32
    const uint32_t myslot = sbase + OFF_SLOTS + (uint32_t)(SL_CRIT + gw) * (SLOT_F * 4);
    // chunk-tile index of each critical phase inside this warp's tensor-memory slice
    constexpr int TC_P1 = 0, TC_P2 = 4, TC_P3 = 8, TC_P4 = 10, TC_P5 = 14, TC_P9 = 18, TC_P10 = 22, TC_P11 = 26, TC_P12 = 30;
    auto tload = [&](int tc0, int n) {
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (k < n) tmem_ld8(tq + (uint32_t)(tc0 + k) * 8u, wa[2 * k], wa[2 * k + 1]);
    };
    auto twait = [&]() {
      tmem_wait_ld();
#pragma unroll
      for (int k = 0; k < 4; ++k) reg_fence(wa[2 * k], wa[2 * k + 1]);
    };
    // late part: chunks c0 .. c0+n-1 of the operand that has just arrived, times the preloaded chunk-tiles -> this warp's slot
    auto late = [&](uint32_t xaddr, int n) {
      float hh[4] = {0.f, 0.f, 0.f, 0.f}, hl[4] = {0.f, 0.f, 0.f, 0.f}, lh[4] = {0.f, 0.f, 0.f, 0.f};
      uint4 xf[4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (i < n) xf[i] = lds128(xaddr + (uint32_t)i * csb);
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (i < n) {
          mma16816(hh, wa[2 * i], xf[i].x, xf[i].y);       // W_hi * x_hi
          if (!BF16) {
            mma16816(lh, wa[2 * i + 1], xf[i].x, xf[i].y);   // W_lo * x_hi
            mma16816(hl, wa[2 * i], xf[i].z, xf[i].w);       // W_hi * x_lo
          }
        }
      store_tile(myslot, g, t, hh, hl, lh);
    };
    const int al_pp = tid - 12 * 32, al_n = (p0 + al_pp) % S, al_j = (p0 + al_pp) / S;   // the pair this thread writes the alignment of
    // wait for an exchange of this step, then re-arm its mbarrier for the next step (the phase that has just completed cannot be
    // disturbed any more; one lane of one critical warp, so no burst of twelve arrivals at the top of a step)
    auto wait_rearm = [&](int mb, uint32_t parity, uint32_t bytes) {
      mbar_wait(mb0 + (uint32_t)mb * 8u, parity);
      if (tid == (12 + (mb & 3)) * 32) mbar_expect_tx(mb0 + (uint32_t)mb * 8u, bytes);
    };
    tload(TC_P2, 4);   // step 0 has no late part in P1 (zero go frame / zero state)
    for (int step = 0; step < a.steps; ++step) {
      const uint32_t par = (uint32_t)step & 1u;
      const uint32_t XHAc = XHA + 16 * par, XH1c = XH1 + 16 * par, XH2c = XH2 + 16 * par;
      bool late1 = false;
      if (step > 0) wait_rearm(MB_P12, par ^ 1u, BLK);   // y2 of the previous step has landed
      TRM(0);
      if (TRACE && a.trace != nullptr && blockIdx.x == a.trace_cta && tid == 12 * 32 && step < 100) a.trace[400 + step] = clock64();   // step starts
      // ================= P1: decoder prenet dense_1 + ReLU.  free run: W_f y2 (late: the h2' term) + W_1c ctx; teacher: background only ====
      if (free_run && step > 0) {
        late(XADDR(XY2 + 4 * gw), 4);
        tload(TC_P2, 4);
        late1 = true;                        // (the handoff barrier below counts the critical threads too: no NB_CRIT sync needed)
      }
      TRM(50); nb_sync(NB_H1, 256); TRM(51);
      {
        float v = sum4(red_nc, SL_P1E) + BIAS(late1 ? BI_P1 : BI_P1S0);
        if (late1) v += sum4(red_nc, SL_CRIT);
        stage_x(stg_n, rc, fmaxf(v, 0.f));
        send_rows(OFF_X + (uint32_t)(XP1 + q) * csb, MB_P1, false);
      }
      twait();
      TRM(1);
      wait_rearm(MB_P1, par, BLK);
      TRM(2);
      // ================= P2: prenet dense_2 + ReLU (CTA pair 2c, 2c+1 computes chunk c; each feeds the peers of its parity) ====
      late(XADDR(XP1 + 4 * gw), 4);
      tload(TC_P3, 2);
      nb_sync(NB_CRIT, 128);
      stage_x(stg_n, rc, fmaxf(sum4(red_nc, SL_CRIT) + BIAS(BI_P2), 0.f));
      send_rows(OFF_X + (uint32_t)(XP2 + (q >> 1)) * csb, MB_P2, true);
      twait();
      TRM(3);
      wait_rearm(MB_P2, par, BLK / 2);
      TRM(4);
      // ================= P3: attention GRU reset gate on [prenet | h_att]; r * h_att goes out ====
      late(XADDR(XP2 + 2 * gw), 2);
      tload(TC_P4, 4);
      TRM(52); nb_sync(NB_H3, 256); TRM(53);
      stage_x(stg_n, rc, sigmoid_f(sum4(red_nc, SL_CRIT) + sum4(red_nc, SL_RE0) + BIAS(BI_RA)) * st_ha);
      send_rows(OFF_X + (uint32_t)(XRA + q) * csb, MB_P3, false);
      twait();
      TRM(5);
      wait_rearm(MB_P3, par, BLK);
      TRM(6);
      // ================= P4: candidate; h_att' = u h + (1-u) tanh(c_h + c_x + b) ====
      late(XADDR(XRA + 4 * gw), 4);
      tload(TC_P5, 4);
      TRM(54); nb_sync(NB_H4, 384); TRM(55);
      {
        const float u = sigmoid_f(sum4(red_nc, SL_U) + BIAS(BI_UA));
        const float c = tanh_f(sum4(red_nc, SL_CRIT) + sum4(red_nc, SL_CX) + BIAS(BI_CA));
        st_ha = u * st_ha + (1.0f - u) * c;
        stage_x(stg_n, rc, st_ha);
        send_rows(OFF_X + (uint32_t)(XHAc + q) * csb, MB_P4, false);
      }
      twait();
      TRM(7);
      wait_rearm(MB_P4, par, BLK);
      TRM(8);
      // ================= P5: query layer; pushed as e^{2 pq} (fp32) for the score phase ====
      late(XADDR(XHAc + 4 * gw), 4);
      tload(TC_P9, 4);
      nb_sync(NB_CRIT, 128);
      sts_f(stg_n + rc * 4, __expf(2.0f * fminf(fmaxf(sum4(red_nc, SL_CRIT), -30.f), 30.f)));
      send_rows(L.pq + (uint32_t)q * csb, MB_P5, false);
      twait();
      TRM(9);
      wait_rearm(MB_P5, par, BLK);
      // h1' / h2' of the previous step landed long ago (nobody pushes them again before this step's P10 / P12): their mbarriers are
      // re-armed here instead of at the top of the step, where the critical group would wait for the trailing h2' push
      if (step > 0) { wait_rearm(MB_H1, par ^ 1u, BLK); wait_rearm(MB_H2, par ^ 1u, BLK); }
      TRM(10);
      // ================= P6 / P7: attention (all warps; the critical group alone when S <= 2) ====
      if (small_att) {
        p6_compute(8);
        nb_sync(NB_CRIT, 128);
        TRM(11);
        p6_send_crit();
        wait_rearm(MB_P6, par, (uint32_t)NQ * 16u);
        TRM(12);
        p7_compute_crit(myslot);
        nb_sync(NB_CRIT, 128);
        TRM(13);
        const float* reds = reinterpret_cast<const float*>(smem_raw + OFF_REDS) + rn;
        const float inv = rcp_approx((reds[0] + reds[8]) + (reds[16] + reds[24]));
        stage_x(stg_n, rc, sum4(red_nc, SL_CRIT) * inv);
        if (rc == 0) reinterpret_cast<float*>(smem_raw + OFF_INV)[rn] = inv;
        send_rows(OFF_X + (uint32_t)(XC + q) * csb, MB_P7, false);
      } else {
      p6_compute(2 * NW);
      TRW(112);
      __syncthreads();
      TRM(11);
      p6_send();
      wait_rearm(MB_P6, par, (uint32_t)NQ * 16u);
      TRM(12);
      TRW(128);
      p7_compute();
      TRW(144);
      __syncthreads();
      TRM(13);
      {
        const float* reds = reinterpret_cast<const float*>(smem_raw + OFF_REDS) + rn;
        float s0 = 0.f, s1 = 0.f, c0 = 0.f, c1 = 0.f;
#pragma unroll
        for (int s = 0; s < NW; s += 2) {
          s0 += reds[s * 8]; s1 += reds[s * 8 + 8];
          c0 += lds_f(red_nc + (SL_CTX + s) * SLOT_F * 4); c1 += lds_f(red_nc + (SL_CTX + s + 1) * SLOT_F * 4);
        }
        const float inv = rcp_approx(s0 + s1);
        stage_x(stg_n, rc, (c0 + c1) * inv);
        if (rc == 0) reinterpret_cast<float*>(smem_raw + OFF_INV)[rn] = inv;
        send_rows(OFF_X + (uint32_t)(XC + q) * csb, MB_P7, false);
      }
      }
      TRM(14);
      wait_rearm(MB_P7, par, BLK);
      TRM(15);
      // ================= P9: GRU-1 reset gate on [h_att' | ctx'] (512->256 projection folded in) and h1 ====
      late(XADDR(XC + 4 * gw), 4);
      tload(TC_P10, 4);
      TRM(56); nb_sync(NB_H9, 256); TRM(57);
      stage_x(stg_n, rc, sigmoid_f(sum4(red_nc, SL_CRIT) + sum4(red_nc, SL_RE1) + BIAS(BI_R1)) * st_h1);
      send_rows(OFF_X + (uint32_t)(XR1 + q) * csb, MB_P9, false);
      twait();
      if (a.align_out != nullptr) {
        // alignments of this CTA's pairs (tacotron.py:104: [N,T_in,steps]); the normalisers were written before the barrier above
        const float* stage = reinterpret_cast<const float*>(smem_raw + L.stage);
        const float* invs = reinterpret_cast<const float*>(smem_raw + OFF_INV);
        const float* mxs = reinterpret_cast<const float*>(smem_raw + OFF_MX);
        for (int pp = tid - 12 * 32; pp < npq; pp += 128) {
          const bool first = pp < 128;
          const int n = first ? al_n : (int)smem_raw[L.pn + pp], j = first ? al_j : (p0 + pp - n) / S;
          const float e = exact ? __expf(stage[pp] - mxs[n]) : stage[pp];
          a.align_out[((size_t)(n0 + n) * T_in + j) * a.max_steps + step] = e * invs[n];
        }
      }
      TRM(16);
      wait_rearm(MB_P9, par, BLK);
      TRM(17);
      // ================= P10: GRU-1 candidate, h1' ====
      late(XADDR(XR1 + 4 * gw), 4);
      tload(TC_P11, 4);
      TRM(58); nb_sync(NB_H10, 512); TRM(59);
      {
        const float u = sigmoid_f(sum4(red_nc, SL_U) + BIAS(BI_U1));
        const float c = tanh_f(sum4(red_nc, SL_CRIT) + sum4(red_nc, SL_CX) + BIAS(BI_C1));
        st_h1 = u * st_h1 + (1.0f - u) * c;
        st_y1 = lds_f(sbase + OFF_Y0S + (uint32_t)(rn * 16 + rc) * 4u) + st_h1;     // ResidualWrapper: y1 = y0 + h1'
        stage_x(stg_n, rc, st_y1);
        send_rows(OFF_X + (uint32_t)(XY1 + q) * csb, MB_P10, false);             // critical: GRU 2's gates wait for y1
        __syncwarp();
        stage_x(stg_n, rc, st_h1);
        send_rows(OFF_X + (uint32_t)(XH1c + q) * csb, MB_H1, false);             // the state itself: first needed in the next step
      }
      twait();
      TRM(18);
      wait_rearm(MB_P10, par, BLK);
      TRM(19);
      // ================= P11: GRU-2 reset gate on [y1 = y0 + h1' | h2] (late: the h1' term) ====
      late(XADDR(XY1 + 4 * gw), 4);
      TRM(45);
      tload(TC_P12, 4);
      TRM(46);
      TRM(60); nb_sync(NB_H11, 256); TRM(61);
      stage_x(stg_n, rc, sigmoid_f(sum4(red_nc, SL_CRIT) + sum4(red_nc, SL_RE2) + BIAS(BI_R2)) * st_h2);
      TRM(47);
      send_rows(OFF_X + (uint32_t)(XR2 + q) * csb, MB_P11, false);
      TRM(48);
      twait();
      TRM(20);
      wait_rearm(MB_P11, par, BLK);
      TRM(21);
      // ================= P12: GRU-2 candidate, h2' ====
      late(XADDR(XR2 + 4 * gw), 4);
      if (free_run) tload(TC_P1, 4); else tload(TC_P2, 4);
      TRM(62); nb_sync(NB_H12, 384); TRM(63);
      {
        const float u = sigmoid_f(sum4(red_nc, SL_U) + BIAS(BI_U2));
        const float c = tanh_f(sum4(red_nc, SL_CRIT) + sum4(red_nc, SL_CX) + BIAS(BI_C2));
        st_h2 = u * st_h2 + (1.0f - u) * c;
        stage_x(stg_n, rc, st_y1 + st_h2);                                        // y2 = y1 + h2': the next prenet and the frames need it
        send_rows(OFF_X + (uint32_t)(XY2 + q) * csb, MB_P12, false);
        __syncwarp();
        stage_x(stg_n, rc, st_h2);
        send_rows(OFF_X + (uint32_t)(XH2c + q) * csb, MB_H2, false);
      }
      twait();
      TRM(22);
      if (step == 0) TRX(27);
    }
    TRX(26);
  } else {
    // =====================================================================================================================
    // BACKGROUND GROUPS: A = warps 0-3 (update gates), B = 4-7 (candidate x-parts, output projection), C = 8-11 (early parts of the
    // critical tiles, y0).  Each warp walks its item list; weights come from tensor memory or from a per-warp ring that cp.async
    // keeps `D` chunk-tiles ahead of the consumer (the stream is laid out in consumption order, one step per lap).
    // =====================================================================================================================
    const uint4* rsrc = reinterpret_cast<const uint4*>(w.ring) + ((size_t)(q * 12 + warp) * w.ring_stride) * 64 + lane;
    const int rn_len = w.ring_len[warp];
    const int D = rn_len < w.ring_kb ? rn_len : w.ring_kb;
    const bool resident = D == rn_len;            // the whole lap fits: filled once, never refilled
    const uint32_t rbase = sbase + L.ring + (uint32_t)(warp * w.ring_kb) * 1024u + (uint32_t)lane * 16u;
    int rp = 0, kf = 0;                           // ring slot of the oldest entry; stream index of the next entry to request
    auto refill = [&](int cnt) {                  // request the next cnt entries into the slots consumed last
      if (resident) return;
      int rf = rp - cnt;
      if (rf < 0) rf += D;
      for (int k = 0; k < cnt; ++k) {
        const uint4* src = rsrc + (size_t)kf * 64;
        const uint32_t dst = rbase + (uint32_t)rf * 1024u;
        cp_async16(dst, src);
        cp_async16(dst + 512u, src + 32);
        cp_async_commit();
        rf = rf + 1 == D ? 0 : rf + 1;
        kf = kf + 1 == rn_len ? 0 : kf + 1;
      }
    };
    {   // fill the ring
      for (int k = 0; k < D; ++k) {
        const uint4* src = rsrc + (size_t)k * 64;
        cp_async16(rbase + (uint32_t)k * 1024u, src);
        cp_async16(rbase + (uint32_t)k * 1024u + 512u, src + 32);
        cp_async_commit();
      }
      kf = D == rn_len ? 0 : D;
    }
    float hh[4] = {0.f, 0.f, 0.f, 0.f}, hl[4] = {0.f, 0.f, 0.f, 0.f}, lh[4] = {0.f, 0.f, 0.f, 0.f};   // live across items (and the attention phases)
    uint4 wa[8];
    const int fb_lane_n = min(g, S - 1);
    auto run_items = [&](const Item* items, int n_items, int step) {
      const uint32_t par = (uint32_t)step & 1u;
#define ITSTAMP(k) do { if (TRACE && a.trace != nullptr && step == 8 && blockIdx.x == a.trace_cta && warp == a.trace_warp && lane == 0) a.trace[320 + (items == prog.post[warp] ? 40 : 0) + it * 4 + (k)] = clock64(); } while (0)
      for (int it = 0; it < n_items; ++it) {
        ITSTAMP(0);
        const uint32_t w0 = items[it].w[0];
        const int n = (int)(w0 & 7u), nops = (int)((w0 >> 19) & 3u);
        if (w0 & 16u) {
#pragma unroll
          for (int k = 0; k < 4; ++k) { hh[k] = 0.f; hl[k] = 0.f; lh[k] = 0.f; }
        }
        if (n > 0) {
          // ---- A fragments ----
          if (w0 & 8u) {
            const uint32_t tc = items[it].w[1];
#pragma unroll
            for (int k = 0; k < 4; ++k)
              if (k < n) tmem_ld8(tq + (tc + (uint32_t)k) * 8u, wa[2 * k], wa[2 * k + 1]);
            tmem_wait_ld();
#pragma unroll
            for (int k = 0; k < 4; ++k) reg_fence(wa[2 * k], wa[2 * k + 1]);
          } else {
            if (!resident) cp_async_wait_pending(D - n); else cp_async_wait_pending(0);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              if (k < n) {
                const uint32_t src = rbase + (uint32_t)rp * 1024u;
                wa[2 * k] = lds128(src);
                wa[2 * k + 1] = lds128(src + 512u);
                rp = rp + 1 == D ? 0 : rp + 1;
              }
            // the slots are free as soon as the fragments sit in registers: request the next entries NOW, before the operand
            // waits and the MMAs of this item (the refill then lands while this item runs)
#pragma unroll
            for (int k = 0; k < 4; ++k) reg_fence(wa[2 * k], wa[2 * k + 1]);
            refill(n);
          }
          ITSTAMP(1);
          // ---- operands ----
          for (int o = 0; o < nops; ++o) {
            const uint32_t od = items[it].w[2 + o];
            const uint32_t mb = (od >> 10) & 31u;
            if (mb) mbar_wait(mb0 + (mb - 1u) * 8u, (od & 0x10000u) ? par ^ 1u : par);
            const uint32_t pb = (od >> 8) & 3u;
            const uint32_t chunk = (od & 255u) + (pb == 1u ? 16u * par : (pb == 2u ? 16u * (par ^ 1u) : 0u));
            uint4 xf[4];
            if (od & 0x8000u) {
              // teacher forcing: the frame fed at step+1 is mel_targets[:, step*r + r-1, :]  (helpers.py:48,75)
              const float* src = a.targets + ((size_t)(n0 + fb_lane_n) * a.T_tgt + (size_t)step * a.r + a.r - 1) * M;
#pragma unroll
              for (int i = 0; i < 4; ++i)
                if (i < n) {
                  const int k0 = ((int)(od & 255u) + i) * 16;
                  const float2 lo2 = __ldg(reinterpret_cast<const float2*>(src + k0 + 2 * t));
                  const float2 hi2 = __ldg(reinterpret_cast<const float2*>(src + k0 + 2 * t + 8));
                  split2(lo2.x, lo2.y, xf[i].x, xf[i].z);
                  split2(hi2.x, hi2.y, xf[i].y, xf[i].w);
                }
            } else {
              const uint32_t xaddr = XADDR(chunk);
#pragma unroll
              for (int i = 0; i < 4; ++i)
                if (i < n) xf[i] = lds128(xaddr + (uint32_t)i * csb);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (i < n) {
                mma16816(hh, wa[2 * i], xf[i].x, xf[i].y);
                if (!BF16) {
                  mma16816(lh, wa[2 * i + 1], xf[i].x, xf[i].y);
                  mma16816(hl, wa[2 * i], xf[i].z, xf[i].w);
                }
              }
          }
        }
        ITSTAMP(2);
        if (w0 & 32u) {
          const uint32_t slot = (w0 >> 6) & 63u;
          store_tile(sbase + OFF_SLOTS + slot * (SLOT_F * 4), g, t, hh, hl, lh);
        }
        const uint32_t post = (w0 >> 12) & 7u;
        if (post == POST_ARRIVE) {
          const int nb = (int)((w0 >> 15) & 15u);
          __syncwarp();
          nb_arrive(nb, nb == NB_H10 ? 512 : ((nb == NB_H4 || nb == NB_H12) ? 384 : 256));
        } else if (post == POST_Y0) {
          // y0 tile of this CTA = [h_att' | ctx'] W_p + b_p: reduce the group's four partial tiles into the local fp32 copy that the
          // candidate phase of GRU 1 adds to h1' (nothing is exchanged: every consumer of y0 reads y1 or y2)
          nb_sync(NB_CGRP, 128);
          sts_f(sbase + OFF_Y0S + (uint32_t)(rn * 16 + rc) * 4u, sum4(red_nc, SL_Y0) + BIAS(BI_Y0));
          __syncwarp();
          nb_arrive(NB_H10, 512);
        } else if (post == POST_OUT) {
          // frames of this step: tiles 2q and 2q+1 of y2 W_o + b_o  (tacotron.py:83)
          nb_sync(NB_BGRP, 128);
          const int ntiles = Dout >> 4;
          const float oa = sum4(red_nc, SL_O) + BIAS(BI_OA), ob = sum4(red_nc, SL_O + 4) + BIAS(BI_OB);
          if (rn < S) {
            float* dst = a.dec_out + ((size_t)(n0 + rn) * a.max_steps + step) * Dout + rc;
            if (2 * q < ntiles) dst[(2 * q) * 16] = oa;
            if (2 * q + 1 < ntiles) dst[(2 * q + 1) * 16] = ob;
          }
        }
        ITSTAMP(3);
      }
    };
    if (warp < 4) { __syncwarp(); nb_arrive(NB_H1, 256); }   // P1 of step 0: zero context, zero go frame -> the (zeroed) early slots are complete
    for (int step = 0; step < a.steps; ++step) {
      const uint32_t par = (uint32_t)step & 1u;
      run_items(prog.pre[warp], prog.n_pre[warp], step);
      TRW(64);
      if (small_att) {
        mbar_wait(mb0 + MB_P6 * 8, par);   // pacing only: the attention phases run on the critical group
      } else {
      mbar_wait(mb0 + MB_P5 * 8, par);
      TRW(160);
      {
        const int reps = (TRACE && a.trace != nullptr && step == 8) ? 3 : 1;
#pragma unroll 1
        for (int rep = 0; rep < reps; ++rep) { p6_compute(2 * NW); TRW(112 + 64 * rep); }
      }
      __syncthreads();
      p6_send();
      mbar_wait(mb0 + MB_P6 * 8, par);
      TRW(128);
      {   // trace build: the phase runs three times at the stamped step (same code, warm on the repeats)
        const int reps = (TRACE && a.trace != nullptr && step == 8) ? 3 : 1;
#pragma unroll 1
        for (int rep = 0; rep < reps; ++rep) { p7_compute(); TRW(144 + 64 * rep); }
      }
      __syncthreads();
      }
      TRW(80);
      run_items(prog.post[warp], prog.n_post[warp], step);
      TRW(96);
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  }
  // nobody may exit while a peer can still write into its shared memory
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  cluster_sync_all();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(lds32(sbase + OFF_TMEM)) : "memory");
}

}  // namespace

size_t decoder_cw_smem_bytes(int s_max, int T_in, int att_res, int ring_kb) { return make_dyn(s_max, T_in, att_res, ring_kb).total; }

// Residency of the attention operands, in order of preference, each with the deepest weight ring (>= 4 KB per background warp:
// an item takes up to four chunk-tiles at once) that fits 227 KB of shared memory:
//   3 keys and memory in shared memory (weights fill tensor memory: TL_WIDE), the plan of every S <= 5 at T_in <= 100;
//   ATT_TMEM keys and memory in tensor memory (TL_ATT: 26 background chunk-tiles per quarter move to the ring), if they fit its
//     224 free columns: S = 8 up to T_in = 105;
//   1 keys only, 2 memory only, 0 neither (P6 reloads keys from global memory and recomputes their exponentials, P7 walks the
//     memory rows serially): long inputs.
bool decoder_cw_plan(int s_max, int T_in, int* att_res, int* ring_kb, size_t* smem) {
  static const int masks[5] = {3, ATT_TMEM, 1, 2, 0};
  static const int rings[3] = {6, 5, 4};
  for (int m = 0; m < 5; ++m) {
    if (masks[m] == ATT_TMEM && att_tmem_cols(s_max, T_in) > TMEM_ATT_COLS) continue;
    for (int k = 0; k < 3; ++k) {
      const size_t b = decoder_cw_smem_bytes(s_max, T_in, masks[m], rings[k]);
      if (b <= 227 * 1024) { *att_res = masks[m]; *ring_kb = rings[k]; *smem = b; return true; }
    }
  }
  return false;
}

int decoder_cw_max_clusters() {
  auto kern = decoder_cw_kernel<false, false, false>;
  const int smem = 200 * 1024;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess ||
      cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(CS);
  cfg.blockDim = dim3(NT);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

cudaError_t launch_decoder_cw(const cw::Weights& wt, const DecoderArgs& a_in, int nclusters, cudaStream_t st, bool bf16_only) {
  if (a_in.N <= 0 || a_in.steps <= 0) return cudaSuccess;
  if (nclusters < 1 || nclusters > a_in.N) return cudaErrorInvalidValue;
  DecoderArgs a = a_in;
  a.s_max = (a.N + nclusters - 1) / nclusters;
  if (a.s_max > 8 || (wt.M & 15) || (wt.Dout & 15) || wt.M > 128 || wt.Dout > 512) return cudaErrorInvalidValue;
  const int mode = a.targets != nullptr ? 1 : 0;
  int ring_kb = 0;
  size_t smem = 0;
  if (!decoder_cw_plan(a.s_max, a.T_in, &a.att_res, &ring_kb, &smem)) return cudaErrorInvalidValue;
  const int lay = (a.att_res & ATT_TMEM) ? TL_ATT : TL_WIDE;
  if (a.s_max <= 2) {   // small batches: let the ring hold a whole lap if it fits (no refills at all)
    int longest = 0;
    for (int i = 0; i < 12; ++i) longest = wt.ring_len[lay][mode][i] > longest ? wt.ring_len[lay][mode][i] : longest;
    if (longest <= 7 && decoder_cw_smem_bytes(a.s_max, a.T_in, a.att_res, longest) <= 227 * 1024) {
      ring_kb = longest;
      smem = decoder_cw_smem_bytes(a.s_max, a.T_in, a.att_res, ring_kb);
    }
  }
  Args k{};
  k.tmem_img = wt.tmem_img[lay];
  k.ring = reinterpret_cast<const char*>(wt.ring[lay]) + (size_t)mode * 16 * 12 * wt.ring_stride * 1024;
  for (int i = 0; i < 12; ++i) k.ring_len[i] = wt.ring_len[lay][mode][i];
  k.ring_stride = wt.ring_stride;
  k.bias = wt.bias;
  k.att_v = wt.att_v;
  k.M = wt.M; k.Dout = wt.Dout;
  k.exact_softmax = wt.v_l1 > 40.0f ? 1 : 0;
  k.ring_kb = ring_kb;
  const bool small = a.s_max <= 2;
  auto kern = a.trace != nullptr ? (small ? decoder_cw_kernel<true, false, true> : decoder_cw_kernel<true, false, false>)
              : bf16_only ? (small ? decoder_cw_kernel<false, true, true> : decoder_cw_kernel<false, true, false>)
                          : (small ? decoder_cw_kernel<false, false, true> : decoder_cw_kernel<false, false, false>);
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  if (e != cudaSuccess) return e;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(nclusters * CS);
  cfg.blockDim = dim3(NT);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, k, wt.prog[lay][mode], a, nclusters);
}

}  // namespace taco
