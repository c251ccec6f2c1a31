// K7 (v6) "critical warps": layout shared by the kernel (decoder_cw.cu) and the host-side packer (decoder_cw_pack.inc).
//
// Operator: tf.contrib.seq2seq.dynamic_decode(BasicDecoder(output_cell, helper, zero_state), max_iters) of reference
// models/tacotron.py:66-94 (rnn_wrappers.py:22-24,50-52; helpers.py:26-38,68-77; SURVEY Appendix B.2/B.3/B.5).
//
// A cluster of 16 CTAs owns S <= 8 utterances; CTA q owns output columns [16q, 16q+16) of every 256-wide layer.
// Inside a CTA the 16 warps are four groups of four (one warp per SM sub-partition each):
//   D = warps 12-15  the CRITICAL group: per phase, wait for the operand that has just been exchanged, multiply it with at
//                    most four 16x16 weight chunk-tiles per warp (from tensor memory), cross-reduce the four partial tiles,
//                    finish the gate math on register-resident state and push the result to the 16 peers;
//   A, B, C = warps 0-3, 4-7, 8-11: BACKGROUND groups that run a host-written item list: every product whose operand is
//                    complete earlier than the critical one (recurrent states, previous context, ...), every tile that is
//                    only needed one phase later (update gates, candidate x-parts, the 512->256 projection), the output
//                    projection, and their share of the attention phases.  Results meet the critical group in
//                    shared-memory partial-tile slots behind named barriers (bar.arrive / bar.sync).
#pragma once
#include <stdint.h>

namespace taco {
namespace cw {

constexpr int CS = 16, NT = 512, NW = 16;
constexpr int DHID = 256;
constexpr int RS = 20;            // floats per sample row of a partial tile (16 + pad: conflict-free fragment stores)
constexpr int SLOT_F = 8 * RS;    // floats per partial-tile slot

// ---- activation buffers in MMA B-fragment order; sizes in 16-row chunks (one chunk = S x 64 bytes) ----------------
// XHA / XH1 / XH2 hold the recurrent states and are double buffered by step parity (background warps read the value of
// step s while the exchange of step s+1 lands).
// y1 = y0 + h1' and y2 = y1 + h2' are formed by the critical reducers from CTA-local tiles (y0 never leaves its CTA) and pushed as
// the critical exchanges of the GRU candidate phases; h1' / h2' themselves follow on mbarriers nobody waits for before the next step.
enum { XC = 0, XP1 = 16, XP2 = 32, XHA = 40, XRA = 72, XY1 = 88, XH1 = 104, XR1 = 136, XH2 = 152, XR2 = 184, XY2 = 200, X_CHUNKS = 216 };

// ---- partial-tile slots ------------------------------------------------------------------------------------------
enum { SL_CRIT = 0, SL_P1E = 4, SL_RE0 = 8, SL_RE1 = 12, SL_RE2 = 16, SL_U = 20, SL_CX = 24, SL_Y0 = 28, SL_CTX = 32,
       SL_O = SL_CTX /* the output projection reuses the context partials */, N_SLOTS = 48 };

// ---- mbarriers (one per exchange) -----------------------------------------------------------------------------------
enum { MB_P1 = 0, MB_P2, MB_P3, MB_P4, MB_P5, MB_P6, MB_P7, MB_P9, MB_H1 /* h1' (not critical) */, MB_P10 /* y1 */, MB_P11,
       MB_P12 /* y2 */, MB_H2 /* h2' (not critical) */, N_MBAR = 16 };

// ---- named barriers ---------------------------------------------------------------------------------------------------
enum { NB_SYNC = 0, NB_CRIT = 1, NB_H1 = 2, NB_H3 = 3, NB_H4 = 4, NB_H9 = 5, NB_H10 = 6, NB_H11 = 7, NB_H12 = 8, NB_CGRP = 9,
       NB_AGRP = 10, NB_BGRP = 11 };

// ---- background items ---------------------------------------------------------------------------------------------
// One item = up to four weight chunk-tiles (A fragments: tensor memory or the next entries of the warp's ring) times up
// to three activation operands (the same weights multiply y0, h1' and h2' where a sum of activations is never formed).
//   w0: n (0-4) | tmem << 3 | zero_acc << 4 | flush << 5 | slot << 6 (6 bits) | post << 12 (3 bits) | nb << 15 (4 bits: named barrier of
//       POST_ARRIVE) | nops << 19 (2 bits)
//   w1: tensor-memory column of the first chunk-tile (tmem items)
//   w2..w4: operands: chunk index (8 bits) | pbuf << 8 (0 single, 1 parity of this step, 2 parity of the previous step)
//           | (mbarrier + 1) << 10 (5 bits; 0 = no wait) | frames << 15 (operand = teacher-forcing frame chunks from global memory)
//           | prev << 16 (wait for the PREVIOUS step's phase of that mbarrier: recurrent states h1, h2)
enum { POST_NONE = 0, POST_ARRIVE = 1, POST_Y0 = 2 /* reduce the y0 tile into the CTA-local fp32 copy, then arrive */, POST_OUT = 3 };
struct Item { uint32_t w[5]; };
constexpr int MAX_ITEMS = 8;      // per warp and half step (before the attention phases / after them)
struct Program {
  Item pre[NW][MAX_ITEMS];        // items of step s that run before the attention phases of step s
  Item post[NW][MAX_ITEMS];       // ... and after them
  uint8_t n_pre[NW], n_post[NW];
};

// ---- critical phases: late operand of each phase for critical warp cw (chunks c0 .. c0+n-1 of buffer `xbuf`) ------------
enum { CP_P1 = 0, CP_P2, CP_P3, CP_P4, CP_P5, CP_P9, CP_P10, CP_P11, CP_P12, N_CPHASE };
// chunk-tiles per critical warp and phase in tensor memory (P3 multiplies the 128-wide prenet output: 2 per warp)
constexpr int CP_N[N_CPHASE] = {4, 4, 2, 4, 4, 4, 4, 4, 4};
constexpr int CP_TOTAL = 34;      // sum of CP_N: chunk-tiles 0..33 of the quarter belong to the critical warp
constexpr int TMEM_BG0 = CP_TOTAL;   // background chunk-tiles start here (30 per lane quarter)
constexpr int TMEM_TILES = 64;    // chunk-tiles per lane quarter (512 columns / 8)

// ---- tensor-memory layouts -------------------------------------------------------------------------------------------
// TL_WIDE: all 64 chunk-tiles of a lane quarter are weights.  TL_ATT: only the first TMEM_ATT_TILES are (the critical tiles and
// two background tiles; every other background tile streams through the ring), and columns TMEM_ATT_COL0..511 hold this CTA's
// attention operands, so that eight utterances per cluster keep them on chip (shared memory has room for neither).  In lane
// quarter gq (the quarter the P6 / P7 warps w with w & 3 == gq can read):
//   * exp(2 key) row of pair pp, (pp >> 1) & 3 == gq, at column TMEM_ATT_COL0 + 8 (2 (pp >> 3) + (pp & 1)); lane l holds
//     elements 4l..4l+3 and 128+4l..128+4l+3 (the registers pair_sum works on);
//   * memory columns of position j, j & 3 == gq, at column TMEM_ATT_COL0 + att_key_cols + 4 (j >> 2); lane 4 n + t holds
//     memory[n][j][16 q + 4 t .. + 3] (zero for n >= S).
enum { TL_WIDE = 0, TL_ATT = 1 };
constexpr int TMEM_ATT_TILES = 36;
constexpr int TMEM_ATT_COL0 = TMEM_ATT_TILES * 8, TMEM_ATT_COLS = 512 - TMEM_ATT_COL0;
constexpr int ATT_TMEM = 4;       // att_res bit: attention operands in tensor memory (layout TL_ATT)
__host__ __device__ constexpr int att_key_cols(int S, int T_in) { return 16 * (((T_in * S) / CS + 4 + 7) / 8); }
__host__ __device__ constexpr int att_tmem_cols(int S, int T_in) { return att_key_cols(S, T_in) + 4 * ((T_in + 3) / 4); }

// ---- bias table per CTA (floats) ----------------------------------------------------------------------------------
enum { BI_P1 = 0, BI_P1S0 = 16 /* step 0 of a free run: the go frame is zero, not W_o y + b_o */, BI_P2 = 32, BI_RA = 48, BI_UA = 64,
       BI_CA = 80, BI_Y0 = 96, BI_R1 = 112, BI_U1 = 128, BI_C1 = 144, BI_R2 = 160, BI_U2 = 176, BI_C2 = 192, BI_OA = 208,
       BI_OB = 224, N_BIAS = 240 };

struct Weights {
  int M, Dout;
  const void* tmem_img[2]; // by layout: [16 CTAs][4 quarters][64 chunk-tiles][2][32 lanes] uint4 (TL_ATT: tiles >= 36 unused)
  const void* ring[2];     // by layout: [2 modes][16 CTAs][12 background warps][ring_stride] chunk-tiles of 1 KB, consumption order
  int ring_len[2][2][12];  // chunk-tiles per step of each background warp (by layout, mode)
  int ring_stride;         // chunk-tiles reserved per warp in `ring`
  const float* bias;       // [2 modes][16 CTAs][N_BIAS]
  const float* att_v;      // [256]
  float v_l1;              // ||attention_v||_1
  Program prog[2][2];     // by layout, then [0] free running, [1] teacher forcing
};

}  // namespace cw
}  // namespace taco
