// Shared between the replicated-state forward (gnca_rep.cu) and the resident backward (gnca_rep_bwd.cu):
// layout of what the forward keeps for BPTT instead of the dense x_t / u_t history.
#pragma once
#include <stdint.h>

namespace gnca {

// One record per ACTIVE cell (fire & pre-alive) of a step, in cell order, at
//   rec[((t*B + b)*HW + slot) * kRecStride],  slot = rank of the cell among the active cells of (t, b).
// Forward writes  y[48] (perception: identity | sobel_x | sobel_y), u[16] (masked pre-norm update),
// xs[16] (gathered sender state sum_i w x(q_i) A(q_i)), th[16] = tanh(Wm xs + bm as) and as.
// The backward overwrites u with gd = dL/du and th with gm = dL/d(Wm xs + bm as); the batched weight-gradient
// kernel then needs nothing but the records.
constexpr int kRecY = 0, kRecU = 48, kRecXs = 64, kRecTh = 80, kRecAs = 96, kRecStride = 100;
// The backward additionally keeps, per record, the hidden layer h[128] and its gradient gh[128] (unit order permuted:
// index 4*l + jj <-> unit l + 32*jj) at hgh[((t*B + b)*HW + slot) * kHghStride]: the weight-gradient pass then is a pure
// stream of outer products.
constexpr int kHghStride = 256;
// bitmaps of a step: [0] sender-alive (graph_alpha_thr), [1] active = fire & pre-alive, [2] post-alive
constexpr int kMaskWords = 64;
// blocks of the batched weight-gradient kernel (two per SM)
constexpr int kMaxWgradBlocks = 296;

// Zero-padded graph shift (k_rep_fwd<16, true>): what the forward keeps beyond the records for the attention backward.
// Rank 0 of a sample's cluster writes them on every step with the message on; other steps leave them unwritten.
struct ZpRec {
  float* w;                   // [T][B][16] softmax weight of offset i (0 for i >= k)
  float* rowsum;              // [T][B][C][H] per-(channel, row) sums of x_t
};
// ... and what the resident backward (k_rep_bwd<16, kFrames, true>) reads and writes.
struct ZpBwd {
  const float* x;             // [T+1][B][C][HW] x_t, the state step t consumes (after the damage)
  const float* w;             // ZpRec::w
  const float* rowsum;        // ZpRec::rowsum
  float* bg;                  // [B][HW] bm . gm of the active cells of the current step, by cell
  float* pw;                  // [B][2dC + 2d + 1] per-sample wq | bq | wk | bk | scaling gradients (k_attn_bwd layout)
  int d;                      // d_model
};
// floats of the backward's shared-memory tail for the attention backward (behind the plain carve)
constexpr int kZpSmemFloats = 64 * 16 /*row sums*/ + 16 /*w*/ + 16 * 16 /*warp gw*/ + 8 * 16 /*cluster gw*/ +
                              4 * 16 /*gL, logits, row range*/ + 16 /*bm*/ + 3 * 16 + 2 * 32 /*xbar, wkq, gxb, qp, gqp*/ +
                              16 * 16 /*S*/ + 16 * 32 /*KP*/ + 64 /*row sums of gL*/ + 16 /*misc*/;

}  // namespace gnca
