// Streaming backward of one graph-NCA step (SURVEY Appendix A).  Saved from the forward: x_in, the masked
// pre-norm update u (valid on active cells) and the GroupNorm statistics (mean, rstd); everything else
// (perception, hidden layer, masks, message) is recomputed.
//
//   k_bwd_norm   : post-alive gate, tanh', GroupNorm partial sums (S1,S2,dgamma,dbeta) per tile, gz on active
//                  cells, active/post byte masks.
//   k_bwd_stats  : per-sample S1/N, S2/N (deterministic), dgamma/dbeta -> gparams.
//   k_bwd_mlp    : persistent blocks; batches of active cells staged in shared memory and pushed through the
//                  five small GEMMs of the MLP backward with register tiles (FFMA); message backward;
//                  weight-gradient partials per block (deterministic, no atomics).
//   k_bwd_gather : dL/dx = gate path + perception transpose (gather from active neighbours) + message transpose
//                  (gather from active receivers at +offset) + the gradient of a recorded frame of x, if any.
//   k_bwd_reduce : gparams += sum over blocks of the partials.
#include "gnca_common.cuh"
#include "gnca_internal.h"

namespace gnca {

constexpr int kBThreads = 256;
constexpr int kBChunk = 1024;
constexpr int kBChunkSmall = 256;
constexpr int kBTileW = 32, kBTileH = 8;
constexpr int kMaxBwdBlocks = 296;      // two resident blocks per SM when the staged batch is 32 cells (C >= 16)

template <int C>
struct BwdCfg {
  static constexpr int NB = (C < 16) ? 64 : 32;    // active cells per staged batch (32: two blocks fit an SM at C = 16)
  static constexpr int NBP = NB + 4;               // padded row stride (floats): conflict-free float4 rows
  static constexpr int TPC = kBThreads / NB;       // threads per cell in the cell-parallel phases
  static constexpr int CQ = C / TPC;               // channels per thread there
  static constexpr int TK = ((3 * C) % 8 == 0) ? (3 * C) / 8 : 3;   // dW1 tile width in k
  static constexpr int KG = (3 * C) / TK;
  static_assert(C % TPC == 0 && CQ >= 1, "channel split");
};

struct BwdArgs {
  StepArgs s;
  const float* gout;        // dL/dx'
  float* gx;                // dL/dx
  const float* u;           // saved masked pre-norm update
  const float* stats;       // saved (mean, rstd) [B][2]
  // scratch
  unsigned char* actmask;   // [B][HW]
  unsigned char* postmask;  // [B][HW]
  float* gz;                // [B][C][HW]   (active cells)
  float* gy;                // [B][3C][HW]  (active cells)
  float* gxs;               // [B][C][HW]   (active cells)
  double* tile_part;        // [B][ntiles][2+2C]
  float* sums;              // [B][2]  S1/N, S2/N
  float* wpart;             // [nblocks][canonical total]
  int ntiles, nblocks, n_items, nchunks, bchunk;
  int64_t wtotal;
  gnca_layout L;
  const float* zp_rowsum;   // row sums of x (zero-padded shift)
  AttnBwdScratch zp_scratch;
  float* gw_part;           // [B][nchunks][GNCA_MAX_K] dL/dw_i partials (zero-padded shift) or null
  const float* grow;        // [B][C][H] additive row term of dL/dx from the attention weights, or null
  const float* gframe;      // [B][C][HW] dL/dx of a recorded frame (the state this step consumes), or null
};

// ------------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(kBThreads) k_bwd_norm(BwdArgs A, Packed P, const float* __restrict__ packed) {
  const StepArgs& a = A.s;
  const int b = blockIdx.y;
  const int H = a.H, W = a.W, HW = H * W;
  const int tiles_x = (W + kBTileW - 1) / kBTileW;
  const int ty0 = (blockIdx.x / tiles_x) * kBTileH, tx0 = (blockIdx.x % tiles_x) * kBTileW;
  const int lx = threadIdx.x % kBTileW, ly = threadIdx.x / kBTileW;
  const int y = ty0 + ly, x = tx0 + lx;
  const bool inside = y < H && x < W;
  double* part = A.tile_part + ((size_t)b * A.ntiles + blockIdx.x) * (2 + 2 * C);
  if (!sample_active(a, b)) {
    if (threadIdx.x < 2 + 2 * C) part[threadIdx.x] = 0.0;
    if (inside) { A.actmask[(size_t)b * HW + y * W + x] = 0; A.postmask[(size_t)b * HW + y * W + x] = 1; }
    return;
  }
  __shared__ float s_sc[C], s_bi[C], s_gam[C], s_idle_th[C];
  __shared__ float s_alpha[kBTileH + 2][kBTileW + 2 + 1];
  __shared__ unsigned char s_act[kBTileH + 2][kBTileW + 2];
  __shared__ double s_red[kBThreads / 32][2 + 2 * C];
  const float fr = step_fire_rate(a);
  const bool gn = (a.flags & GNCA_F_GROUPNORM) != 0;
  const float mu = gn ? A.stats[b * 2] : 0.f, rstd = gn ? A.stats[b * 2 + 1] : 1.f;
  if (threadIdx.x < C) {
    const int c = threadIdx.x;
    float sc = 1.f, bi = 0.f, gam = 1.f;
    if (gn) { gam = packed[P.gamma + c]; sc = rstd * gam; bi = packed[P.beta + c] - mu * sc; }
    s_sc[c] = sc; s_bi[c] = bi; s_gam[c] = gam;
    s_idle_th[c] = tanhf(bi);
  }
  __syncthreads();
  const float* xs_base = a.x_in + (size_t)b * C * HW;
  const float* alpha = xs_base + 3 * HW;
  const float* ub = A.u + (size_t)b * C * HW;
  for (int i = threadIdx.x; i < (kBTileH + 2) * (kBTileW + 2); i += kBThreads) {
    const int hy = i / (kBTileW + 2), hx = i % (kBTileW + 2);
    const int yy = ty0 + hy - 1, xx = tx0 + hx - 1;
    float v = -INFINITY;
    unsigned char act = 0;
    if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
      const int cell = yy * W + xx;
      act = alive_at(alpha, yy, xx, H, W, a.alpha_thr) && fires(a, fr, b, cell);
      v = updated_alpha(alpha[cell], act, act ? ub[3 * HW + cell] : 0.f, s_sc[3], s_bi[3],
                        __fmul_rn(s_idle_th[3], a.update_gain), a.update_gain);
    }
    s_alpha[hy][hx] = v;
    s_act[hy][hx] = act;
  }
  __syncthreads();
  double acc[2 + 2 * C];
#pragma unroll
  for (int i = 0; i < 2 + 2 * C; ++i) acc[i] = 0.0;
  if (inside) {
    const int cell = y * W + x;
    const bool act = s_act[ly + 1][lx + 1] != 0;
    float mx = -INFINITY;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) mx = fmaxf(mx, s_alpha[ly + i][lx + j]);
    const bool post = mx > a.alpha_thr;
    A.actmask[(size_t)b * HW + cell] = act ? 1 : 0;
    A.postmask[(size_t)b * HW + cell] = post ? 1 : 0;
    const float* go = A.gout + (size_t)b * C * HW + cell;
    float s1 = 0.f, s2 = 0.f;
    // all loads of the cell before the first use (one L2 round trip instead of one per channel: the conditional u load
    // made every channel its own basic block); u of an inactive cell is read and dropped
    float gv[C], uv[C];
#pragma unroll
    for (int c = 0; c < C; ++c) { gv[c] = go[(size_t)c * HW]; uv[c] = ub[(size_t)c * HW + cell]; }
#pragma unroll
    for (int c = 0; c < C; ++c) {
      float g = gv[c];
      if (c == 3 && !post) g = 0.f;
      const float uu = act ? uv[c] : 0.f;
      const float th = act ? tanhf(fmaf(uu, s_sc[c], s_bi[c])) : s_idle_th[c];
      const float gz = g * a.update_gain * (1.f - th * th);
      if (act) A.gz[((size_t)b * C + c) * HW + cell] = gz;
      if (gn) {
        const float uh = (uu - mu) * rstd;
        const float gu = gz * s_gam[c];
        s1 += gu;
        s2 = fmaf(gu, uh, s2);
        acc[2 + c] = (double)(gz * uh);
        acc[2 + C + c] = (double)gz;
      }
    }
    acc[0] = (double)s1; acc[1] = (double)s2;
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int i = 0; i < 2 + 2 * C; ++i) {
    const double v = warp_sum(acc[i]);
    if (lane == 0) s_red[warp][i] = v;
  }
  __syncthreads();
  if (threadIdx.x < 2 + 2 * C) {
    double t = 0.0;
    for (int w = 0; w < kBThreads / 32; ++w) t += s_red[w][threadIdx.x];
    part[threadIdx.x] = t;
  }
}

// one block per sample (blockDim >= 2+2C): deterministic reduction over tiles
template <int C>
__global__ void k_bwd_stats(BwdArgs A, float* __restrict__ gparams) {
  const int b = blockIdx.x;
  const StepArgs& a = A.s;
  __shared__ double s_dg[2 * C];
  const int i = threadIdx.x;
  if (i < 2 + 2 * C) {
    double t = 0.0;
    for (int tl = 0; tl < A.ntiles; ++tl) t += A.tile_part[((size_t)b * A.ntiles + tl) * (2 + 2 * C) + i];
    if (i < 2) {
      const double n = (double)C * (double)a.H * (double)a.W;
      A.sums[b * 2 + i] = (float)(t / n);
    } else {
      // per-sample dgamma/dbeta go to a per-sample slot; summed over samples (in order) by block 0 below
      A.tile_part[((size_t)b * A.ntiles) * (2 + 2 * C) + i] = t;
    }
  }
  (void)s_dg; (void)gparams;
}

template <int C>
__global__ void k_bwd_affine_reduce(BwdArgs A, float* __restrict__ gparams) {
  const int i = threadIdx.x;   // 0..2C-1
  if (i >= 2 * C) return;
  if (!(A.s.flags & GNCA_F_GROUPNORM)) return;
  double t = 0.0;
  for (int b = 0; b < A.s.B; ++b) t += A.tile_part[((size_t)b * A.ntiles) * (2 + 2 * C) + 2 + i];
  const int64_t dst = (i < C) ? A.L.gamma + i : A.L.beta + (i - C);
  gparams[dst] += (float)t;
}

// ------------------------------------------------------------------------------------------------
// Shared-memory plan of k_bwd_mlp.  WG = false stages W1T and W1 next to W2; WG = true reads those two from global memory
// (L1-cached), for the C = 32 models with a hidden layer wide enough (>= 164 graph, >= 180 classic) that the staged plan
// exceeds the 226 KB a block may use.
template <int C>
struct BwdSmem {
  using K = BwdCfg<C>;
  static size_t floats(int hid, bool graph, bool wg) {
    size_t f = (wg ? 0 : (size_t)2 * 3 * C * hid) + pad4(hid) + (size_t)C * hid;            // [W1T, W1,] b1, W2
    f += C;                                                                                // gamma
    if (graph) f += C * C + C;                                                             // Wm, bm
    f += (size_t)(3 * C + C + 2 * hid) * K::NBP;                                           // Yt, GDt, Ht, GHt
    if (graph) f += (size_t)(3 * C + 2) * K::NBP;                                          // XSt, GAt, GXSt, AS, GB
    return f;
  }
  static size_t bytes(int hid, bool graph, bool wg) {
    return floats(hid, graph, wg) * sizeof(float) + kBChunk * sizeof(uint16_t) + K::NB * sizeof(int);
  }
};

constexpr size_t kBwdSmemLimit = 226 * 1024;

// Accumulation into a partial that ONE thread owns (this block's weight-gradient slot / this chunk's dL/dw slot): a
// reduction without return value instead of load - add - store.  The thread does not wait for the L2 round trip (the
// read-modify-writes of a batch held 18 % of the kernel's stall samples and the block barrier behind them another 19 %),
// and the result is the same sequence of fp32 additions: operations of one thread on one address stay in program order
// (the instruction is REDG.E.ADD.F32.FTZ.RN: round to nearest like the FADD it replaces; subnormal sums flush to zero).
__device__ __forceinline__ void red_add(float* p, float v) {
  asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}

__device__ __forceinline__ float dot4(const float4& a, const float4& b) {
  return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, a.w * b.w)));
}

template <int C, int CH, bool WG>
__global__ void __launch_bounds__(kBThreads, 2) k_bwd_mlp(BwdArgs A, Packed P, int hid, const float* __restrict__ packed) {
  using K = BwdCfg<C>;
  constexpr int NB = K::NB, NBP = K::NBP, TPC = K::TPC, CQ = K::CQ, C3 = 3 * C;
  const StepArgs& a = A.s;
  const int H = a.H, W = a.W, HW = H * W;
  const bool graph = (a.flags & GNCA_F_GRAPH) != 0;
  const bool gn = (a.flags & GNCA_F_GROUPNORM) != 0;
  const bool torus = (a.flags & GNCA_F_TORUS) != 0;
  const bool a2a = (a.flags & GNCA_F_ALIVE_TO_ALIVE) != 0;
  const float gain_m = graph ? step_message_gain(a) : 0.f;
  const bool msg_on = graph && gain_m != 0.f && a.k > 0;
  const int c_lo = ((a.flags & GNCA_F_HIDDEN_ONLY) && C >= 4) ? 4 : 0;

  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* sW1T = reinterpret_cast<float*>(smem_raw);
  float* sb1 = sW1T + (WG ? 0 : C3 * hid);
  float* sW2 = sb1 + pad4(hid);
  float* sW1 = sW2 + C * hid;
  float* sgam = sW1 + (WG ? 0 : hid * C3);
  // W1T / W1 rows as float4: shared memory, or the packed buffer in global memory (WG)
  const float* W1T = WG ? packed + P.w1t : sW1T;
  const float* W1 = WG ? packed + P.w1 : sW1;
  auto w4 = [](const float* p) -> float4 {
    if constexpr (WG) return __ldg(reinterpret_cast<const float4*>(p));
    else return *reinterpret_cast<const float4*>(p);
  };
  float* sWm = sgam + C;
  float* sbm = sWm + (graph ? C * C : 0);
  float* Yt = sbm + (graph ? C : 0);
  float* GDt = Yt + C3 * NBP;
  float* Ht = GDt + C * NBP;
  float* GHt = Ht + hid * NBP;
  float* XSt = GHt + hid * NBP;
  float* GAt = XSt + (graph ? C * NBP : 0);
  float* GXSt = GAt + (graph ? C * NBP : 0);
  float* AS = GXSt + (graph ? C * NBP : 0);
  float* GB = AS + (graph ? NBP : 0);
  float* endf = GB + (graph ? NBP : 0);
  uint16_t* slist = reinterpret_cast<uint16_t*>(endf);
  int* scell = reinterpret_cast<int*>(slist + kBChunk);
  __shared__ int s_nact;
  __shared__ int swcount[kBThreads / 32], swbase[kBThreads / 32 + 1];
  __shared__ int s_ody[GNCA_MAX_K], s_odx[GNCA_MAX_K];      // the step's sender offsets (reduced modulo the grid on a torus)
  __shared__ float s_owt[GNCA_MAX_K];                        // and the sample's weights

  if (!WG) block_copy(sW1T, packed + P.w1t, C3 * hid);
  block_copy(sb1, packed + P.b1, pad4(hid));
  block_copy(sW2, packed + P.w2, C * hid);
  if (!WG) block_copy(sW1, packed + P.w1, hid * C3);
  if (threadIdx.x < C) sgam[threadIdx.x] = packed[P.gamma + threadIdx.x];
  if (graph) { block_copy(sWm, packed + P.wm, C * C); block_copy(sbm, packed + P.bm, C); }
  __syncthreads();

  float* wp = A.wpart + (size_t)blockIdx.x * A.wtotal;   // this block's weight-gradient partial (pre-zeroed)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cell_l = threadIdx.x / TPC, part = threadIdx.x % TPC;

  for (int item = blockIdx.x; item < A.n_items; item += gridDim.x) {
    const int b = item / A.nchunks, chunk = item % A.nchunks;
    if (!sample_active(a, b)) continue;
    const float* xs_base = a.x_in + (size_t)b * C * HW;
    const unsigned char* am = A.actmask + (size_t)b * HW;
    const int cell0 = chunk * CH;
    // ---- compaction of the chunk's active cells (same deterministic order as the forward) ----------
    {
      constexpr int kPerWarp = CH / (kBThreads / 32);
      uint32_t bal[kPerWarp / 32];
      int cnt = 0;
#pragma unroll
      for (int it = 0; it < kPerWarp / 32; ++it) {
        const int cell = cell0 + warp * kPerWarp + it * 32 + lane;
        const bool act = cell < HW && am[cell] != 0;
        bal[it] = __ballot_sync(0xffffffffu, act);
        cnt += __popc(bal[it]);
      }
      __syncthreads();   // previous item fully consumed slist / swbase
      if (msg_on && threadIdx.x < a.k) {
        int dy, dx;
        step_offset(a, threadIdx.x, dy, dx);
        s_ody[threadIdx.x] = torus ? dy % H : dy;
        s_odx[threadIdx.x] = torus ? dx % W : 0;
        s_owt[threadIdx.x] = a.attn_w ? __ldg(a.attn_w + (size_t)b * a.k + threadIdx.x) : 1.0f / (float)a.k;
      }
      if (lane == 0) swcount[warp] = cnt;
      __syncthreads();
      if (threadIdx.x == 0) {
        int s = 0;
        for (int w = 0; w < kBThreads / 32; ++w) { swbase[w] = s; s += swcount[w]; }
        swbase[kBThreads / 32] = s;
        s_nact = s;
      }
      __syncthreads();
      int base = swbase[warp];
#pragma unroll
      for (int it = 0; it < kPerWarp / 32; ++it) {
        if (bal[it] & (1u << lane))
          slist[base + __popc(bal[it] & ((1u << lane) - 1u))] = (uint16_t)(warp * kPerWarp + it * 32 + lane);
        base += __popc(bal[it]);
      }
      __syncthreads();
    }
    const int nact = s_nact;
    const float mu = gn ? A.stats[b * 2] : 0.f, rstd = gn ? A.stats[b * 2 + 1] : 1.f;
    const float s1n = gn ? A.sums[b * 2] : 0.f, s2n = gn ? A.sums[b * 2 + 1] : 0.f;

    for (int base = 0; base < nact; base += NB) {
      const int nb = min(NB, nact - base);
      // ---- (a) stage y, gd (and the gathered sender state) ------------------------------------------
      float gdv[CQ];
      {
        const bool valid = cell_l < nb;
        int cell = 0, y = 0, x = 0;
        if (valid) { cell = cell0 + (int)slist[base + cell_l]; y = cell / W; x = cell - y * W; }
        if (part == 0 && cell_l < NB) scell[cell_l] = valid ? cell : -1;
        // All loads of the phase are requested before the first use, without branches (the edge taps of the perception
        // and of the senders' alive windows come from a clamped address; an idle lane reads cell 0 and drops it): the
        // original per-channel / per-sender basic blocks paid ~2 k dependent L2 round trips per batch.
        const bool up = y > 0, dn = y < H - 1, lf = x > 0, rt = x < W - 1;
        const int oU = up ? -W : 0, oD = dn ? W : 0, oL = lf ? -1 : 0, oR = rt ? 1 : 0;
        float pv[CQ][9], gzv[CQ], uv[CQ];
#pragma unroll
        for (int cc = 0; cc < CQ; ++cc) {
          const int c = part * CQ + cc;
          const float* p = xs_base + (size_t)c * HW + cell;
          pv[cc][0] = __ldg(p + (oU + oL)); pv[cc][1] = __ldg(p + oU); pv[cc][2] = __ldg(p + (oU + oR));
          pv[cc][3] = __ldg(p + oL);        pv[cc][4] = __ldg(p);      pv[cc][5] = __ldg(p + oR);
          pv[cc][6] = __ldg(p + (oD + oL)); pv[cc][7] = __ldg(p + oD); pv[cc][8] = __ldg(p + (oD + oR));
          gzv[cc] = A.gz[((size_t)b * C + c) * HW + cell];
          uv[cc] = gn ? A.u[((size_t)b * C + c) * HW + cell] : 0.f;
        }
#pragma unroll
        for (int cc = 0; cc < CQ; ++cc) {
          const int c = part * CQ + cc;
          float vid = 0.f, vsx = 0.f, vsy = 0.f, gd = 0.f;
          if (valid) {
            const float a00 = (up && lf) ? pv[cc][0] : 0.f, a01 = up ? pv[cc][1] : 0.f, a02 = (up && rt) ? pv[cc][2] : 0.f;
            const float a10 = lf ? pv[cc][3] : 0.f, a12 = rt ? pv[cc][5] : 0.f;
            const float a20 = (dn && lf) ? pv[cc][6] : 0.f, a21 = dn ? pv[cc][7] : 0.f, a22 = (dn && rt) ? pv[cc][8] : 0.f;
            vid = pv[cc][4];
            vsx = (a00 - a02) + 2.f * (a10 - a12) + (a20 - a22);
            vsy = (a00 + 2.f * a01 + a02) - (a20 + 2.f * a21 + a22);
            const float gz = gzv[cc];
            if (gn) {
              const float uh = (uv[cc] - mu) * rstd;
              gd = rstd * (gz * sgam[c] - s1n - uh * s2n);
            } else {
              gd = gz;
            }
          }
          Yt[c * NBP + cell_l] = vid;
          Yt[(C + c) * NBP + cell_l] = vsx;
          Yt[(2 * C + c) * NBP + cell_l] = vsy;
          GDt[c * NBP + cell_l] = gd;
          gdv[cc] = gd;
        }
        if (msg_on) {
          float xsv[CQ];
#pragma unroll
          for (int cc = 0; cc < CQ; ++cc) xsv[cc] = 0.f;
          float as = 0.f;
          const float* alpha = xs_base + 3 * HW;
          constexpr int SB = 4;                                  // senders per round
#pragma unroll 1
          for (int i0 = 0; i0 < a.k; i0 += SB) {
            float w[SB], v[SB][CQ], al[SB][9];
            int qy[SB], qx[SB];
#pragma unroll
            for (int sI = 0; sI < SB; ++sI) {
              const int ii = min(i0 + sI, a.k - 1);
              const int dy = s_ody[ii], dx = s_odx[ii];
              int yy = y - dy, xx = torus ? x - dx : x;
              bool ok = valid && i0 + sI < a.k;
              if (torus) {
                yy = yy < 0 ? yy + H : (yy >= H ? yy - H : yy);
                xx = xx < 0 ? xx + W : (xx >= W ? xx - W : xx);
              } else {
                ok = ok && yy >= 0 && yy < H;
                yy = ok ? yy : y;
              }
              qy[sI] = yy; qx[sI] = xx;
              w[sI] = ok ? s_owt[ii] : 0.f;
            }
#pragma unroll
            for (int sI = 0; sI < SB; ++sI) {
#pragma unroll
              for (int cc = 0; cc < CQ; ++cc)
                v[sI][cc] = __ldg(xs_base + (size_t)(part * CQ + cc) * HW + qy[sI] * W + qx[sI]);
            }
            if (a2a) {
#pragma unroll
              for (int sI = 0; sI < SB; ++sI) {
                const int ru = (qy[sI] > 0 ? qy[sI] - 1 : qy[sI]) * W, rc = qy[sI] * W, rd = (qy[sI] < H - 1 ? qy[sI] + 1 : qy[sI]) * W;
                const int xl = qx[sI] > 0 ? qx[sI] - 1 : qx[sI], xc = qx[sI], xr = qx[sI] < W - 1 ? qx[sI] + 1 : qx[sI];
                al[sI][0] = __ldg(alpha + ru + xl); al[sI][1] = __ldg(alpha + ru + xc); al[sI][2] = __ldg(alpha + ru + xr);
                al[sI][3] = __ldg(alpha + rc + xl); al[sI][4] = __ldg(alpha + rc + xc); al[sI][5] = __ldg(alpha + rc + xr);
                al[sI][6] = __ldg(alpha + rd + xl); al[sI][7] = __ldg(alpha + rd + xc); al[sI][8] = __ldg(alpha + rd + xr);
              }
            }
#pragma unroll
            for (int sI = 0; sI < SB; ++sI) {
              float ww = w[sI];
              if (a2a) {
                const float m = fmaxf(fmaxf(fmaxf(fmaxf(al[sI][0], al[sI][1]), fmaxf(al[sI][2], al[sI][3])),
                                            fmaxf(fmaxf(al[sI][4], al[sI][5]), fmaxf(al[sI][6], al[sI][7]))), al[sI][8]);
                ww = m > a.graph_alpha_thr ? ww : 0.f;
              }
#pragma unroll
              for (int cc = 0; cc < CQ; ++cc) xsv[cc] = fmaf(ww, v[sI][cc], xsv[cc]);
              as += ww;
            }
          }
#pragma unroll
          for (int cc = 0; cc < CQ; ++cc) XSt[(part * CQ + cc) * NBP + cell_l] = xsv[cc];
          if (part == 0) AS[cell_l] = as;
        }
      }
      __syncthreads();
      // ---- (b1) message: agg = Wm xs + bm as ; g_agg = gd * gain * (1 - tanh^2 agg) on the gated channels ---
      if (msg_on) {
#pragma unroll
        for (int cc = 0; cc < CQ; ++cc) {
          const int c = part * CQ + cc;
          float agg = sbm[c] * AS[cell_l];
          for (int ci = 0; ci < C; ++ci) agg = fmaf(sWm[c * C + ci], XSt[ci * NBP + cell_l], agg);
          const float t = tanhf(agg);
          GAt[c * NBP + cell_l] = (c >= c_lo) ? gdv[cc] * gain_m * (1.f - t * t) : 0.f;
        }
      }
      // ---- (b2) G1: h = relu(Y W1^T + b1) ; G2: gh = (GD W2) * [h > 0]  -> Ht, GHt ----------------------
      {
        constexpr int CG = NB / 4, JG = kBThreads / CG;
        const int cg = threadIdx.x % CG, jg0 = threadIdx.x / CG;
        for (int jt = jg0; jt * 4 < hid; jt += JG) {
          const int j = jt * 4;
          float acc[4][4];
          const float4 bb = *reinterpret_cast<const float4*>(sb1 + j);
#pragma unroll
          for (int m = 0; m < 4; ++m) { acc[m][0] = bb.x; acc[m][1] = bb.y; acc[m][2] = bb.z; acc[m][3] = bb.w; }
#pragma unroll 4
          for (int k = 0; k < C3; ++k) {
            const float4 yv = *reinterpret_cast<const float4*>(Yt + k * NBP + 4 * cg);
            const float4 w = w4(W1T + k * hid + j);
            const float ym[4] = {yv.x, yv.y, yv.z, yv.w};
#pragma unroll
            for (int m = 0; m < 4; ++m) {
              acc[m][0] = fmaf(ym[m], w.x, acc[m][0]); acc[m][1] = fmaf(ym[m], w.y, acc[m][1]);
              acc[m][2] = fmaf(ym[m], w.z, acc[m][2]); acc[m][3] = fmaf(ym[m], w.w, acc[m][3]);
            }
          }
          float g2[4][4];
#pragma unroll
          for (int m = 0; m < 4; ++m)
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) g2[m][jj] = 0.f;
#pragma unroll 4
          for (int c = 0; c < C; ++c) {
            const float4 gv = *reinterpret_cast<const float4*>(GDt + c * NBP + 4 * cg);
            const float4 w = *reinterpret_cast<const float4*>(sW2 + c * hid + j);
            const float gm[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
            for (int m = 0; m < 4; ++m) {
              g2[m][0] = fmaf(gm[m], w.x, g2[m][0]); g2[m][1] = fmaf(gm[m], w.y, g2[m][1]);
              g2[m][2] = fmaf(gm[m], w.z, g2[m][2]); g2[m][3] = fmaf(gm[m], w.w, g2[m][3]);
            }
          }
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            float4 hv, gv;
            hv.x = fmaxf(acc[0][jj], 0.f); hv.y = fmaxf(acc[1][jj], 0.f);
            hv.z = fmaxf(acc[2][jj], 0.f); hv.w = fmaxf(acc[3][jj], 0.f);
            gv.x = acc[0][jj] > 0.f ? g2[0][jj] : 0.f; gv.y = acc[1][jj] > 0.f ? g2[1][jj] : 0.f;
            gv.z = acc[2][jj] > 0.f ? g2[2][jj] : 0.f; gv.w = acc[3][jj] > 0.f ? g2[3][jj] : 0.f;
            *reinterpret_cast<float4*>(Ht + (j + jj) * NBP + 4 * cg) = hv;
            *reinterpret_cast<float4*>(GHt + (j + jj) * NBP + 4 * cg) = gv;
          }
        }
      }
      __syncthreads();
      // ---- (c1) G3: gy = GH W1  -> global gy (active cells) ------------------------------------------------
      {
        constexpr int CG = NB / 4, KQ = C3 / 4;
        for (int tile = threadIdx.x; tile < CG * KQ; tile += kBThreads) {
          const int cg = tile % CG, kq = tile / CG;
          float acc[4][4];
#pragma unroll
          for (int m = 0; m < 4; ++m)
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) acc[m][kk] = 0.f;
#pragma unroll 4
          for (int j = 0; j < hid; ++j) {
            const float4 gv = *reinterpret_cast<const float4*>(GHt + j * NBP + 4 * cg);
            const float4 w = w4(W1 + j * C3 + 4 * kq);
            const float gm[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
            for (int m = 0; m < 4; ++m) {
              acc[m][0] = fmaf(gm[m], w.x, acc[m][0]); acc[m][1] = fmaf(gm[m], w.y, acc[m][1]);
              acc[m][2] = fmaf(gm[m], w.z, acc[m][2]); acc[m][3] = fmaf(gm[m], w.w, acc[m][3]);
            }
          }
#pragma unroll
          for (int m = 0; m < 4; ++m) {
            const int cl = 4 * cg + m;
            if (cl >= nb) continue;
            float* gyp = A.gy + ((size_t)b * C3 + 4 * kq) * HW + scell[cl];
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) gyp[(size_t)kk * HW] = acc[m][kk];
          }
        }
      }
      // ---- (c2) G4: dW1 += GH^T Y, db1 += colsum(GH) -------------------------------------------------------
      {
        constexpr int TK = K::TK, KG = K::KG;
        const int JQ = hid / 4;
        for (int tile = threadIdx.x; tile < JQ * KG; tile += kBThreads) {
          const int kg = tile % KG, jg = tile / KG;
          float acc[4][TK];
          float accb[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int jj = 0; jj < 4; ++jj)
#pragma unroll
            for (int kk = 0; kk < TK; ++kk) acc[jj][kk] = 0.f;
          for (int c4 = 0; c4 < NB / 4; ++c4) {
            float4 g[4];
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) g[jj] = *reinterpret_cast<const float4*>(GHt + (jg + JQ * jj) * NBP + 4 * c4);
#pragma unroll
            for (int kk = 0; kk < TK; ++kk) {
              const float4 yv = *reinterpret_cast<const float4*>(Yt + (kg + KG * kk) * NBP + 4 * c4);
#pragma unroll
              for (int jj = 0; jj < 4; ++jj) acc[jj][kk] += dot4(g[jj], yv);
            }
            if (kg == 0) {
#pragma unroll
              for (int jj = 0; jj < 4; ++jj) accb[jj] += (g[jj].x + g[jj].y) + (g[jj].z + g[jj].w);
            }
          }
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            const int j = jg + JQ * jj;
#pragma unroll
            for (int kk = 0; kk < TK; ++kk) red_add(wp + A.L.w1 + (int64_t)j * C3 + (kg + KG * kk), acc[jj][kk]);
            if (kg == 0) red_add(wp + A.L.b1 + j, accb[jj]);
          }
        }
      }
      // ---- (c3) G5: dW2 += GD^T H ----------------------------------------------------------------------------
      {
        const int JQ = hid / 4;
        constexpr int CQ4 = C / 4;
        for (int tile = threadIdx.x; tile < JQ * CQ4; tile += kBThreads) {
          const int cq = tile % CQ4, jg = tile / CQ4;
          float acc[4][4];
#pragma unroll
          for (int cc = 0; cc < 4; ++cc)
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) acc[cc][jj] = 0.f;
          for (int c4 = 0; c4 < NB / 4; ++c4) {
            float4 hh[4];
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) hh[jj] = *reinterpret_cast<const float4*>(Ht + (jg + JQ * jj) * NBP + 4 * c4);
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
              const float4 gv = *reinterpret_cast<const float4*>(GDt + (cq + CQ4 * cc) * NBP + 4 * c4);
#pragma unroll
              for (int jj = 0; jj < 4; ++jj) acc[cc][jj] += dot4(gv, hh[jj]);
            }
          }
#pragma unroll
          for (int cc = 0; cc < 4; ++cc)
#pragma unroll
            for (int jj = 0; jj < 4; ++jj)
              red_add(wp + A.L.w2 + (int64_t)(cq + CQ4 * cc) * hid + (jg + JQ * jj), acc[cc][jj]);
        }
      }
      // ---- (c4) message weight grads and g_xs = Wm^T g_agg -> global (active receivers) -----------------------
      if (msg_on) {
        for (int idx = threadIdx.x; idx < C * C + C; idx += kBThreads) {
          float acc = 0.f;
          if (idx < C * C) {
            const int co = idx / C, ci = idx % C;
            for (int cl = 0; cl < nb; ++cl) acc = fmaf(GAt[co * NBP + cl], XSt[ci * NBP + cl], acc);
            red_add(wp + A.L.wm + idx, acc);
          } else {
            const int c = idx - C * C;
            for (int cl = 0; cl < nb; ++cl) acc = fmaf(GAt[c * NBP + cl], AS[cl], acc);
            red_add(wp + A.L.bm + c, acc);
          }
        }
        for (int idx = threadIdx.x; idx < NB * C; idx += kBThreads) {
          const int cl = idx % NB, ci = idx / NB;
          float v = 0.f;
          if (cl < nb) {
#pragma unroll 4
            for (int co = 0; co < C; ++co) v = fmaf(sWm[co * C + ci], GAt[co * NBP + cl], v);
            A.gxs[((size_t)b * C + ci) * HW + scell[cl]] = v;
          }
          GXSt[ci * NBP + cl] = v;
        }
        if (A.gw_part) {   // zero-padded shift: dL/dw_i += sum_p [ g_xs(p) . A x(q_i(p)) + (bm . g_agg(p)) A(q_i(p)) ]
          for (int cl = threadIdx.x; cl < NB; cl += kBThreads) {
            float gb = 0.f;
            for (int c = 0; c < C; ++c) gb = fmaf(sbm[c], GAt[c * NBP + cl], gb);
            GB[cl] = gb;
          }
          __syncthreads();        // GB / GXSt are complete and every thread is past (c3): Ht is free until the next batch
          // one (receiver, offset) pair per thread -- 8 threads walking 64 receivers each with two dependent global
          // round trips per receiver held the whole block at a barrier for ~100 k cycles --, then the same fixed-order
          // sum over the receivers as before (a skipped pair adds an exact 0)
          float* PV = Ht;         // [kcap][NB] over Ht | GHt (2 * hid * NBP floats)
          const int kcap = (2 * hid * NBP) / NB;
          for (int o0 = 0; o0 < a.k; o0 += kcap) {
            const int kc = min(kcap, a.k - o0);
            for (int idx = threadIdx.x; idx < kc * NB; idx += kBThreads) {
              const int cl = idx % NB, oi = o0 + idx / NB;
              float v = 0.f;
              if (cl < nb) {
                int dy, dx, qy, qx;
                step_offset(a, oi, dy, dx);
                const int pc = scell[cl], py = pc / W, px = pc - py * W;
                if (sender_of(py, px, dy, dx, H, W, torus, qy, qx) &&
                    !(a2a && !alive_at(xs_base + 3 * HW, qy, qx, H, W, a.graph_alpha_thr))) {
                  float xq[C];
#pragma unroll
                  for (int c = 0; c < C; ++c) xq[c] = __ldg(xs_base + (size_t)c * HW + qy * W + qx);
                  v = GB[cl];
#pragma unroll
                  for (int c = 0; c < C; ++c) v = fmaf(GXSt[c * NBP + cl], xq[c], v);
                }
              }
              PV[idx] = v;
            }
            __syncthreads();
            for (int oi = threadIdx.x; oi < kc; oi += kBThreads) {
              float acc = 0.f;
              for (int cl = 0; cl < nb; ++cl) acc += PV[oi * NB + cl];
              red_add(A.gw_part + ((size_t)b * A.nchunks + chunk) * GNCA_MAX_K + o0 + oi, acc);
            }
            if (o0 + kcap < a.k) __syncthreads();
          }
        }
      }
      __syncthreads();
    }
  }
}

// ------------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(256) k_bwd_gather(BwdArgs A) {
  const StepArgs& a = A.s;
  const int b = blockIdx.y, H = a.H, W = a.W, HW = H * W;
  const int cell = blockIdx.x * blockDim.x + threadIdx.x;
  if (cell >= HW) return;
  const float* go = A.gout + (size_t)b * C * HW + cell;
  float* gxp = A.gx + (size_t)b * C * HW + cell;
  const float* gf = A.gframe ? A.gframe + (size_t)b * C * HW + cell : nullptr;
  if (!sample_active(a, b)) {
#pragma unroll
    for (int c = 0; c < C; ++c) gxp[(size_t)c * HW] = gf ? go[(size_t)c * HW] + gf[(size_t)c * HW] : go[(size_t)c * HW];
    return;
  }
  const int y = cell / W, x = cell - y * W;
  const unsigned char* am = A.actmask + (size_t)b * HW;
  const bool post = A.postmask[(size_t)b * HW + cell] != 0;
  float g[C];
#pragma unroll
  for (int c = 0; c < C; ++c) g[c] = go[(size_t)c * HW];
  if (!post) g[3] = 0.f;
  // perception transpose: output cells n = (y-i, x-j) whose stencil tap (i,j) read this cell
  const float kx[3][3] = {{1.f, 0.f, -1.f}, {2.f, 0.f, -2.f}, {1.f, 0.f, -1.f}};
  const float ky[3][3] = {{1.f, 2.f, 1.f}, {0.f, 0.f, 0.f}, {-1.f, -2.f, -1.f}};
  const float* gyb = A.gy + (size_t)b * 3 * C * HW;
#pragma unroll
  for (int i = -1; i <= 1; ++i) {
#pragma unroll
    for (int j = -1; j <= 1; ++j) {
      const int yy = y - i, xx = x - j;
      if (yy < 0 || yy >= H || xx < 0 || xx >= W) continue;
      const int n = yy * W + xx;
      if (!am[n]) continue;
      const float wx = kx[i + 1][j + 1], wy = ky[i + 1][j + 1];
#pragma unroll
      for (int c = 0; c < C; ++c) {
        float v = g[c];
        if (i == 0 && j == 0) v += gyb[(size_t)c * HW + n];
        if (wx != 0.f) v = fmaf(wx, gyb[(size_t)(C + c) * HW + n], v);
        if (wy != 0.f) v = fmaf(wy, gyb[(size_t)(2 * C + c) * HW + n], v);
        g[c] = v;
      }
    }
  }
  // message transpose: receivers p with sender_of(p, offset i) == this cell
  const bool graph = (a.flags & GNCA_F_GRAPH) != 0;
  const float gain_m = graph ? step_message_gain(a) : 0.f;
  if (graph && gain_m != 0.f && a.k > 0) {
    const bool torus = (a.flags & GNCA_F_TORUS) != 0;
    const float* xs_base = a.x_in + (size_t)b * C * HW;
    if (!(a.flags & GNCA_F_ALIVE_TO_ALIVE) || alive_at(xs_base + 3 * HW, y, x, H, W, a.graph_alpha_thr)) {
      const float wuni = 1.0f / (float)a.k;
      const float* gxsb = A.gxs + (size_t)b * C * HW;
      for (int i = 0; i < a.k; ++i) {
        int dy, dx;
        step_offset(a, i, dy, dx);
        int py, px;
        if (torus) {
          py = ((y + dy) % H + H) % H;
          px = ((x + dx) % W + W) % W;
        } else {
          py = y + dy; px = x;
          if (py < 0 || py >= H) continue;
        }
        const int pc = py * W + px;
        if (!am[pc]) continue;
        const float w = a.attn_w ? a.attn_w[(size_t)b * a.k + i] : wuni;
#pragma unroll
        for (int c = 0; c < C; ++c) g[c] = fmaf(w, gxsb[(size_t)c * HW + pc], g[c]);
      }
    }
  }
  if (A.grow) {
#pragma unroll
    for (int c = 0; c < C; ++c) g[c] += A.grow[((size_t)b * C + c) * H + y];
  }
  if (gf) {
#pragma unroll
    for (int c = 0; c < C; ++c) g[c] += gf[(size_t)c * HW];
  }
#pragma unroll
  for (int c = 0; c < C; ++c) gxp[(size_t)c * HW] = g[c];
}

__global__ void k_bwd_reduce(int nblocks, int64_t total, const float* __restrict__ wpart, float* __restrict__ gparams) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int bk = 0; bk < nblocks; ++bk) s += wpart[(size_t)bk * total + i];
    gparams[i] += s;
  }
}

// ------------------------------------------------------------------------------------------------
// host
// ------------------------------------------------------------------------------------------------
static inline size_t align_up_b(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct BwdWorkspace {
  unsigned char *actmask, *postmask;
  float *gz, *gy, *gxs, *sums, *wpart;
  double* tile_part;
  size_t bytes;
  size_t wpart_bytes;
  AttnBwdScratch attn;
  size_t gw_bytes;
};

static BwdWorkspace carve_bwd(void* base, const gnca_model& m, int B, int H, int W) {
  BwdWorkspace w;
  const size_t HW = (size_t)H * W;
  const int ntiles = ((W + kBTileW - 1) / kBTileW) * ((H + kBTileH - 1) / kBTileH);
  const gnca_layout L = make_layout(m);
  char* p = reinterpret_cast<char*>(base);
  size_t o = 0;
  w.actmask = reinterpret_cast<unsigned char*>(p + o); o = align_up_b(o + B * HW, 256);
  w.postmask = reinterpret_cast<unsigned char*>(p + o); o = align_up_b(o + B * HW, 256);
  w.gz = reinterpret_cast<float*>(p + o); o = align_up_b(o + (size_t)B * m.C * HW * 4, 256);
  w.gy = reinterpret_cast<float*>(p + o); o = align_up_b(o + (size_t)B * 3 * m.C * HW * 4, 256);
  w.gxs = reinterpret_cast<float*>(p + o); o = align_up_b(o + (size_t)B * m.C * HW * 4, 256);
  w.tile_part = reinterpret_cast<double*>(p + o); o = align_up_b(o + (size_t)B * ntiles * (2 + 2 * m.C) * 8, 256);
  w.sums = reinterpret_cast<float*>(p + o); o = align_up_b(o + (size_t)B * 2 * 4, 256);
  w.wpart = reinterpret_cast<float*>(p + o);
  w.wpart_bytes = (size_t)kMaxBwdBlocks * L.total * 4;
  o = align_up_b(o + w.wpart_bytes, 256);
  const int nchunks = (H * W + kBChunkSmall - 1) / kBChunkSmall;   // sized for the small chunk
  w.attn = carve_attn_bwd(p + o, m, B, H, nchunks);
  w.gw_bytes = (size_t)B * nchunks * GNCA_MAX_K * 4;
  o += ((m.flags & GNCA_F_GRAPH) ? attn_bwd_scratch_bytes(m, B, H, nchunks) : 0);
  w.bytes = o;
  return w;
}

size_t bwd_workspace_bytes(const gnca_model& m, int B, int H, int W) { return carve_bwd(nullptr, m, B, H, W).bytes; }

// persistent blocks: as many as are resident at once (two per SM when the shared memory of a block allows it)
template <int C, int CH, bool WG>
static int launch_bwd_mlp(const gnca_model& m, const Packed& P, const float* packed, const BwdArgs& A, size_t smem,
                          cudaStream_t st) {
  static int n_sm = 0;
  if (n_sm == 0) {
    int dev = 0;
    GNCA_CHECK_CUDA(cudaGetDevice(&dev));
    GNCA_CHECK_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  }
  int per_sm = 1;
  GNCA_CHECK_CUDA(cudaFuncSetAttribute(k_bwd_mlp<C, CH, WG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_bwd_mlp<C, CH, WG>, kBThreads, smem) != cudaSuccess || per_sm < 1) { cudaGetLastError(); per_sm = 1; }
  const int nblk = min(A.n_items, min(kMaxBwdBlocks, per_sm * n_sm));
  k_bwd_mlp<C, CH, WG><<<nblk, kBThreads, smem, st>>>(A, P, m.hidden, packed);
  return 0;
}

template <int C>
static int launch_step_bwd(const gnca_model& m, const Packed& P, const float* packed, BwdArgs& A, float* gparams,
                           cudaStream_t st) {
  const StepArgs& a = A.s;
  const bool graph = (m.flags & GNCA_F_GRAPH) != 0;
  // the shared-memory plan is settled before the first launch: a rejected configuration leaves gparams untouched
  const bool wg = BwdSmem<C>::bytes(m.hidden, graph, false) > kBwdSmemLimit;
  const size_t smem = BwdSmem<C>::bytes(m.hidden, graph, wg);
  if (smem > kBwdSmemLimit) return GNCA_ERR_UNSUPPORTED;
  dim3 g1(A.ntiles, a.B);
  k_bwd_norm<C><<<g1, kBThreads, 0, st>>>(A, P, packed);
  GNCA_LAUNCH_CHECK();
  k_bwd_stats<C><<<a.B, 128, 0, st>>>(A, gparams);
  GNCA_LAUNCH_CHECK();
  k_bwd_affine_reduce<C><<<1, 64, 0, st>>>(A, gparams);
  GNCA_LAUNCH_CHECK();
  prof_begin(PROF_BWD_MLP, st);
  int rc;
  if (A.bchunk == kBChunkSmall)
    rc = wg ? launch_bwd_mlp<C, kBChunkSmall, true>(m, P, packed, A, smem, st)
            : launch_bwd_mlp<C, kBChunkSmall, false>(m, P, packed, A, smem, st);
  else
    rc = wg ? launch_bwd_mlp<C, kBChunk, true>(m, P, packed, A, smem, st)
            : launch_bwd_mlp<C, kBChunk, false>(m, P, packed, A, smem, st);
  if (rc) return rc;
  prof_end(PROF_BWD_MLP, st);
  GNCA_LAUNCH_CHECK();
  if (A.gw_part) {
    rc = run_attn_bwd(m, P, packed, a, A.zp_rowsum, A.zp_scratch, A.nchunks, gparams, st, /*defer_reduce=*/true);
    if (rc) return rc;
  }
  dim3 g3((a.H * a.W + 255) / 256, a.B);
  k_bwd_gather<C><<<g3, 256, 0, st>>>(A);
  GNCA_LAUNCH_CHECK();
  return 0;
}

int dispatch_step_bwd(const gnca_model& m, const Packed& P, const float* packed, BwdArgs& A, float* gparams,
                      cudaStream_t st) {
  switch (m.C) {
    case 4: return launch_step_bwd<4>(m, P, packed, A, gparams, st);
    case 8: return launch_step_bwd<8>(m, P, packed, A, gparams, st);
    case 16: return launch_step_bwd<16>(m, P, packed, A, gparams, st);
    case 32: return launch_step_bwd<32>(m, P, packed, A, gparams, st);
  }
  return GNCA_ERR_UNSUPPORTED;
}


int run_step_bwd(const gnca_model& m, const Packed& P, const float* packed, const StepArgs& a_in, const float* stats,
                 const float* gout, float* gx, float* gparams, const FwdWorkspace& fws, void* bwd_ws, bool zero_partials,
                 bool reduce_partials, cudaStream_t st, const float* gframe) {
  BwdWorkspace w = carve_bwd(bwd_ws, m, a_in.B, a_in.H, a_in.W);
  StepArgs a = a_in;
  // zero-padded shift: the per-sample softmax weights depend on x, Wq, Wk, scaling -> recompute them here and
  // back-propagate through them after the cell phase
  const bool zp = (m.flags & GNCA_F_GRAPH) && !(m.flags & GNCA_F_TORUS) && a.k > 0;
  if (zp) {
    int rc = run_attn_prepass(m, P, packed, a, fws, st);
    if (rc) return rc;
    GNCA_CHECK_CUDA(cudaMemsetAsync(w.attn.gw_part, 0, w.gw_bytes, st));
    // per-sample gradients of query_proj / key_proj / scaling: summed over the steps of a BPTT in place, reduced over the
    // samples once after its last step (zero_partials / reduce_partials bracket the steps)
    if (zero_partials)
      GNCA_CHECK_CUDA(cudaMemsetAsync(w.attn.pw, 0, (size_t)a.B * (2 * m.d_model * m.C + 2 * m.d_model + 1) * sizeof(float), st));
  }
  BwdArgs A{};
  A.s = a;
  A.gw_part = zp ? w.attn.gw_part : nullptr;
  A.grow = zp ? w.attn.grow : nullptr;
  A.zp_rowsum = zp ? fws.rowsum : nullptr;
  A.zp_scratch = w.attn;
  A.gout = gout; A.gx = gx; A.u = a.u; A.stats = stats; A.gframe = gframe;
  A.actmask = w.actmask; A.postmask = w.postmask; A.gz = w.gz; A.gy = w.gy; A.gxs = w.gxs;
  A.tile_part = w.tile_part; A.sums = w.sums; A.wpart = w.wpart;
  A.ntiles = ((a.W + kBTileW - 1) / kBTileW) * ((a.H + kBTileH - 1) / kBTileH);
  A.bchunk = ((long long)a.B * ((a.H * a.W + kBChunk - 1) / kBChunk) < 2 * 148) ? kBChunkSmall : kBChunk;
  A.nchunks = (a.H * a.W + A.bchunk - 1) / A.bchunk;
  A.n_items = a.B * A.nchunks;
  A.nblocks = A.n_items < kMaxBwdBlocks ? A.n_items : kMaxBwdBlocks;
  A.L = make_layout(m);
  A.wtotal = A.L.total;
  if (zero_partials) GNCA_CHECK_CUDA(cudaMemsetAsync(w.wpart, 0, w.wpart_bytes, st));
  int rc = dispatch_step_bwd(m, P, packed, A, gparams, st);
  if (rc) return rc;
  if (reduce_partials) {
    k_bwd_reduce<<<(int)((A.wtotal + 255) / 256), 256, 0, st>>>(kMaxBwdBlocks, A.wtotal, w.wpart, gparams);
    GNCA_LAUNCH_CHECK();
    if (zp) { rc = run_attn_param_reduce(m, a.B, w.attn, gparams, st); if (rc) return rc; }
  }
  return 0;
}

}  // namespace gnca

using namespace gnca;

extern "C" int gnca_step_bwd(const gnca_model* m, const float* packed_dev, int B, int H, int W, const float* x_in_dev,
                             const float* fire_u_dev, float fire_rate, const int32_t* offsets_host, int k,
                             float message_gain, const float* u_dev, const float* stats_dev, const float* gout_dev,
                             float* gx_dev, float* gparams_dev, void* workspace_dev, size_t workspace_bytes,
                             void* stream) {
  if (!m || !packed_dev || !x_in_dev || !u_dev || !stats_dev || !gout_dev || !gx_dev || !gparams_dev || !workspace_dev)
    return GNCA_ERR_ARG;
  if (B <= 0 || H <= 0 || W <= 0) return GNCA_ERR_ARG;
  if (!model_supported(*m)) return GNCA_ERR_UNSUPPORTED;
  if (fire_rate < 1.0f && !fire_u_dev) return GNCA_ERR_ARG;
  const bool graph = (m->flags & GNCA_F_GRAPH) != 0;
  FwdWorkspace fws = carve_fwd_workspace(workspace_dev, *m, B, H, W);
  if (fws.bytes + bwd_workspace_bytes(*m, B, H, W) > workspace_bytes) return GNCA_ERR_WORKSPACE;
  StepArgs a;
  fill_step_args(a, *m, B, H, W);
  int rc = set_host_offsets(a, offsets_host, graph ? k : 0);
  if (rc) return rc;
  a.fire_rate = fire_rate; a.message_gain = message_gain;
  a.fire_u = fire_u_dev;
  a.x_in = x_in_dev; a.u = const_cast<float*>(u_dev);
  const Packed P = make_packed(m->C, m->hidden, m->d_model, graph);
  return run_step_bwd(*m, P, packed_dev, a, stats_dev, gout_dev, gx_dev, gparams_dev, fws,
                      reinterpret_cast<char*>(workspace_dev) + fws.bytes, true, true, (cudaStream_t)stream);
}
