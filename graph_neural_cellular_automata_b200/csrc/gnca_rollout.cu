// Rollout entry points (the loop of train_graph_augmented_nca.py:302-324 as ONE call).
//   impl 1 (streaming): per-step kernels of gnca_fwd.cu / gnca_bwd.cu driven by a device-resident schedule --
//                       no host synchronisation inside the loop, so the whole call can sit in a CUDA graph.
//   impl 2 (resident):  cluster kernel of gnca_resident.cu (state stays in shared memory across steps).
// BPTT stores only x_t (x_hist); u, the hidden layer, masks and the message are recomputed in the backward.
#include "gnca_common.cuh"
#include "gnca_internal.h"
#include "gnca_metrics.cuh"
#include "gnca_rep.h"

namespace gnca {

__global__ void k_mul_inplace(size_t n, float* __restrict__ x, DamageView d, int C, int HW) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const size_t bc = i / HW;
    x[i] *= d.at((int)(bc / C), (int)(bc % C), (int)(i - bc * HW), C, HW);
  }
}

// out = a + b: dL/dx_T plus the gradient of the last frame when that frame is x_T (T % every == 0)
__global__ void k_add(size_t n, float* __restrict__ out, const float* __restrict__ a, const float* __restrict__ b) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    out[i] = a[i] + b[i];
}

// Frame metrics of one state buffer x ([B][C][HW]) on the streaming path: block (p, b) reduces cells
// [p * cells, (p + 1) * cells) of sample b into part[b][p] -- the first level of a two-level reduction whose second is
// k_metrics_reduce, both in a fixed order.
constexpr int kMetThreads = 256;
constexpr int kMetCells = 4096;                    // cells per block of k_frame_metrics

static inline int frame_metrics_parts(int HW) { return (HW + kMetCells - 1) / kMetCells; }

__global__ void __launch_bounds__(kMetThreads) k_frame_metrics(const float* __restrict__ x, int C, int HW,
                                                                const float* __restrict__ tgt, float eps, float thr,
                                                                double* __restrict__ part) {
  const int p = blockIdx.x, P = gridDim.x, b = blockIdx.y;
  const int lo = p * kMetCells, hi = min(HW, lo + kMetCells);
  const float* xb = x + (size_t)b * C * HW;
  MetAcc acc{0.0, 0.0, 0, 0};
  for (int cell = lo + (int)threadIdx.x; cell < hi; cell += kMetThreads)
    met_cell(acc, xb[cell], xb[HW + cell], xb[2 * (size_t)HW + cell], xb[3 * (size_t)HW + cell], tgt, cell, HW, eps,
             thr);
  met_warp_sum(acc);
  __shared__ double s_met[kMetThreads / 32][4];
  if ((threadIdx.x & 31) == 0) met_put(s_met[threadIdx.x >> 5], acc);
  __syncthreads();
  if (threadIdx.x == 0) met_sum_parts(part + ((size_t)b * P + p) * 4, &s_met[0][0], 0, kMetThreads / 32, 4);
}

// sums / counts of each (frame, sample) row from its P partials, in part order
__global__ void k_metrics_reduce(int rows, int P, const double* __restrict__ part, double* __restrict__ sums,
                                 int* __restrict__ counts) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  double s[4];
  met_sum_parts(s, part + (size_t)r * P * 4, 0, P, 4);
  sums[2 * (size_t)r] = s[0];
  sums[2 * (size_t)r + 1] = s[1];
  counts[2 * (size_t)r] = (int)s[2];
  counts[2 * (size_t)r + 1] = (int)s[3];
}

int run_metrics_reduce(int rows, int P, const double* part, double* sums, int* counts, cudaStream_t st) {
  k_metrics_reduce<<<(rows + 127) / 128, 128, 0, st>>>(rows, P, part, sums, counts);
  GNCA_LAUNCH_CHECK();
  return 0;
}

// metrics of frame f (the state x) on the streaming path.  per < B: one launch per block of `per` samples, block i
// against target + i * tstride (a stack with per-model targets), into the same partial rows
static int frame_metrics(const FrameMetrics& met, const float* x, int f, int B, int C, int HW, float thr, int per,
                         int tstride, cudaStream_t st) {
  const int P = frame_metrics_parts(HW);
  for (int b0 = 0; b0 < B; b0 += per) {
    k_frame_metrics<<<dim3(P, per), kMetThreads, 0, st>>>(x + (size_t)b0 * C * HW, C, HW,
                                                          met.target + (size_t)(b0 / per) * tstride, met.eps, thr,
                                                          met.part + (size_t)b0 * P * 4);
    GNCA_LAUNCH_CHECK();
  }
  return run_metrics_reduce(B, P, met.part, met.sums + (size_t)f * B * 2, met.counts + (size_t)f * B * 2, st);
}

// SSIM of one state buffer x ([B][C][HW]): block (p, b) sums ssim_cell over the interior cells among
// [p * kSsimCells, (p + 1) * kSsimCells) of sample b into part[b][p]; k_ssim_reduce is the second level.  Both in a fixed
// order.  Backs gnca_ssim_rgb and the kept steps of the streaming path.
constexpr int kSsimCells = 1024;                   // cells per block of k_frame_ssim

static inline int frame_ssim_parts(int HW) { return (HW + kSsimCells - 1) / kSsimCells; }

__global__ void __launch_bounds__(kMetThreads) k_frame_ssim(const float* __restrict__ x, int C, int H, int W,
                                                             const float* __restrict__ tgt, double* __restrict__ part) {
  const int p = blockIdx.x, P = gridDim.x, b = blockIdx.y, HW = H * W;
  const int lo = p * kSsimCells, hi = min(HW, lo + kSsimCells);
  const float* xb = x + (size_t)b * C * HW;
  auto state = [&](int yy, int xx) {
    const int cell = yy * W + xx;
    return make_float4(xb[cell], xb[HW + cell], xb[2 * (size_t)HW + cell], xb[3 * (size_t)HW + cell]);
  };
  double s = 0.0;
  for (int cell = lo + (int)threadIdx.x; cell < hi; cell += kMetThreads) {
    const int y = cell / W, xx = cell - y * W;
    if (ssim_interior(y, xx, H, W)) s += ssim_cell(state, tgt, y, xx, W, HW);
  }
  s = warp_sum_f64(s);
  __shared__ double s_ss[kMetThreads / 32];
  if ((threadIdx.x & 31) == 0) s_ss[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < kMetThreads / 32; ++w) t += s_ss[w];
    part[(size_t)b * P + p] = t;
  }
}

// ssim[r] = (sum of the P partials of row r, in part order) / (3 (H-6)(W-6))
__global__ void k_ssim_reduce(int rows, int P, const double* __restrict__ part, double inv_cells,
                              double* __restrict__ ssim) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  double s = 0.0;
  for (int p = 0; p < P; ++p) s += part[(size_t)r * P + p];
  ssim[r] = s * inv_cells;
}

int run_ssim_reduce(int rows, int P, const double* part, double* ssim, int H, int W, cudaStream_t st) {
  const double inv_cells = 1.0 / (3.0 * (double)(H - 2 * kSsimR) * (double)(W - 2 * kSsimR));
  k_ssim_reduce<<<(rows + 127) / 128, 128, 0, st>>>(rows, P, part, inv_cells, ssim);
  GNCA_LAUNCH_CHECK();
  return 0;
}

// SSIM of the B samples of x into ssim[B], through part (>= B * frame_ssim_parts(H * W) doubles); per / tstride as in
// frame_metrics
static int frame_ssim(const float* x, int B, int C, int H, int W, const float* tgt, double* part, double* ssim,
                      cudaStream_t st, int per = 0, int tstride = 0) {
  const int P = frame_ssim_parts(H * W);
  if (per == 0) per = B;
  for (int b0 = 0; b0 < B; b0 += per) {
    k_frame_ssim<<<dim3(P, per), kMetThreads, 0, st>>>(x + (size_t)b0 * C * H * W, C, H, W,
                                                       tgt + (size_t)(b0 / per) * tstride, part + (size_t)b0 * P);
    GNCA_LAUNCH_CHECK();
  }
  return run_ssim_reduce(B, P, part, ssim, H, W, st);
}

// the metrics of frame f on the streaming path, with its SSIM when ss is set.  A stack with a target stride: each
// model's samples against its own target (x_0 of a stack at T = 0: a stack runs no streaming step)
static int frame_quality(const FrameMetrics& met, const SsimFrames* ss, const float* x, int f, int B, int C, int H,
                         int W, float thr, cudaStream_t st, const ModelStack* ms, int target_stride) {
  const bool own = ms && target_stride;
  const int per = own ? ms->per_model : B, tstride = own ? target_stride : 0;
  int rc = frame_metrics(met, x, f, B, C, H * W, thr, per, tstride, st);
  if (rc || !ss) return rc;
  return frame_ssim(x, B, C, H, W, met.target, ss->part, ss->ssim + (size_t)f * B, st, per, tstride);
}

static int launch_add(size_t n, float* out, const float* a, const float* b, cudaStream_t st) {
  k_add<<<(int)((n + 1023) / 1024 < 2368 ? (n + 1023) / 1024 : 2368), 256, 0, st>>>(n, out, a, b);
  GNCA_LAUNCH_CHECK();
  return 0;
}

// g0 of a rollout whose backward starts at step T: gT, plus dL/dframe_{T/every} when frame T / every is x_T
static int fold_last_frame(size_t N, int T, int every, const float* g_frames, const float* gT, float* out,
                           cudaStream_t st) {
  return launch_add(N, out, gT, g_frames + (size_t)(T / every) * N, st);
}

struct RolloutWorkspace {
  float* ping;     // [B][C][H][W]
  float* pong;
  float* u;        // [B][C][H][W]
  float* stats;    // [B][2]
  float* g_a;      // gradient ping-pong
  float* g_b;
  float* alpha_tmp;  // [B][H][W] (resident kernel)
  char* step_ws;   // forward + backward per-step workspace
  size_t step_bytes;
  size_t bytes;
};

static inline size_t al(size_t v) { return (v + 255) / 256 * 256; }

static RolloutWorkspace carve_rollout(void* base, const gnca_model& m, int B, int H, int W) {
  RolloutWorkspace r;
  const size_t N = (size_t)B * m.C * H * W * sizeof(float);
  char* p = reinterpret_cast<char*>(base);
  size_t o = 0;
  r.ping = reinterpret_cast<float*>(p + o); o = al(o + N);
  r.pong = reinterpret_cast<float*>(p + o); o = al(o + N);
  r.u = reinterpret_cast<float*>(p + o); o = al(o + N);
  r.g_a = reinterpret_cast<float*>(p + o); o = al(o + N);
  r.g_b = reinterpret_cast<float*>(p + o); o = al(o + N);
  r.stats = reinterpret_cast<float*>(p + o); o = al(o + (size_t)B * 2 * sizeof(float));
  r.alpha_tmp = reinterpret_cast<float*>(p + o); o = al(o + (size_t)B * H * W * sizeof(float));
  r.step_ws = p + o;
  r.step_bytes = carve_fwd_workspace(nullptr, m, B, H, W).bytes + bwd_workspace_bytes(m, B, H, W);
  o = al(o + r.step_bytes);
  r.bytes = o;
  return r;
}

static void schedule_to_args(StepArgs& a, const gnca_schedule& s, int t, int B, int H, int W) {
  a.t = t;
  a.k = s.k;
  a.fire_rate_dev = s.fire_rate;
  a.message_gain_dev = s.message_gain;
  a.offsets_dev = s.offsets;
  a.steps = s.steps;
  a.fire_u = s.fire_u ? s.fire_u + (size_t)t * B * H * W : nullptr;
  a.philox_seed = s.philox_seed;
  a.philox_offset = s.philox_offset;
}

static int launch_damage(size_t N, float* x, const gnca_schedule& s, int C, int HW, cudaStream_t st) {
  k_mul_inplace<<<(int)((N + 1023) / 1024 < 2368 ? (N + 1023) / 1024 : 2368), 256, 0, st>>>(N, x, DamageView{s.damage, s.damage_layout}, C, HW);
  GNCA_LAUNCH_CHECK();
  return 0;
}

// Where the backward finds the forward of the steps from t0 on: x_t0 at `x0`, x_t (t > t0) at rest[t - t0 - 1], u_t and
// stats_t at slot t - t0 of `u` / `stats` (NULL: recomputed per step).  The dense history is {x_hist, x_hist + N, u_hist,
// stats_hist, 0}; a checkpoint segment is {ckpt[j], its recomputed states, ..., j * every}.
struct SavedSteps {
  const float* x0;
  const float* rest;
  const float* u;
  const float* stats;
  int t0;
};

// g of the rollout's last state: gT, plus the last frame's gradient when that frame is x_T; T == 0 writes g0 directly
static int bwd_begin(size_t N, int T, int every, const float* g_frames, const float* gT, float* g0,
                     const RolloutWorkspace& r, const float** gcur, cudaStream_t st) {
  *gcur = gT;
  if (T == 0) {
    if (g_frames) return fold_last_frame(N, T, every, g_frames, gT, g0, st);
    GNCA_CHECK_CUDA(cudaMemcpyAsync(g0, gT, N * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
  }
  if (g_frames && T % every == 0) {          // g_b is not written before the second step (t = T - 2)
    int rc = fold_last_frame(N, T, every, g_frames, gT, r.g_b, st);
    if (rc) return rc;
    *gcur = r.g_b;
  }
  return 0;
}

// The per-step backward of steps t_hi - 1 down to t_lo of a T-step rollout.  *gcur enters as dL/dx_{t_hi} and leaves as
// dL/dx_{t_lo}.  The gradient ping-pong and the weight-gradient partials follow the global t: the partials are zeroed at
// t = T - 1 and reduced into gparams at t = 0, so a caller may split [0, T) into ranges run last to first.
static int bwd_steps(const gnca_model& m, const Packed& P, const float* packed, int B, int H, int W,
                     const gnca_schedule& s, const SavedSteps& sv, int t_lo, int t_hi, int every, const float* g_frames,
                     const float** gcur, float* g0, float* gparams, const RolloutWorkspace& r, const FwdWorkspace& fws,
                     char* bws, cudaStream_t st) {
  const size_t N = (size_t)B * m.C * H * W;
  const bool graph = (m.flags & GNCA_F_GRAPH) != 0;
  const int T = s.T;
  for (int t = t_hi - 1; t >= t_lo; --t) {
    StepArgs a;
    fill_step_args(a, m, B, H, W);
    schedule_to_args(a, s, t, B, H, W);
    if (!graph) a.k = 0;
    a.x_in = const_cast<float*>(t == sv.t0 ? sv.x0 : sv.rest + (size_t)(t - sv.t0 - 1) * N);
    a.x_out = nullptr;
    const float* stats_t = r.stats;
    int rc = 0;
    if (sv.u && sv.stats) {
      a.u = const_cast<float*>(sv.u) + (size_t)(t - sv.t0) * N;
      stats_t = sv.stats + (size_t)(t - sv.t0) * B * 2;
    } else {
      a.u = r.u;
      a.stats = r.stats;
      rc = dispatch_step_recompute(m, P, packed, a, fws, st);
      if (rc) return rc;
    }
    float* gnext = (t == 0) ? g0 : (((T - 1 - t) & 1) ? r.g_b : r.g_a);
    // the frame of step t is x_t after the damage: its gradient joins dL/dx_t before the damage mask multiplies it
    const float* gframe = (g_frames && t % every == 0) ? g_frames + (size_t)(t / every) * N : nullptr;
    rc = run_step_bwd(m, P, packed, a, stats_t, *gcur, gnext, gparams, fws, bws, t == T - 1, t == 0, st, gframe);
    if (rc) return rc;
    if (s.damage && t == s.damage_step) {
      rc = launch_damage(N, gnext, s, m.C, H * W, st);
      if (rc) return rc;
    }
    *gcur = gnext;
  }
  return 0;
}

// Segment buffer of gnca_rollout_bwd_ckpt: the recomputed x_t of a segment's steps after its first, then u_t and stats_t
// of every step of the segment
struct Segment {
  float* x;       // [every - 1][B][C][H][W]
  float* u;       // [every][B][C][H][W]
  float* stats;   // [every][B][2]
  size_t bytes;
};

static Segment carve_segment(void* base, const gnca_model& m, int B, int H, int W, int every) {
  Segment s;
  const size_t N = (size_t)B * m.C * H * W * sizeof(float);
  char* p = reinterpret_cast<char*>(base);
  size_t o = 0;
  s.x = reinterpret_cast<float*>(p + o); o = al(o + (size_t)(every - 1) * N);
  s.u = reinterpret_cast<float*>(p + o); o = al(o + (size_t)every * N);
  s.stats = reinterpret_cast<float*>(p + o); o = al(o + (size_t)every * B * 2 * sizeof(float));
  s.bytes = o;
  return s;
}

// gnca_rollout_fwd with a strided history: x_t of every step t % every == 0 goes to x_hist slot t / every
// (every == 1: the full [T+1] history of gnca_rollout_fwd).
// met: the per-frame metrics of gnca_rollout_metrics (stride met->every), by the kernel that runs the steps
// ss (with met only): the SSIM of the same frames (gnca_rollout_metrics_ssim)
// ms: a stack of models (gnca_rollout_*_models): the steps run on a cluster kernel or not at all, since only those stage
// their weights per sample.  T = 0 reads no weight and takes the copy path below.
// target_stride (with met and ms): model i's metrics against met->target + i * target_stride (gnca_rollout_metrics_targets)
static int rollout_fwd(const gnca_model* m, const float* packed_dev, int B, int H, int W, const gnca_schedule* sched,
                       const float* x0_dev, float* xT_dev, float* x_hist_dev, int every, float* stats_hist_dev,
                       float* u_hist_dev, void* workspace_dev, size_t workspace_bytes, int impl, void* stream,
                       const FrameMetrics* met = nullptr, const ModelStack* ms = nullptr,
                       const SsimFrames* ss = nullptr, int target_stride = 0) {
  if (!m || !packed_dev || !sched || !x0_dev || !xT_dev || !workspace_dev) return GNCA_ERR_ARG;
  if (B <= 0 || H <= 0 || W <= 0 || sched->T < 0) return GNCA_ERR_ARG;
  if (!model_supported(*m)) return GNCA_ERR_UNSUPPORTED;
  const bool graph = (m->flags & GNCA_F_GRAPH) != 0;
  if (sched->T > 0 && (!sched->fire_rate || (graph && !sched->message_gain))) return GNCA_ERR_ARG;
  if (graph && sched->k > 0 && !sched->offsets) return GNCA_ERR_ARG;
  if (sched->k < 0 || sched->k > GNCA_MAX_K) return GNCA_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  RolloutWorkspace r = carve_rollout(workspace_dev, *m, B, H, W);
  if (r.bytes > workspace_bytes) return GNCA_ERR_WORKSPACE;
  const size_t N = (size_t)B * m->C * H * W;
  const Packed P = make_packed(m->C, m->hidden, m->d_model, graph);
  FwdWorkspace fws = carve_fwd_workspace(r.step_ws, *m, B, H, W);
  const int T = sched->T;
  if (impl != 1 && T > 0) {
    // auto: small samples (the launch-latency-bound regime) go to the cluster-resident kernel
    const bool want = impl == 2 || impl == 3 || ms || (size_t)H * W <= 16384;
    if (want) {
      const ModelStack one{0, 0};
      int rc = GNCA_ERR_UNSUPPORTED;
      if (impl != 3)
        rc = run_rep_fwd(*m, P, packed_dev, B, H, W, *sched, x0_dev, xT_dev, x_hist_dev, stats_hist_dev, u_hist_dev,
                         nullptr, nullptr, r.ping, st, every, 0, nullptr, met, ms ? *ms : one, ss, target_stride);
      if (rc == GNCA_ERR_UNSUPPORTED)
        rc = run_resident_fwd(*m, P, packed_dev, B, H, W, *sched, x0_dev, xT_dev, x_hist_dev, stats_hist_dev,
                              u_hist_dev, r.ping, r.pong, r.alpha_tmp, st, every, met, ms ? *ms : one, ss,
                              target_stride);
      if (rc != GNCA_ERR_UNSUPPORTED || impl == 2 || impl == 3 || ms) return rc;
    }
  }

  // where x_t lives: its x_hist slot when step t is kept, else ping/pong (x_T straight into xT_dev).  A step reads x_t
  // and writes x_{t+1}: two history slots, or a slot and the ping/pong buffer of the other parity -- never one buffer.
  auto x_at = [&](int t) -> float* {
    if (x_hist_dev && t % every == 0) return x_hist_dev + (size_t)(t / every) * N;
    if (t == T) return xT_dev;
    return (t & 1) ? r.pong : r.ping;
  };
  GNCA_CHECK_CUDA(cudaMemcpyAsync(x_at(0), x0_dev, N * sizeof(float), cudaMemcpyDeviceToDevice, st));
  for (int t = 0; t < T; ++t) {
    if (sched->damage && t == sched->damage_step) {
      int rc = launch_damage(N, x_at(t), *sched, m->C, H * W, st);
      if (rc) return rc;
    }
    if (met && t % met->every == 0) {
      int rc = frame_quality(*met, ss, x_at(t), t / met->every, B, m->C, H, W, m->alpha_thr, st, ms, target_stride);
      if (rc) return rc;
    }
    StepArgs a;
    fill_step_args(a, *m, B, H, W);
    schedule_to_args(a, *sched, t, B, H, W);
    if (!graph) a.k = 0;
    a.x_in = x_at(t);
    a.x_out = x_at(t + 1);
    a.u = u_hist_dev ? u_hist_dev + (size_t)t * N : r.u;
    a.stats = stats_hist_dev ? stats_hist_dev + (size_t)t * B * 2 : r.stats;
    int rc = dispatch_step_fwd(*m, P, packed_dev, a, fws, nullptr, st);
    if (rc) return rc;
  }
  if ((x_hist_dev && T % every == 0) || T == 0)
    GNCA_CHECK_CUDA(cudaMemcpyAsync(xT_dev, x_at(T), N * sizeof(float), cudaMemcpyDeviceToDevice, st));
  if (met && T % met->every == 0)
    return frame_quality(*met, ss, xT_dev, T / met->every, B, m->C, H, W, m->alpha_thr, st, ms, target_stride);
  return 0;
}

// gnca_rollout_fwd_bptt with a strided history: x_t of every step t % every == 0 goes to x_hist slot t / every
static int rollout_fwd_bptt(const gnca_model* m, const float* packed_dev, int B, int H, int W, const gnca_schedule* sched,
                            const float* x0_dev, float* xT_dev, float* x_hist_dev, int every, void* bptt_dev,
                            size_t bptt_bytes, void* workspace_dev, size_t workspace_bytes, void* stream) {
  if (!m || !packed_dev || !sched || !x0_dev || !xT_dev || !bptt_dev || !workspace_dev) return GNCA_ERR_ARG;
  if (B <= 0 || H <= 0 || W <= 0 || sched->T < 0) return GNCA_ERR_ARG;
  if (!model_supported(*m)) return GNCA_ERR_UNSUPPORTED;
  if (sched->k < 0 || sched->k > GNCA_MAX_K) return GNCA_ERR_UNSUPPORTED;
  const size_t need = gnca_bptt_bytes(m, B, H, W, sched->T);
  if (need == 0) return GNCA_ERR_UNSUPPORTED;
  if (need > bptt_bytes) return GNCA_ERR_WORKSPACE;
  RolloutWorkspace r = carve_rollout(workspace_dev, *m, B, H, W);
  if (r.bytes > workspace_bytes) return GNCA_ERR_WORKSPACE;
  const bool graph = (m->flags & GNCA_F_GRAPH) != 0;
  // the records are only worth writing if the resident backward can consume them for this batch / shape
  if (!rep_bwd_supported(*m, B, H, W, graph ? sched->k : 0)) return GNCA_ERR_UNSUPPORTED;
  const Packed P = make_packed(m->C, m->hidden, m->d_model, graph);
  float *rec, *stats;
  uint32_t* masks;
  rep_bptt_carve(bptt_dev, B, H, W, sched->T, &rec, &masks, &stats);
  if (sched->T == 0) {
    cudaMemcpyAsync(xT_dev, x0_dev, (size_t)B * m->C * H * W * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
    if (x_hist_dev)
      cudaMemcpyAsync(x_hist_dev, x0_dev, (size_t)B * m->C * H * W * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
    return 0;
  }
  return run_rep_fwd(*m, P, packed_dev, B, H, W, *sched, x0_dev, xT_dev, x_hist_dev, stats, nullptr, rec, masks, r.ping,
                     (cudaStream_t)stream, every);
}

// The schedule of steps [t0, t0 + n) as a launch of its own: per-step arrays and fire_u start at t0, the Philox counter
// is advanced by the blocks of t0 steps (the resident kernels key block ((t*B + b)*HW >> 2) + q + philox_offset, and
// H*W % 4 == 0 there, so this is exact), and damage_step becomes local.  `damage_at_start`: whether a damage step at t0
// itself stays in the segment -- the backward must multiply its gradient, while a recomputed forward starts from a
// checkpoint that is already post-damage.  steps[b] stays absolute (the kernels take t0 for it).
static gnca_schedule segment_schedule(const gnca_schedule& s, int t0, int n, int B, int H, int W, bool damage_at_start) {
  gnca_schedule r = s;
  const size_t HW = (size_t)H * W;
  r.T = n;
  r.fire_rate = s.fire_rate ? s.fire_rate + t0 : nullptr;
  r.message_gain = s.message_gain ? s.message_gain + t0 : nullptr;
  r.offsets = s.offsets ? s.offsets + (size_t)t0 * s.k * 2 : nullptr;
  r.fire_u = s.fire_u ? s.fire_u + (size_t)t0 * B * HW : nullptr;
  r.philox_offset = s.philox_offset + (uint64_t)t0 * (uint64_t)B * (HW >> 2);
  const int lo = damage_at_start ? t0 : t0 + 1;
  if (s.damage && s.damage_step >= lo && s.damage_step < t0 + n) {
    r.damage_step = s.damage_step - t0;
  } else {
    r.damage = nullptr;
    r.damage_step = 0;
  }
  return r;
}

// Segment buffer of gnca_rollout_bwd_bptt_ckpt: the records of `every` steps (rep_bptt_carve layout of the segment's
// step count), the gradient carried between segments, and x_T of the recomputed forward (not needed, but the kernel
// writes it).  Neither may live in the rollout workspace: the resident backward's scratch (GZ, RG, partials) starts at
// its base, where the recomputed forward also keeps its u overflow.
struct RepSegment {
  void* bptt;
  size_t bptt_bytes;
  float* g;       // [B][C][H][W]
  float* xT;      // [B][C][H][W]
  size_t bytes;
};

static RepSegment carve_rep_segment(void* base, const gnca_model& m, int B, int H, int W, int every) {
  RepSegment s;
  const size_t N = (size_t)B * m.C * H * W * sizeof(float);
  char* p = reinterpret_cast<char*>(base);
  size_t o = 0;
  s.bptt = p;
  s.bptt_bytes = rep_bptt_bytes(m, B, H, W, every);
  o = al(o + s.bptt_bytes);
  s.g = reinterpret_cast<float*>(p + o); o = al(o + N);
  s.xT = reinterpret_cast<float*>(p + o); o = al(o + N);
  s.bytes = o;
  return s;
}

}  // namespace gnca

using namespace gnca;

extern "C" {

size_t gnca_rollout_workspace_bytes(const gnca_model* m, int B, int H, int W, int T) {
  (void)T;
  if (!m || B <= 0 || H <= 0 || W <= 0) return 0;
  const size_t a = carve_rollout(nullptr, *m, B, H, W).bytes;
  const size_t b = (m->C == 16) ? rep_bwd_workspace_bytes(*m, B, H, W) : 0;
  return a > b ? a : b;
}

int gnca_rollout_fwd(const gnca_model* m, const float* packed_dev, int B, int H, int W, const gnca_schedule* sched,
                     const float* x0_dev, float* xT_dev, float* x_hist_dev, float* stats_hist_dev, float* u_hist_dev,
                     void* workspace_dev, size_t workspace_bytes, int impl, void* stream) {
  return rollout_fwd(m, packed_dev, B, H, W, sched, x0_dev, xT_dev, x_hist_dev, 1, stats_hist_dev, u_hist_dev,
                     workspace_dev, workspace_bytes, impl, stream);
}

int gnca_record_frames(int T, int every) {
  if (T < 0 || every <= 0) return GNCA_ERR_ARG;
  return T / every + 1;
}

int gnca_rollout_record(const gnca_model* m, const float* packed_dev, int B, int H, int W, const gnca_schedule* sched,
                        const float* x0_dev, float* xT_dev, int every, float* frames_dev, float* attn_dev,
                        void* workspace_dev, size_t workspace_bytes, int impl, void* stream) {
  if (!m || !packed_dev || !sched || !x0_dev || !xT_dev || !frames_dev || !workspace_dev) return GNCA_ERR_ARG;
  if (B <= 0 || H <= 0 || W <= 0 || sched->T < 0 || every <= 0) return GNCA_ERR_ARG;
  if (!model_supported(*m)) return GNCA_ERR_UNSUPPORTED;
  const bool graph = (m->flags & GNCA_F_GRAPH) != 0;
  if (attn_dev && !graph) return GNCA_ERR_ARG;
  if (sched->k < 0 || sched->k > GNCA_MAX_K) return GNCA_ERR_UNSUPPORTED;
  int rc = rollout_fwd(m, packed_dev, B, H, W, sched, x0_dev, xT_dev, frames_dev, every, nullptr, nullptr,
                       workspace_dev, workspace_bytes, impl, stream);
  if (rc || !attn_dev) return rc;
  // Attention map of every recorded step t = f * every < T, from the frame (the state step t consumes) and step t's
  // offsets -- the map gnca_step_fwd returns for that step.  Every sample gets one, frozen ones included, whatever the
  // step's fire rate and message gain: the map depends on neither.
  cudaStream_t st = (cudaStream_t)stream;
  const size_t N = (size_t)B * m->C * H * W;
  const Packed P = make_packed(m->C, m->hidden, m->d_model, graph);
  const FwdWorkspace fws = carve_fwd_workspace(carve_rollout(workspace_dev, *m, B, H, W).step_ws, *m, B, H, W);
  const bool zero_pad = !(m->flags & GNCA_F_TORUS);
  for (int f = 0; (size_t)f * every < (size_t)sched->T; ++f) {
    StepArgs a;
    fill_step_args(a, *m, B, H, W);
    schedule_to_args(a, *sched, f * every, B, H, W);
    a.steps = nullptr;
    a.fire_u = nullptr;
    a.x_in = frames_dev + (size_t)f * N;
    a.partials = fws.partials;
    a.attn_w = nullptr;
    if (zero_pad && a.k > 0) {
      rc = run_attn_prepass(*m, P, packed_dev, a, fws, st);
      if (rc) return rc;
    }
    rc = run_attn_map(*m, P, packed_dev, a, fws, attn_dev + (size_t)f * B * H * W, st);
    if (rc) return rc;
  }
  return 0;
}

size_t gnca_metrics_scratch_bytes(const gnca_model* m, int B, int H, int W, int T, int every) {
  if (!m || B <= 0 || H <= 0 || W <= 0 || T < 0 || every <= 0 || m->C < 4) return 0;
  // the cluster kernels keep one partial per rank (<= 8) of every frame; the streaming path reuses one frame's blocks
  const size_t F = (size_t)(T / every + 1);
  const size_t cluster = F * B * 8, streaming = (size_t)B * frame_metrics_parts(H * W);
  return (cluster > streaming ? cluster : streaming) * 4 * sizeof(double);
}

static int model_stack(const gnca_model& m, int n_models, int B, int impl, ModelStack* ms);

// the shared body of gnca_rollout_metrics[_ssim][_models] and gnca_rollout_metrics_targets: n_models = 0 runs one
// model, ssim_dev = NULL skips SSIM.  own_targets (a stack only): target_dev is [n_models][4][H][W], one per model;
// otherwise one [4][H][W] target for every sample
static int rollout_metrics(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                           const gnca_schedule* sched, const float* x0_dev, float* xT_dev, int every,
                           const float* target_dev, bool own_targets, float eps, double* sums_dev, int32_t* counts_dev,
                           double* ssim_dev, bool want_ssim, void* scratch_dev, size_t scratch_bytes,
                           void* workspace_dev, size_t workspace_bytes, int impl, void* stream) {
  if (!m || !packed_dev || !sched || !x0_dev || !xT_dev || !target_dev || !sums_dev || !counts_dev || !scratch_dev ||
      !workspace_dev || (want_ssim && !ssim_dev))
    return GNCA_ERR_ARG;
  if (B <= 0 || H <= 0 || W <= 0 || sched->T < 0 || every <= 0 || m->C < 4) return GNCA_ERR_ARG;
  if (want_ssim && (H < kSsimWin || W < kSsimWin)) return GNCA_ERR_ARG;
  if (!(eps >= 0.f)) return GNCA_ERR_ARG;
  ModelStack ms{0, 0};
  if (n_models > 0) {
    int rc = model_stack(*m, n_models, B, impl, &ms);
    if (rc) return rc;
  }
  const long long target_stride = own_targets ? 4LL * H * W : 0;     // an int in the kernels
  if (target_stride > 0x7fffffffLL) return GNCA_ERR_UNSUPPORTED;
  if (!model_supported(*m)) return GNCA_ERR_UNSUPPORTED;
  if (sched->k < 0 || sched->k > GNCA_MAX_K) return GNCA_ERR_UNSUPPORTED;
  const size_t met_bytes = gnca_metrics_scratch_bytes(m, B, H, W, sched->T, every);
  const size_t need = want_ssim ? gnca_metrics_ssim_scratch_bytes(m, B, H, W, sched->T, every) : met_bytes;
  if (need > scratch_bytes) return GNCA_ERR_WORKSPACE;
  const FrameMetrics met{target_dev, reinterpret_cast<double*>(scratch_dev), sums_dev, counts_dev, eps, every};
  const SsimFrames ss{reinterpret_cast<double*>(static_cast<char*>(scratch_dev) + met_bytes), ssim_dev};
  return rollout_fwd(m, packed_dev, B, H, W, sched, x0_dev, xT_dev, nullptr, 1, nullptr, nullptr, workspace_dev,
                     workspace_bytes, impl, stream, &met, n_models > 0 ? &ms : nullptr, want_ssim ? &ss : nullptr,
                     (int)target_stride);
}

int gnca_rollout_metrics(const gnca_model* m, const float* packed_dev, int B, int H, int W, const gnca_schedule* sched,
                         const float* x0_dev, float* xT_dev, int every, const float* target_dev, float eps,
                         double* sums_dev, int32_t* counts_dev, void* scratch_dev, size_t scratch_bytes,
                         void* workspace_dev, size_t workspace_bytes, int impl, void* stream) {
  return rollout_metrics(m, packed_dev, 0, B, H, W, sched, x0_dev, xT_dev, every, target_dev, false, eps, sums_dev,
                         counts_dev, nullptr, false, scratch_dev, scratch_bytes, workspace_dev, workspace_bytes, impl,
                         stream);
}

size_t gnca_metrics_ssim_scratch_bytes(const gnca_model* m, int B, int H, int W, int T, int every) {
  const size_t met = gnca_metrics_scratch_bytes(m, B, H, W, T, every);
  if (met == 0 || H < kSsimWin || W < kSsimWin) return 0;
  // one SSIM partial per rank of every frame on the cluster kernels, per block of one frame on the streaming path
  const size_t F = (size_t)(T / every + 1);
  const size_t cluster = F * B * 8, streaming = (size_t)B * frame_ssim_parts(H * W);
  return met + (cluster > streaming ? cluster : streaming) * sizeof(double);
}

int gnca_rollout_metrics_ssim(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                              const gnca_schedule* sched, const float* x0_dev, float* xT_dev, int every,
                              const float* target_dev, float eps, double* sums_dev, int32_t* counts_dev,
                              double* ssim_dev, void* scratch_dev, size_t scratch_bytes, void* workspace_dev,
                              size_t workspace_bytes, int impl, void* stream) {
  return rollout_metrics(m, packed_dev, 0, B, H, W, sched, x0_dev, xT_dev, every, target_dev, false, eps, sums_dev,
                         counts_dev, ssim_dev, true, scratch_dev, scratch_bytes, workspace_dev, workspace_bytes, impl,
                         stream);
}

size_t gnca_ssim_rgb_scratch_bytes(int B, int H, int W) {
  if (B <= 0 || H < kSsimWin || W < kSsimWin) return 0;
  return (size_t)B * frame_ssim_parts(H * W) * sizeof(double);
}

int gnca_ssim_rgb(const float* x_dev, int B, int C, int H, int W, const float* target_dev, double* ssim_dev,
                  void* scratch_dev, size_t scratch_bytes, void* stream) {
  if (!x_dev || !target_dev || !ssim_dev || !scratch_dev) return GNCA_ERR_ARG;
  if (B <= 0 || C < 4 || H < kSsimWin || W < kSsimWin) return GNCA_ERR_ARG;
  if (gnca_ssim_rgb_scratch_bytes(B, H, W) > scratch_bytes) return GNCA_ERR_WORKSPACE;
  return frame_ssim(x_dev, B, C, H, W, target_dev, reinterpret_cast<double*>(scratch_dev), ssim_dev,
                    (cudaStream_t)stream);
}

/* ---- a stack of same-architecture models in one launch: sample b runs model b / (B / n_models) ---- */
// the argument checks of the two stacked entry points that gnca_rollout_record / gnca_rollout_metrics do not make
static int model_stack(const gnca_model& m, int n_models, int B, int impl, ModelStack* ms) {
  if (n_models < 1 || B % n_models != 0 || impl < 0 || impl > 3) return GNCA_ERR_ARG;
  if (impl == 1) return GNCA_ERR_UNSUPPORTED;        // the streaming kernels stage weights per tile, not per sample
  ms->stride = make_packed(m.C, m.hidden, m.d_model, (m.flags & GNCA_F_GRAPH) != 0).total;
  ms->per_model = B / n_models;
  return 0;
}

int gnca_rollout_record_models(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                               const gnca_schedule* sched, const float* x0_dev, float* xT_dev, int every,
                               float* frames_dev, void* workspace_dev, size_t workspace_bytes, int impl, void* stream) {
  if (!m || !packed_dev || !sched || !x0_dev || !xT_dev || !frames_dev || !workspace_dev) return GNCA_ERR_ARG;
  if (B <= 0 || H <= 0 || W <= 0 || sched->T < 0 || every <= 0) return GNCA_ERR_ARG;
  ModelStack ms;
  int rc = model_stack(*m, n_models, B, impl, &ms);
  if (rc) return rc;
  if (!model_supported(*m)) return GNCA_ERR_UNSUPPORTED;
  if (sched->k < 0 || sched->k > GNCA_MAX_K) return GNCA_ERR_UNSUPPORTED;
  return rollout_fwd(m, packed_dev, B, H, W, sched, x0_dev, xT_dev, frames_dev, every, nullptr, nullptr, workspace_dev,
                     workspace_bytes, impl, stream, nullptr, &ms);
}

int gnca_rollout_metrics_models(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                                const gnca_schedule* sched, const float* x0_dev, float* xT_dev, int every,
                                const float* target_dev, float eps, double* sums_dev, int32_t* counts_dev,
                                void* scratch_dev, size_t scratch_bytes, void* workspace_dev, size_t workspace_bytes,
                                int impl, void* stream) {
  if (n_models < 1) return GNCA_ERR_ARG;
  return rollout_metrics(m, packed_dev, n_models, B, H, W, sched, x0_dev, xT_dev, every, target_dev, false, eps,
                         sums_dev, counts_dev, nullptr, false, scratch_dev, scratch_bytes, workspace_dev,
                         workspace_bytes, impl, stream);
}

int gnca_rollout_metrics_ssim_models(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                                     const gnca_schedule* sched, const float* x0_dev, float* xT_dev, int every,
                                     const float* target_dev, float eps, double* sums_dev, int32_t* counts_dev,
                                     double* ssim_dev, void* scratch_dev, size_t scratch_bytes, void* workspace_dev,
                                     size_t workspace_bytes, int impl, void* stream) {
  if (n_models < 1) return GNCA_ERR_ARG;
  return rollout_metrics(m, packed_dev, n_models, B, H, W, sched, x0_dev, xT_dev, every, target_dev, false, eps,
                         sums_dev, counts_dev, ssim_dev, true, scratch_dev, scratch_bytes, workspace_dev,
                         workspace_bytes, impl, stream);
}

int gnca_rollout_metrics_targets(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                                 const gnca_schedule* sched, const float* x0_dev, float* xT_dev, int every,
                                 const float* targets_dev, float eps, double* sums_dev, int32_t* counts_dev,
                                 double* ssim_dev, void* scratch_dev, size_t scratch_bytes, void* workspace_dev,
                                 size_t workspace_bytes, int impl, void* stream) {
  if (!targets_dev || n_models < 1 || B % n_models != 0) return GNCA_ERR_ARG;
  return rollout_metrics(m, packed_dev, n_models, B, H, W, sched, x0_dev, xT_dev, every, targets_dev, true, eps,
                         sums_dev, counts_dev, ssim_dev, ssim_dev != nullptr, scratch_dev, scratch_bytes, workspace_dev,
                         workspace_bytes, impl, stream);
}

int gnca_rollout_bwd_frames(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                            const gnca_schedule* sched, const float* x_hist_dev, const float* stats_hist_dev,
                            const float* u_hist_dev, int every, const float* g_frames_dev, const float* gT_dev,
                            float* g0_dev, float* gparams_dev, void* workspace_dev, size_t workspace_bytes, int impl,
                            void* stream) {
  if (!m || !packed_dev || !sched || !x_hist_dev || !gT_dev || !g0_dev || !gparams_dev || !workspace_dev)
    return GNCA_ERR_ARG;
  if (B <= 0 || H <= 0 || W <= 0 || sched->T < 0) return GNCA_ERR_ARG;
  if (g_frames_dev && every <= 0) return GNCA_ERR_ARG;
  if (!model_supported(*m)) return GNCA_ERR_UNSUPPORTED;
  if (sched->k < 0 || sched->k > GNCA_MAX_K) return GNCA_ERR_UNSUPPORTED;
  (void)impl;             // the backward currently always takes the streaming kernels (x_hist layout is shared)
  const bool graph = (m->flags & GNCA_F_GRAPH) != 0;
  cudaStream_t st = (cudaStream_t)stream;
  RolloutWorkspace r = carve_rollout(workspace_dev, *m, B, H, W);
  if (r.bytes > workspace_bytes) return GNCA_ERR_WORKSPACE;
  const size_t N = (size_t)B * m->C * H * W;
  const Packed P = make_packed(m->C, m->hidden, m->d_model, graph);
  FwdWorkspace fws = carve_fwd_workspace(r.step_ws, *m, B, H, W);
  const int T = sched->T;
  const float* gcur;
  int rc = bwd_begin(N, T, every, g_frames_dev, gT_dev, g0_dev, r, &gcur, st);
  if (rc || T == 0) return rc;
  // u and the statistics are recomputed per step unless both histories are given
  const SavedSteps sv{x_hist_dev, x_hist_dev + N, u_hist_dev, stats_hist_dev, 0};
  return bwd_steps(*m, P, packed_dev, B, H, W, *sched, sv, 0, T, every, g_frames_dev, &gcur, g0_dev, gparams_dev, r, fws,
                   r.step_ws + fws.bytes, st);
}

size_t gnca_ckpt_segment_bytes(const gnca_model* m, int B, int H, int W, int every) {
  if (!m || B <= 0 || H <= 0 || W <= 0 || every <= 0) return 0;
  return carve_segment(nullptr, *m, B, H, W, every).bytes;
}

int gnca_rollout_bwd_ckpt(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                          const gnca_schedule* sched, const float* ckpt_dev, int every,
                          const float* g_frames_dev, const float* gT_dev, float* g0_dev, float* gparams_dev,
                          void* segment_dev, size_t segment_bytes,
                          void* workspace_dev, size_t workspace_bytes, void* stream) {
  if (!m || !packed_dev || !sched || !ckpt_dev || !gT_dev || !g0_dev || !gparams_dev || !segment_dev || !workspace_dev)
    return GNCA_ERR_ARG;
  if (B <= 0 || H <= 0 || W <= 0 || sched->T < 0 || every <= 0) return GNCA_ERR_ARG;
  if (!model_supported(*m)) return GNCA_ERR_UNSUPPORTED;
  const bool graph = (m->flags & GNCA_F_GRAPH) != 0;
  if (sched->T > 0 && (!sched->fire_rate || (graph && !sched->message_gain))) return GNCA_ERR_ARG;
  if (graph && sched->k > 0 && !sched->offsets) return GNCA_ERR_ARG;
  if (sched->k < 0 || sched->k > GNCA_MAX_K) return GNCA_ERR_UNSUPPORTED;
  const Segment seg = carve_segment(segment_dev, *m, B, H, W, every);
  if (seg.bytes > segment_bytes) return GNCA_ERR_WORKSPACE;
  RolloutWorkspace r = carve_rollout(workspace_dev, *m, B, H, W);
  if (r.bytes > workspace_bytes) return GNCA_ERR_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t N = (size_t)B * m->C * H * W;
  const Packed P = make_packed(m->C, m->hidden, m->d_model, graph);
  // The recomputed forward writes only the segment, r.ping and the forward workspace: the weight-gradient partials in
  // the backward workspace stay live from t = T - 1 to t = 0
  FwdWorkspace fws = carve_fwd_workspace(r.step_ws, *m, B, H, W);
  char* bws = r.step_ws + fws.bytes;
  const int T = sched->T;
  const float* gcur;
  int rc = bwd_begin(N, T, every, g_frames_dev, gT_dev, g0_dev, r, &gcur, st);
  if (rc || T == 0) return rc;
  for (int j = (T - 1) / every; j >= 0; --j) {
    const int t_lo = j * every, t_hi = t_lo + every < T ? t_lo + every : T;
    const SavedSteps sv{ckpt_dev + (size_t)j * N, seg.x, seg.u, seg.stats, t_lo};
    for (int t = t_lo; t < t_hi; ++t) {
      float* x_in = const_cast<float*>(t == t_lo ? sv.x0 : seg.x + (size_t)(t - t_lo - 1) * N);
      // a checkpoint is the state after the damage: only a damage step inside the segment is applied here
      if (sched->damage && t == sched->damage_step && t != t_lo) {
        rc = launch_damage(N, x_in, *sched, m->C, H * W, st);
        if (rc) return rc;
      }
      StepArgs a;
      fill_step_args(a, *m, B, H, W);
      schedule_to_args(a, *sched, t, B, H, W);
      if (!graph) a.k = 0;
      a.x_in = x_in;
      // the segment's last output (the next checkpoint, or x_T) is not needed by the backward
      a.x_out = t + 1 < t_hi ? seg.x + (size_t)(t - t_lo) * N : r.ping;
      a.u = seg.u + (size_t)(t - t_lo) * N;
      a.stats = seg.stats + (size_t)(t - t_lo) * B * 2;
      rc = dispatch_step_fwd(*m, P, packed_dev, a, fws, nullptr, st);
      if (rc) return rc;
    }
    rc = bwd_steps(*m, P, packed_dev, B, H, W, *sched, sv, t_lo, t_hi, every, g_frames_dev, &gcur, g0_dev, gparams_dev,
                   r, fws, bws, st);
    if (rc) return rc;
  }
  return 0;
}

int gnca_rollout_bwd(const gnca_model* m, const float* packed_dev, int B, int H, int W, const gnca_schedule* sched,
                     const float* x_hist_dev, const float* stats_hist_dev, const float* u_hist_dev,
                     const float* gT_dev, float* g0_dev,
                     float* gparams_dev, void* workspace_dev, size_t workspace_bytes, int impl, void* stream) {
  return gnca_rollout_bwd_frames(m, packed_dev, B, H, W, sched, x_hist_dev, stats_hist_dev, u_hist_dev, 0, nullptr,
                                 gT_dev, g0_dev, gparams_dev, workspace_dev, workspace_bytes, impl, stream);
}


/* ---- resident BPTT: records instead of the dense x_t / u_t history (gnca_rep.cu / gnca_rep_bwd.cu) ---- */
size_t gnca_bptt_bytes(const gnca_model* m, int B, int H, int W, int T) {
  if (!m || B <= 0 || H <= 0 || W <= 0 || T < 0) return 0;
  if ((m->flags & GNCA_F_GRAPH) && !(m->flags & GNCA_F_TORUS)) return 0;
  return rep_bptt_bytes(*m, B, H, W, T);
}

int gnca_rollout_fwd_bptt_record(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                                 const gnca_schedule* sched, const float* x0_dev, float* xT_dev, int every,
                                 float* frames_dev, void* bptt_dev, size_t bptt_bytes, void* workspace_dev,
                                 size_t workspace_bytes, void* stream) {
  if (!frames_dev || every <= 0) return GNCA_ERR_ARG;
  return rollout_fwd_bptt(m, packed_dev, B, H, W, sched, x0_dev, xT_dev, frames_dev, every, bptt_dev, bptt_bytes,
                          workspace_dev, workspace_bytes, stream);
}

int gnca_rollout_fwd_bptt(const gnca_model* m, const float* packed_dev, int B, int H, int W, const gnca_schedule* sched,
                          const float* x0_dev, float* xT_dev, float* x_hist_dev, void* bptt_dev, size_t bptt_bytes,
                          void* workspace_dev, size_t workspace_bytes, void* stream) {
  return rollout_fwd_bptt(m, packed_dev, B, H, W, sched, x0_dev, xT_dev, x_hist_dev, 1, bptt_dev, bptt_bytes,
                          workspace_dev, workspace_bytes, stream);
}

int gnca_rollout_bwd_bptt_frames(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                                 const gnca_schedule* sched, void* bptt_dev, size_t bptt_bytes, int every,
                                 const float* g_frames_dev, const float* gT_dev, float* g0_dev, float* gparams_dev,
                                 void* workspace_dev, size_t workspace_bytes, void* stream) {
  if (!m || !packed_dev || !sched || !bptt_dev || !gT_dev || !g0_dev || !gparams_dev || !workspace_dev) return GNCA_ERR_ARG;
  if (B <= 0 || H <= 0 || W <= 0 || sched->T < 0) return GNCA_ERR_ARG;
  if (g_frames_dev && every <= 0) return GNCA_ERR_ARG;
  if (!model_supported(*m)) return GNCA_ERR_UNSUPPORTED;
  if (sched->k < 0 || sched->k > GNCA_MAX_K) return GNCA_ERR_UNSUPPORTED;
  const size_t need = gnca_bptt_bytes(m, B, H, W, sched->T);
  if (need == 0) return GNCA_ERR_UNSUPPORTED;
  if (need > bptt_bytes) return GNCA_ERR_WORKSPACE;
  if (rep_bwd_workspace_bytes(*m, B, H, W) > workspace_bytes) return GNCA_ERR_WORKSPACE;
  const bool graph = (m->flags & GNCA_F_GRAPH) != 0;
  const Packed P = make_packed(m->C, m->hidden, m->d_model, graph);
  if (sched->T == 0) {
    const size_t N = (size_t)B * m->C * H * W;
    if (g_frames_dev) return fold_last_frame(N, 0, every, g_frames_dev, gT_dev, g0_dev, (cudaStream_t)stream);
    cudaMemcpyAsync(g0_dev, gT_dev, N * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
    return 0;
  }
  return run_rep_bwd(*m, P, packed_dev, B, H, W, *sched, bptt_dev, gT_dev, g0_dev, gparams_dev, workspace_dev,
                     (cudaStream_t)stream, g_frames_dev, every);
}

int gnca_rollout_bwd_bptt(const gnca_model* m, const float* packed_dev, int B, int H, int W, const gnca_schedule* sched,
                          void* bptt_dev, size_t bptt_bytes, const float* gT_dev, float* g0_dev, float* gparams_dev,
                          void* workspace_dev, size_t workspace_bytes, void* stream) {
  return gnca_rollout_bwd_bptt_frames(m, packed_dev, B, H, W, sched, bptt_dev, bptt_bytes, 0, nullptr, gT_dev, g0_dev,
                                      gparams_dev, workspace_dev, workspace_bytes, stream);
}

/* ---- resident BPTT of the zero-padded graph shift: records plus x_t, softmax weights and row sums ---- */
size_t gnca_bptt_zp_bytes(const gnca_model* m, int B, int H, int W, int T) {
  if (!m || B <= 0 || H <= 0 || W <= 0 || T < 0) return 0;
  if (!model_supported(*m)) return 0;
  return rep_bptt_zp_bytes(*m, B, H, W, T);
}

int gnca_rollout_fwd_bptt_zp(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                             const gnca_schedule* sched, const float* x0_dev, float* xT_dev, int every, float* frames_dev,
                             void* bptt_dev, size_t bptt_bytes, void* workspace_dev, size_t workspace_bytes,
                             void* stream) {
  if (!m || !packed_dev || !sched || !x0_dev || !xT_dev || !bptt_dev || !workspace_dev) return GNCA_ERR_ARG;
  if (B <= 0 || H <= 0 || W <= 0 || sched->T < 0) return GNCA_ERR_ARG;
  if (frames_dev && every <= 0) return GNCA_ERR_ARG;
  if (!model_supported(*m)) return GNCA_ERR_UNSUPPORTED;
  if (sched->T > 0 && (!sched->fire_rate || !sched->message_gain)) return GNCA_ERR_ARG;
  if (sched->k > 0 && !sched->offsets) return GNCA_ERR_ARG;
  if (sched->k < 0 || sched->k > GNCA_MAX_K) return GNCA_ERR_UNSUPPORTED;
  const size_t need = gnca_bptt_zp_bytes(m, B, H, W, sched->T);
  if (need == 0) return GNCA_ERR_UNSUPPORTED;
  if (need > bptt_bytes) return GNCA_ERR_WORKSPACE;
  RolloutWorkspace r = carve_rollout(workspace_dev, *m, B, H, W);
  if (r.bytes > workspace_bytes) return GNCA_ERR_WORKSPACE;
  if (!rep_bwd_supported(*m, B, H, W, sched->k, true)) return GNCA_ERR_UNSUPPORTED;
  const int T = sched->T;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t N = (size_t)B * m->C * H * W;
  float *rec, *stats, *xs;
  uint32_t* masks;
  ZpRec zr;
  rep_bptt_carve(bptt_dev, B, H, W, T, &rec, &masks, &stats);
  rep_bptt_zp_carve(bptt_dev, *m, B, H, W, T, &xs, &zr, nullptr);
  if (T == 0) {
    GNCA_CHECK_CUDA(cudaMemcpyAsync(xT_dev, x0_dev, N * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (frames_dev) GNCA_CHECK_CUDA(cudaMemcpyAsync(frames_dev, x0_dev, N * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
  }
  // x_t of every step is what the backward reads (the dL/dw_i sums); the frames are a copy of every `every`-th state (a
  // copy, not a view: a caller editing a frame in place cannot corrupt what the backward reads).  The full history
  // (every = 1) is one contiguous copy; a strided 2D copy is avoided because every * state bytes can exceed the
  // largest pitch the copy engine takes.
  const Packed P = make_packed(m->C, m->hidden, m->d_model, true);
  int rc = run_rep_fwd(*m, P, packed_dev, B, H, W, *sched, x0_dev, xT_dev, xs, stats, nullptr, rec, masks, r.ping, st, 1,
                       0, &zr);
  if (rc || !frames_dev) return rc;
  if (every == 1) {
    GNCA_CHECK_CUDA(cudaMemcpyAsync(frames_dev, xs, (size_t)(T + 1) * N * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
  }
  for (int f = 0; (size_t)f * every <= (size_t)T; ++f)
    GNCA_CHECK_CUDA(cudaMemcpyAsync(frames_dev + (size_t)f * N, xs + (size_t)f * every * N, N * sizeof(float),
                                    cudaMemcpyDeviceToDevice, st));
  return 0;
}

int gnca_rollout_bwd_bptt_zp(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                             const gnca_schedule* sched, void* bptt_dev, size_t bptt_bytes, int every,
                             const float* g_frames_dev, const float* gT_dev, float* g0_dev, float* gparams_dev,
                             void* workspace_dev, size_t workspace_bytes, void* stream) {
  if (!m || !packed_dev || !sched || !bptt_dev || !gT_dev || !g0_dev || !gparams_dev || !workspace_dev) return GNCA_ERR_ARG;
  if (B <= 0 || H <= 0 || W <= 0 || sched->T < 0) return GNCA_ERR_ARG;
  if (g_frames_dev && every <= 0) return GNCA_ERR_ARG;
  if (!model_supported(*m)) return GNCA_ERR_UNSUPPORTED;
  if (sched->T > 0 && !sched->message_gain) return GNCA_ERR_ARG;
  if (sched->k > 0 && !sched->offsets) return GNCA_ERR_ARG;
  if (sched->k < 0 || sched->k > GNCA_MAX_K) return GNCA_ERR_UNSUPPORTED;
  const size_t need = gnca_bptt_zp_bytes(m, B, H, W, sched->T);
  if (need == 0) return GNCA_ERR_UNSUPPORTED;
  if (need > bptt_bytes) return GNCA_ERR_WORKSPACE;
  if (rep_bwd_workspace_bytes(*m, B, H, W) > workspace_bytes) return GNCA_ERR_WORKSPACE;
  if (!rep_bwd_supported(*m, B, H, W, sched->k, true)) return GNCA_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  if (sched->T == 0) {
    const size_t N = (size_t)B * m->C * H * W;
    if (g_frames_dev) return fold_last_frame(N, 0, every, g_frames_dev, gT_dev, g0_dev, st);
    GNCA_CHECK_CUDA(cudaMemcpyAsync(g0_dev, gT_dev, N * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
  }
  ZpBwd zb;
  rep_bptt_zp_carve(bptt_dev, *m, B, H, W, sched->T, nullptr, nullptr, &zb);
  const Packed P = make_packed(m->C, m->hidden, m->d_model, true);
  return run_rep_bwd(*m, P, packed_dev, B, H, W, *sched, bptt_dev, gT_dev, g0_dev, gparams_dev, workspace_dev, st,
                     g_frames_dev, every, 0, &zb);
}

/* ---- resident BPTT of a stack of same-architecture models: sample b runs model b / (B / n_models) ---- */
size_t gnca_rollout_workspace_models_bytes(const gnca_model* m, int n_models, int B, int H, int W, int T) {
  if (!m || n_models < 1 || B <= 0 || H <= 0 || W <= 0) return 0;
  const size_t a = gnca_rollout_workspace_bytes(m, B, H, W, T);
  const size_t b = (m->C == 16) ? rep_bwd_workspace_bytes(*m, B, H, W, n_models) : 0;
  return a > b ? a : b;
}

// the checks of the four stacked BPTT entry points after their pointer checks, all before any launch.  zp: the
// zero-padded graph shift's buffer (gnca_bptt_zp_bytes), else the records of gnca_bptt_bytes
static int bptt_models_check(const gnca_model* m, int n_models, int B, int H, int W, const gnca_schedule* sched,
                             bool zp, size_t bptt_bytes, size_t workspace_bytes, ModelStack* ms) {
  if (B <= 0 || H <= 0 || W <= 0 || sched->T < 0) return GNCA_ERR_ARG;
  const int rc = model_stack(*m, n_models, B, 0, ms);
  if (rc) return rc;
  if (!model_supported(*m)) return GNCA_ERR_UNSUPPORTED;
  const bool graph = (m->flags & GNCA_F_GRAPH) != 0;
  if (sched->T > 0 && (!sched->fire_rate || (graph && !sched->message_gain))) return GNCA_ERR_ARG;
  if (graph && sched->k > 0 && !sched->offsets) return GNCA_ERR_ARG;
  if (sched->k < 0 || sched->k > GNCA_MAX_K) return GNCA_ERR_UNSUPPORTED;
  const size_t need = zp ? gnca_bptt_zp_bytes(m, B, H, W, sched->T) : gnca_bptt_bytes(m, B, H, W, sched->T);
  if (need == 0) return GNCA_ERR_UNSUPPORTED;
  if (need > bptt_bytes) return GNCA_ERR_WORKSPACE;
  if (gnca_rollout_workspace_models_bytes(m, n_models, B, H, W, sched->T) > workspace_bytes) return GNCA_ERR_WORKSPACE;
  // no streaming fallback: the records are only written when the resident backward takes this batch and shape
  if (!rep_bwd_supported(*m, B, H, W, graph ? sched->k : 0, zp)) return GNCA_ERR_UNSUPPORTED;
  return 0;
}

static int fwd_bptt_models(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                           const gnca_schedule* sched, const float* x0_dev, float* xT_dev, void* bptt_dev,
                           size_t bptt_bytes, void* workspace_dev, size_t workspace_bytes, void* stream, bool zp) {
  if (!m || !packed_dev || !sched || !x0_dev || !xT_dev || !bptt_dev || !workspace_dev) return GNCA_ERR_ARG;
  ModelStack ms;
  const int rc = bptt_models_check(m, n_models, B, H, W, sched, zp, bptt_bytes, workspace_bytes, &ms);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int T = sched->T;
  if (T == 0) {
    GNCA_CHECK_CUDA(cudaMemcpyAsync(xT_dev, x0_dev, (size_t)B * m->C * H * W * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
  }
  RolloutWorkspace r = carve_rollout(workspace_dev, *m, B, H, W);
  const Packed P = make_packed(m->C, m->hidden, m->d_model, (m->flags & GNCA_F_GRAPH) != 0);
  float *rec, *stats, *xs = nullptr;
  uint32_t* masks;
  ZpRec zr;
  rep_bptt_carve(bptt_dev, B, H, W, T, &rec, &masks, &stats);
  if (zp) rep_bptt_zp_carve(bptt_dev, *m, B, H, W, T, &xs, &zr, nullptr);
  return run_rep_fwd(*m, P, packed_dev, B, H, W, *sched, x0_dev, xT_dev, xs, stats, nullptr, rec, masks, r.ping, st, 1,
                     0, zp ? &zr : nullptr, nullptr, ms);
}

static int bwd_bptt_models(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                           const gnca_schedule* sched, void* bptt_dev, size_t bptt_bytes, const float* gT_dev,
                           float* g0_dev, float* gparams_dev, void* workspace_dev, size_t workspace_bytes, void* stream,
                           bool zp) {
  if (!m || !packed_dev || !sched || !bptt_dev || !gT_dev || !g0_dev || !gparams_dev || !workspace_dev)
    return GNCA_ERR_ARG;
  ModelStack ms;
  const int rc = bptt_models_check(m, n_models, B, H, W, sched, zp, bptt_bytes, workspace_bytes, &ms);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (sched->T == 0) {
    GNCA_CHECK_CUDA(cudaMemcpyAsync(g0_dev, gT_dev, (size_t)B * m->C * H * W * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
  }
  const Packed P = make_packed(m->C, m->hidden, m->d_model, (m->flags & GNCA_F_GRAPH) != 0);
  ZpBwd zb;
  if (zp) rep_bptt_zp_carve(bptt_dev, *m, B, H, W, sched->T, nullptr, nullptr, &zb);
  return run_rep_bwd(*m, P, packed_dev, B, H, W, *sched, bptt_dev, gT_dev, g0_dev, gparams_dev, workspace_dev, st,
                     nullptr, 1, 0, zp ? &zb : nullptr, true, ms);
}

int gnca_rollout_fwd_bptt_models(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                                 const gnca_schedule* sched, const float* x0_dev, float* xT_dev, void* bptt_dev,
                                 size_t bptt_bytes, void* workspace_dev, size_t workspace_bytes, void* stream) {
  return fwd_bptt_models(m, packed_dev, n_models, B, H, W, sched, x0_dev, xT_dev, bptt_dev, bptt_bytes, workspace_dev,
                         workspace_bytes, stream, false);
}

int gnca_rollout_bwd_bptt_models(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                                 const gnca_schedule* sched, void* bptt_dev, size_t bptt_bytes, const float* gT_dev,
                                 float* g0_dev, float* gparams_dev, void* workspace_dev, size_t workspace_bytes,
                                 void* stream) {
  return bwd_bptt_models(m, packed_dev, n_models, B, H, W, sched, bptt_dev, bptt_bytes, gT_dev, g0_dev, gparams_dev,
                         workspace_dev, workspace_bytes, stream, false);
}

int gnca_rollout_fwd_bptt_zp_models(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                                    const gnca_schedule* sched, const float* x0_dev, float* xT_dev, void* bptt_dev,
                                    size_t bptt_bytes, void* workspace_dev, size_t workspace_bytes, void* stream) {
  return fwd_bptt_models(m, packed_dev, n_models, B, H, W, sched, x0_dev, xT_dev, bptt_dev, bptt_bytes, workspace_dev,
                         workspace_bytes, stream, true);
}

int gnca_rollout_bwd_bptt_zp_models(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                                    const gnca_schedule* sched, void* bptt_dev, size_t bptt_bytes, const float* gT_dev,
                                    float* g0_dev, float* gparams_dev, void* workspace_dev, size_t workspace_bytes,
                                    void* stream) {
  return bwd_bptt_models(m, packed_dev, n_models, B, H, W, sched, bptt_dev, bptt_bytes, gT_dev, g0_dev, gparams_dev,
                         workspace_dev, workspace_bytes, stream, true);
}

/* ---- checkpointed resident BPTT: x_{j*every} only; each segment's records are recomputed in the backward ---- */
size_t gnca_bptt_ckpt_bytes(const gnca_model* m, int B, int H, int W, int every) {
  if (!m || B <= 0 || H <= 0 || W <= 0 || every <= 0) return 0;
  if (gnca_bptt_bytes(m, B, H, W, every) == 0) return 0;
  return carve_rep_segment(nullptr, *m, B, H, W, every).bytes;
}

int gnca_rollout_fwd_bptt_ckpt(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                               const gnca_schedule* sched, const float* x0_dev, float* xT_dev, int every, float* ckpt_dev,
                               void* workspace_dev, size_t workspace_bytes, void* stream) {
  if (!m || !packed_dev || !sched || !x0_dev || !xT_dev || !ckpt_dev || !workspace_dev) return GNCA_ERR_ARG;
  if (B <= 0 || H <= 0 || W <= 0 || sched->T < 0 || every <= 0) return GNCA_ERR_ARG;
  if (!model_supported(*m)) return GNCA_ERR_UNSUPPORTED;
  const bool graph = (m->flags & GNCA_F_GRAPH) != 0;
  if (sched->T > 0 && (!sched->fire_rate || (graph && !sched->message_gain))) return GNCA_ERR_ARG;
  if (graph && sched->k > 0 && !sched->offsets) return GNCA_ERR_ARG;
  if (sched->k < 0 || sched->k > GNCA_MAX_K) return GNCA_ERR_UNSUPPORTED;
  if (gnca_bptt_bytes(m, B, H, W, 1) == 0) return GNCA_ERR_UNSUPPORTED;
  RolloutWorkspace r = carve_rollout(workspace_dev, *m, B, H, W);
  if (r.bytes > workspace_bytes) return GNCA_ERR_WORKSPACE;
  // checkpoints are only worth keeping if the resident backward can recompute from them for this batch / shape
  if (!rep_bwd_supported(*m, B, H, W, graph ? sched->k : 0)) return GNCA_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  if (sched->T == 0) {
    const size_t nb = (size_t)B * m->C * H * W * sizeof(float);
    GNCA_CHECK_CUDA(cudaMemcpyAsync(xT_dev, x0_dev, nb, cudaMemcpyDeviceToDevice, st));
    GNCA_CHECK_CUDA(cudaMemcpyAsync(ckpt_dev, x0_dev, nb, cudaMemcpyDeviceToDevice, st));
    return 0;
  }
  const Packed P = make_packed(m->C, m->hidden, m->d_model, graph);
  // the same kernel, scratch and launch configuration as the recompute of gnca_rollout_bwd_bptt_ckpt: no records
  return run_rep_fwd(*m, P, packed_dev, B, H, W, *sched, x0_dev, xT_dev, ckpt_dev, nullptr, nullptr, nullptr, nullptr,
                     r.ping, st, every, 0);
}

int gnca_rollout_bwd_bptt_ckpt_frames(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                                      const gnca_schedule* sched, const float* frames_dev, int every, int ckpt_every,
                                      const float* g_frames_dev, const float* gT_dev, float* g0_dev, float* gparams_dev,
                                      void* segment_dev, size_t segment_bytes, void* workspace_dev,
                                      size_t workspace_bytes, void* stream) {
  if (!m || !packed_dev || !sched || !frames_dev || !gT_dev || !g0_dev || !gparams_dev || !segment_dev || !workspace_dev)
    return GNCA_ERR_ARG;
  if (B <= 0 || H <= 0 || W <= 0 || sched->T < 0 || every <= 0 || ckpt_every <= 0) return GNCA_ERR_ARG;
  if (ckpt_every % every != 0) return GNCA_ERR_ARG;
  if (!model_supported(*m)) return GNCA_ERR_UNSUPPORTED;
  const bool graph = (m->flags & GNCA_F_GRAPH) != 0;
  if (sched->T > 0 && (!sched->fire_rate || (graph && !sched->message_gain))) return GNCA_ERR_ARG;
  if (graph && sched->k > 0 && !sched->offsets) return GNCA_ERR_ARG;
  if (sched->k < 0 || sched->k > GNCA_MAX_K) return GNCA_ERR_UNSUPPORTED;
  const size_t need = gnca_bptt_ckpt_bytes(m, B, H, W, ckpt_every);
  if (need == 0) return GNCA_ERR_UNSUPPORTED;
  if (need > segment_bytes) return GNCA_ERR_WORKSPACE;
  RolloutWorkspace r = carve_rollout(workspace_dev, *m, B, H, W);
  if (r.bytes > workspace_bytes || rep_bwd_workspace_bytes(*m, B, H, W) > workspace_bytes) return GNCA_ERR_WORKSPACE;
  if (!rep_bwd_supported(*m, B, H, W, graph ? sched->k : 0)) return GNCA_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t N = (size_t)B * m->C * H * W;
  const int T = sched->T;
  if (T == 0) {
    if (g_frames_dev) return fold_last_frame(N, 0, every, g_frames_dev, gT_dev, g0_dev, st);
    GNCA_CHECK_CUDA(cudaMemcpyAsync(g0_dev, gT_dev, N * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
  }
  const Packed P = make_packed(m->C, m->hidden, m->d_model, graph);
  const RepSegment seg = carve_rep_segment(segment_dev, *m, B, H, W, ckpt_every);
  const int nseg = (T - 1) / ckpt_every + 1;
  const size_t per_ckpt = (size_t)(ckpt_every / every);           // frames between consecutive checkpoints
  // dL/dx_{j*ckpt_every} goes to g0 for even j and to the segment's slot for odd j: segment 0 ends in g0, and no launch
  // reads the buffer it writes
  auto g_at = [&](int j) -> float* { return (j & 1) ? seg.g : g0_dev; };
  // The last frame, when it is x_T, goes into g_T here, once: each segment's backward leaves it out of its own g_T
  // (there it would be the next segment's first frame, added already).  g_at(nseg) is the buffer the last segment
  // does not write.
  const float* gT = gT_dev;
  if (g_frames_dev && T % every == 0) {
    int rc = fold_last_frame(N, T, every, g_frames_dev, gT_dev, g_at(nseg), st);
    if (rc) return rc;
    gT = g_at(nseg);
  }
  for (int j = nseg - 1; j >= 0; --j) {
    const int t0 = j * ckpt_every, n = T - t0 < ckpt_every ? T - t0 : ckpt_every;
    float *rec, *stats;
    uint32_t* masks;
    rep_bptt_carve(seg.bptt, B, H, W, n, &rec, &masks, &stats);
    // the checkpoint is x_t0 after a damage at t0: the recompute applies only a damage step inside the segment
    const gnca_schedule sf = segment_schedule(*sched, t0, n, B, H, W, false);
    int rc = run_rep_fwd(*m, P, packed_dev, B, H, W, sf, frames_dev + (size_t)j * per_ckpt * N, seg.xT, nullptr, stats,
                         nullptr, rec, masks, r.ping, st, 1, t0);
    if (rc) return rc;
    // frames t0 / every ... of the segment are added at their local steps t % every == 0 (t0 is a multiple of every)
    const gnca_schedule sb = segment_schedule(*sched, t0, n, B, H, W, true);
    const float* gfr = g_frames_dev ? g_frames_dev + (size_t)(t0 / every) * N : nullptr;
    rc = run_rep_bwd(*m, P, packed_dev, B, H, W, sb, seg.bptt, j == nseg - 1 ? gT : g_at(j + 1), g_at(j),
                     gparams_dev, workspace_dev, st, gfr, every, t0, nullptr, false);
    if (rc) return rc;
  }
  return 0;
}

int gnca_rollout_bwd_bptt_ckpt(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                               const gnca_schedule* sched, const float* ckpt_dev, int every, const float* gT_dev,
                               float* g0_dev, float* gparams_dev, void* segment_dev, size_t segment_bytes,
                               void* workspace_dev, size_t workspace_bytes, void* stream) {
  // the checkpoints are the frames of stride `every`, each one a checkpoint
  return gnca_rollout_bwd_bptt_ckpt_frames(m, packed_dev, B, H, W, sched, ckpt_dev, every, every, nullptr, gT_dev,
                                           g0_dev, gparams_dev, segment_dev, segment_bytes, workspace_dev,
                                           workspace_bytes, stream);
}

/* ---- host-side schedule construction: T x random.sample(range(n), k) on CPython's MT19937 state ----
 * CPython: random.sample on a short population is a partial Fisher-Yates over a copy of the population driven by
 * _randbelow(m) = { k = m.bit_length(); do r = getrandbits(k) while (r >= m); }, getrandbits(k <= 32) =
 * genrand_uint32() >> (32 - k)   (Lib/random.py, Modules/_randommodule.c).  `mt` is the 624-word state, *mti the
 * position (the 625th element of random.getstate()[1]); both are advanced in place. */
int gnca_host_sample_indices(uint32_t* mt, int32_t* mti, int n, int k, int T, int32_t* out_idx) {
  if (!mt || !mti || !out_idx || n <= 0 || k < 0 || k > n || n > 4096 || T < 0) return GNCA_ERR_ARG;
  int pos = *mti;
  auto next_u32 = [&]() -> uint32_t {
    if (pos >= 624) {
      const uint32_t UPPER = 0x80000000u, LOWER = 0x7fffffffu, MATRIX = 0x9908b0dfu;
      int kk;
      for (kk = 0; kk < 624 - 397; ++kk) {
        const uint32_t y = (mt[kk] & UPPER) | (mt[kk + 1] & LOWER);
        mt[kk] = mt[kk + 397] ^ (y >> 1) ^ ((y & 1u) ? MATRIX : 0u);
      }
      for (; kk < 623; ++kk) {
        const uint32_t y = (mt[kk] & UPPER) | (mt[kk + 1] & LOWER);
        mt[kk] = mt[kk + (397 - 624)] ^ (y >> 1) ^ ((y & 1u) ? MATRIX : 0u);
      }
      const uint32_t y = (mt[623] & UPPER) | (mt[0] & LOWER);
      mt[623] = mt[396] ^ (y >> 1) ^ ((y & 1u) ? MATRIX : 0u);
      pos = 0;
    }
    uint32_t y = mt[pos++];
    y ^= (y >> 11);
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= (y >> 18);
    return y;
  };
  int32_t pool[4096];
  for (int t = 0; t < T; ++t) {
    for (int i = 0; i < n; ++i) pool[i] = i;
    for (int i = 0; i < k; ++i) {
      const uint32_t m = (uint32_t)(n - i);
      int bits = 0;
      for (uint32_t v = m; v; v >>= 1) ++bits;
      uint32_t r;
      do { r = next_u32() >> (32 - bits); } while (r >= m);
      out_idx[t * k + i] = pool[r];
      pool[r] = pool[n - i - 1];
    }
  }
  *mti = pos;
  return 0;
}

// The same draws from a block of raw MT19937 outputs the caller pulled with random.getrandbits(32 * n_words): no
// state conversion on the python side (getstate -> numpy -> setstate costs more than the sampling).  Writes the
// chosen offsets straight from the table; *used = words consumed (the caller restores the state and skips exactly
// that many outputs).  Returns GNCA_ERR_UNSUPPORTED when the block is too short (the caller retries with more).
int gnca_host_sample_offsets_words(const uint32_t* words, int n_words, const int8_t* table /*[n][2]*/, int n, int k,
                                   int T, int8_t* out_off /*[T][k][2]*/, int32_t* used) {
  if (!words || !table || !out_off || !used || n <= 0 || k < 0 || k > n || n > 4096 || T < 0) return GNCA_ERR_ARG;
  int pos = 0;
  int32_t pool[4096];
  for (int t = 0; t < T; ++t) {
    for (int i = 0; i < n; ++i) pool[i] = i;
    for (int i = 0; i < k; ++i) {
      const uint32_t m = (uint32_t)(n - i);
      int bits = 0;
      for (uint32_t v = m; v; v >>= 1) ++bits;
      uint32_t r;
      do {
        if (pos >= n_words) return GNCA_ERR_UNSUPPORTED;
        r = words[pos++] >> (32 - bits);
      } while (r >= m);
      const int src = pool[r];
      out_off[((size_t)t * k + i) * 2] = table[2 * src];
      out_off[((size_t)t * k + i) * 2 + 1] = table[2 * src + 1];
      pool[r] = pool[n - i - 1];
    }
  }
  *used = pos;
  return 0;
}
}  // extern "C"
