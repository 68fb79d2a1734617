/*
 * gnca.h -- C ABI of libgnca.so: the B200 (sm_100a) graph-NCA step / rollout kernels.
 *
 * This is the drop-in boundary for the hot path of Psylocibe23/Graph_Neural_Cellular_Automata.  The
 * reference has no FFI layer (it is pure PyTorch); what these entry points replace are the bodies of
 *
 *   FixedSobelPerception.forward      src/modules/perception.py:21-26            -> gnca_perception_fwd/_bwd
 *   NeuralCA._alive_mask              src/modules/nca.py:55-62                   -> gnca_alive_mask
 *   GraphAugmentation.forward         src/modules/graph_augmentation.py:104-169  -> gnca_graph_fwd/_bwd
 *   NeuralCA.forward                  src/modules/nca.py:64-105                  -> gnca_step_fwd/_bwd (GNCA_F_GRAPH clear)
 *   NeuralCAGraph.forward             src/modules/ncagraph.py:106-168            -> gnca_step_fwd/_bwd (GNCA_F_GRAPH set)
 *   the rollout loop                  src/training/train_graph_augmented_nca.py:302-324 -> gnca_rollout_fwd/_bwd
 *   the recording loop                test_graph_augmented_regeneration.py:183-194     -> gnca_rollout_record
 *   losses on recorded states         (eager autograd through every x_t)               -> gnca_rollout_bwd_frames
 *   loss_premult_rgba (+ its grad)    src/training/train_graph_augmented_nca.py:52-61,337-339 -> gnca_loss_premult_rgba
 *   grad normalise + Adam             src/training/train_graph_augmented_nca.py:370-375 -> gnca_normalize_adam
 *   multiplicative damage             src/utils/damage.py:16-98                  -> gnca_apply_mask
 *
 * Conventions
 *   - every pointer named *_dev / documented "device" is a CUDA device pointer; tensors are fp32,
 *     contiguous NCHW exactly as the reference's modules take them;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises;
 *   - return value: 0 = ok, >0 = a cudaError_t, <0 = one of GNCA_ERR_*.  Nothing throws;
 *   - no call ever falls back to the host: an unsupported configuration returns GNCA_ERR_UNSUPPORTED.
 *
 * Parameters travel as ONE flat fp32 device buffer in the canonical order of gnca_param_layout()
 * (same orientation as the reference's state_dict tensors).  gnca_pack_weights() derives the
 * kernel-side buffer (adds transposed copies for the forward MLP); gradients come back in the canonical
 * layout.
 */
#ifndef GNCA_H_
#define GNCA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GNCA_VERSION 106

#define GNCA_ERR_ARG (-1)         /* null pointer / bad size */
#define GNCA_ERR_UNSUPPORTED (-2) /* shape or flag combination without a kernel */
#define GNCA_ERR_WORKSPACE (-3)   /* workspace too small */

#define GNCA_F_GRAPH 1u          /* NeuralCAGraph (else classic NeuralCA) */
#define GNCA_F_TORUS 2u          /* graph shift = torch.roll (graph_zero_padded_shift=False) */
#define GNCA_F_HIDDEN_ONLY 4u    /* ncagraph.py:98-101 */
#define GNCA_F_ALIVE_TO_ALIVE 8u /* graph_augmentation.py:116-117,130-133 */
#define GNCA_F_GROUPNORM 16u     /* use_groupnorm */

#define GNCA_MAX_K 64 /* chosen offsets per step */

typedef struct gnca_model {
  int32_t C;       /* n_channels: 4, 8, 16 or 32 */
  int32_t hidden;  /* update_hidden, multiple of 4, <= 256 */
  int32_t d_model; /* graph_d_model (used by the zero-padded-shift attention only), <= 64 */
  uint32_t flags;  /* GNCA_F_* */
  float update_gain;
  float alpha_thr;       /* model.alpha_thr  (pre / post alive) */
  float graph_alpha_thr; /* model.graph.alpha_thr (sender alive) */
  float gn_eps;          /* 1e-3 in the reference */
} gnca_model;

/* offsets (in floats) of each tensor inside the canonical flat parameter / gradient buffer; -1 = absent */
typedef struct gnca_layout {
  int64_t w1, b1, w2;   /* update_net.0.weight [hidden,3C], update_net.0.bias [hidden], update_net.2.weight [C,hidden] */
  int64_t gamma, beta;  /* norm.weight, norm.bias [C] (present even when GroupNorm is off) */
  int64_t wm, bm;       /* graph.msg_proj [C,C],[C] */
  int64_t wq, bq;       /* graph.query_proj [d,C],[d] */
  int64_t wk, bk;       /* graph.key_proj [d,C],[d] */
  int64_t scaling;      /* graph.scaling [1] */
  int64_t total;        /* floats in the canonical buffer */
  int64_t packed_total; /* floats in the packed (kernel-side) buffer */
} gnca_layout;

/* Per-step schedule of a rollout; every array lives on the DEVICE. */
typedef struct gnca_schedule {
  int32_t T;                  /* steps */
  int32_t k;                  /* offsets per step (0 for classic) */
  const float* fire_rate;     /* [T]   fire_rate of step t (>= 1 -> no mask) */
  const float* message_gain;  /* [T]   model.message_gain at step t (0 -> message skipped) */
  const int8_t* offsets;      /* [T][k][2] (dy,dx) drawn by random.sample at step t */
  const int32_t* steps;       /* [B] per-sample step counts (sample b advances while steps[b] > t) or NULL */
  const float* fire_u;        /* [T][B][H][W] uniforms (the reference's torch.rand draws) or NULL */
  uint64_t philox_seed;       /* used when fire_u == NULL: in-kernel Philox4x32-10 uniforms */
  uint64_t philox_offset;
  const float* damage;        /* multiplicative mask applied to x BEFORE step damage_step, or NULL; layout below */
  int32_t damage_step;
  int32_t max_offset;         /* max(|dy|,|dx|) over all offsets (halo depth of the resident kernel); 0 = unknown */
  int32_t damage_layout;      /* GNCA_DMG_DENSE [B][C][H][W] | GNCA_DMG_PLANE [B][H][W] on every channel |
                                 GNCA_DMG_PLANE_ALPHA [B][H][W] on the alpha channel only (salt & pepper) */
  int32_t reserved_;
} gnca_schedule;

#define GNCA_DMG_DENSE 0
#define GNCA_DMG_PLANE 1
#define GNCA_DMG_PLANE_ALPHA 2

/* Damage DESCRIPTOR (src/utils/damage.py:16-98, policy :101-138): one kind + one size for the whole batch, per-sample
 * geometry.  gnca_damage_plane evaluates it in closed form into a per-cell plane [B][H][W] (square / circle / stripes /
 * gaussian from the positions; alpha_drop / saltpepper from the caller's uniforms), which the rollout kernels multiply
 * in at `damage_step` (schedule.damage with layout GNCA_DMG_PLANE / GNCA_DMG_PLANE_ALPHA) -- no [B][C][H][W] mask. */
#define GNCA_DK_SQUARE 1      /* cutout_square_  :16-24   pos[b] = top-left (y, x), side `size`                         */
#define GNCA_DK_CIRCLE 2      /* cutout_circle_  :27-37   pos[b] = centre, radius `size`                                */
#define GNCA_DK_STRIPE_H 3    /* stripe_wipe_    :40-51   rows  [pos[0][0], +size) of EVERY sample                      */
#define GNCA_DK_STRIPE_V 4    /*                           cols  [pos[0][0], +size)                                      */
#define GNCA_DK_GAUSSIAN 5    /* gaussian_hole_  :87-98   clamp(1 - exp(-r2 / (2 (size*softness)^2)), 0, 1)             */
#define GNCA_DK_ALPHA_DROP 6  /* alpha_dropout_  :54-66   0 where rand < p and alpha > alpha_thr (hard: all channels)   */
#define GNCA_DK_SALTPEPPER 7  /* salt_pepper_alpha_ :69-73  0 where rand < p, alpha channel only                        */
typedef struct gnca_damage {
  int32_t kind;
  int32_t size;
  float softness;             /* gaussian */
  float p;                    /* alpha_drop / saltpepper */
  float alpha_thr;            /* alpha_drop */
  int32_t reserved_;
  const int64_t* pos;         /* device [B][2] (y, x) -- what torch.randint drew, never read back by the host */
  const float* rand;          /* device [B][H][W] uniforms (torch.rand_like(alpha)) for kinds 6, 7 */
} gnca_damage;
/* plane[b][y][x] of the descriptor; `state` ([B][C][H][W]) is read for alpha_drop only.  *layout_out = the schedule
 * layout the plane must be applied with. */
int gnca_damage_plane(const gnca_damage* d, int B, int C, int H, int W, const float* state_dev, float* plane_dev,
                      int32_t* layout_out, void* stream);
/* state *= plane (layout GNCA_DMG_PLANE or GNCA_DMG_PLANE_ALPHA), in place */
int gnca_apply_plane(int B, int C, int H, int W, float* state_dev, const float* plane_dev, int32_t layout, void* stream);

int gnca_version(void);
const char* gnca_error_string(int code);
/* number of CUDA kernels this library has launched in this process (bench.py reports it as gpu_launches) */
unsigned long long gnca_launch_count(void);
/* Optional per-kernel timing (CUDA events on the launching stream around each launch of the kernel family):
 * ids 0 k_update, 1 k_apply, 2 resident forward rollout, 3 k_bwd_mlp, 6 resident backward.  read() waits for the
 * recorded events, returns the summed duration and launch count since the last read, and clears them. */
int gnca_profile_enable(int on);
int gnca_profile_read(int kernel_id, double* total_ms, unsigned long long* launches);

int gnca_param_layout(const gnca_model* m, gnca_layout* out);
/* canonical flat params -> packed kernel-side buffer (packed_total floats) */
int gnca_pack_weights(const gnca_model* m, const float* params_dev, float* packed_dev, void* stream);

/* ------------------------------------------------------------------ single operators ------- */
/* perception.py:21-26 : x [B,C,H,W] -> y [B,3C,H,W] = [identity | sobel_x | sobel_y], zero halo */
int gnca_perception_fwd(int B, int C, int H, int W, const float* x_dev, float* y_dev, void* stream);
/* transpose: gy [B,3C,H,W] -> gx [B,C,H,W] */
int gnca_perception_bwd(int B, int C, int H, int W, const float* gy_dev, float* gx_dev, void* stream);
/* nca.py:55-62 : (maxpool3x3(x[:,3]) > thr) as float [B,1,H,W] */
int gnca_alive_mask(int B, int C, int H, int W, const float* x_dev, float thr, float* mask_dev, void* stream);

/* ------------------------------------------------------------------ one CA step ------------- */
size_t gnca_step_workspace_bytes(const gnca_model* m, int B, int H, int W);

/*
 * x_out = step(x_in).  fire_u_dev: [B,H,W] uniforms or NULL (required iff fire_rate < 1).
 * offsets_host: k (dy,dx) pairs, HOST memory (the module's random.sample result); k may be 0.
 * u_dev [B,C,H,W] and stats_dev [B,2] receive the masked pre-norm update and (mean, rstd): scratch for
 * inference, saved tensors for gnca_step_bwd.  attn_dev: optional [B,H,W] normalised attention map.
 */
int gnca_step_fwd(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                  const float* x_in_dev, float* x_out_dev,
                  const float* fire_u_dev, float fire_rate,
                  const int32_t* offsets_host, int k, float message_gain,
                  float* u_dev, float* stats_dev, float* attn_dev,
                  void* workspace_dev, size_t workspace_bytes, void* stream);

/*
 * Backward of gnca_step_fwd.  gx_dev = dL/dx_in (overwritten); gparams_dev (canonical layout) is
 * ACCUMULATED into (+=) so a rollout can sum over steps; zero it first for a single step.
 */
int gnca_step_bwd(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                  const float* x_in_dev, const float* fire_u_dev, float fire_rate,
                  const int32_t* offsets_host, int k, float message_gain,
                  const float* u_dev, const float* stats_dev,
                  const float* gout_dev, float* gx_dev, float* gparams_dev,
                  void* workspace_dev, size_t workspace_bytes, void* stream);

/* GraphAugmentation.forward alone: m [B,C,H,W] (+ optional attn [B,H,W]); bwd accumulates into gparams */
int gnca_graph_fwd(const gnca_model* m, const float* packed_dev, int B, int H, int W, const float* x_dev,
                   const int32_t* offsets_host, int k, float* msg_dev, float* attn_dev,
                   void* workspace_dev, size_t workspace_bytes, void* stream);
int gnca_graph_bwd(const gnca_model* m, const float* packed_dev, int B, int H, int W, const float* x_dev,
                   const int32_t* offsets_host, int k, const float* gmsg_dev, float* gx_dev,
                   float* gparams_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ rollout ----------------- */
size_t gnca_rollout_workspace_bytes(const gnca_model* m, int B, int H, int W, int T);

/*
 * T steps in one call.  x_hist_dev: NULL for inference, else [T+1][B][C][H][W] receives x_0..x_T
 * (what the backward recomputes from; x_T is also written to xT_dev).  stats_hist_dev: [T][B][2] or NULL.
 * u_hist_dev: optional [T][B][C][H][W]; when given (together with stats_hist_dev) the masked pre-norm update of
 * the ACTIVE cells of every step is kept, and gnca_rollout_bwd skips recomputing the forward MLP.
 * `impl`: 0 = auto, 1 = streaming per-step kernels (any shape), 2 = cluster-resident kernels
 * (state lives in shared memory across all T steps; needs the sample to fit, torus or classic: the
 * replicated-state kernel when the whole sample fits one CTA, else the banded one), 3 = banded kernel only.
 */
int gnca_rollout_fwd(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                     const gnca_schedule* sched, const float* x0_dev, float* xT_dev,
                     float* x_hist_dev, float* stats_hist_dev, float* u_hist_dev,
                     void* workspace_dev, size_t workspace_bytes, int impl, void* stream);

/*
 * Recording rollout for inference: the T steps of gnca_rollout_fwd (same `impl`, dispatch and fallbacks, same
 * GNCA_ERR_UNSUPPORTED combinations), keeping every `every`-th state and, optionally, the attention map of each kept step.
 *   - frames: F = gnca_record_frames(T, every) = T / every + 1; frames_dev[f] ([F][B][C][H][W]) = x_{f*every}, the
 *     state step f*every consumes (after the schedule's damage when f*every == damage_step).  A frozen sample
 *     (steps[b] <= t) shows its frozen state.  xT_dev always receives x_T, whether or not T % every == 0.
 *   - attention (attn_dev != NULL, graph models only): FA = ceil(T / every) maps, one per kept step f*every < T;
 *     attn_dev[f] ([FA][B][H][W]) is exactly the attention map gnca_step_fwd returns for x_{f*every} with that step's
 *     offsets (and, zero-padded shift, the per-sample softmax weights of that state).  It is computed for every
 *     sample, frozen ones included, and depends on neither the fire rate nor the message gain of the step.
 *   - T == 0: F = 1 (x_0) and FA = 0; every > T: F = 1.
 * No BPTT buffers: the workspace is the one of gnca_rollout_workspace_bytes.  Argument errors (every <= 0, frames_dev
 * NULL, attention on a classic model; k outside [0, GNCA_MAX_K] is GNCA_ERR_UNSUPPORTED) return before any launch.
 */
int gnca_record_frames(int T, int every); /* T / every + 1, or GNCA_ERR_ARG (T < 0, every <= 0) */
int gnca_rollout_record(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                        const gnca_schedule* sched, const float* x0_dev, float* xT_dev,
                        int every, float* frames_dev, float* attn_dev,
                        void* workspace_dev, size_t workspace_bytes, int impl, void* stream);

/*
 * Monitoring rollout: the T steps of gnca_rollout_fwd (same `impl`, dispatch and GNCA_ERR_UNSUPPORTED combinations;
 * xT_dev receives the same x_T), reducing each frame gnca_rollout_record would keep against a target instead of
 * keeping it.  Frame f (F = gnca_record_frames(T, every)) is x_{f*every}, as in gnca_rollout_record; per frame and
 * sample, with p = the premultiplied RGBA of the frame (rgb * alpha, alpha = channel 3) and d = p - target:
 *   - sums_dev[F][B][2]   = { sum of d^2 over the 4 channels and H*W cells,
 *                             sum of (clip(p, 0, 1) - clip(target, 0, 1))^2 over the 3 RGB channels };
 *   - counts_dev[F][B][2] = { cells with |d| < eps on all 4 channels, cells with alpha > m->alpha_thr }.
 * target_dev: [4][H][W] fp32, premultiplied.  The products and differences are rounded one operation at a time (no
 * FMA), the squares are summed in double over a fixed partition in a fixed order: two calls give bit-identical sums.
 * scratch_dev: gnca_metrics_scratch_bytes(m, B, H, W, T, every) bytes (0: bad arguments); the workspace is the one of
 * gnca_rollout_workspace_bytes.  No BPTT buffer.  Argument errors (a NULL pointer, every <= 0, eps < 0, C < 4) are
 * GNCA_ERR_ARG, a scratch or workspace too small is GNCA_ERR_WORKSPACE, k outside [0, GNCA_MAX_K] is
 * GNCA_ERR_UNSUPPORTED, all before any launch.
 */
size_t gnca_metrics_scratch_bytes(const gnca_model* m, int B, int H, int W, int T, int every);
int gnca_rollout_metrics(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                         const gnca_schedule* sched, const float* x0_dev, float* xT_dev, int every,
                         const float* target_dev, float eps, double* sums_dev, int32_t* counts_dev,
                         void* scratch_dev, size_t scratch_bytes, void* workspace_dev, size_t workspace_bytes,
                         int impl, void* stream);

/*
 * Many models in one rollout: gnca_rollout_record / gnca_rollout_metrics for a stack of n_models models that share the
 * descriptor `m`, the schedule and (metrics) the target -- e.g. the saved checkpoints of one training run.
 * packed_dev is [n_models][packed_total] (gnca_param_layout().packed_total floats per model, each buffer from
 * gnca_pack_weights).  B counts all samples and must be a multiple of n_models: sample b runs model b / (B / n_models),
 * so x0, frames, x_T, sums and counts keep their single-model shapes with the model-major B.  Each sample's cluster stages
 * its own model's weights, so the M * B samples fill the GPU the way one large batch does.
 *   - impl: 0 (auto) = the replicated-state kernel where it runs, else the banded one; 2 / 3 as in gnca_rollout_fwd.
 *     impl 1 (streaming) is GNCA_ERR_UNSUPPORTED, and so is a shape or model neither cluster kernel takes: there is no
 *     fallback to the streaming kernels.  T == 0 launches no step.
 *   - No attention maps and no BPTT.  With n_models == 1 the results are bit-identical to the single-model call on the
 *     same impl; model i's block equals the single-model call with model i on the same B, schedule and impl.
 * Argument errors return before any launch: those of gnca_rollout_record / gnca_rollout_metrics, n_models < 1,
 * B % n_models != 0 or impl outside [0, 3] are GNCA_ERR_ARG.  Scratch and workspace sizes are those of the total B.
 */
int gnca_rollout_record_models(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                               const gnca_schedule* sched, const float* x0_dev, float* xT_dev, int every,
                               float* frames_dev, void* workspace_dev, size_t workspace_bytes, int impl, void* stream);
int gnca_rollout_metrics_models(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                                const gnca_schedule* sched, const float* x0_dev, float* xT_dev, int every,
                                const float* target_dev, float eps, double* sums_dev, int32_t* counts_dev,
                                void* scratch_dev, size_t scratch_bytes, void* workspace_dev, size_t workspace_bytes,
                                int impl, void* stream);

/*
 * SSIM on the device.  The SSIM of a state is skimage's structural_similarity(pred, tgt, channel_axis=-1,
 * data_range=1.0) with every other argument at its default, where pred = clip(premultiplied RGB of the state, 0, 1)
 * (r * alpha rounded as for gnca_rollout_metrics, alpha = channel 3) and tgt = clip(target RGB, 0, 1).  Per channel: 7x7
 * uniform windows, cov_norm = 49/48, C1 = 0.01^2, C2 = 0.03^2, S = (2 ux uy + C1)(2 vxy + C2) / ((ux^2 + uy^2 + C1)
 * (vx + vy + C2)) averaged over the (H-6)(W-6) interior cells (the windows that lie inside the grid); SSIM is the mean
 * of the three channel means.  The window moments are taken in double and summed over a fixed partition in a fixed
 * order: two calls give bit-identical results.
 *
 * gnca_ssim_rgb: ssim_dev[B] (double) of the states x_dev [B][C][H][W] against target_dev [4][H][W] (premultiplied).
 * scratch_dev: gnca_ssim_rgb_scratch_bytes(B, H, W) bytes (0: bad arguments).
 *
 * gnca_rollout_metrics_ssim[_models]: gnca_rollout_metrics[_models] with, in addition, ssim_dev[F][B] (double) = the
 * SSIM of each frame.  sums, counts and x_T are those of the call without SSIM.  scratch_dev:
 * gnca_metrics_ssim_scratch_bytes(m, B, H, W, T, every) bytes (0: bad arguments, H or W < 7).
 *
 * Argument errors return before any launch: a NULL pointer, C < 4, H or W < 7, every <= 0 (and the other argument
 * errors of the calls without SSIM) are GNCA_ERR_ARG, a scratch too small is GNCA_ERR_WORKSPACE, k outside
 * [0, GNCA_MAX_K] or a shape no kernel family takes is GNCA_ERR_UNSUPPORTED.
 */
size_t gnca_ssim_rgb_scratch_bytes(int B, int H, int W);
int gnca_ssim_rgb(const float* x_dev, int B, int C, int H, int W, const float* target_dev, double* ssim_dev,
                  void* scratch_dev, size_t scratch_bytes, void* stream);
size_t gnca_metrics_ssim_scratch_bytes(const gnca_model* m, int B, int H, int W, int T, int every);
int gnca_rollout_metrics_ssim(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                              const gnca_schedule* sched, const float* x0_dev, float* xT_dev, int every,
                              const float* target_dev, float eps, double* sums_dev, int32_t* counts_dev,
                              double* ssim_dev, void* scratch_dev, size_t scratch_bytes, void* workspace_dev,
                              size_t workspace_bytes, int impl, void* stream);
int gnca_rollout_metrics_ssim_models(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                                     const gnca_schedule* sched, const float* x0_dev, float* xT_dev, int every,
                                     const float* target_dev, float eps, double* sums_dev, int32_t* counts_dev,
                                     double* ssim_dev, void* scratch_dev, size_t scratch_bytes, void* workspace_dev,
                                     size_t workspace_bytes, int impl, void* stream);

/*
 * A target per model: gnca_rollout_metrics_ssim_models where model i (samples [i * B / n_models, (i + 1) * B /
 * n_models)) is measured against targets_dev[i] ([n_models][4][H][W], premultiplied RGBA), for a target sweep.
 * ssim_dev = NULL skips the SSIM (gnca_rollout_metrics_models).  Scratch from gnca_metrics_scratch_bytes, or
 * gnca_metrics_ssim_scratch_bytes with ssim_dev.  With every targets_dev[i] equal to one target the results are
 * bit-identical to the _models calls with that target; model i's block equals block i of the _models call with the
 * target targets_dev[i].
 * Argument errors return before any launch: a NULL targets_dev, n_models < 1 and B % n_models != 0 are GNCA_ERR_ARG;
 * every other case is that of the _models calls (GNCA_ERR_UNSUPPORTED for impl 1 and for shapes no cluster kernel
 * takes).
 */
int gnca_rollout_metrics_targets(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                                 const gnca_schedule* sched, const float* x0_dev, float* xT_dev, int every,
                                 const float* targets_dev, float eps, double* sums_dev, int32_t* counts_dev,
                                 double* ssim_dev, void* scratch_dev, size_t scratch_bytes, void* workspace_dev,
                                 size_t workspace_bytes, int impl, void* stream);

/* BPTT: given gT = dL/dx_T and the x_hist of the forward, produce g0 = dL/dx_0 and ACCUMULATE gparams. */
int gnca_rollout_bwd(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                     const gnca_schedule* sched, const float* x_hist_dev, const float* stats_hist_dev,
                     const float* u_hist_dev,
                     const float* gT_dev, float* g0_dev, float* gparams_dev,
                     void* workspace_dev, size_t workspace_bytes, int impl, void* stream);

/*
 * Differentiable frames: BPTT of a loss on the strided frames of a recording rollout (frame f = x_{f*every}, exactly the
 * frames of gnca_rollout_record) and on x_T.  g_frames_dev ([F][B][C][H][W], F = gnca_record_frames(T, every)) holds
 * dL/dframe_f; NULL is exactly gnca_rollout_bwd / gnca_rollout_bwd_bptt (which are these functions with NULL).
 *   - At step t = f*every, dL/dx_t = (backward of step t) + dL/dframe_f.  The damage mask of damage_step multiplies that
 *     SUM: the frame is the state after the damage.  A frozen sample (steps[b] <= t) passes g through and still
 *     receives its frame gradients.
 *   - When T % every == 0, frame F-1 and x_T hold equal values but are two outputs: their gradients add.  T == 0:
 *     g0 = gT + g_frames[0].
 * The result equals autograd through T sequential steps with the same schedule.  Argument errors return before any
 * launch: `every <= 0` with a frame gradient, or a NULL required pointer, is GNCA_ERR_ARG; k outside [0, GNCA_MAX_K]
 * is GNCA_ERR_UNSUPPORTED.  The workspaces are those of gnca_rollout_workspace_bytes.
 */
int gnca_rollout_bwd_frames(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                            const gnca_schedule* sched, const float* x_hist_dev, const float* stats_hist_dev,
                            const float* u_hist_dev, int every, const float* g_frames_dev,
                            const float* gT_dev, float* g0_dev, float* gparams_dev,
                            void* workspace_dev, size_t workspace_bytes, int impl, void* stream);

/*
 * Checkpointed BPTT: memory that does not grow with T on the streaming path.  The forward is gnca_rollout_record with
 * impl = 1 (streaming): its frames x_{j*every} are the checkpoints.  They must come from the streaming kernels, because
 * the backward recomputes every segment with them and relies on reproducing the forward bit for bit.  The backward
 * keeps the checkpoints plus one segment: (every - 1) states, `every` pre-norm updates and `every` [B][2] statistics
 * instead of the T + 1 states and T updates of the dense history.
 *
 * gnca_ckpt_segment_bytes: bytes of that segment buffer, each region 256-byte aligned; 0 on bad arguments.
 *
 * gnca_rollout_bwd_ckpt: ckpt_dev [T/every+1][B][C][H][W] = the frames gnca_rollout_record(..., every, impl = 1) wrote.
 * Segments are processed last to first.  For each one, the forward of its steps is recomputed from its checkpoint into
 * segment_dev, with the streaming kernels, the same schedule and the absolute step indices (Philox, steps[b], fire_u and
 * the offsets key on them); a checkpoint at damage_step is already post-damage, a damage step inside a segment is applied
 * to the recomputed state.  Then the per-step backward runs over the segment.  g_frames_dev (optional, same shape as
 * ckpt_dev) has the semantics of gnca_rollout_bwd_frames.  The result equals gnca_rollout_bwd on the full streaming
 * history.  gparams is ACCUMULATED.  Argument errors return before any launch: a NULL required pointer, every <= 0 or
 * T < 0 is GNCA_ERR_ARG; a segment or workspace (gnca_rollout_workspace_bytes) too small is GNCA_ERR_WORKSPACE; k
 * outside [0, GNCA_MAX_K] is GNCA_ERR_UNSUPPORTED.
 */
size_t gnca_ckpt_segment_bytes(const gnca_model* m, int B, int H, int W, int every);
int gnca_rollout_bwd_ckpt(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                          const gnca_schedule* sched, const float* ckpt_dev, int every,
                          const float* g_frames_dev, const float* gT_dev, float* g0_dev, float* gparams_dev,
                          void* segment_dev, size_t segment_bytes,
                          void* workspace_dev, size_t workspace_bytes, void* stream);

/*
 * Resident BPTT (16-channel / 128-hidden models, classic or torus graph, grids up to 2048 cells with W % 4 == 0).
 * Instead of the dense x_t / u_t history the forward keeps one compact record per ACTIVE cell and step (perception,
 * pre-norm update, gathered sender state ...) plus three bitmaps and the GroupNorm statistics per step, in the opaque
 * buffer `bptt_dev` (gnca_bptt_bytes; 0 = configuration not supported -> use gnca_rollout_fwd/_bwd).  The backward
 * is one cluster-resident kernel for the propagation of dL/dx plus one batched pass over all records for the weight
 * gradients.  x_hist_dev may be NULL (it is not needed by the backward).  gparams_dev is ACCUMULATED into.
 */
size_t gnca_bptt_bytes(const gnca_model* m, int B, int H, int W, int T);
int gnca_rollout_fwd_bptt(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                          const gnca_schedule* sched, const float* x0_dev, float* xT_dev, float* x_hist_dev,
                          void* bptt_dev, size_t bptt_bytes, void* workspace_dev, size_t workspace_bytes,
                          void* stream);
int gnca_rollout_bwd_bptt(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                          const gnca_schedule* sched, void* bptt_dev, size_t bptt_bytes, const float* gT_dev,
                          float* g0_dev, float* gparams_dev, void* workspace_dev, size_t workspace_bytes,
                          void* stream);
/* The record-based forward of gnca_rollout_fwd_bptt keeping the frames of gnca_rollout_record instead of a full
 * history: frames_dev[f] = x_{f*every} ([F][B][C][H][W], non-NULL, every > 0); xT_dev always receives x_T. */
int gnca_rollout_fwd_bptt_record(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                                 const gnca_schedule* sched, const float* x0_dev, float* xT_dev, int every,
                                 float* frames_dev, void* bptt_dev, size_t bptt_bytes, void* workspace_dev,
                                 size_t workspace_bytes, void* stream);
/* gnca_rollout_bwd_bptt with the frame gradients of gnca_rollout_bwd_frames */
int gnca_rollout_bwd_bptt_frames(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                                 const gnca_schedule* sched, void* bptt_dev, size_t bptt_bytes, int every,
                                 const float* g_frames_dev, const float* gT_dev, float* g0_dev, float* gparams_dev,
                                 void* workspace_dev, size_t workspace_bytes, void* stream);

/*
 * Resident BPTT of the zero-padded graph shift (the graph default: GNCA_F_GRAPH without GNCA_F_TORUS), for
 * 16-channel / 128-hidden models with d_model <= 32, at most 16 offsets per step, grids up to 2048 cells with W % 4 == 0.
 * gnca_bptt_bytes stays 0 for these models; this path has its own buffer and entry points.
 *
 * gnca_bptt_zp_bytes: bytes of `bptt_dev`: the records, bitmaps and statistics of gnca_bptt_bytes, then x_t of every
 * step ([T+1][B][C][H][W]), the softmax weights and per-(channel, row) sums of x_t of every step with the message on,
 * one per-cell scratch and the per-sample Q/K/scaling gradients.  0 for a classic or torus model, an unsupported
 * model or shape, or bad arguments.
 *
 * gnca_rollout_fwd_bptt_zp: the T steps on the resident zero-pad forward kernel, keeping that buffer.  frames_dev
 * (optional, [T/every+1][B][C][H][W]) receives x_{f*every} (every > 0; every = 1 is the full history); xT_dev always
 * receives x_T, bit-equal to gnca_rollout_fwd.  GNCA_ERR_UNSUPPORTED (before any launch) where the forward or the
 * backward has no resident kernel for the batch, shape or offsets (a grid no taller or wider than the largest offset).
 *
 * gnca_rollout_bwd_bptt_zp: from that buffer (same schedule), gT = dL/dx_T and the optional frame gradients of
 * gnca_rollout_bwd_bptt_frames, produce g0 = dL/dx_0 and ACCUMULATE gparams, the attention's wq, bq, wk, bk and
 * scaling included.  One cluster-resident launch propagates dL/dx through the message, the softmax weights and the
 * pooled query / keys; the weight gradients follow as in gnca_rollout_bwd_bptt.  Workspace: gnca_rollout_workspace_bytes.
 *
 * Argument errors return before any launch: a NULL required pointer, B, H or W <= 0, T < 0, or every <= 0 with frames
 * is GNCA_ERR_ARG; a buffer or workspace too small is GNCA_ERR_WORKSPACE; k outside [0, GNCA_MAX_K] or an unsupported
 * configuration is GNCA_ERR_UNSUPPORTED.
 */
size_t gnca_bptt_zp_bytes(const gnca_model* m, int B, int H, int W, int T);
int gnca_rollout_fwd_bptt_zp(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                             const gnca_schedule* sched, const float* x0_dev, float* xT_dev, int every, float* frames_dev,
                             void* bptt_dev, size_t bptt_bytes, void* workspace_dev, size_t workspace_bytes,
                             void* stream);
int gnca_rollout_bwd_bptt_zp(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                             const gnca_schedule* sched, void* bptt_dev, size_t bptt_bytes, int every,
                             const float* g_frames_dev, const float* gT_dev, float* g0_dev, float* gparams_dev,
                             void* workspace_dev, size_t workspace_bytes, void* stream);

/*
 * Training many models in one rollout: the resident BPTT (gnca_rollout_fwd_bptt / _bwd_bptt, and the _zp pair for the
 * zero-padded graph shift) for a stack of n_models models that share the descriptor `m` and the schedule -- e.g. the
 * seeds or learning rates of a sweep.  packed_dev is [n_models][packed_total] as in gnca_rollout_record_models; B counts
 * all samples and must be a multiple of n_models: sample b runs model b / (B / n_models), so x0, x_T, gT and g0 keep
 * their single-model shapes with the model-major B.  The record buffer is that of the single-model call on the total B
 * (gnca_bptt_bytes / gnca_bptt_zp_bytes).
 *   - The forward writes no history or frames; x_T equals gnca_rollout_record_models on the same impl 0.
 *   - The backward ACCUMULATES gparams_dev[n_models][param_total]: model i's gradients in row i, summed over its own
 *     samples only, in a fixed order (no float atomics: two calls are bit-identical).  With n_models == 1 every output
 *     is bit-identical to the single-model call.  Model i's block of g0 equals the single-model call of model i on the
 *     whole batch with gT zero outside block i; its parameter gradients equal that call's up to the summation order.
 *   - Workspace: gnca_rollout_workspace_models_bytes, which holds at least one weight-gradient partial per model (0 on
 *     bad arguments).
 *   - No frame gradients, no checkpoints and no streaming fallback: a batch or shape the resident BPTT has no
 *     configuration for is GNCA_ERR_UNSUPPORTED.
 * Errors return before any launch: a NULL required pointer, n_models < 1, B % n_models != 0, B, H or W <= 0 or T < 0 is
 * GNCA_ERR_ARG; a buffer or workspace too small is GNCA_ERR_WORKSPACE; k outside [0, GNCA_MAX_K] or an unsupported
 * model, batch or shape is GNCA_ERR_UNSUPPORTED.
 */
size_t gnca_rollout_workspace_models_bytes(const gnca_model* m, int n_models, int B, int H, int W, int T);
int gnca_rollout_fwd_bptt_models(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                                 const gnca_schedule* sched, const float* x0_dev, float* xT_dev, void* bptt_dev,
                                 size_t bptt_bytes, void* workspace_dev, size_t workspace_bytes, void* stream);
int gnca_rollout_bwd_bptt_models(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                                 const gnca_schedule* sched, void* bptt_dev, size_t bptt_bytes, const float* gT_dev,
                                 float* g0_dev, float* gparams_dev, void* workspace_dev, size_t workspace_bytes,
                                 void* stream);
int gnca_rollout_fwd_bptt_zp_models(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                                    const gnca_schedule* sched, const float* x0_dev, float* xT_dev, void* bptt_dev,
                                    size_t bptt_bytes, void* workspace_dev, size_t workspace_bytes, void* stream);
int gnca_rollout_bwd_bptt_zp_models(const gnca_model* m, const float* packed_dev, int n_models, int B, int H, int W,
                                    const gnca_schedule* sched, void* bptt_dev, size_t bptt_bytes, const float* gT_dev,
                                    float* g0_dev, float* gparams_dev, void* workspace_dev, size_t workspace_bytes,
                                    void* stream);

/*
 * Checkpointed resident BPTT: the resident backward with memory that does not grow with T.  The forward keeps only the
 * states x_{j*every}; the backward recomputes the records of one `every`-step segment at a time, last segment first,
 * with the resident forward kernel, and runs the resident backward over them.  Eligible configurations are those of
 * gnca_bptt_bytes (0 = not supported), and the launch must have a resident backward for the batch and shape.
 *
 * gnca_bptt_ckpt_bytes: bytes of the segment buffer: the records, bitmaps and statistics of `every` steps
 * (gnca_bptt_bytes(m, B, H, W, every)), then one [B][C][H][W] gradient carried across segment boundaries and one
 * [B][C][H][W] x_T scratch of the recompute, each 256-byte aligned.  0 on bad arguments or an ineligible configuration.
 *
 * gnca_rollout_fwd_bptt_ckpt: the T steps on the resident forward kernel, without records; ckpt_dev
 * ([T/every+1][B][C][H][W], the frames of gnca_rollout_record) receives x_{j*every}, after the schedule's damage when
 * j*every == damage_step; xT_dev receives x_T.  It uses the kernel and launch configuration of the recompute (they depend
 * on B and H*W only), so the backward reproduces every step bit for bit.  GNCA_ERR_UNSUPPORTED where the resident
 * backward does not exist for the model, batch or shape.
 *
 * gnca_rollout_bwd_bptt_ckpt: from the checkpoints of gnca_rollout_fwd_bptt_ckpt (same schedule and `every`) and
 * gT = dL/dx_T, produce g0 = dL/dx_0 and ACCUMULATE gparams.  Segment j covers steps [j*every, min((j+1)*every, T)); its
 * forward restarts from ckpt[j] at that absolute step (fire rates, gains, offsets, fire_u, the Philox counter and
 * steps[b] keep their absolute indices), without re-applying a damage at the checkpoint; the backward still multiplies
 * dL/dx by the mask at damage_step.  g0 equals the unsegmented gnca_rollout_bwd_bptt bit for bit; gparams match it up to
 * the summation order.  segment_dev: gnca_bptt_ckpt_bytes(every) bytes; workspace: gnca_rollout_workspace_bytes.
 * Argument errors return before any launch: a NULL required pointer, every <= 0 or T < 0 is GNCA_ERR_ARG; a segment
 * or workspace too small is GNCA_ERR_WORKSPACE; k outside [0, GNCA_MAX_K] is GNCA_ERR_UNSUPPORTED.  It is
 * gnca_rollout_bwd_bptt_ckpt_frames with frames_dev = ckpt_dev, ckpt_every = every and no frame gradients.
 *
 * gnca_rollout_bwd_bptt_ckpt_frames: the same backward with frame gradients, for a loss on recorded frames.  frames_dev
 * ([T/every+1][B][C][H][W]) holds x_{f*every}, written by gnca_rollout_fwd_bptt_ckpt(..., every, frames_dev); the
 * checkpoints are frames_dev[j * ckpt_every / every], so segments are ckpt_every steps long.  g_frames_dev (optional,
 * same shape) holds dL/dx_{f*every}: segment j adds frames [t0/every, (t0+n)/every) at their steps, before the damage
 * mask, with the semantics of gnca_rollout_bwd_bptt_frames; when T % every == 0 the last frame is x_T and is added to
 * gT once, before the last segment.  T = 0 gives g0 = gT + g_frames[0].  segment_dev: gnca_bptt_ckpt_bytes(ckpt_every)
 * bytes.  A ckpt_every that is not a positive multiple of every is GNCA_ERR_ARG; the other argument errors are those
 * of gnca_rollout_bwd_bptt_ckpt, and a configuration without the checkpointed resident BPTT (gnca_bptt_ckpt_bytes
 * = 0, e.g. the zero-padded graph shift) is GNCA_ERR_UNSUPPORTED, all before any launch.
 */
size_t gnca_bptt_ckpt_bytes(const gnca_model* m, int B, int H, int W, int every);
int gnca_rollout_fwd_bptt_ckpt(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                               const gnca_schedule* sched, const float* x0_dev, float* xT_dev, int every, float* ckpt_dev,
                               void* workspace_dev, size_t workspace_bytes, void* stream);
int gnca_rollout_bwd_bptt_ckpt(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                               const gnca_schedule* sched, const float* ckpt_dev, int every, const float* gT_dev,
                               float* g0_dev, float* gparams_dev, void* segment_dev, size_t segment_bytes,
                               void* workspace_dev, size_t workspace_bytes, void* stream);
int gnca_rollout_bwd_bptt_ckpt_frames(const gnca_model* m, const float* packed_dev, int B, int H, int W,
                                      const gnca_schedule* sched, const float* frames_dev, int every, int ckpt_every,
                                      const float* g_frames_dev, const float* gT_dev, float* g0_dev, float* gparams_dev,
                                      void* segment_dev, size_t segment_bytes, void* workspace_dev,
                                      size_t workspace_bytes, void* stream);

/*
 * HOST function (no device work): T consecutive `random.sample(range(n), k)` draws of CPython's `random` module on
 * its own MT19937 state (`mt[624]`, `*mti` = random.getstate()[1][:624], [624]); state advanced in place so the caller
 * can `random.setstate` it back -- the python RNG stream stays exactly what T reference `forward` calls consume
 * (graph_augmentation.py:120-121).  out_idx: [T][k] indices into the offset table.
 */
int gnca_host_sample_indices(uint32_t* mt, int32_t* mti, int n, int k, int T, int32_t* out_idx);
/*
 * HOST function: the same T draws taken from `n_words` raw MT19937 outputs (the caller pulled them with
 * random.getrandbits(32 * n_words), first output = word 0); writes the chosen (dy, dx) pairs of `table` [n][2] to
 * out_off [T][k][2] and the number of words consumed to *used -- the caller restores the saved state and skips exactly
 * `used` outputs, so the python stream again equals T reference forward calls.  GNCA_ERR_UNSUPPORTED: block too short.
 */
int gnca_host_sample_offsets_words(const uint32_t* words, int n_words, const int8_t* table, int n, int k, int T,
                                   int8_t* out_off, int32_t* used);

/* ------------------------------------------------------------------ training glue ----------- */
/* per_sample[b] = mean_{4HW}([rgb*a, a] - target)^2 ; gx (optional) = d(scale * sum_b per_sample[b])/dx, [B,C,H,W] */
int gnca_loss_premult_rgba(int B, int C, int H, int W, const float* x_dev, const float* target_dev /*[4,H,W]*/,
                           float* per_sample_dev, float* gx_dev, float scale, void* stream);
/* the same with one target per block of B / n_targets samples: sample b against targets_dev[b / (B / n_targets)]
 * ([n_targets][4][H][W]); n_targets == 1 is bit-identical to gnca_loss_premult_rgba.  n_targets < 1 or
 * B % n_targets != 0 is GNCA_ERR_ARG. */
int gnca_loss_premult_rgba_targets(int B, int C, int H, int W, const float* x_dev, const float* targets_dev,
                                   int n_targets, float* per_sample_dev, float* gx_dev, float scale, void* stream);
/*
 * For each of n_seg parameter tensors (seg_off[i]..seg_off[i+1] in the flat buffers, host array of n_seg+1):
 * g /= (||g||_2 + 1e-8) unless seg_has_grad[i]==0 (skipped like a None grad), then torch.optim.Adam
 * with coupled L2 weight decay.  step is 1-based.
 */
int gnca_normalize_adam(float* params_dev, float* grads_dev, float* exp_avg_dev, float* exp_avg_sq_dev,
                        const int64_t* seg_off_host, const int32_t* seg_has_grad_host, int n_seg,
                        int normalize, float lr, float beta1, float beta2, float eps, float weight_decay,
                        int64_t step, void* stream);
/* x *= mask (damage.py as multiplicative masks); mask [B,C,H,W] */
int gnca_apply_mask(int64_t n, float* x_dev, const float* mask_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GNCA_H_ */
