"""Train M same-architecture models at once: one training iteration of GraphNCATrainer (fire="philox") for each of
them, with the rollout, loss and BPTT of all M as ONE stacked resident BPTT (rollout.rollout_models_fwd_raw /
rollout_models_bwd_raw).  At the batch sizes the reference trains with (16, 32) one model leaves most of the GPU idle,
because a sample's cluster of at most 8 CTAs sets the step time; a seed or learning-rate sweep fills it instead.

Each model keeps its own SamplePool and FusedNormalizedAdam, so its checkpoints (utils/checkpoint.py, torch_state_dict)
are those of a single-model run.  The models share the schedule of an iteration (step counts, fire rates, offsets, the
Philox stream) and the damage policy draw; the pools are drawn model by model.  They share the target too, or each
trains towards its own (a target sweep: one model per image).
"""
from __future__ import annotations

import random
from typing import Dict, Optional, Sequence

import numpy as np
import torch

from ..rollout import _model_stack, _stack_packed, rollout_models_bwd_raw, rollout_models_fwd_raw
from ..utils.damage import sample_damage_mask
from .dp import Shard, worst_k_indices
from .optim import FusedNormalizedAdam
from .pool import SamplePool
from .trainer import GraphNCATrainer, TrainConfig, premult_loss


class PopulationTrainer(GraphNCATrainer):
    """`train_step(epoch)` = per model: pool sample; once for the stacked batch: damage policy, schedule
    (GraphNCATrainer._draw_schedule over M*B samples), stacked forward with records, premultiplied loss at scale 1/B,
    stacked BPTT; per model: normalise + Adam at its learning rate under the StepLR schedule, worst-k and random reseed,
    pool replace.  With one model it consumes the host RNG exactly as GraphNCATrainer(fire="philox") and gives
    bit-identical parameters, Adam moments, losses and pool.

    `target`: [4, H, W] premultiplied RGBA shared by every model, or [M, 4, H, W], model i training towards target[i]
    (premult_loss with per-model targets; nothing else about the iteration changes).

    `learning_rates`: one base learning rate per model (default cfg.learning_rate for all).  Production mode only:
    fire="torch", a BPTT budget, rollout_impl other than "auto" / "resident", more than one rank, or a learning-rate list
    whose length is not M, or a [M', 4, H, W] target with M' != M raise ValueError."""

    def __init__(self, models: Sequence, target: torch.Tensor, cfg: TrainConfig, *,
                 learning_rates: Optional[Sequence[float]] = None, seed_fn=None):
        models = list(models)
        if cfg.fire != "philox":
            raise ValueError("PopulationTrainer: fire must be 'philox' (there is no reference torch.rand stream to "
                             "replay for a population)")
        if cfg.bptt_budget_bytes is not None:
            raise ValueError("PopulationTrainer: bptt_budget_bytes is not supported (a stack has no checkpointed BPTT)")
        if cfg.rollout_impl not in ("auto", "resident"):
            raise ValueError(f"PopulationTrainer: rollout_impl must be 'auto' or 'resident', got {cfg.rollout_impl!r}")
        if Shard(cfg.batch_size).world > 1:
            raise ValueError("PopulationTrainer: runs on one rank (no data-parallel populations)")
        _model_stack(models, None, "PopulationTrainer", cfg.rollout_impl)
        M = len(models)
        if target.dim() == 4 and target.shape[0] != M:
            raise ValueError(f"PopulationTrainer: {target.shape[0]} targets for {M} models")
        lrs = [cfg.learning_rate] * M if learning_rates is None else [float(v) for v in learning_rates]
        if len(lrs) != M:
            raise ValueError(f"PopulationTrainer: {len(lrs)} learning rates for {M} models")
        super().__init__(models[0], target, cfg, seed_fn=seed_fn)
        self.models, self.learning_rates = models, lrs
        self.opt.lr = lrs[0]
        self.pools = [self.pool] + [SamplePool(cfg.pool_size, self.seed_fn, device=self.device) for _ in models[1:]]
        self.opts = [self.opt] + [FusedNormalizedAdam(m, lr=lr, weight_decay=cfg.weight_decay, normalize=True)
                                  for m, lr in zip(models[1:], lrs[1:])]
        self.shard = Shard(M * cfg.batch_size)      # _draw_schedule sizes the schedule by the local batch

    def lr_at(self, epoch: int, i: int = 0) -> float:
        """Model i's StepLR rate (GraphNCATrainer.lr_at with its own base rate)."""
        return self.learning_rates[i] * self.cfg.scheduler_gamma ** ((epoch - 1) // self.cfg.scheduler_step_size)

    def train_step(self, epoch: int = 1) -> Dict:
        cfg = self.cfg
        B, M = cfg.batch_size, len(self.models)
        draws = [pool.sample(B) for pool in self.pools]
        idx = [d[0] for d in draws]
        state = torch.cat([d[1] for d in draws]) if M > 1 else draws[0][1]
        D = sample_damage_mask(state, cfg.damage, epoch, fast=True) if cfg.damage else None
        sched, steps_host = self._draw_schedule(epoch, M * B, state)
        if D is not None:
            sched.damage, sched.damage_layout, sched.damage_step = D.plane, D.layout, 0
        desc, packed = self.model.model_desc(), _stack_packed(self.models)
        xT, hist = rollout_models_fwd_raw(desc, packed, state.contiguous(), sched)
        per, gxT = premult_loss(xT, self.target, 1.0 / B)                 # each model: the mean over its own B
        _, gflat = rollout_models_bwd_raw(desc, packed, hist, sched, gxT)
        for i, opt in enumerate(self.opts):
            opt.step(gflat[i], lr=self.lr_at(epoch, i))
        per = per.view(M, B)
        worst_all = []
        for i in range(M):
            worst = worst_k_indices(per[i], cfg.reset_worst_prob)
            rand_idx = int(torch.randint(0, B, (1,)).item()) if random.random() < cfg.random_reseed_prob else None
            new_states = xT[i * B:(i + 1) * B]
            if worst is not None and worst.numel() > 0:
                new_states = new_states.clone()
                new_states[worst] = self.seed_fn(len(worst))
            if rand_idx is not None:
                new_states = new_states.clone()
                new_states[rand_idx:rand_idx + 1] = self.seed_fn(1)
            self.pools[i].replace(idx[i], new_states)
            worst_all.append(worst)
        self.last = {"per_sample": per, "loss": per.mean(1), "steps": steps_host, "worst": worst_all, "gflat": gflat,
                     "x_T": xT, "cell_updates": int(np.minimum(steps_host, sched.T).sum()) * self.img * self.img}
        return self.last
