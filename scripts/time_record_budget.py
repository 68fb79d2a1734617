"""Cost and memory of frame losses under a BPTT budget: record_rollout(..., differentiable=True, bptt_budget=N) against
record_rollout(..., checkpoint=True) (streaming checkpoints) and, where they fit, the unbudgeted records.  Timed with
CUDA events around whole forward + loss + backward calls through the public autograd API.

Cases (trained torus weights, 40x40x16, B = 32, a grown pattern, fire rate 0.5 on the in-kernel Philox stream, a frame
every 50 steps, L = sum over frames of mean(frame[:, :4]^2) + mean(x_T[:, :4]^2)):
  T = 1000: checkpoint=True against budgets of 3 and 4 GiB (the record buffer would take 72.9 GB, above
      BPTT_MAX_BYTES).  One resident segment of 50 steps takes 3.40 GiB, so 3 GiB plans the streaming checkpoints and
      4 GiB the resident ones;
  T = 300: the unbudgeted records against a 4 GiB budget below them, and checkpoint=True.
Each arm records the plan its forward took.  Peak memory = torch.cuda.max_memory_allocated over the first timed call,
above what was allocated before it.  The arms of a case alternate (forward order, then reverse), so the spread shows.

Reads the card's name and power limit in the same run and writes profiles/r06_record_budget.json (or --out).  Needs a
CUDA device; it has no CPU path.

    python scripts/time_record_budget.py [--out profiles/r06_record_budget.json]
"""
from __future__ import annotations

import argparse
import json
import os
import random
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import graph_neural_cellular_automata_b200 as G  # noqa: E402
from graph_neural_cellular_automata_b200.rollout import make_schedule, record_rollout, rollout  # noqa: E402
from graph_neural_cellular_automata_b200.utils.nca_init import make_seed  # noqa: E402

EVERY = 50


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def arm(m, x0, s, **kw):
    """one forward + loss + backward; returns the plan the forward took (None without a budget)"""
    def run():
        for q in m.parameters():
            q.grad = None
        xg = x0.clone().requires_grad_(True)
        tr = record_rollout(m, xg, s, every=EVERY, differentiable=True, **kw)
        loss = (tr.states[:, :, :4] ** 2).mean(dim=(1, 2, 3, 4)).sum() + (tr.x_T[:, :4] ** 2).mean()
        plan = getattr(tr.x_T.grad_fn, "plan", None)
        loss.backward()
        return plan
    return run


def time_ms(fn, reps, warmup=1):
    """mean time of fn() between two CUDA events over `reps` calls after `warmup` untimed ones, the peak bytes allocated
    above the starting point during the first timed call, and fn's result"""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for i in range(reps):
        a.record()
        out = fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
        if i == 0:
            peak = torch.cuda.max_memory_allocated() - base
    return sum(ms) / len(ms), peak, out


def measure(fns, reps):
    out = {k: {"ms": [], "peak_gb": None, "plan": None} for k in fns}
    for rnd in range(2):
        for k in (list(fns) if rnd == 0 else list(reversed(list(fns)))):
            ms, peak, plan = time_ms(fns[k], reps)
            out[k]["ms"].append(round(ms, 3))
            out[k]["peak_gb"] = round(peak / 1e9, 3)
            out[k]["plan"] = list(plan) if plan is not None else None
            torch.cuda.empty_cache()
    return out


def report(dev, name, r):
    print(f"[{dev}] {name}: ms per call (two alternating runs), peak GB, plan")
    for k, v in r.items():
        print(f"  {k:20s} {v['ms'][0]:10.2f} {v['ms'][1]:10.2f} ms   peak {v['peak_gb']:8.3f} GB   {v['plan']}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_record_budget.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_record_budget.py needs a CUDA device")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import load_params      # tests/conftest.py: the trained-weight fixture loader
    dev = card()
    res = {"card": dev, "every": EVERY, "cases": {}}
    torch.manual_seed(42); random.seed(42)
    m = G.NeuralCAGraph(16, update_hidden=128, img_size=40, update_gain=0.05, alpha_thr=0.12, message_gain=0.25,
                        hidden_only=True, graph_zero_padded_shift=False)
    m.load_state_dict(load_params("weights_graph_ep960.npz"), strict=False)
    m = m.cuda()
    B, H = 32, 40
    with torch.no_grad():
        x0 = rollout(m, make_seed(16, H, B, device="cuda"), make_schedule(m, B, H, H, 48, fire_rate=0.6, seed=4))

    for T, reps, fns in (
            (1000, 2, lambda s: {"checkpoint": arm(m, x0, s, checkpoint=True),
                                 "budget_3GiB": arm(m, x0, s, bptt_budget=3 << 30),
                                 "budget_4GiB": arm(m, x0, s, bptt_budget=4 << 30)}),
            (300, 4, lambda s: {"records": arm(m, x0, s),
                                "budget_4GiB": arm(m, x0, s, bptt_budget=4 << 30),
                                "checkpoint": arm(m, x0, s, checkpoint=True)})):
        s = make_schedule(m, B, H, H, T, fire_rate=0.5, seed=7 + T)
        r = measure(fns(s), reps)
        name = f"40x40x16_torus_B32_T{T}_every{EVERY}"
        res["cases"][name] = r
        report(dev, name, r)

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
