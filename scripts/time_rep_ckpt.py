"""Cost and memory of the checkpointed resident BPTT against the unsegmented resident BPTT and, at T = 1000, against
the dense-history streaming fallback that rollout() takes there without a budget.  Timed with CUDA events around whole
forward + loss + backward calls (rollout_fwd_raw / rollout_bwd_raw, the calls of GraphNCATrainer.train_step).

Cases (trained torus weights, 40x40x16, B = 32, a grown pattern, fire rate 0.5 on the in-kernel Philox stream):
  T = 64 and T = 400: unsegmented records against checkpoint strides K in {8, 16, 32, 64};
  T = 1000: the streaming fallback (the record buffer would exceed BPTT_MAX_BYTES) against the resident checkpointed
      path under a 4 GiB budget (the stride bptt_plan picks).
Peak memory = torch.cuda.max_memory_allocated over one call, above what was allocated before it.  The variants of a
case alternate (forward order, then reverse), so the spread shows.

Reads the card's name and power limit in the same run and writes profiles/r04_rep_ckpt.json (or --out).  Needs a CUDA
device; it has no CPU path.

    python scripts/time_rep_ckpt.py [--out profiles/r04_rep_ckpt.json]
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
from graph_neural_cellular_automata_b200.rollout import (_ckpt_bwd_raw, _ckpt_fwd_raw, bptt_plan,  # noqa: E402
                                                         make_schedule, rollout, rollout_bwd_raw, rollout_fwd_raw)
from graph_neural_cellular_automata_b200.utils.nca_init import make_seed  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def time_ms(fn, reps, warmup=1):
    """mean time of fn() between two CUDA events over `reps` calls after `warmup` untimed ones, and the peak bytes
    allocated above the starting point during the first timed call"""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for i in range(reps):
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
        if i == 0:
            peak = torch.cuda.max_memory_allocated() - base
    return sum(ms) / len(ms), peak


def loss_grad(xT):
    """dL/dx_T of L = mean(x_T[:, :4]^2)"""
    g = torch.zeros_like(xT)
    g[:, :4] = 2.0 * xT[:, :4] / xT[:, :4].numel()
    return g


def variants(m, x0, s, ks, *, unsegmented=True, fallback=False, budget=None):
    desc, packed = m.model_desc(), m.packed_weights()

    def plain(impl):
        def run():
            xT, hist = rollout_fwd_raw(desc, packed, x0, s, history=True, impl=impl, keep_x=False)
            rollout_bwd_raw(desc, packed, hist, s, loss_grad(xT), impl=impl)
        return run

    def seg(k):
        def run():
            xT, ckpt = _ckpt_fwd_raw(desc, packed, x0, s, k, resident=True)
            _ckpt_bwd_raw(desc, packed, ckpt, s, k, True, loss_grad(xT))
        return run

    def budgeted():
        xT, hist = rollout_fwd_raw(desc, packed, x0, s, history=True, keep_x=False, bptt_budget=budget)
        rollout_bwd_raw(desc, packed, hist, s, loss_grad(xT))

    fns = {}
    if unsegmented:
        fns["unsegmented"] = plain(0)
    if fallback:
        fns["streaming_fallback"] = plain(0)
    for k in ks:
        fns[f"K{k}"] = seg(k)
    if budget is not None:
        fns["budget"] = budgeted
    return fns


def measure(fns, reps):
    out = {k: {"ms": [], "peak_gb": None} for k in fns}
    for rnd in range(2):
        for k in (list(fns) if rnd == 0 else list(reversed(list(fns)))):
            ms, peak = time_ms(fns[k], reps)
            out[k]["ms"].append(round(ms, 3))
            out[k]["peak_gb"] = round(peak / 1e9, 3)
            torch.cuda.empty_cache()
    return out


def report(dev, name, r):
    print(f"[{dev}] {name}: ms per call (two alternating runs), peak GB")
    for k, v in r.items():
        if isinstance(v, dict) and "ms" in v:
            print(f"  {k:20s} {v['ms'][0]:10.2f} {v['ms'][1]:10.2f} ms   peak {v['peak_gb']:8.3f} GB")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_rep_ckpt.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_rep_ckpt.py needs a CUDA device")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import load_params      # tests/conftest.py: the trained-weight fixture loader
    dev = card()
    res = {"card": dev, "cases": {}}
    torch.manual_seed(42); random.seed(42)
    m = G.NeuralCAGraph(16, update_hidden=128, img_size=40, update_gain=0.05, alpha_thr=0.12, message_gain=0.25,
                        hidden_only=True, graph_zero_padded_shift=False)
    m.load_state_dict(load_params("weights_graph_ep960.npz"), strict=False)
    m = m.cuda()
    B, H = 32, 40
    with torch.no_grad():
        x0 = rollout(m, make_seed(16, H, B, device="cuda"), make_schedule(m, B, H, H, 48, fire_rate=0.6, seed=4))
    for T, reps in ((64, 20), (400, 4)):
        s = make_schedule(m, B, H, H, T, fire_rate=0.5, seed=5 + T)
        r = measure(variants(m, x0, s, (8, 16, 32, 64)), reps)
        name = f"40x40x16_torus_B32_T{T}"
        res["cases"][name] = r
        report(dev, name, r)

    T, budget = 1000, 4 << 30
    s = make_schedule(m, B, H, H, T, fire_rate=0.5, seed=7)
    plan = bptt_plan(m, B, H, H, T, budget)
    r = measure(variants(m, x0, s, (), unsegmented=False, fallback=True, budget=budget), 2)
    r["budget_bytes"], r["plan"] = budget, list(plan)
    name = "40x40x16_torus_B32_T1000"
    res["cases"][name] = r
    report(dev, f"{name} (budget {budget >> 30} GiB: {plan[0]}, K = {plan[1]}, {plan[2] / 1e9:.2f} GB)", r)

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
