"""Cost of differentiable frames (record_rollout(..., differentiable=True)), timed with CUDA events: forward + loss +
backward per call, graph NCA, 16 channels, 40x40 torus, trained weights, resident kernels.

Variants at each shape:
  xT        the loss on x_T only through rollout() (what training pays today);
  S8, S1    a loss on every frame and on x_T through one differentiable recording, every 8 / every step;
  chain8    the same loss at S = 8 without this entry point: T / 8 chained rollout() calls of 8 steps each.
Shapes: the training shape (B = 32, T = 64, ragged steps in [48, 80)) and bench.py's (B = 8, T = 96).  Every variant
is timed twice, in alternating order, so that the spread shows next to the differences.

Prints the card's name and power limit with the numbers, and one JSON line.  Needs a CUDA device; it has no CPU path.

    python scripts/time_record_grad.py [--reps 20]
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


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def time_ms(fn, reps, warmup=3):
    """mean wall time of fn() between two CUDA events, over `reps` calls after `warmup` untimed ones"""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def ell(x):
    return (x[:, :4] ** 2).mean()


def shape(m, B, T, steps, reps):
    H = W = 40
    with torch.no_grad():
        x0 = make_seed(16, H, B, device="cuda")
        x0 = rollout(m, x0, make_schedule(m, B, H, W, 48, fire_rate=0.6, seed=1), impl="streaming")
    s = make_schedule(m, B, H, W, T, fire_rate=0.5, steps=steps, seed=2)
    S = 8
    st = torch.tensor(steps if steps is not None else [T] * B)
    segs = []
    for i in range(T // S):          # the workaround: one schedule (own Philox stream) per segment of S steps
        seg_steps = (st - i * S).clamp(0, S).tolist()
        segs.append(make_schedule(m, B, H, W, S, fire_rate=0.5, steps=seg_steps, seed=100 + i))

    def zero():
        for q in m.parameters():
            q.grad = None

    def xT():
        zero()
        ell(rollout(m, x0.clone().requires_grad_(True), s, impl="resident")).backward()

    def frames(every):
        def run():
            zero()
            tr = record_rollout(m, x0.clone().requires_grad_(True), s, every=every, impl="resident", differentiable=True)
            (sum(ell(tr.states[f]) for f in range(tr.states.shape[0])) + ell(tr.x_T)).backward()
        return run

    def chain():
        zero()
        x = x0.clone().requires_grad_(True)
        loss = ell(x)
        for sg in segs:
            x = rollout(m, x, sg, impl="resident")
            loss = loss + ell(x)
        (loss + ell(x)).backward()

    fns = {"xT": xT, "S8": frames(8), "S1": frames(1), "chain8": chain}
    out = {k: [] for k in fns}
    for rnd in range(2):
        for k in (list(fns) if rnd == 0 else list(reversed(list(fns)))):
            out[k].append(time_ms(fns[k], reps))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_record_grad.py needs a CUDA device")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import load_params      # tests/conftest.py: the trained-weight fixture loader
    dev = card()
    torch.manual_seed(42); random.seed(42)
    m = G.NeuralCAGraph(16, update_hidden=128, img_size=40, update_gain=0.05, alpha_thr=0.12, message_gain=0.25,
                        hidden_only=True, graph_zero_padded_shift=False)
    m.load_state_dict(load_params("weights_graph_ep960.npz"), strict=False)
    m = m.cuda()
    res = {}
    steps = torch.randint(48, 80, (32,), generator=torch.Generator().manual_seed(0)).tolist()
    for name, B, T, st in (("B32_T64_ragged", 32, 64, steps), ("B8_T96", 8, 96, None)):
        r = shape(m, B, T, st, args.reps)
        res[name] = r
        base = sum(r["xT"]) / 2
        print(f"[{dev}] 40x40x16 torus, {name}, resident: ms per forward + backward (two alternating runs)")
        for k, v in r.items():
            print(f"  {k:8s} {v[0]:9.3f} {v[1]:9.3f} ms   ({sum(v) / 2 / base:.3f}x xT)")
    print(json.dumps({"card": dev, "ms": res}))


if __name__ == "__main__":
    main()
