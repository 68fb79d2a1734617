"""Cost and memory of checkpointed BPTT (rollout(..., checkpoint_every=K)) against the dense streaming BPTT, timed with
CUDA events around whole forward + loss + backward calls.

Cases:
  256x256x32 torus, B = 16, T = 200: dense and K in {8, 14, 32}; also the forward alone (no grad, streaming);
  256x256x32 torus, B = 16, T = 1000 (the regeneration length), K = 32: checkpointed only -- the dense history would need
      (2T + 1) * B * C * H * W * 4 bytes, printed, not attempted;
  40x40x16 zero-padded shift, B = 32, T = 64: dense and K = 8, the overhead at the small shape.
The large shape uses random weights and a random state inside a disk (about 28 % of the cells alive at the start);
the small one the trained weights and a grown pattern.  Peak memory = torch.cuda.max_memory_allocated over one call,
above what was allocated before it.  Each variant is timed twice, in alternating order, so the spread shows.

Reads the card's name and power limit in the same run and writes profiles/r03_ckpt.json (or --out).  Needs a CUDA
device; it has no CPU path.

    python scripts/time_ckpt.py [--reps 3] [--out profiles/r03_ckpt.json]
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
from graph_neural_cellular_automata_b200.rollout import make_schedule, rollout  # noqa: E402
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
    a.record()
    fn()
    b.record()
    b.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    ms = [a.elapsed_time(b)]
    for _ in range(reps - 1):
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return sum(ms) / len(ms), peak


def ell(x):
    return (x[:, :4] ** 2).mean()


def variants(m, x0, s, ks, dense):
    def zero():
        for q in m.parameters():
            q.grad = None

    def train(**kw):
        def run():
            zero()
            ell(rollout(m, x0.clone().requires_grad_(True), s, **kw)).backward()
        return run

    def fwd():
        with torch.no_grad():
            rollout(m, x0, s, impl="streaming")

    fns = {"forward_only": fwd}
    if dense:
        fns["dense"] = train(impl="streaming")
    for k in ks:
        fns[f"K{k}"] = train(checkpoint_every=k)
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


def blob(B, C, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    disk = (((yy - H / 2) ** 2 + (xx - W / 2) ** 2) < (0.3 * min(H, W)) ** 2).float()
    return (torch.rand(B, C, H, W, generator=g) * disk).cuda()


def report(dev, name, r):
    print(f"[{dev}] {name}: ms per call (two alternating runs), peak GB")
    fwd = sum(r["forward_only"]["ms"]) / 2
    dense = sum(r["dense"]["ms"]) / 2 if "dense" in r else None
    for k, v in r.items():
        t = sum(v["ms"]) / 2
        extra = f"   dense + {(t - dense) / fwd:.2f} x forward" if dense is not None and k.startswith("K") else ""
        print(f"  {k:13s} {v['ms'][0]:10.1f} {v['ms'][1]:10.1f} ms   peak {v['peak_gb']:8.3f} GB{extra}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_ckpt.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_ckpt.py needs a CUDA device")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import load_params      # tests/conftest.py: the trained-weight fixture loader
    dev = card()
    res = {"card": dev, "cases": {}}

    torch.manual_seed(42); random.seed(42)
    big = G.NeuralCAGraph(32, update_hidden=128, img_size=256, update_gain=0.1, alpha_thr=0.1, message_gain=0.3,
                          hidden_only=True, graph_zero_padded_shift=False)
    with torch.no_grad():
        big.update_net[2].weight.normal_(0, 0.05)
    big = big.cuda()
    B, C, H = 16, 32, 256
    x0 = blob(B, C, H, H, 1)
    s = make_schedule(big, B, H, H, 200, fire_rate=0.5, seed=2)
    r = measure(variants(big, x0, s, (8, 14, 32), dense=True), args.reps)
    res["cases"]["256x256x32_B16_T200"] = r
    report(dev, "256x256x32 torus, B = 16, T = 200", r)

    T = 1000
    dense_bytes = (2 * T + 1) * B * C * H * H * 4
    print(f"  T = {T}: the dense history would need {dense_bytes / 1e9:.1f} GB (x_hist[T+1] + u_hist[T]); not attempted")
    s = make_schedule(big, B, H, H, T, fire_rate=0.5, seed=3)
    r = measure(variants(big, x0, s, (32,), dense=False), 1)
    r["dense_history_bytes_not_run"] = dense_bytes
    res["cases"]["256x256x32_B16_T1000"] = r
    report(dev, "256x256x32 torus, B = 16, T = 1000", {k: v for k, v in r.items() if isinstance(v, dict)})

    small = G.NeuralCAGraph(16, update_hidden=128, img_size=40, update_gain=0.05, alpha_thr=0.12, message_gain=0.25,
                            hidden_only=True, graph_zero_padded_shift=True)
    small.load_state_dict(load_params("weights_graph_ep960.npz"), strict=False)
    small = small.cuda()
    B, H, T = 32, 40, 64
    with torch.no_grad():
        x0 = rollout(small, make_seed(16, H, B, device="cuda"), make_schedule(small, B, H, H, 48, fire_rate=0.6, seed=4))
    s = make_schedule(small, B, H, H, T, fire_rate=0.5, seed=5)
    r = measure(variants(small, x0, s, (8,), dense=True), 10 * args.reps)
    res["cases"]["40x40x16_zeropad_B32_T64"] = r
    report(dev, "40x40x16 zero-padded shift, B = 32, T = 64", r)

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
