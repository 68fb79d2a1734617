"""Cost of a checkpoint sweep: M models of one architecture over one regeneration schedule, as M sequential
monitor_rollout calls against one stacked call (monitor_rollout over the list, gnca_rollout_metrics_models).

Setup: 40x40x16 graph NCA (zero-padded shift, the module default, and torus), T = 1000 steps from a grown pattern,
damage at t = 500, a frame every 10 steps; M in {1, 16, 64, 148, 300} models at B = 1 and B = 8 samples per model.
The models are seeded perturbations of the trained ep960 weights (a sweep's timing does not depend on the values).
Each arm is timed with CUDA events around whole sweeps after a warm-up sweep, the two arms alternated within each of
two rounds.  Reported: wall time per sweep, cell updates per second (M * B * H * W * T / time), and the cluster size
the stacked launch took.

Prints the card's name and power limit with the numbers and writes them to profiles/r08_sweep.json (or --out).
Needs a CUDA device; it has no CPU path.

    python scripts/time_sweep.py [--ms 1,16,64,148,300] [--out profiles/r08_sweep.json]
"""
from __future__ import annotations

import argparse
import json
import os
import random
import re
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import graph_neural_cellular_automata_b200 as G  # noqa: E402
from graph_neural_cellular_automata_b200.rollout import make_schedule, monitor_rollout, rollout  # noqa: E402
from graph_neural_cellular_automata_b200.utils import metrics as UM  # noqa: E402
from graph_neural_cellular_automata_b200.utils.nca_init import make_seed  # noqa: E402

H = W = 40
T, DAMAGE_STEP, EVERY = 1000, 500, 10


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def models(n, torus, params):
    out = []
    for i in range(n):
        m = G.NeuralCAGraph(16, update_hidden=128, img_size=H, update_gain=0.05, alpha_thr=0.12, message_gain=0.25,
                            hidden_only=True, graph_zero_padded_shift=not torus)
        m.load_state_dict(params, strict=False)
        if i:
            g = torch.Generator().manual_seed(i)
            with torch.no_grad():
                for name, p in m.named_parameters():
                    if "perception" not in name and p.requires_grad:
                        p.add_(0.03 * p.abs().mean() * torch.randn(p.shape, generator=g))
        out.append(m.cuda())
    return out


def time_ms(fn):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def stacked_cluster_size(ms, x0, s, tgt):
    """the NC the replicated-state kernel printed for the stacked launch (GNCA_DEBUG goes to fd 2)"""
    with tempfile.TemporaryFile(mode="w+") as f:
        fd = os.dup(2)
        os.dup2(f.fileno(), 2)
        os.environ["GNCA_DEBUG"] = "1"
        try:
            monitor_rollout(ms, x0, s, tgt, every=EVERY)
            torch.cuda.synchronize()
        finally:
            del os.environ["GNCA_DEBUG"]
            os.dup2(fd, 2)
            os.close(fd)
        f.seek(0)
        nc = re.findall(r"NC=(\d+)", f.read())
    return int(nc[-1]) if nc else None


def sweep(torus, M, B, pool, x_grown, rounds=2):
    ms = pool[:M]
    n = M * B
    x0 = x_grown[:1].expand(n, -1, -1, -1).contiguous()
    tgt = UM.premultiply(x_grown[:1])[0].contiguous()
    dmg = torch.ones(n, 16, H, W, device="cuda")
    dmg[:, :, H // 4:H // 2, H // 4:H // 2] = 0.0
    random.seed(3)
    s = make_schedule(ms[0], n, H, W, T, fire_rate=0.5, seed=4, damage=dmg, damage_step=DAMAGE_STEP)
    random.seed(3)          # the same offsets for the per-model calls, on B samples each
    s_one = make_schedule(ms[0], B, H, W, T, fire_rate=0.5, seed=4, damage=dmg[:B], damage_step=DAMAGE_STEP)
    arms = {"sequential": lambda: [monitor_rollout(m, x0[i * B:(i + 1) * B], s_one, tgt, every=EVERY)
                                   for i, m in enumerate(ms)],
            "stacked": lambda: monitor_rollout(ms, x0, s, tgt, every=EVERY)}
    times = {k: [] for k in arms}
    with torch.no_grad():
        for fn in arms.values():
            fn()                                           # warm-up: modules, allocator, launch configuration
        for _ in range(rounds):
            for k, fn in arms.items():
                times[k].append(time_ms(fn))
        nc = stacked_cluster_size(ms, x0, s, tgt)
    cells = n * H * W * T
    return {"model": "torus" if torus else "zeropad", "M": M, "B": B, "ms": times,
            "cell_updates_per_s": {k: cells / (min(v) / 1e3) for k, v in times.items()},
            "speedup": min(times["sequential"]) / min(times["stacked"]), "stacked_NC": nc}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ms", default="1,16,64,148,300")
    ap.add_argument("--bs", default="1,8")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_sweep.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_sweep.py needs a CUDA device")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import load_params      # tests/conftest.py: the trained-weight fixture loader
    params = load_params("weights_graph_ep960.npz")
    Ms = [int(v) for v in args.ms.split(",")]
    Bs = [int(v) for v in args.bs.split(",")]
    dev = card()
    rows = []
    for torus in (False, True):
        pool = models(max(Ms), torus, params)
        with torch.no_grad():
            x_grown = rollout(pool[0], make_seed(16, H, 1, device="cuda"),
                              make_schedule(pool[0], 1, H, W, 64, fire_rate=0.5, seed=1))
        for B in Bs:
            for M in Ms:
                r = sweep(torus, M, B, pool, x_grown)
                rows.append(r)
                print(f"[{dev}] {r['model']:7s} M={M:3d} B={B}: sequential "
                      f"{' '.join(f'{v:9.1f}' for v in r['ms']['sequential'])} ms, stacked "
                      f"{' '.join(f'{v:8.1f}' for v in r['ms']['stacked'])} ms, {r['speedup']:.2f}x, "
                      f"{r['cell_updates_per_s']['stacked']:.3e} cell-updates/s stacked, NC={r['stacked_NC']}",
                      flush=True)
    res = {"card": dev, "setup": f"40x40x16, T={T}, damage at t={DAMAGE_STEP}, a frame every {EVERY} steps",
           "rows": rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
