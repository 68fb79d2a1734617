"""Training iteration of the zero-padded graph shift (the module default) at B = 32 with the resident zero-pad BPTT
(rollout_impl="auto") against the dense history + streaming backward it replaces, and the torus model's resident BPTT for
reference, alternating in one process; per-kernel event timings of each (ids of include/gnca.h: 2 resident fwd,
3 k_bwd_mlp / k_rep_wgrad, 6 resident bwd).

The dense path is selected in the same build by not offering the zero-pad buffer to a zero-pad model (the forward then
keeps the dense history and the backward takes the streaming kernels, as before this path existed; no zero-pad forward
runs on that path).

usage: python scripts/time_zp_bptt.py [--iters N] [--out FILE.json]"""
import argparse, ctypes, json, os, random, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
import graph_neural_cellular_automata_b200 as G
from graph_neural_cellular_automata_b200 import _lib
from graph_neural_cellular_automata_b200 import rollout as R
from graph_neural_cellular_automata_b200.training.trainer import GraphNCATrainer, TrainConfig

ap = argparse.ArgumentParser()
ap.add_argument("--iters", type=int, default=10)
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--out", default=None)
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("time_zp_bptt: no CUDA device")
lib = _lib.load()
target = torch.from_numpy(np.load(os.path.join(ROOT, "tests/golden/target_gecko_surrogate.npy"))).cuda()
_orig = R._records_fwd_raw


def _dense_only(desc, packed, x0, sched, every, keep_x):
    """the record path as it was before the zero-pad buffer: none for a zero-pad model, so rollout_fwd_raw keeps the
    dense history (nothing of the zero-pad forward runs)"""
    B, _, H, W = x0.shape
    if (lib.gnca_bptt_bytes(ctypes.byref(desc), B, H, W, sched.T) == 0
            and lib.gnca_bptt_zp_bytes(ctypes.byref(desc), B, H, W, sched.T) > 0):
        return None
    return _orig(desc, packed, x0, sched, every, keep_x)


def trainer(long_prob, zero_pad=True):
    torch.manual_seed(1234); random.seed(1234)
    m = G.NeuralCAGraph(16, update_hidden=128, img_size=40, update_gain=0.05, alpha_thr=0.12, message_gain=0.25,
                        hidden_only=True, graph_zero_padded_shift=zero_pad)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in
                       np.load(os.path.join(ROOT, "tests/golden/weights_graph_ep960.npz")).items()}, strict=False)
    return GraphNCATrainer(m.cuda(), target, TrainConfig(batch_size=32, pool_size=1024, long_rollout_prob=long_prob,
                                                         fire="philox"))


def timed(tr, n):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        tr.train_step(epoch=300)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / n * 1e3


def kernels(tr):
    for kid in range(8):
        lib.gnca_profile_read(kid, ctypes.byref(ctypes.c_double(0)), ctypes.byref(ctypes.c_ulonglong(0)))
    lib.gnca_profile_enable(1)
    for _ in range(3):
        tr.train_step(epoch=300)
    torch.cuda.synchronize()
    lib.gnca_profile_enable(0)
    out = {}
    for kid in range(8):
        a, c = ctypes.c_double(0), ctypes.c_ulonglong(0)
        lib.gnca_profile_read(kid, ctypes.byref(a), ctypes.byref(c))
        if c.value:
            out["id%d" % kid] = {"ms_per_iter": a.value / 3, "launches_per_iter": c.value // 3}
    return out


gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
res = {"gpu": gpu, "shape": "B=32, 40x40x16, hidden 128, k=8, d_model 16, message_every 3, philox fire", "regimes": {}}
for name, long_prob in (("short", 0.0), ("long", 1.0)):
    # torus_resident: the trainer's torus model on its resident BPTT, for reference (same shapes and schedule draws)
    trs = {"zp_resident": trainer(long_prob), "dense_streaming": trainer(long_prob),
           "torus_resident": trainer(long_prob, zero_pad=False)}
    paths = {"zp_resident": _orig, "dense_streaming": _dense_only, "torus_resident": _orig}
    times = {k: [] for k in trs}
    for k in trs:                                  # warm-up (allocations of the largest step count included)
        R._records_fwd_raw = paths[k]
        timed(trs[k], 3)
    for _ in range(args.rounds):                   # alternate the paths
        for k in trs:
            R._records_fwd_raw = paths[k]
            times[k].append(timed(trs[k], args.iters))
    kern = {}
    for k in trs:
        R._records_fwd_raw = paths[k]
        kern[k] = kernels(trs[k])
    R._records_fwd_raw = _orig
    res["regimes"][name] = {k: {"ms_per_iter": sorted(v), "median": sorted(v)[len(v) // 2], "kernels": kern[k]}
                            for k, v in times.items()}
    print(name, json.dumps(res["regimes"][name]), flush=True)
print(json.dumps({"gpu": gpu}))
if args.out:
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
