#!/usr/bin/env python
"""Successive halving on the GPU: what running only the active sets costs and what a halving run gives.

indirection: k_run_hp through an agent list against the identity path (thread t runs agent t) on C2 (1 M agents), C4
             (2 M), C3 (4 M) and Taxi Q(lambda) on the lazy store (102 400), the configurations of profiles/hp_cost.txt.
             Both engines hold two sets.  On the list engine the last agent alone is set 1, and set 1 is paused, so
             its launch runs agents 0 .. N-2 through the list: every agent but one.  Training steps/s from the
             kernels' CUDA events, the two engines alternating chunk by chunk in one process, `--reps` chunks each
             after a warm-up chunk; medians.
scaling:     one 100-episode chunk of the 64-set x 16 384-agent Taxi Q-learning f32 grid with 64, 32, 16, 8 and 4 sets
             active (the first k sets, contiguous): training steps/s from the kernel's CUDA events, and the agents the
             launch covers.  The sets are reconstructed (rlb_engine_set_hparams) before every chunk; each k runs
             `--reps` times, alternating, medians.
end to end:  tools/rl_sweep.py's run against tools/rl_halving.py's (--min_episodes 100 --eta 2) over that grid, 1000
             episodes: wall time of train + evaluate, training steps, the best set and its evaluate mean return.  One
             run each: neither number has a spread.
The card's name, power limit and SM clock are read (nvidia-smi --query-gpu, read-only) in the same process.
    python tools/halving_cost.py --out DIR          (writes DIR/halving_cost.txt)"""
import argparse
import importlib
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
abi = importlib.import_module("rl-rust_b200._abi")
W = importlib.import_module("rl-rust_b200.workloads")
driver = importlib.import_module("rl-rust_b200.driver")
hp_ab = importlib.import_module("tools.hp_ab")

POINTS, PER_POINT, N_EP = 64, 16384, 1000
LRS = [float(x) for x in np.geomspace(0.01, 0.5, 8)]
EXPLORATION = [float(x) for x in np.linspace(0.2, 0.9, 8)]


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip()
    except Exception as exc:   # noqa: BLE001
        return "nvidia-smi unavailable: %s" % exc


def indirection(reps, lines):
    lines.append("indirection: k_run_hp through an agent list (every agent but the last) against the identity path; "
                 "training steps/s (train_steps / kernel_ms of each chunk), alternating")
    for name, n, over in hp_ab.COST:
        w = dict(W.WORKLOADS[name]) if name in W.WORKLOADS else dict(over)
        c, h = W.combo(w, 0), W.workload_hyper(w)
        chunk = w["chunk"]
        store = 4 if name == "taxi_qlambda_lazy" else 0
        one = hp_ab.one_set(h)
        ident = W.make_engine(c, h, n, store_kind=store)
        listed = W.make_engine(c, h, n, store_kind=store)
        group = np.zeros(n, np.uint32)
        group[-1] = 1
        for e in (ident, listed):
            e.set_hparams([one, one], group)
        listed.set_active_sets([True, False])
        rates = {"identity": [], "list": []}
        ep = 0
        for r in range(reps + 1):
            for label, eng in (("identity", ident), ("list", listed)):
                res = eng.train(ep + chunk, max(1, w["n_episodes"] // 10), ep_begin=ep)
                if r:
                    rates[label].append(res["train_steps"] / (res["kernel_ms"] * 1e-3))
            ep += chunk
        a, b = np.array(rates["identity"]), np.array(rates["list"])
        lines.append("  %-18s agents=%-8d store=%d  identity %s  list %s  ratio(median) %.4f" % (
            name, n, ident.store_kind(), " ".join("%.4g" % x for x in a), " ".join("%.4g" % x for x in b), np.median(b) / np.median(a)))
        print(lines[-1], flush=True)
        ident.close()
        listed.close()


def scaling(reps, lines):
    c, h = W.combo(W.WORKLOADS["c4"], 0), W.hyper(N_EP)
    sets = [dict(learning_rate=lr, initial_epsilon=1.0, epsilon_decay=1.0 / (x * N_EP)) for lr in LRS for x in EXPLORATION]
    group = np.repeat(np.arange(POINTS, dtype=np.uint32), PER_POINT)
    eng = W.make_engine(c, h, POINTS * PER_POINT)
    ks = (64, 32, 16, 8, 4)
    rates = {k: [] for k in ks}
    for r in range(reps + 1):
        for k in ks:
            eng.set_hparams(sets, group)
            mask = np.zeros(POINTS, bool)
            mask[:k] = True
            eng.set_active_sets(mask)
            res = eng.train(100, N_EP // 10)
            if r:
                rates[k].append(res["train_steps"] / (res["kernel_ms"] * 1e-3))
    eng.close()
    lines.append("scaling: one 100-episode chunk of the Taxi Q-learning f32 grid, %d sets x %d agents, k sets active; "
                 "training steps/s (kernel CUDA events), %d reps each, alternating" % (POINTS, PER_POINT, reps))
    base = np.median(rates[64])
    for k in ks:
        m = np.median(rates[k])
        lines.append("  %2d sets active (%8d agents, %6d CTAs of 128): median %.4g steps/s (%s), %.3f of 64 sets' rate"
                     % (k, k * PER_POINT, k * PER_POINT // 128, m, " ".join("%.4g" % x for x in rates[k]), m / base))
    print("\n".join(lines[-6:]), flush=True)


def end_to_end(lines):
    grid = {"learning_rate": LRS, "exploration_time": EXPLORATION}
    kw = dict(agents_per_point=PER_POINT, n_episodes=N_EP, real="f32", verbose=False)
    driver.run_sweep("taxi", {"learning_rate": LRS[:2]}, agents_per_point=64, n_episodes=20, real="f32", verbose=False)   # warm-up
    sweep = driver.run_sweep("taxi", grid, **kw)
    halving = driver.run_halving("taxi", grid, min_episodes=100, eta=2, **kw)
    lines.append("end to end: Taxi Q-learning f32 grid, %d points (learning_rate x exploration_time) x %d agents, %d episodes; "
                 "one run each (no spread)" % (POINTS, PER_POINT, N_EP))
    for name, r in (("sweep (rl_sweep)", sweep), ("halving (rl_halving, --min_episodes 100 --eta 2)", halving)):
        best = r["ranking"][0]
        p = r["points"][best]
        lines.append("  %-50s %.3f s wall (train + evaluate), %d training steps; best set %d %s: evaluate mean return %.4f"
                     % (name, r["seconds"], r["train_steps"], best, p["params"], p["eval_mean_return"]))
    lines.append("  halving rungs: %s" % ", ".join("%d eps x %d sets" % (r["episodes"][1] - r["episodes"][0], len(r["active"]))
                                                   for r in halving["rungs"]))
    same = halving["points"][halving["ranking"][0]]["eval_mean_return"] == sweep["points"][halving["ranking"][0]]["eval_mean_return"]
    lines.append("  halving's best set has the sweep's evaluate return for that point, bit for bit: %s" % same)
    print("\n".join(lines[-5:]), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for halving_cost.txt")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    lines = ["card (name, power limit, SM clock, max SM clock): %s" % card()]
    print(lines[0], flush=True)
    indirection(a.reps, lines)
    scaling(a.reps, lines)
    end_to_end(lines)
    lines.append("card at the end: %s" % card())
    open(os.path.join(a.out, "halving_cost.txt"), "w").write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
