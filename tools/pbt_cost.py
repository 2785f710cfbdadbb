#!/usr/bin/env python
"""Population-based training on the GPU: what its exploit step costs and what a PBT run gives against the plain grid.

clone: the 64-point Taxi Q-learning f32 population (16 384 agents per point) after one chunk of training; a quarter of
       the agents (the 16 weakest sets) take the state of agents of the top 16 sets.  rlb_agent_clone is timed with CUDA
       events on the engine's stream over `--reps` calls (the id upload and k_clone_agents), and k_clone_agents alone
       with torch.profiler in a separate pass; bytes moved = 2 x pairs x (per-agent Q bytes) + the scalars (eps, ucb_t,
       flag) + the ids read, over kernel time, against the B200's 7.7 TB/s.  Against it: the host round trip that does
       the same job without the call (rlb_download_tables + rlb_get_agent_states, the copy on the host, the uploads),
       wall time over `--rt_reps` repetitions.
run:   tools/rl_pbt.py's run (interval 100, fraction 0.25) against tools/rl_sweep.py's over the same 64-point grid,
       16 384 agents per point and 1000 episodes: wall time of train + evaluate and the best set's evaluate mean return.
The card's name and power limit are read (nvidia-smi --query-gpu, read-only) in the same process.
    python tools/pbt_cost.py --out DIR          (writes DIR/pbt_cost.txt)"""
import argparse
import importlib
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
abi = importlib.import_module("rl-rust_b200._abi")
W = importlib.import_module("rl-rust_b200.workloads")
driver = importlib.import_module("rl-rust_b200.driver")
hp_ab = importlib.import_module("tools.hp_ab")

POINTS, PER_POINT, N_EP = 64, 16384, 1000
LRS = [float(x) for x in np.geomspace(0.01, 0.5, 8)]
EXPLORATION = [float(x) for x in np.linspace(0.2, 0.9, 8)]
HBM_BYTES_PER_S = 7.7e12


def clone_cost(lines, reps, rt_reps):
    import torch
    c = dict(W.combo(W.WORKLOADS["c4"], 0))
    h = W.hyper(N_EP)
    n = POINTS * PER_POINT
    eng = W.make_engine(c, h, n)
    sets = [dict(learning_rate=lr, initial_epsilon=1.0, epsilon_decay=1.0 / (x * N_EP)) for lr in LRS for x in EXPLORATION]
    eng.set_hparams(sets, np.repeat(np.arange(POINTS, dtype=np.uint32), PER_POINT))
    stream = torch.cuda.Stream()
    eng.set_stream(stream.cuda_stream)
    res = eng.train(100, N_EP // 10)
    order = np.argsort(-res["sums"][:, :, 1].sum(0), kind="stable")
    quarter = POINTS // 4
    j = np.arange(PER_POINT, dtype=np.uint32)
    winners = order[:quarter][np.random.default_rng(1).integers(0, quarter, quarter)]
    src = np.concatenate([w * PER_POINT + j for w in winners]).astype(np.uint32)
    dst = np.concatenate([l * PER_POINT + j for l in order[POINTS - quarter:]]).astype(np.uint32)
    pairs = len(dst)
    q_stride = eng.S * eng.T * eng.A * (4 if eng.real == abi.REAL_F32 else 8)
    moved = 2 * pairs * (q_stride + 8 + 8 + 1) + 8 * pairs
    eng.clone_agents(src, dst)                                     # warm-up
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        eng.clone_agents(src, dst)
        e1.record(stream)
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    t0 = time.perf_counter()
    for _ in range(reps):
        eng.clone_agents(src, dst)
    call_s = (time.perf_counter() - t0) / reps
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            eng.clone_agents(src, dst)
        torch.cuda.synchronize()
    kern_us = [ev.device_time for ev in prof.events() if "k_clone_agents" in ev.name]
    # the same job today: a host round trip of every table and state
    rt = []
    for _ in range(rt_reps):
        t0 = time.perf_counter()
        q, _ = eng.download_tables(counts=False)
        st = eng.states()
        q[dst] = q[src]
        for f in ("epsilon", "ucb_t", "policy_flag"):
            st[f][dst] = st[f][src]
        eng.upload_tables(q, None)
        eng.set_states(st)
        rt.append(time.perf_counter() - t0)
        del q
    eng.close()
    k_med = float(np.median(kern_us)) * 1e-6 if kern_us else float("nan")
    lines.append("rlb_agent_clone: Taxi Q-learning f32, %d sets x %d agents, %d pairs (a quarter of the agents as destinations), "
                 "%d B of Q per agent" % (POINTS, PER_POINT, pairs, q_stride))
    lines.append("  CUDA events around the call (id upload + k_clone_agents), %d reps: median %.3f ms, min %.3f ms, max %.3f ms"
                 % (reps, np.median(ms), min(ms), max(ms)))
    lines.append("  host clock per call (validation on the host, upload, kernel, synchronise): %.3f ms" % (call_s * 1e3))
    lines.append("  k_clone_agents (torch.profiler, %d launches): median %.3f ms; %.3f GB moved -> %.2f TB/s = %.1f %% of 7.7 TB/s (HBM-bound)"
                 % (len(kern_us), k_med * 1e3, moved / 1e9, moved / k_med / 1e12, 100.0 * moved / k_med / HBM_BYTES_PER_S))
    lines.append("  host round trip (download tables + states, copy, upload), %d reps: %s s (%.0fx the call)"
                 % (rt_reps, " ".join("%.2f" % x for x in rt), np.median(rt) / (np.median(ms) * 1e-3)))
    print("\n".join(lines[-5:]), flush=True)


def run_cost(lines, interval=100, fraction=0.25):
    grid = {"learning_rate": LRS, "exploration_time": EXPLORATION}
    kw = dict(agents_per_point=PER_POINT, n_episodes=N_EP, real="f32", verbose=False)
    driver.run_sweep("taxi", {"learning_rate": LRS[:2]}, agents_per_point=64, n_episodes=20, real="f32", verbose=False)   # warm-up
    sweep = driver.run_sweep("taxi", grid, **kw)
    pbt = driver.run_pbt("taxi", grid, interval=interval, fraction=fraction, **kw)
    lines.append("Taxi Q-learning f32 grid: %d points (learning_rate x exploration_time) x %d agents, %d episodes" % (POINTS, PER_POINT, N_EP))
    for name, r in (("grid (rl_sweep)", sweep), ("PBT (rl_pbt, interval %d, fraction %.2f)" % (interval, fraction), pbt)):
        best = r["ranking"][0]
        p = r["points"][best]
        lines.append("  %-42s %.3f s wall (train + evaluate); best set %d %s: evaluate mean return %.4f"
                     % (name, r["seconds"], best, p.get("final_params", p["params"]), p["eval_mean_return"]))
    print("\n".join(lines[-3:]), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for pbt_cost.txt")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rt_reps", type=int, default=3)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    lines = ["card: %s" % hp_ab.card()]
    print(lines[0], flush=True)
    clone_cost(lines, a.reps, a.rt_reps)
    run_cost(lines)
    open(os.path.join(a.out, "pbt_cost.txt"), "w").write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
