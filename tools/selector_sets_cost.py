#!/usr/bin/env python
"""The action selector per hyper-parameter set on the GPU: what it costs and what it buys.

cost:    k_run against k_run_hp holding one set equal to the configuration, its selector given through
         rlb_engine_set_selectors, on C2 (hybrid store), C4, C3 and Taxi Q(lambda) on the lazy store: training steps/s from
         the kernels' CUDA events, the two engines alternating chunk by chunk in one process, `--reps` chunks each after a
         warm-up chunk; medians and the range of the chunk ratios.
mixed:   the Taxi Q-learning grid selector {eps, ucb} x learning_rate {0.05, 0.1, 0.2, 0.5} (16 384 agents per point, 1000
         episodes of train(n, n/10)) as one engine with the two selectors' launches concurrent (the default build), as one
         engine with them back to back (a library built with -DRLB_SEL_CONCURRENT=0: `--seq_lib`, run in a child process),
         and as two engines of four sets, one per selector, on two streams.  Every point's per-episode sums are checked bit
         for bit between the three first; then `--reps` timed runs each, alternating, wall time to the last wait.
c5:      C5's one-step cells (4 envs x {Basic, Double}, each with 2 selectors x 3 targets) at 8 192 and 102 400 agents per
         cell: 8 engines of six sets against the 16 engines of three sets (one per selector) that tools/target_sets_cost.py
         runs, async on 8 streams, after the same bit-for-bit check.
The card's name, power limit and SM clocks are read (nvidia-smi --query-gpu, read-only) in the same process.
    python tools/selector_sets_cost.py --out DIR [--seq_lib rl-rust_b200/ab/librlb_selseq.so]   (writes DIR/selector_sets_cost.txt)"""
import argparse
import importlib
import os
import subprocess
import sys
import time

import numpy as np

TOOLS = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(TOOLS))
sys.path.insert(0, TOOLS)
abi = importlib.import_module("rl-rust_b200._abi")
W = importlib.import_module("rl-rust_b200.workloads")
from target_sets_cost import alternate, card, fmt, one_set   # noqa: E402

COST = [("c2", 1 << 20, {}), ("c4", 1 << 21, {}), ("c3", 1 << 22, {}),
        ("taxi_qlambda_lazy", 102400, dict(env=3, agent=1, selector=0, policy=0, target=1, n_episodes=1000, chunk=100))]
LRS = [0.05, 0.1, 0.2, 0.5]
PER, N_EP = 16384, 1000


def cost(reps, lines):
    for name, n, over in COST:
        w = dict(W.WORKLOADS[name]) if name in W.WORKLOADS else dict(over)
        c, h = W.combo(w, 0), W.workload_hyper(w)
        store = 4 if name == "taxi_qlambda_lazy" else 0
        plain = W.make_engine(c, h, n, store_kind=store)
        hp = W.make_engine(c, h, n, store_kind=store)
        hp.set_hparams([one_set(h)], np.zeros(n, np.uint32))
        hp.set_selectors(np.array([c["selector"]], np.int32))
        a, b, same = alternate(plain, hp, w, reps)
        lines.append(fmt(name, n, plain.store_kind(), a, b, same))
        print(lines[-1], flush=True)
        plain.close()
        hp.close()


def grid_sets(h):
    return [dict(one_set(h), learning_rate=lr) for _ in (0, 1) for lr in LRS]


def mixed_one(h):
    """The grid as one engine (created with UCB, as grid_engine does): its engine and every point's sums per run."""
    c = dict(env=3, agent=0, selector=1, policy=0, target=1, real=0)
    e = W.make_engine(c, h, 8 * PER)
    e.set_hparams(grid_sets(h), np.repeat(np.arange(8, dtype=np.uint32), PER))
    e.set_selectors(np.array([0] * 4 + [1] * 4, np.int32))
    return e


def run_timed(engines):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for e in engines:
        e.train(N_EP, N_EP // 10, wait=False)
    parts = [e.train_wait()[0] for e in engines]
    return time.perf_counter() - t0, parts


def child_seq(reps, path):
    """The one-engine grid under the back-to-back library (this process was started with RLB_LIB)."""
    h = W.hyper(N_EP)
    times, sums = [], None
    for r in range(reps + 1):
        dt, parts = run_timed_fresh(lambda: [mixed_one(h)])
        if r == 0:
            sums = parts[0]["sums"]
        else:
            times.append(dt)
    np.savez(path, times=np.array(times), sums=sums)


def mixed(reps, lines, seq_lib, out):
    import torch
    h = W.hyper(N_EP)
    strm = [torch.cuda.Stream() for _ in range(2)]

    def two():
        out_e = []
        for k in (0, 1):   # the four sets of one selector, with the agent ids they have in the one-engine grid
            e = W.make_engine(dict(env=3, agent=0, selector=k, policy=0, target=1, real=0), h, 4 * PER, 4 * k * PER)
            e.set_hparams(grid_sets(h)[4 * k:4 * k + 4], np.repeat(np.arange(4, dtype=np.uint32), PER))
            e.set_stream(strm[k].cuda_stream)
            out_e.append(e)
        return out_e

    seq = None
    if seq_lib:
        path = os.path.join(out, "selector_seq_child.npz")
        subprocess.check_call([sys.executable, os.path.abspath(__file__), "--child_seq", path, "--reps", str(reps)],
                              env=dict(os.environ, RLB_LIB=os.path.abspath(seq_lib)))
        z = np.load(path)
        seq = (list(z["times"]), z["sums"])
        os.remove(path)
    t_one, t_two, s_one, s_two = [], [], None, None
    for r in range(reps + 1):   # alternating: one engine, then the two engines; the first run of each checks bits, unmeasured
        ta, pa = run_timed_fresh(lambda: [mixed_one(h)])
        tb, pb = run_timed_fresh(two)
        if r == 0:
            s_one, s_two = pa[0]["sums"], np.concatenate([p["sums"] for p in pb], axis=1)
        else:
            t_one.append(ta)
            t_two.append(tb)
    bits = lambda x, y: x is not None and y is not None and np.array_equal(x.view(np.uint64), y.view(np.uint64))
    lines.append("Taxi Q-learning grid selector {eps, ucb} x learning_rate %s = 8 points x %d agents, %d episodes (train(n, n/10))" % (LRS, PER, N_EP))
    lines.append("  per-point sums bit-identical: one engine concurrent vs two engines %s; vs one engine back to back %s"
                 % (bits(s_one, s_two), bits(s_one, seq[1]) if seq else "not measured"))
    lines.append("  one engine, concurrent launches (default): wall %s s, median %.3f" % (" ".join("%.3f" % t for t in t_one), np.median(t_one)))
    if seq:
        lines.append("  one engine, back to back (RLB_SEL_CONCURRENT=0, separate process): wall %s s, median %.3f"
                     % (" ".join("%.3f" % t for t in seq[0]), np.median(seq[0])))
    else:
        lines.append("  one engine, back to back: not measured")
    lines.append("  two engines of four sets on two streams: wall %s s, median %.3f" % (" ".join("%.3f" % t for t in t_two), np.median(t_two)))
    print("\n".join(lines[-5:]), flush=True)


def run_timed_fresh(make):
    engines = make()
    dt, parts = run_timed(engines)
    for e in engines:
        e.close()
    return dt, parts


def c5(lines, streams=8):
    import torch
    strm = [torch.cuda.Stream() for _ in range(streams)]
    w = W.WORKLOADS["c5"]
    n_ep = w["n_episodes"]
    h = W.hyper(n_ep, slippery=True)
    tg = [abi.TARGET_SARSA, abi.TARGET_QLEARNING, abi.TARGET_EXPECTED_SARSA]
    combos = sorted({(x["env"], x["policy"]) for x in w["cells"] if x["agent"] == 0})

    def drive(engines):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for e in engines:
            e.train(n_ep, max(1, n_ep // 10), wait=False)
        parts = [e.train_wait()[0] for e in engines]
        return time.perf_counter() - t0, parts

    for per in (8192, 102400):
        six = []
        for k, (env, pol) in enumerate(combos):   # 2 selectors x 3 targets per engine: set g = sel * 3 + target
            e = W.make_engine(dict(env=env, agent=0, selector=1, policy=pol, target=tg[0], real=0), h, 6 * per)
            e.set_hparams([one_set(h)] * 6, np.repeat(np.arange(6, dtype=np.uint32), per))
            e.set_targets(np.array(tg * 2, np.int32))
            e.set_selectors(np.array([0] * 3 + [1] * 3, np.int32))
            e.set_stream(strm[k % streams].cuda_stream)
            six.append(e)
        t6, p6 = drive(six)
        for e in six:
            e.close()
        three, j = [], 0
        for env, pol in combos:
            for sel in (0, 1):   # the agent ids these sets have in the six-set engine
                e = W.make_engine(dict(env=env, agent=0, selector=sel, policy=pol, target=tg[0], real=0), h, 3 * per, 3 * sel * per)
                e.set_hparams([one_set(h)] * 3, np.repeat(np.arange(3, dtype=np.uint32), per))
                e.set_targets(np.array(tg, np.int32))
                e.set_stream(strm[j % streams].cuda_stream)
                three.append(e)
                j += 1
        t3, p3 = drive(three)
        for e in three:
            e.close()
        same = all(np.array_equal(p6[k]["sums"][:, 3 * s:3 * s + 3].view(np.uint64), p3[2 * k + s]["sums"].view(np.uint64))
                   for k in range(len(combos)) for s in (0, 1))
        s6, s3 = sum(p["train_steps"] for p in p6), sum(p["train_steps"] for p in p3)
        lines.append("C5 one-step cells: %d (env, policy) x 2 selectors x 3 targets, %d agents per cell, %d episodes" % (len(combos), per, n_ep))
        lines.append("  %d engines of six sets, async on %d streams:   %.3f s wall  (%d train steps, %.4g steps/s)" % (len(combos), streams, t6, s6, s6 / t6))
        lines.append("  %d engines of three sets, async on %d streams: %.3f s wall  (%d train steps, %.4g steps/s)" % (2 * len(combos), streams, t3, s3, s3 / t3))
        lines.append("  speed-up %.3fx; per-set sums bit-identical between the two: %s" % (t3 / t6, same))
        print("\n".join(lines[-4:]), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="directory for selector_sets_cost.txt")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seq_lib", default=None, help="librlb built with -DRLB_SEL_CONCURRENT=0 (tools/build_variant.sh)")
    ap.add_argument("--child_seq", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child_seq:
        child_seq(a.reps, a.child_seq)
        return
    if not a.out:
        ap.error("--out is required")
    os.makedirs(a.out, exist_ok=True)
    lines = ["card (name, power limit, SM clock, max SM clock): %s" % card(),
             "training steps/s (train_steps / kernel_ms of each chunk), k_run and k_run_hp alternating"]
    print(lines[0], flush=True)
    cost(a.reps, lines)
    mixed(a.reps, lines, a.seq_lib, a.out)
    c5(lines)
    lines.append("card after the runs: %s" % card())
    open(os.path.join(a.out, "selector_sets_cost.txt"), "w").write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
