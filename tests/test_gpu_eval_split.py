"""The evaluate blocks of the on-chip stores run in k_eval launches of their own (rlb_engine.cu, run_chunk) from
RLB_EVAL_SPLIT_MIN_AGENTS = 2^17 agents on, so these engines hold N_SPLIT agents.  An engine on
the thread-group (2) or hybrid (3) store must give, bit for bit, what the same agents give on the HBM store (1), which
keeps its evaluate blocks inside k_run, and what the CPU oracle gives: records, sums, totals, tables and agent states,
over ranges that start off the eval_at grid, evaluate after every episode, never evaluate, and end right after their
trigger episode; on the blocking, pipelined, asynchronous and evaluate call paths, with taps, and under hyper-parameter
sets with both selectors and a mask."""
import importlib

import numpy as np
import pytest

import parity as P
from oracle import oracle_py as O
from test_gpu_hparams import as_set
from test_gpu_targets import fields_equal

pytestmark = pytest.mark.gpu

abi = importlib.import_module("rl-rust_b200._abi")

N_SPLIT = 1 << 17   # RLB_EVAL_SPLIT_MIN_AGENTS: fewer agents run their evaluate blocks fused

# env x selector x policy x target (Sarsa(lambda), Q(lambda)) x real: every trace agent of the envs with on-chip stores
SPLIT_CASES = [dict(env=env, agent=1, selector=sel, policy=pol, target=tgt, real=real)
               for env in (1, 2) for sel in (0, 1) for pol in (0, 1) for tgt in (0, 1) for real in (0, 1)]


def on_store(c, h, n, first, store):
    """An engine on `store`, or None when the store cannot hold this agent (the engine refuses it)."""
    try:
        eng = P.make_engine(c, h, n, first, store_kind=store)
    except abi.RlbError as exc:
        if store != 1 and exc.status == abi.ERR_UNSUPPORTED:
            return None
        raise
    if eng.store_kind() != store:
        eng.close()
        return None
    return eng


def same_result(ra, rb, what):
    for k in ("train_steps", "eval_steps", "eval_episodes", "eval_return_sum", "trace_rows", "steps"):   # not kernel_launches
        if k in ra:
            assert ra[k] == rb[k], (what, k, ra[k], rb[k])
    for k in ("sums",):
        if ra.get(k) is not None:
            assert P.bits_equal(ra[k], rb[k]), (what, k, P.first_diff(ra[k], rb[k]))
    for k in ("episodes", "traj"):
        if ra.get(k) is not None:
            assert fields_equal(ra[k], rb[k]), (what, k)
    for k in ("traj_count", "td_count"):
        if ra.get(k) is not None:
            assert np.array_equal(ra[k], rb[k]), (what, k)
    if ra.get("td_steps") is not None:
        assert P.bits_equal(ra["td_steps"], rb["td_steps"]), (what, "td_steps")


def same_state(a, b, what):
    qa, ca = a.download_tables()
    qb, cb = b.download_tables()
    assert P.bits_equal(qa, qb), (what, "Q", P.first_diff(qa, qb))
    assert np.array_equal(ca, cb), (what, "counts")
    assert fields_equal(a.states(), b.states()), (what, "states")


def twin_calls(a, b):
    """The same calls on both engines, compared after each: every kind of range and call path."""
    calls = [
        ("ends after its trigger", lambda e: e.train(7, 3, sums=True, episodes=True)),            # triggers 0, 3, 6
        ("off the grid", lambda e: e.train(12, 5, ep_begin=7, sums=True, episodes=True)),         # trigger 10
        ("eval_at 1", lambda e: e.train(15, 1, ep_begin=12, sums=True, episodes=True)),
        ("eval_at beyond", lambda e: e.train(21, 1000, ep_begin=15, sums=True, episodes=True)),
        ("pipelined", lambda e: e.train(37, 4, ep_begin=21, sums=True, episodes=True)),           # 4 launches, host records
        ("taps", lambda e: e.train(43, 2, ep_begin=37, sums=True, episodes=True, traj_capacity=100, td_capacity=50)),
        ("evaluate", lambda e: e.evaluate(9, sums=True, episodes=True)),
    ]
    for what, call in calls:
        ra, rb = call(a), call(b)
        same_result(ra, rb, what)
        if what == "ends after its trigger":   # the split path ran: train 0, evaluate, train 1-3, evaluate, train 4-6, evaluate
            assert (ra["kernel_launches"], rb["kernel_launches"]) == (6, 1), (ra["kernel_launches"], rb["kernel_launches"])
        if what in ("ends after its trigger", "taps", "evaluate"):
            same_state(a, b, what)
    ra = a.train(50, 3, ep_begin=43, sums=True, episodes=True, wait=False)                     # the asynchronous call
    rb = b.train(50, 3, ep_begin=43, sums=True, episodes=True, wait=False)
    a.train_wait()
    b.train_wait()
    same_result(ra, rb, "async")
    same_state(a, b, "async")


@pytest.mark.parametrize("c", SPLIT_CASES, ids=P.combo_id)
def test_split_matches_the_fused_hbm_store(c):
    h = P.hyper(50, max_steps=40)
    n, first = N_SPLIT, 12345
    ran = 0
    for store in (2, 3):
        eng = on_store(c, h, n, first, store)
        if eng is None:
            continue
        with eng, P.make_engine(c, h, n, first, store_kind=1) as ref:
            twin_calls(eng, ref)
        ran += 1
    if c["real"] == 0 and c["selector"] == 0:
        assert ran, "no on-chip store ran %s" % P.combo_id(c)


def compare_agents(g, o, c, k):
    """The first k agents of the engine's run against the oracle's k agents: records, tables and agent state (the call's
    totals cover every agent; the twin tests compare them against the HBM store)."""
    tag = P.combo_id(c)
    for f in ("len", "ret", "tdsum", "tdabs", "q"):
        assert P.bits_equal(g[f][:k], o[f]), (tag, f, P.first_diff(g[f][:k], o[f]))
    if c["selector"] == 1:
        assert np.array_equal(g["counts"][:k], o["counts"]), (tag, "counts")
    for f in ("rng_n", "policy_flag", "ucb_t" if c["selector"] else "epsilon"):
        assert P.bits_equal(g["state"][f][:k], o["state"][f]), (tag, f)


@pytest.mark.parametrize("c", [dict(env=1, agent=1, selector=0, policy=0, target=0, real=0),   # the C2 family
                               dict(env=2, agent=1, selector=1, policy=1, target=1, real=1),
                               dict(env=1, agent=1, selector=1, policy=0, target=1, real=0)], ids=P.combo_id)
@pytest.mark.parametrize("eval_at", [1, 3, 1000])
def test_split_matches_the_oracle(c, eval_at):
    n_ep, k = 8, 48
    h = P.hyper(n_ep)
    o = O.batch_train(P.oracle_config(c, h), 0, k, n_ep, eval_at, n_threads=4)
    ran = 0
    for store in (2, 3):
        eng = on_store(c, h, N_SPLIT, 0, store)
        if eng is None:
            continue
        eng.close()
        compare_agents(P.gpu_run(c, h, N_SPLIT, n_ep, eval_at, store_kind=store), o, c, k)
        ran += 1
    assert ran or c["selector"] == 1


def engine_with_sets(c, h, n, first, store, sets, group, mask):
    """An engine with sets[group[i]] and the selectors eps-greedy, UCB, eps-greedy per set, or None when the store cannot
    hold the agent or the UCB selector (refused, as rlb.h says)."""
    eng = on_store(c, h, n, first, store)
    if eng is None:
        return None
    try:
        eng.set_hparams([as_set(s) for s in sets], group)
        eng.set_selectors(np.array([0, 1, 0], np.int32))
    except abi.RlbError as exc:
        eng.close()
        assert store != 1 and exc.status == abi.ERR_UNSUPPORTED
        return None
    if mask is not None:
        eng.set_active_sets(mask)
    return eng


@pytest.mark.parametrize("real", [0, 1])
@pytest.mark.parametrize("mask", [None, [True, True, False]], ids=["all", "masked"])
def test_split_under_sets_with_both_selectors(real, mask):
    c = dict(env=1, agent=1, selector=0, policy=0, target=0, real=real)
    h = P.hyper(50, max_steps=40)
    sets = [dict(h, lr=0.1, ucb_c=0.3), dict(h, lr=0.05, eps0=0.5, ucb_c=0.7), dict(h, lr=0.2, gamma=0.9, ucb_c=1.1)]
    n = N_SPLIT
    group = (np.arange(n) % 3).astype(np.uint32)
    ran = 0
    for store in (2, 3):
        eng = engine_with_sets(c, h, n, 777, store, sets, group, mask)
        if eng is None:
            continue
        with eng, engine_with_sets(c, h, n, 777, 1, sets, group, mask) as ref:
            twin_calls(eng, ref)
        ran += 1
    assert ran or real == 1
