"""Per-agent hyper-parameter sets (rlb_engine_set_hparams) on the GPU.  The contract is constructor equivalence: after
set_hparams(S, n, g) agent i gives, bit for bit, what agent 0 of an engine built with S[g[i]], n_agents = 1 and
first_agent_id + i gives — checked against the CPU oracle on every env x agent x selector x policy and every table store
the case fits, and against separate engines for the grouped per-episode sums, the call paths, the step-level calls, the
resets, snapshots and the multi-GPU gather."""
import ctypes as C
import importlib

import numpy as np
import pytest

import parity as P
from oracle import oracle_py as O

pytestmark = pytest.mark.gpu

abi = importlib.import_module("rl-rust_b200._abi")
snapshot = importlib.import_module("rl-rust_b200.snapshot")

# the value lists of test_gpu_random_configs.py: negative gamma*lambda, -0.0 and large defaults, lr 7.0, eps0 0
LR = [0.05, 0.5, 1.0, 1.5, 1e-3, 7.0]
GAMMA = [0.95, 1.0, 0.0, -0.7, 0.5]
LAMBDA = [0.5, 1.0, 0.0, -0.9, 0.99]
EPS0 = [1.0, 0.3, 0.0, 0.999]
EPS_FINAL = [0.0, 0.05, 0.5]
UCB_C = [0.5, 0.0, 2.0, -1.0]
DEFAULT_Q = [0.0, -0.0, 1.0, -3.5, 100.0]


def draw_set(rng, decay_kind, n_ep):
    h = dict(lr=float(rng.choice(LR)), gamma=float(rng.choice(GAMMA)), lambda_=float(rng.choice(LAMBDA)),
             eps0=float(rng.choice(EPS0)), eps_final=float(rng.choice(EPS_FINAL)), ucb_c=float(rng.choice(UCB_C)),
             default_q=float(rng.choice(DEFAULT_Q)))
    h["eps_decay"] = float(rng.choice([0.9, 0.5, 0.999])) if decay_kind == 1 else float(rng.choice([1.0 / (0.5 * n_ep), 0.01, 0.3]))
    return h


def as_set(h):
    return dict(learning_rate=h["lr"], discount_factor=h["gamma"], lambda_factor=h["lambda_"], initial_epsilon=h["eps0"],
                epsilon_decay=h["eps_decay"], final_epsilon=h["eps_final"], confidence_level=h["ucb_c"], default_value=h["default_q"])


def run_with_sets(c, h, sets, group, n_ep, eval_at, first=0, store_kind=0):
    with P.make_engine(c, h, len(group), first, store_kind=store_kind) as eng:
        eng.set_hparams([as_set(s) for s in sets], group)
        res = eng.train(n_ep, eval_at, sums=True, episodes=True)
        q, counts = eng.download_tables()
        st = eng.states()
    eps = res["episodes"]
    return dict(ret=eps["ret"].T.astype(np.float64), len=eps["length"].T.astype(np.uint64), tdsum=eps["td_sum"].T.astype(np.float64),
                tdabs=eps["td_abs_sum"].T.astype(np.float64), q=q.astype(np.float64), counts=counts.astype(np.uint64), state=st,
                sums=res["sums"], train_steps=res["train_steps"], eval_steps=res["eval_steps"], records=eps)


def agent_slice(g, i):
    return {k: (g[k][i:i + 1] if k in ("ret", "len", "tdsum", "tdabs", "q", "counts", "state") else g[k]) for k in g}


CASES = [dict(env=env, agent=agent, selector=sel, policy=pol) for env in range(4) for agent in (0, 1) for sel in (0, 1) for pol in (0, 1)]


@pytest.mark.parametrize("k", range(len(CASES)), ids=["%s-%s-%s-%s" % (P.ENV_NAMES[c["env"]], "traces" if c["agent"] else "onestep",
                                                                     "ucb" if c["selector"] else "eps", "double" if c["policy"] else "basic") for c in CASES])
def test_sets_match_the_oracle_agent_by_agent(k):
    rng = np.random.default_rng(7000 + k)
    c = dict(CASES[k], target=int(rng.integers(0, 3)), real=int(rng.integers(0, 2)))
    n_ep, eval_at = int(rng.integers(3, 7)), int(rng.integers(2, 4))
    n_agents, first = int(rng.integers(40, 71)), int(rng.integers(0, 2 ** 40))
    base = P.hyper(n_ep, map_id=int(rng.integers(0, 2)), slippery=bool(rng.integers(0, 2)), max_steps=int(rng.choice([17, 64, 100])),
                   decay_kind=int(rng.integers(0, 2)), seed=int(rng.integers(0, 2 ** 63)))
    sets = [dict(base, **draw_set(rng, base["decay_kind"], n_ep)) for _ in range(4)]
    group = np.arange(n_agents, dtype=np.uint32) % 4          # neighbouring lanes hold different sets
    oracle = [O.batch_train(P.oracle_config(c, sets[group[i]]), first + i, 1, n_ep, eval_at, n_threads=1) for i in range(n_agents)]
    ran = 0
    for store in ((1, 2, 3) if c["env"] in (1, 2) else (1,)) + ((4,) if c["agent"] == 1 else ()):
        try:
            g = run_with_sets(c, base, sets, group, n_ep, eval_at, first=first, store_kind=store)
        except abi.RlbError as exc:
            if store != 1 and exc.status == abi.ERR_UNSUPPORTED:   # this configuration does not fit that store
                continue
            raise
        ran += 1
        for i in range(n_agents):
            o = oracle[i]
            P.compare(agent_slice(g, i), dict(o, train_steps=g["train_steps"], eval_steps=g["eval_steps"]), c)
        assert g["train_steps"] == sum(o["train_steps"] for o in oracle)
        assert g["eval_steps"] == sum(o["eval_steps"] for o in oracle)
    assert ran >= 1


def separate_engines(c, h, sets, per_set, n_ep, eval_at):
    outs = []
    for gi, s in enumerate(sets):
        hs = dict(h, **s)
        outs.append(P.gpu_run(c, hs, per_set, n_ep, eval_at, first_agent_id=gi * per_set))
    return outs


@pytest.mark.parametrize("wl", ["c2", "c4"])
def test_one_engine_with_sets_equals_separate_engines(wl):
    w = P._W.WORKLOADS[wl]
    c = P._W.combo(w, 0)
    n_ep, eval_at, per_set = 20, 10, 3000
    h = P._W.workload_hyper(w)
    h["eps_decay"] = 1.0 / (0.5 * n_ep)
    sets = [dict(lr=0.05, gamma=0.95, lambda_=0.5, eps0=1.0, eps_decay=h["eps_decay"], eps_final=0.0, ucb_c=0.5, default_q=0.0),
            dict(lr=0.2, gamma=0.9, lambda_=0.8, eps0=0.5, eps_decay=0.01, eps_final=0.05, ucb_c=1.0, default_q=-1.0),
            dict(lr=0.01, gamma=0.99, lambda_=0.3, eps0=1.0, eps_decay=0.2, eps_final=0.1, ucb_c=2.0, default_q=0.5)]
    group = np.repeat(np.arange(3, dtype=np.uint32), per_set)
    g = run_with_sets(c, h, sets, group, n_ep, eval_at)
    assert g["sums"].shape == (n_ep, 3, 4)
    for gi, o in enumerate(separate_engines(c, h, sets, per_set, n_ep, eval_at)):
        sl = slice(gi * per_set, (gi + 1) * per_set)
        for key in ("ret", "len", "tdsum", "tdabs", "q", "counts"):
            assert P.bits_equal(g[key][sl], o[key]), (wl, gi, key)
        for key in ("rng_n", "epsilon", "ucb_t", "policy_flag"):
            assert P.bits_equal(g["state"][key][sl], o["state"][key]), (wl, gi, key)
        assert P.bits_equal(g["sums"][:, gi], o["sums"]), (wl, gi, P.first_diff(g["sums"][:, gi], o["sums"]))
    # one set of all agents, equal to the configuration: the engine without sets, sums included
    one = dict(lr=h["lr"], gamma=h["gamma"], lambda_=h["lambda_"], eps0=h["eps0"], eps_decay=h["eps_decay"], eps_final=h["eps_final"],
               ucb_c=h["ucb_c"], default_q=h["default_q"])
    n = 2 * per_set
    g1 = run_with_sets(c, h, [one], np.zeros(n, np.uint32), n_ep, eval_at)
    o1 = P.gpu_run(c, h, n, n_ep, eval_at)
    assert g1["sums"].shape == (n_ep, 1, 4)
    assert P.bits_equal(g1["sums"][:, 0], o1["sums"])
    for key in ("ret", "len", "tdsum", "tdabs", "q"):
        assert P.bits_equal(g1[key], o1[key]), key


def make_c4_with_sets(n_sets=3, per_set=700):
    w = P._W.WORKLOADS["c4"]
    c, h = P._W.combo(w, 0), P._W.workload_hyper(w)
    eng = P.make_engine(c, h, n_sets * per_set)
    sets = [dict(learning_rate=0.05 * (g + 1), discount_factor=0.9 + 0.03 * g, initial_epsilon=1.0 - 0.2 * g,
                 epsilon_decay=0.02 * (g + 1), final_epsilon=0.01 * g, default_value=-0.5 * g) for g in range(n_sets)]
    eng.set_hparams(sets, np.arange(n_sets * per_set, dtype=np.uint32) % n_sets)
    return eng, sets


def test_grouped_sums_identical_across_call_paths():
    n_ep, eval_at = 24, 6
    results = {}
    with make_c4_with_sets()[0] as eng:                       # blocking, sums only
        results["blocking"] = eng.train(n_ep, eval_at)["sums"]
        results["evaluate"] = eng.evaluate(30)["sums"]
    with make_c4_with_sets()[0] as eng:                       # chunked (ep_begin)
        parts = [eng.train(e, eval_at, ep_begin=b)["sums"] for b, e in ((0, 7), (7, 15), (15, 24))]
        results["chunked"] = np.concatenate(parts)
        results["evaluate_chunked"] = eng.evaluate(30)["sums"]
    with make_c4_with_sets()[0] as eng:                       # asynchronous, two calls in flight
        eng.train(12, eval_at, wait=False)
        eng.train(24, eval_at, ep_begin=12, wait=False)
        done = eng.train_wait()
        results["async"] = np.concatenate([d["sums"] for d in done])
    with make_c4_with_sets()[0] as eng:                       # pipelined host records
        r = eng.train(n_ep, eval_at, episodes=True)
        results["pipelined"] = r["sums"]
        assert r["episodes"].shape == (n_ep, eng.N)
    assert results["blocking"].shape == (n_ep, 3, 4)
    for k in ("chunked", "async", "pipelined"):
        assert P.bits_equal(results[k], results["blocking"]), k
    assert results["evaluate"].shape == (30, 3, 4)
    assert P.bits_equal(results["evaluate_chunked"], results["evaluate"])


def test_evaluate_sums_per_set_equal_separate_engines():
    w = P._W.WORKLOADS["c4"]
    c, h = P._W.combo(w, 1), P._W.workload_hyper(w)
    per_set = 500
    sets = [dict(lr=0.1, gamma=0.9, lambda_=0.5, eps0=1.0, eps_decay=0.05, eps_final=0.0, ucb_c=0.5, default_q=0.0),
            dict(lr=0.3, gamma=0.99, lambda_=0.5, eps0=0.2, eps_decay=0.01, eps_final=0.0, ucb_c=0.5, default_q=1.0)]
    with P.make_engine(c, h, 2 * per_set) as eng:
        eng.set_hparams([as_set(s) for s in sets], np.repeat(np.arange(2, dtype=np.uint32), per_set))
        eng.train(10, 5, sums=False)
        ev = eng.evaluate(15)["sums"]
    for gi, s in enumerate(sets):
        with P.make_engine(c, dict(h, **s), per_set, gi * per_set) as e1:
            e1.train(10, 5, sums=False)
            assert P.bits_equal(ev[:, gi], e1.evaluate(15)["sums"]), gi


def test_step_level_calls_and_resets_use_each_agents_set():
    w = P._W.WORKLOADS["c4"]
    c, h = P._W.combo(w, 0), P._W.workload_hyper(w)
    per_set = 64
    sets = [dict(lr=0.1, gamma=0.9, lambda_=0.5, eps0=0.8, eps_decay=0.05, eps_final=0.1, ucb_c=0.5, default_q=2.0),
            dict(lr=0.7, gamma=0.5, lambda_=0.5, eps0=0.3, eps_decay=0.2, eps_final=0.0, ucb_c=0.5, default_q=-1.5)]
    group = np.repeat(np.arange(2, dtype=np.uint32), per_set)
    eng = P.make_engine(c, h, 2 * per_set)
    eng.set_hparams([as_set(s) for s in sets], group)
    singles = [P.make_engine(c, dict(h, **s), per_set, gi * per_set) for gi, s in enumerate(sets)]
    # a host loop over rlb_agent_step: every field of every agent equals its own engine's
    for _ in range(60):
        a = eng.agent_step()
        for gi, e1 in enumerate(singles):
            b = e1.agent_step()
            sl = slice(gi * per_set, (gi + 1) * per_set)
            for key in ("kind", "obs", "action", "reward", "terminated", "td"):
                assert P.bits_equal(a[key][sl].astype(np.float64), b[key].astype(np.float64)), key
    q, _ = eng.download_tables()
    for gi, e1 in enumerate(singles):
        assert P.bits_equal(q[gi * per_set:(gi + 1) * per_set], e1.download_tables()[0])
    # rlb_selector_update decays each epsilon with its own k and floor
    eng.selector_reset()
    for _ in range(5):
        eng.selector_update()
    eps = eng.states()["epsilon"]
    for gi, s in enumerate(sets):
        e = s["eps0"]
        for _ in range(5):
            n = e - s["eps_decay"]
            e = e if s["eps_final"] > n else n
        assert np.all(eps[group == gi] == e), gi
    # resets refill per agent: epsilon to the set's initial value, and (agent reset, a new agent) the tables to its default
    for name, reset, refills_q in (("agent_reset", eng.agent_reset, True), ("set_agent_kind", lambda: eng.set_agent_kind(1), True),
                                   ("set_selector", lambda: eng.set_selector(abi.SEL_EPS_GREEDY), False)):
        eng.train(3, 2, sums=False)
        reset()
        q, _ = eng.download_tables()
        st = eng.states()
        for gi, s in enumerate(sets):
            if refills_q:
                assert np.all(q[group == gi] == np.float32(s["default_q"])), (name, gi)
            assert np.all(st["epsilon"][group == gi] == s["eps0"]), (name, gi)
    eng.set_selector(abi.SEL_UCB)
    q, counts = eng.download_tables()
    assert not counts.any() and np.all(eng.states()["ucb_t"] == 1)
    eng.set_hparams(None, None)                                # back to the configuration's values
    assert eng.hparam_sets() == 0
    assert np.all(eng.download_tables()[0] == np.float32(h["default_q"]))
    for e1 in singles:
        e1.close()
    eng.close()


def raw_set(eng, sets, n, group):
    return abi.lib.rlb_engine_set_hparams(eng.h, abi.ptr(sets), n, abi.ptr(group))


def test_errors_leave_the_engine_untouched():
    w = P._W.WORKLOADS["c4"]
    c, h = P._W.combo(w, 0), P._W.workload_hyper(w)
    with P.make_engine(c, h, 100) as eng:
        sets = eng.hparams_array([dict(default_value=3.0), dict(default_value=4.0)])
        eng.set_hparams(sets, np.arange(100) % 2)
        eng.train(4, 2, sums=False)
        q0, st0 = eng.download_tables()[0], eng.states()
        bad = np.arange(100, dtype=np.uint32) % 2
        bad[57] = 2
        assert raw_set(eng, sets, 2, bad) == abi.ERR_INVALID_ARG                       # group id out of range
        assert raw_set(eng, sets, 0, None) == abi.ERR_INVALID_ARG                      # n_sets 0 with a pointer
        assert raw_set(eng, None, 0, bad) == abi.ERR_INVALID_ARG
        big = np.zeros(abi.MAX_HPARAM_SETS + 1, abi.HPARAMS_DTYPE)
        assert raw_set(eng, big, abi.MAX_HPARAM_SETS + 1, np.zeros(100, np.uint32)) == abi.ERR_INVALID_ARG
        assert abi.lib.rlb_agent_set_model(eng.h, 10) == abi.ERR_UNSUPPORTED          # Dyna after sets
        assert eng.hparam_sets() == 2
        assert P.bits_equal(eng.download_tables()[0], q0)
        st = eng.states()
        for key in ("epsilon", "rng_n", "ucb_t", "policy_flag"):
            assert P.bits_equal(st[key], st0[key]), key
        assert eng.train(2, 1)["sums"].shape == (2, 2, 4)
    with P.make_engine(c, dict(h, planning_steps=10), 100) as eng:                     # sets after Dyna
        assert raw_set(eng, eng.hparams_array([{}]), 1, np.zeros(100, np.uint32)) == abi.ERR_UNSUPPORTED
        assert eng.hparam_sets() == 0


def test_snapshot_with_sets_resumes_bit_identically(tmp_path):
    path = str(tmp_path / "snap.npz")
    eng, sets = make_c4_with_sets(per_set=300)
    eng.train(10, 5, sums=False)
    snapshot.save_snapshot(eng, path)
    want = eng.train(20, 5, ep_begin=10, episodes=True)
    q_want = eng.download_tables()[0]
    eng.close()
    w = P._W.WORKLOADS["c4"]
    with P.make_engine(P._W.combo(w, 0), P._W.workload_hyper(w), 900) as eng2:
        snapshot.load_snapshot(eng2, path)
        assert eng2.hparam_sets() == 3
        got = eng2.train(20, 5, ep_begin=10, episodes=True)
        assert P.bits_equal(got["sums"], want["sums"])
        assert np.array_equal(got["episodes"], want["episodes"])
        assert P.bits_equal(eng2.download_tables()[0], q_want)


@pytest.mark.skipif(abi.lib.rlb_device_count() < 2, reason="needs two GPUs")
def test_two_gpu_gather_of_grouped_sums():
    import torch
    w = P._W.WORKLOADS["c4"]
    c, h = P._W.combo(w, 0), P._W.workload_hyper(w)
    n_sets, half, n_ep = 3, 900, 12
    group = np.arange(2 * half, dtype=np.uint32) % n_sets
    sets = [dict(learning_rate=0.05 * (g + 1), default_value=-0.5 * g) for g in range(n_sets)]
    engines = [P.make_engine(c, h, half, r * half, device=r) for r in range(2)]
    for r, e in enumerate(engines):
        e.set_hparams(sets, group[r * half:(r + 1) * half])
    comms = abi.Comm.init_all([0, 1])
    sums = [torch.zeros((n_ep, n_sets, 4), dtype=torch.float64, device="cuda:%d" % r) for r in range(2)]
    gathered = torch.zeros((2, n_ep, n_sets, 4), dtype=torch.float64, device="cuda:0")
    for r, e in enumerate(engines):
        e.train(n_ep, 4, sums_out=sums[r])
    abi.check(abi.lib.rlb_comm_group_begin())
    for r, cm in enumerate(comms):
        abi.check(abi.lib.rlb_comm_gather_episode_sums(cm.h, abi.ptr(sums[r]), n_ep * n_sets, abi.ptr(gathered) if r == 0 else None, 0,
                                                       C.c_void_p(torch.cuda.current_stream(r).cuda_stream)))
    abi.check(abi.lib.rlb_comm_group_end())
    for r in range(2):
        torch.cuda.synchronize(r)
    got = gathered.cpu().numpy()
    for r in range(2):
        with P.make_engine(c, h, half, r * half) as one:
            one.set_hparams(sets, group[r * half:(r + 1) * half])
            assert P.bits_equal(got[r], one.train(n_ep, 4)["sums"]), r
    for e in engines:
        e.close()
    for cm in comms:
        cm.close()
