"""The bootstrap target per hyper-parameter set (rlb_engine_set_targets) on the GPU.  Agent i of an engine with sets and
per-set targets gives, bit for bit, agent 0 of an engine built with sets[group[i]] and target targets[group[i]] —
checked against the CPU oracle agent by agent on every env x agent x selector x policy and every store the case fits
(neighbouring lanes with different targets), against separate engines on four call paths and at the step level, with
Dyna planning counts, and through the lifecycle rules, errors, snapshots and the sweep drivers."""
import importlib
import json

import numpy as np
import pytest

import parity as P
from oracle import oracle_py as O
from test_gpu_dyna import CELLS
from test_gpu_hparams import CASES, agent_slice, as_set, draw_set

pytestmark = pytest.mark.gpu

abi = importlib.import_module("rl-rust_b200._abi")
snapshot = importlib.import_module("rl-rust_b200.snapshot")
driver = importlib.import_module("rl-rust_b200.driver")

F64_CASES = (1, 6, 11, 13, 20, 27, 30)   # a subset of CASES in f64: every env, both agents, both selectors and policies


def run_with_targets(c, h, sets, group, targets, n_ep, eval_at, first=0, store_kind=0):
    with P.make_engine(c, h, len(group), first, store_kind=store_kind) as eng:
        eng.set_hparams([as_set(s) for s in sets], group)
        eng.set_targets(targets)
        store = eng.store_kind()
        res = eng.train(n_ep, eval_at, sums=True, episodes=True)
        q, counts = eng.download_tables()
        st = eng.states()
    eps = res["episodes"]
    return dict(ret=eps["ret"].T.astype(np.float64), len=eps["length"].T.astype(np.uint64), tdsum=eps["td_sum"].T.astype(np.float64),
                tdabs=eps["td_abs_sum"].T.astype(np.float64), q=q.astype(np.float64), counts=counts.astype(np.uint64), state=st,
                sums=res["sums"], train_steps=res["train_steps"], eval_steps=res["eval_steps"], store=store)


@pytest.mark.parametrize("k,real", [(k, 0) for k in range(len(CASES))] + [(k, 1) for k in F64_CASES], ids=lambda v: str(v))
def test_targets_match_the_oracle_agent_by_agent(k, real):
    rng = np.random.default_rng(12000 + 2 * k + real)
    targets = [int(x) for x in rng.permutation(3)]
    c = dict(CASES[k], target=int(rng.integers(0, 3)), real=real)   # the engine-wide target, overridden per set
    n_ep, eval_at = int(rng.integers(3, 7)), int(rng.integers(2, 4))
    n_agents, first = int(rng.integers(40, 71)), int(rng.integers(0, 2 ** 40))
    base = P.hyper(n_ep, map_id=int(rng.integers(0, 2)), slippery=bool(rng.integers(0, 2)), max_steps=int(rng.choice([17, 64, 100])),
                   decay_kind=int(rng.integers(0, 2)), seed=int(rng.integers(0, 2 ** 63)))
    sets = [dict(base, **draw_set(rng, base["decay_kind"], n_ep)) for _ in range(3)]
    group = np.arange(n_agents, dtype=np.uint32) % 3          # neighbouring lanes hold different targets
    oracle = [O.batch_train(P.oracle_config(dict(c, target=targets[group[i]]), sets[group[i]]), first + i, 1, n_ep, eval_at, n_threads=1)
              for i in range(n_agents)]
    ran = set()
    for store in ((1, 2, 3) if c["env"] in (1, 2) else (1,)) + ((4,) if c["agent"] == 1 else ()):
        try:
            g = run_with_targets(c, base, sets, group, targets, n_ep, eval_at, first=first, store_kind=store)
        except abi.RlbError as exc:
            if store != 1 and exc.status == abi.ERR_UNSUPPORTED:   # this configuration does not fit that store
                continue
            raise
        ran.add(g["store"])
        for i in range(n_agents):
            o = oracle[i]
            P.compare(agent_slice(g, i), dict(o, train_steps=g["train_steps"], eval_steps=g["eval_steps"]), dict(c, target=targets[group[i]]))
        assert g["train_steps"] == sum(o["train_steps"] for o in oracle)
        assert g["eval_steps"] == sum(o["eval_steps"] for o in oracle)
    assert 1 in ran
    if c["env"] == 1 and c["agent"] == 1:
        assert 3 in ran                                          # FrozenLake traces: the hybrid store ran
    if c["env"] == 3 and c["agent"] == 1:
        assert 4 in ran                                          # Taxi traces: the lazy store ran


SEP_SETS = [dict(lr=0.05, gamma=0.95, lambda_=0.5, eps0=1.0, eps_decay=0.05, eps_final=0.0, ucb_c=0.5, default_q=0.0),
            dict(lr=0.2, gamma=0.9, lambda_=0.8, eps0=0.5, eps_decay=0.01, eps_final=0.05, ucb_c=1.0, default_q=-1.0),
            dict(lr=0.1, gamma=0.99, lambda_=0.3, eps0=1.0, eps_decay=0.2, eps_final=0.1, ucb_c=2.0, default_q=0.5)]
SEP_TARGETS = [abi.TARGET_EXPECTED_SARSA, abi.TARGET_SARSA, abi.TARGET_QLEARNING]


def engine_with_targets(c, h, group, sets, targets, first=0, store_kind=0):
    eng = P.make_engine(c, h, len(group), first, store_kind=store_kind)
    eng.set_hparams([as_set(s) for s in sets], group)
    eng.set_targets(np.asarray(targets, np.int32))
    return eng


@pytest.mark.parametrize("path", ["blocking", "chunked", "async", "pipelined"])
@pytest.mark.parametrize("wl", ["c2", "c4"])
def test_one_engine_equals_separate_engines(wl, path):
    w = P._W.WORKLOADS[wl]
    c, h = P._W.combo(w, 0), P._W.workload_hyper(w)
    per, n_ep, eval_at = 512, 20, 7
    group = np.repeat(np.arange(3, dtype=np.uint32), per)
    with engine_with_targets(c, h, group, SEP_SETS, SEP_TARGETS) as eng:
        if path == "blocking":
            r = eng.train(n_ep, eval_at, sums=True, episodes=True)
            sums, eps, steps = r["sums"], r["episodes"], r["train_steps"]
        elif path == "chunked":
            parts = [eng.train(e, eval_at, ep_begin=b, sums=True, episodes=True) for b, e in ((0, 6), (6, 13), (13, 20))]
            sums, eps = np.concatenate([p["sums"] for p in parts]), np.concatenate([p["episodes"] for p in parts])
            steps = sum(p["train_steps"] for p in parts)
        elif path == "async":
            eng.train(9, eval_at, sums=True, episodes=True, wait=False)
            eng.train(n_ep, eval_at, ep_begin=9, sums=True, episodes=True, wait=False)
            parts = eng.train_wait()
            sums, eps = np.concatenate([p["sums"] for p in parts]), np.concatenate([p["episodes"] for p in parts])
            steps = sum(p["train_steps"] for p in parts)
        else:   # the record pipeline: the host buffer is filled chunk by chunk while the next chunk runs
            out = np.zeros((n_ep, len(group)), eng.episode_dtype)
            r = eng.train(n_ep, eval_at, sums=True, episodes_out=out)
            sums, eps, steps = r["sums"], out, r["train_steps"]
        q, _ = eng.download_tables()
        st = eng.states()
    outs = [P.gpu_run(dict(c, target=t), dict(h, **s), per, n_ep, eval_at, first_agent_id=gi * per)
            for gi, (s, t) in enumerate(zip(SEP_SETS, SEP_TARGETS))]
    assert steps == sum(o["train_steps"] for o in outs)
    for gi, o in enumerate(outs):
        sl = slice(gi * per, (gi + 1) * per)
        assert P.bits_equal(sums[:, gi], o["sums"]), (wl, path, gi, P.first_diff(sums[:, gi], o["sums"]))
        assert P.bits_equal(eps["ret"][:, sl].T, o["ret"]) and np.array_equal(eps["length"][:, sl].T.astype(np.uint64), o["len"])
        assert P.bits_equal(eps["td_sum"][:, sl].T, o["tdsum"]), (wl, path, gi)
        assert P.bits_equal(q[sl], o["q"]), (wl, path, gi)
        for key in ("rng_n", "epsilon", "ucb_t", "policy_flag"):
            assert P.bits_equal(st[key][sl], o["state"][key]), (wl, path, gi, key)


def test_step_level_update_and_agent_step():
    c = dict(env=2, agent=0, selector=1, policy=1, target=1, real=1)
    h = P.hyper(50)
    per = 16
    sets = [dict(h, **s) for s in SEP_SETS]
    group = np.repeat(np.arange(3, dtype=np.uint32), per)
    rng = np.random.default_rng(21)
    singles = [P.make_engine(dict(c, target=t), sets[gi], per, gi * per) for gi, t in enumerate(SEP_TARGETS)]
    with engine_with_targets(c, h, group, sets, SEP_TARGETS) as eng:
        # rlb_agent_update on caller transitions
        for _ in range(30):
            n = len(group)
            s = rng.integers(0, 37, n).astype(np.uint32)
            a = rng.integers(0, 4, n).astype(np.uint32)
            s2 = rng.integers(0, 48, n).astype(np.uint32)
            r = rng.choice([-1.0, -100.0], n)
            term = (rng.random(n) < 0.2).astype(np.uint8)
            a2 = eng.get_action(s2)
            td = eng.update(s, a, r, term, s2, a2)
            for gi, e1 in enumerate(singles):
                sl = slice(gi * per, (gi + 1) * per)
                assert np.array_equal(a2[sl], e1.get_action(s2[sl])), gi
                assert P.bits_equal(td[sl], e1.update(s[sl], a[sl], r[sl], term[sl], s2[sl], a2[sl])), gi
        # rlb_agent_step: one transition per call
        for _ in range(60):
            got = eng.agent_step()
            for gi, e1 in enumerate(singles):
                want = e1.agent_step()
                sl = slice(gi * per, (gi + 1) * per)
                for key in ("kind", "obs", "action", "reward", "terminated", "td"):
                    assert P.bits_equal(np.asarray(got[key])[sl].astype(np.float64), np.asarray(want[key]).astype(np.float64)), (gi, key)
        q, counts = eng.download_tables()
        for gi, e1 in enumerate(singles):
            sl = slice(gi * per, (gi + 1) * per)
            q1, c1 = e1.download_tables()
            assert P.bits_equal(q[sl], q1) and np.array_equal(counts[sl], c1), gi
    for e1 in singles:
        e1.close()


DYNA_STEPS = [0, 2, 5]


@pytest.mark.parametrize("k", range(len(CELLS)), ids=lambda v: P.combo_id(dict(CELLS[v][0], real=0)))
def test_targets_with_planning_counts_match_the_oracle(k):
    rng = np.random.default_rng(13000 + k)
    c = dict(CELLS[k][0], real=int(rng.integers(0, 2)))
    n_ep, eval_at = int(rng.integers(3, 6)), 100
    n_agents, first = int(rng.integers(24, 41)), int(rng.integers(0, 2 ** 40))
    base = P.hyper(n_ep, max_steps=int(rng.choice([40, 100])), decay_kind=int(rng.integers(0, 2)), seed=int(rng.integers(0, 2 ** 63)))
    sets = [dict(base, **draw_set(rng, base["decay_kind"], n_ep)) for _ in range(3)]
    targets = [int(x) for x in rng.permutation(3)]
    steps = [int(x) for x in rng.permutation(DYNA_STEPS)]
    group = np.arange(n_agents, dtype=np.uint32) % 3
    with engine_with_targets(c, base, group, sets, targets, first) as eng:
        eng.set_planning_steps(np.asarray(steps, np.uint32))
        assert list(eng.targets) == targets
        res = eng.train(n_ep, eval_at, sums=True, episodes=True)
        q, counts = eng.download_tables()
        st = eng.states()
    eps = res["episodes"]
    g = dict(ret=eps["ret"].T.astype(np.float64), len=eps["length"].T.astype(np.uint64), tdsum=eps["td_sum"].T.astype(np.float64),
             tdabs=eps["td_abs_sum"].T.astype(np.float64), q=q.astype(np.float64), counts=counts.astype(np.uint64), state=st)
    for i in range(n_agents):
        ci = dict(c, target=targets[group[i]])
        o = O.batch_train(P.oracle_config(ci, dict(sets[group[i]], planning_steps=steps[group[i]])), first + i, 1, n_ep, eval_at, n_threads=1)
        P.compare(dict(agent_slice(g, i), train_steps=o["train_steps"], eval_steps=o["eval_steps"]), o, ci)


def copy_of(eng, c, h, targets=None):
    """An engine B with the same config and the sets this engine has in force, given its tables, states and model, then
    `targets` (None: the engine-wide target)."""
    q, counts = eng.download_tables()
    st = eng.states()
    sets, group = eng.hparams
    b = P.make_engine(dict(c, target=int(eng.cfg.target_kind), agent=int(eng.cfg.agent_kind)), h, len(group))
    b.set_hparams(sets, group)
    b.upload_tables(q, counts if c["selector"] == 1 else None)
    b.set_states(st)
    if eng.planning is not None:
        b.set_planning_steps(eng.planning)
        b.upload_model(*eng.download_model())
    if targets is not None:
        b.set_targets(np.asarray(targets, np.int32))
    return b


def fields_equal(x, y):
    """Structured arrays (episode records, agent states) equal field by field, floats bit for bit (NaN == NaN: diverging
    f64 agents carry NaN TD sums, which np.array_equal never finds equal)."""
    return x.dtype == y.dtype and all(P.bits_equal(x[f], y[f]) if x.dtype[f].kind == "f" else np.array_equal(x[f], y[f])
                                      for f in x.dtype.names)


def same_run(a, b, ep0, ep1, eval_at):
    ra = a.train(ep1, eval_at, ep_begin=ep0, sums=True, episodes=True)
    rb = b.train(ep1, eval_at, ep_begin=ep0, sums=True, episodes=True)
    assert P.bits_equal(ra["sums"], rb["sums"]) and fields_equal(ra["episodes"], rb["episodes"])
    assert P.bits_equal(a.download_tables()[0], b.download_tables()[0])
    assert fields_equal(a.states(), b.states())


@pytest.mark.parametrize("c", [dict(env=3, agent=0, selector=0, policy=0, target=1, real=0),
                               dict(env=2, agent=1, selector=1, policy=1, target=0, real=1)], ids=P.combo_id)
def test_retarget_and_lifecycle(c):
    h = P.hyper(40)
    sets = [dict(h, **s) for s in SEP_SETS]
    group = (np.arange(96) % 3).astype(np.uint32)
    with engine_with_targets(c, h, group, sets, SEP_TARGETS) as a:
        a.train(10, 5)
        a.set_targets(np.array([1, 2, 0], np.int32))                                # a retarget between chunks
        assert list(a.targets) == [1, 2, 0]
        with copy_of(a, c, h, [1, 2, 0]) as b:
            same_run(a, b, 10, 16, 5)
            ep = 16
            for name, act in (("retune", lambda e: e.retune_hparams([as_set(dict(s, lr=s["lr"] * 1.2)) for s in sets])),
                              ("mask", lambda e: e.set_active_sets([True, False, True])),
                              ("unmask", lambda e: e.set_active_sets(None)),
                              ("agent_reset", lambda e: e.agent_reset()),
                              ("selector_reset", lambda e: e.selector_reset()),
                              ("policy_reset", lambda e: e.policy_reset()),
                              ("set_kind", lambda e: e.set_agent_kind(1 - int(c["agent"])))):
                act(a)
                act(b)
                assert list(a.targets) == [1, 2, 0], name                               # kept
                b.set_states(a.states())
                same_run(a, b, ep, ep + 3, 5)
                ep += 3
        src, dst = np.arange(0, 96, 3), np.arange(1, 96, 3)                         # set 0 -> set 1: dst keeps set 1's target
        with copy_of(a, c, h, [1, 2, 0]) as b:
            a.clone_agents(src, dst)
            q, counts = b.download_tables()
            st = b.states()
            q[dst], counts[dst] = q[src], counts[src]
            for f in ("epsilon", "ucb_t", "policy_flag"):
                st[f][dst] = st[f][src]
            b.upload_tables(q, counts if c["selector"] == 1 else None)
            b.set_states(st)
            same_run(a, b, ep, ep + 5, 5)
        a.set_target(2)                                                             # every agent now uses 2
        assert a.targets is None and int(a.cfg.target_kind) == 2
        with copy_of(a, c, h) as b:
            same_run(a, b, ep + 5, ep + 9, 5)
        a.set_targets(np.array([0, 0, 1], np.int32))
        a.set_hparams(*a.hparams)                                                   # back to the engine-wide target
        assert a.targets is None
        with copy_of(a, c, h) as b:
            same_run(a, b, ep + 9, ep + 13, 5)
        a.set_targets(np.array([2, 2, 2], np.int32))                                # all equal the configured one
        assert a.targets is None


def test_targets_kept_by_planning_counts():
    c = dict(env=2, agent=0, selector=0, policy=0, target=1, real=0)
    h = P.hyper(30)
    sets = [dict(h, **s) for s in SEP_SETS]
    group = (np.arange(90) % 3).astype(np.uint32)
    with engine_with_targets(c, h, group, sets, SEP_TARGETS) as a:
        a.train(5, 5)
        a.set_planning_steps(np.array([3, 0, 1], np.uint32))
        assert list(a.targets) == SEP_TARGETS
        with copy_of(a, c, h, SEP_TARGETS) as b:
            same_run(a, b, 5, 12, 5)


def test_errors_leave_the_engine_untouched():
    c = dict(env=3, agent=0, selector=0, policy=0, target=1, real=0)
    h = P.hyper(10)
    with P.make_engine(c, h, 60) as eng:
        t = np.array([0, 2], np.int32)
        assert abi.lib.rlb_engine_set_targets(eng.h, abi.ptr(t), 2) == abi.ERR_INVALID_ARG           # no sets
        eng.set_hparams([as_set(dict(h, **s)) for s in SEP_SETS[:2]], (np.arange(60) % 2).astype(np.uint32))
        eng.set_targets(t)
        eng.train(4, 2)
        before = (eng.download_tables()[0], eng.states())
        for bad, n in ((t, 3), (t, 1), (None, 2), (t, 0), (None, 0), (np.array([0, 3], np.int32), 2),
                       (np.array([-1, 1], np.int32), 2), (np.array([2, 7], np.int32), 2)):
            assert abi.lib.rlb_engine_set_targets(eng.h, abi.ptr(bad), n) == abi.ERR_INVALID_ARG, (bad, n)
        with pytest.raises(ValueError):
            eng.set_targets(np.array([0, 3]))
        assert P.bits_equal(eng.download_tables()[0], before[0]) and fields_equal(eng.states(), before[1])
        with copy_of(eng, c, h, [0, 2]) as b:                                        # the targets in force are still [0, 2]
            same_run(eng, b, 4, 10, 2)


def test_snapshot_with_targets_and_a_mask_resumes_bit_identically(tmp_path):
    c = dict(env=2, agent=0, selector=1, policy=0, target=1, real=1)
    h = P.hyper(30)
    sets = [dict(h, **s) for s in SEP_SETS]
    group = (np.arange(90) % 3).astype(np.uint32)
    path = str(tmp_path / "snap.npz")
    with engine_with_targets(c, h, group, sets, SEP_TARGETS) as a:
        a.train(10, 5)
        a.set_active_sets([True, False, True])
        snapshot.save_snapshot(a, path)
        assert list(np.load(path)["hp_target"]) == SEP_TARGETS
        with P.make_engine(c, h, 90) as b:
            snapshot.load_snapshot(b, path)
            assert list(b.targets) == SEP_TARGETS and list(b.active_sets) == [True, False, True]
            same_run(a, b, 10, 20, 5)


def sweep_kw(**kw):
    return dict(dict(agents_per_point=128, n_episodes=40, real="f32", verbose=False), **kw)


def test_sweep_with_a_target_axis_equals_one_sweep_per_target():
    grid = {"target": ["sarsa", "qlearning", "expected_sarsa"], "learning_rate": [0.1, 0.5]}
    res = driver.run_sweep("taxi", grid, **sweep_kw())
    assert res["target"] is None and [p["params"]["target"] for p in res["points"]] == ["sarsa"] * 2 + ["qlearning"] * 2 + ["expected_sarsa"] * 2
    per = res["agents_per_point"]
    for ti, name in enumerate(grid["target"]):
        # the same points, seeds and agent ids as a sweep of this target alone: first_agent_id shifts by the points before
        one = driver.run_sweep("taxi", {"learning_rate": [0.1, 0.5]}, target=name, **sweep_kw())
        for j, pt in enumerate(one["points"]):
            g = 2 * ti + j
            env = driver.make_env("taxi", **dict(driver.DEFAULTS, n_episodes=40))
            with abi.Engine(env.kind, n_agents=per, selector=abi.SEL_EPS_GREEDY, target=driver.TARGET_KINDS[name], real=abi.REAL_F32,
                            decay_kind=abi.DECAY_SUB, first_agent_id=g * per, **pt["hparams"], **env._cfg()) as eng:
                r = eng.train(40, 4, sums=True)
                ev = eng.evaluate(40, sums=True)["sums"]
            window = max(1, 40 // driver.DEFAULTS["moving_average_window"])
            assert res["points"][g]["train_rewards"] == driver.moving_average(window, r["sums"][:, 1] / per), (name, j)
            assert res["points"][g]["eval_mean_return"] == float(ev[:, 1].sum()) / (per * 40), (name, j)
            if ti == 0:                                                        # same agent ids as the one-target sweep
                for key in ("train_rewards", "train_episodes_length", "test_rewards", "test_episodes_length", "eval_mean_return"):
                    assert res["points"][g][key] == pt[key], (name, j, key)


def test_pbt_and_halving_with_a_target_axis():
    grid = {"target": ["sarsa", "qlearning", "expected_sarsa"], "learning_rate": [0.1, 0.5], "planning_steps": [0, 2]}
    kw = sweep_kw(agents_per_point=64, n_episodes=60)
    a = driver.run_pbt("cliffwalking", grid, interval=20, fraction=0.34, pbt_seed=5, resample_probability=0.5, **kw)
    b = driver.run_pbt("cliffwalking", grid, interval=20, fraction=0.34, pbt_seed=5, resample_probability=0.5, **kw)
    a.pop("seconds"), b.pop("seconds")
    assert json.dumps(a) == json.dumps(b)
    moved = [p["flags"]["target"] for step in a["lineage"] for p in step["pairs"]]
    assert moved and all(t in driver.TARGET_KINDS for t in moved)
    hv = driver.run_halving("cliffwalking", grid, min_episodes=10, eta=3, **kw)
    sw = driver.run_sweep("cliffwalking", grid, **kw)
    survivors = hv["rungs"][-1]["active"]
    assert survivors
    for g in survivors:                                                        # a survivor is its sweep point, bit for bit
        for key in ("train_rewards", "test_rewards", "test_episodes_length", "eval_mean_return"):
            assert hv["points"][g][key] == sw["points"][g][key], (g, key)
