"""Dyna-Q under hyper-parameter sets (rlb_engine_set_planning_steps) on the GPU.  Agent i of an engine with sets and
per-set planning counts gives, bit for bit, the reference InternalModelAgent built with sets[group[i]] and
steps[group[i]] planning replays (a count of 0: the plain agent, while its model still records what it sees) — checked
against the CPU oracle agent by agent, against separate engines for the grouped sums and the call paths, and through
the lifecycle: retuned counts, resets, masks, clone, errors, snapshots and the sweep drivers."""
import importlib
import json

import numpy as np
import pytest

import parity as P
from oracle import oracle_py as O
from test_gpu_dyna import CELLS, assert_models_equal
from test_gpu_hparams import as_set, draw_set

pytestmark = pytest.mark.gpu

abi = importlib.import_module("rl-rust_b200._abi")
snapshot = importlib.import_module("rl-rust_b200.snapshot")
driver = importlib.import_module("rl-rust_b200.driver")

COUNTS = [0, 1, 3, 10]
F64_CELLS = (0, 2, 5)   # the bin's cell, traces, Taxi


def oracle_agent(c, h, k, agent_id, n_ep, eval_at):
    """One reference agent with planning count k: its records, tables and states, and its model."""
    cfg = P.oracle_config(c, dict(h, planning_steps=k))
    o = O.batch_train(cfg, agent_id, 1, n_ep, eval_at, n_threads=1)
    s = O.Session(cfg, agent_id)
    s.train(n_ep, eval_at)
    m = s.model()
    s.close()
    return o, m


def tap_model(traj, count, A):
    """The first-seen transitions of an agent's own train steps, read from its trajectory tap: a train step (kind 1)
    follows the reset or step that chose its (obs, action) in the same training episode."""
    seen, out = set(), ([], [], [], [])
    t = traj[:count]
    for j in range(1, len(t)):
        if t[j]["kind"] != 1:
            continue
        s, a = int(t[j - 1]["obs"]), int(t[j - 1]["action"])
        if s * A + a in seen:
            continue
        seen.add(s * A + a)
        for lst, v in zip(out, (s, a, int(t[j]["obs"]), float(t[j]["reward"]))):
            lst.append(v)
    return tuple(np.asarray(x) for x in out)


def engine_with_counts(c, h, group, sets, steps, first=0, store_kind=0):
    eng = P.make_engine(c, h, len(group), first, store_kind=store_kind)
    eng.set_hparams([as_set(s) for s in sets], group)
    eng.set_planning_steps(np.asarray(steps, np.uint32))
    return eng


@pytest.mark.parametrize("k,real", [(k, r) for k in range(len(CELLS)) for r in ((0, 1) if k in F64_CELLS else (0,))],
                         ids=lambda v: str(v))
def test_sets_with_counts_match_the_oracle_agent_by_agent(k, real):
    rng = np.random.default_rng(9100 + 2 * k + real)
    cell, _ = CELLS[k]
    c = dict(cell, real=real)
    n_ep, eval_at = int(rng.integers(3, 6)), 100          # one evaluate block, at episode 0
    n_agents, first = int(rng.integers(24, 41)), int(rng.integers(0, 2 ** 40))
    base = P.hyper(n_ep, max_steps=int(rng.choice([40, 100])), decay_kind=int(rng.integers(0, 2)), seed=int(rng.integers(0, 2 ** 63)))
    sets = [dict(base, **draw_set(rng, base["decay_kind"], n_ep)) for _ in range(4)]
    steps = [int(x) for x in rng.permutation(COUNTS)]
    group = np.arange(n_agents, dtype=np.uint32) % 4      # neighbouring lanes hold different sets and counts
    cap = (n_ep + 100) * (base["max_steps"] + 2) if c["env"] != 0 else 4096
    with engine_with_counts(c, base, group, sets, steps, first) as eng:
        res = eng.train(n_ep, eval_at, sums=True, episodes=True, traj_capacity=cap)
        q, counts = eng.download_tables()
        st = eng.states()
        ln, ent = eng.download_model()
        A = eng.A
    eps = res["episodes"]
    g = dict(ret=eps["ret"].T.astype(np.float64), len=eps["length"].T.astype(np.uint64), tdsum=eps["td_sum"].T.astype(np.float64),
             tdabs=eps["td_abs_sum"].T.astype(np.float64), q=q.astype(np.float64), counts=counts.astype(np.uint64), state=st)
    tot_train = tot_eval = 0
    for i in range(n_agents):
        kk = steps[group[i]]
        o, m = oracle_agent(c, sets[group[i]], kk, first + i, n_ep, eval_at)
        sl = {key: (g[key][i:i + 1] if key != "state" else g[key][i:i + 1]) for key in g}
        P.compare(dict(sl, train_steps=o["train_steps"], eval_steps=o["eval_steps"]), o, c)
        tot_train += o["train_steps"]
        tot_eval += o["eval_steps"]
        if kk > 0:
            assert_models_equal(ln[i:i + 1], ent[i:i + 1], [m], "agent %d (count %d)" % (i, kk))
        else:
            assert int(res["traj_count"][i]) <= cap
            assert_models_equal(ln[i:i + 1], ent[i:i + 1], [tap_model(res["traj"][i], int(res["traj_count"][i]), A)],
                                "agent %d (count 0)" % i)
    assert res["train_steps"] == tot_train and res["eval_steps"] == tot_eval


def test_count_zero_is_the_plain_agent():
    c = dict(CELLS[0][0], real=0)
    h = P.hyper(12)
    n = 64
    with engine_with_counts(c, h, np.zeros(n, np.uint32), [h], [0]) as eng:
        assert abi.lib.rlb_model_capacity(eng.h) > 0 and int(eng.cfg.planning_steps) == 1
        r = eng.train(12, 4, sums=True, episodes=True)
        q, _ = eng.download_tables()
        st = eng.states()
    with P.make_engine(c, h, n) as plain:
        pr = plain.train(12, 4, sums=True, episodes=True)
        pq, _ = plain.download_tables()
        pst = plain.states()
    assert P.bits_equal(r["sums"][:, 0], pr["sums"]) and np.array_equal(r["episodes"], pr["episodes"])
    assert P.bits_equal(q, pq) and np.array_equal(st, pst)


def separate(c, h, sets, steps, per, n_ep, eval_at, chunks=None):
    return [P.gpu_run(c, dict(h, **s, planning_steps=k), per, n_ep, eval_at, first_agent_id=gi * per, chunks=chunks)
            for gi, (s, k) in enumerate(zip(sets, steps))]


SEP_SETS = [dict(lr=0.05, gamma=0.95, lambda_=0.5, eps0=1.0, eps_decay=0.05, eps_final=0.0, ucb_c=0.5, default_q=0.0),
            dict(lr=0.2, gamma=0.9, lambda_=0.8, eps0=0.5, eps_decay=0.01, eps_final=0.05, ucb_c=1.0, default_q=-1.0),
            dict(lr=0.1, gamma=0.99, lambda_=0.3, eps0=1.0, eps_decay=0.2, eps_final=0.1, ucb_c=2.0, default_q=0.5)]
SEP_STEPS = [0, 2, 5]


@pytest.mark.parametrize("path", ["blocking", "chunked", "async", "pipelined"])
def test_one_engine_equals_separate_engines(path):
    c = dict(CELLS[0][0], real=0)
    h = P.hyper(20)
    per, n_ep, eval_at = 256, 20, 7
    group = np.repeat(np.arange(3, dtype=np.uint32), per)
    with engine_with_counts(c, h, group, SEP_SETS, SEP_STEPS) as eng:
        if path == "blocking":
            r = eng.train(n_ep, eval_at, sums=True, episodes=True)
            sums, eps, steps = r["sums"], r["episodes"], r["train_steps"]
        elif path == "chunked":
            parts = [eng.train(e, eval_at, ep_begin=b, sums=True, episodes=True) for b, e in ((0, 6), (6, 13), (13, 20))]
            sums = np.concatenate([p["sums"] for p in parts])
            eps = np.concatenate([p["episodes"] for p in parts])
            steps = sum(p["train_steps"] for p in parts)
        elif path == "async":
            eng.train(9, eval_at, sums=True, episodes=True, wait=False)
            eng.train(n_ep, eval_at, ep_begin=9, sums=True, episodes=True, wait=False)
            parts = eng.train_wait()
            sums = np.concatenate([p["sums"] for p in parts])
            eps = np.concatenate([p["episodes"] for p in parts])
            steps = sum(p["train_steps"] for p in parts)
        else:   # the record pipeline: the host buffer is filled chunk by chunk while the next chunk runs
            out = np.zeros((n_ep, len(group)), eng.episode_dtype)
            r = eng.train(n_ep, eval_at, sums=True, episodes_out=out)
            sums, eps, steps = r["sums"], out, r["train_steps"]
        q, _ = eng.download_tables()
        ln, ent = eng.download_model()
    outs = separate(c, h, SEP_SETS, SEP_STEPS, per, n_ep, eval_at)
    assert steps == sum(o["train_steps"] for o in outs)
    for gi, o in enumerate(outs):
        sl = slice(gi * per, (gi + 1) * per)
        assert P.bits_equal(sums[:, gi], o["sums"]), (path, gi, P.first_diff(sums[:, gi], o["sums"]))
        assert P.bits_equal(eps["ret"][:, sl].T, o["ret"]) and np.array_equal(eps["length"][:, sl].T.astype(np.uint64), o["len"])
        assert P.bits_equal(q[sl], o["q"]), (path, gi)
        if SEP_STEPS[gi]:
            assert np.array_equal(ln[sl], o["model_len"]) and np.array_equal(ent[sl], o["model"]), (path, gi)


def test_step_level_update_and_agent_step():
    c = dict(env=2, agent=0, selector=0, policy=1, target=0, real=1)
    h = P.hyper(50)
    n = 8
    sets = [dict(h, **s) for s in SEP_SETS[:2]]
    steps = [3, 0]
    group = (np.arange(n) % 2).astype(np.uint32)
    sess = [O.Session(P.oracle_config(c, dict(sets[group[i]], planning_steps=steps[group[i]])), i) for i in range(n)]
    rng = np.random.default_rng(11)
    with engine_with_counts(c, h, group, sets, steps) as eng:
        for _ in range(40):
            s = rng.integers(0, 37, n).astype(np.uint32)
            a = rng.integers(0, 4, n).astype(np.uint32)
            s2 = rng.integers(0, 48, n).astype(np.uint32)
            r = rng.choice([-1.0, -100.0], n)
            term = (rng.random(n) < 0.2).astype(np.uint8)
            a2 = eng.get_action(s2)
            td = eng.update(s, a, r, term, s2, a2)
            for i, o in enumerate(sess):
                assert int(a2[i]) == o.get_action(int(s2[i]))
                assert P.bits_equal(td[i], o.update(int(s[i]), int(a[i]), float(r[i]), bool(term[i]), int(s2[i]), int(a2[i])))
        q, _ = eng.download_tables()
        st = eng.states()
        ln, ent = eng.download_model()
    for i, o in enumerate(sess):
        oq, _, ost = o.export()
        assert P.bits_equal(q[i], oq) and int(st["rng_n"][i]) == ost.rng_n, i
        if steps[group[i]]:
            assert_models_equal(ln[i:i + 1], ent[i:i + 1], [o.model()], "update, agent %d" % i)
    # rlb_agent_step: one transition per call, each set against an engine with its count engine-wide
    per = 16
    group = np.repeat(np.arange(2, dtype=np.uint32), per)
    with engine_with_counts(c, h, group, sets, [4, 1]) as eng:
        got = [eng.agent_step() for _ in range(60)]
        q, _ = eng.download_tables()
        ln, ent = eng.download_model()
    for gi, k in enumerate([4, 1]):
        with P.make_engine(c, dict(sets[gi], planning_steps=k), per, gi * per) as ref:
            want = [ref.agent_step() for _ in range(60)]
            rq, _ = ref.download_tables()
            rln, rent = ref.download_model()
        sl = slice(gi * per, (gi + 1) * per)
        for a_, b_ in zip(got, want):
            for key in b_:
                assert np.array_equal(np.asarray(a_[key])[sl], np.asarray(b_[key])), (gi, key)
        assert P.bits_equal(q[sl], rq) and np.array_equal(ln[sl], rln) and np.array_equal(ent[sl], rent)


def copy_of(eng, c, h, steps):
    """An engine B with the same config and the sets this engine has in force (retuned values included), given its
    tables, states and model, then `steps`."""
    q, counts = eng.download_tables()
    st = eng.states()
    ln, ent = eng.download_model()
    sets, group = eng.hparams
    b = P.make_engine(c, h, len(group))
    b.set_hparams(sets, group)
    b.upload_tables(q, counts if c["selector"] == 1 else None)
    b.set_states(st)
    b.set_planning_steps(np.asarray(steps, np.uint32))
    b.upload_model(ln, ent)
    return b


def same_run(a, b, ep0, ep1, eval_at):
    ra = a.train(ep1, eval_at, ep_begin=ep0, sums=True, episodes=True)
    rb = b.train(ep1, eval_at, ep_begin=ep0, sums=True, episodes=True)
    assert P.bits_equal(ra["sums"], rb["sums"]) and np.array_equal(ra["episodes"], rb["episodes"])
    assert P.bits_equal(a.download_tables()[0], b.download_tables()[0])
    assert np.array_equal(a.states(), b.states())
    la, ea = a.download_model()
    lb, eb = b.download_model()
    assert np.array_equal(la, lb) and np.array_equal(ea, eb)


@pytest.mark.parametrize("c", [dict(env=2, agent=0, selector=0, policy=0, target=1, real=0),
                               dict(env=3, agent=0, selector=1, policy=1, target=0, real=1)], ids=P.combo_id)
def test_retuned_counts_and_lifecycle_keep_them(c):
    h = P.hyper(40)
    sets = [dict(h, **s) for s in SEP_SETS]
    group = (np.arange(96) % 3).astype(np.uint32)
    with engine_with_counts(c, h, group, sets, [0, 2, 5]) as a:
        a.train(10, 5)
        a.set_planning_steps(np.array([6, 0, 1], np.uint32))      # only the counts change
        assert list(a.planning) == [6, 0, 1] and int(a.cfg.planning_steps) == 6
        with copy_of(a, c, h, [6, 0, 1]) as b:
            same_run(a, b, 10, 20, 5)
            a.retune_hparams([as_set(dict(s, lr=s["lr"] * 1.2)) for s in sets])      # keeps the counts
            b.retune_hparams([as_set(dict(s, lr=s["lr"] * 1.2)) for s in sets])
            same_run(a, b, 20, 25, 5)
            a.agent_reset()                                                          # empties the model, keeps the counts
            assert not a.download_model()[0].any() and list(a.planning) == [6, 0, 1]
            b.agent_reset()
            same_run(a, b, 25, 30, 5)
        a.set_agent_kind(1)                                                          # re-wraps around an empty model
        assert not a.download_model()[0].any() and list(a.planning) == [6, 0, 1]
        assert abi.lib.rlb_model_capacity(a.h) > 0
        with copy_of(a, c, h, [6, 0, 1]) as b:
            b.set_agent_kind(1)
            b.set_states(a.states())
            same_run(a, b, 30, 33, 5)
        a.set_planning_steps(None)                                                   # drops the model
        assert a.planning is None and abi.lib.rlb_model_capacity(a.h) == 0 and a.hparam_sets() == 3


def test_masked_calls_under_a_model():
    c = dict(CELLS[0][0], real=0)
    h = P.hyper(20)
    sets = [dict(h, **s) for s in SEP_SETS]
    group = (np.arange(150) % 3).astype(np.uint32)
    with engine_with_counts(c, h, group, sets, [4, 0, 2]) as full, engine_with_counts(c, h, group, sets, [4, 0, 2]) as m:
        full.train(6, 3)
        m.train(6, 3)
        ln0, ent0 = m.download_model()
        q0 = m.download_tables()[0]
        m.set_active_sets([True, True, False])
        rf = full.train(12, 3, ep_begin=6, sums=True, episodes=True)
        rm = m.train(12, 3, ep_begin=6, sums=True, episodes=True)
        act = group != 2
        assert P.bits_equal(rm["sums"][:, :2], rf["sums"][:, :2]) and not rm["sums"][:, 2].any()
        assert np.array_equal(rm["episodes"][:, act], rf["episodes"][:, act])
        assert not any(rm["episodes"][f][:, ~act].any() for f in rm["episodes"].dtype.names)
        ln, ent = m.download_model()
        lf, ef = full.download_model()
        assert np.array_equal(ln[act], lf[act]) and np.array_equal(ent[act], ef[act])
        assert np.array_equal(ln[~act], ln0[~act]) and np.array_equal(ent[~act], ent0[~act])   # paused: bit for bit
        assert P.bits_equal(m.download_tables()[0][~act], q0[~act])
        m.set_active_sets(np.zeros(3, bool))                                                   # launches nothing
        r0 = m.train(14, 3, ep_begin=12, sums=True)
        assert r0["train_steps"] == 0 and not r0["sums"].any()


def test_clone_with_a_model_under_sets():
    c = dict(env=3, agent=0, selector=1, policy=1, target=1, real=0)
    h = P.hyper(20)
    sets = [dict(h, **s) for s in SEP_SETS]
    group = np.repeat(np.arange(3, dtype=np.uint32), 20)
    src, dst = np.arange(20, 30), np.arange(40, 50)
    with engine_with_counts(c, h, group, sets, [3, 0, 1]) as a, engine_with_counts(c, h, group, sets, [3, 0, 1]) as b:
        a.train(8, 4)
        b.train(8, 4)
        a.clone_agents(src, dst)
        q, counts = b.download_tables()
        st = b.states()
        ln, ent = b.download_model()
        for arr in (q, counts, ln, ent):
            arr[dst] = arr[src]
        for f in ("epsilon", "ucb_t", "policy_flag"):
            st[f][dst] = st[f][src]
        b.upload_tables(q, counts)
        b.set_states(st)
        b.upload_model(ln, ent)
        same_run(a, b, 8, 14, 4)
    ct = dict(c, agent=1)
    with engine_with_counts(ct, h, group, sets, [3, 0, 1]) as t:
        with pytest.raises(abi.RlbError) as ei:
            t.clone_agents(src, dst)
        assert ei.value.status == abi.ERR_UNSUPPORTED


def test_errors_leave_the_engine_untouched():
    c = dict(CELLS[0][0], real=0)
    h = P.hyper(10)
    with P.make_engine(c, h, 32) as eng:
        k = np.array([1, 2], np.uint32)
        assert abi.lib.rlb_engine_set_planning_steps(eng.h, abi.ptr(k), 2) == abi.ERR_INVALID_ARG       # no sets
        eng.set_hparams([as_set(h)] * 2, (np.arange(32) % 2).astype(np.uint32))
        assert abi.lib.rlb_engine_set_planning_steps(eng.h, abi.ptr(k), 3) == abi.ERR_INVALID_ARG       # count mismatch
        assert abi.lib.rlb_engine_set_planning_steps(eng.h, None, 2) == abi.ERR_INVALID_ARG            # NULL with a count
        assert abi.lib.rlb_engine_set_planning_steps(eng.h, abi.ptr(k), 0) == abi.ERR_INVALID_ARG       # a pointer with 0
        assert abi.lib.rlb_model_capacity(eng.h) == 0
        eng.set_planning_steps(k)
        before = (eng.download_tables()[0], eng.states(), eng.download_model())
        assert abi.lib.rlb_engine_set_planning_steps(eng.h, abi.ptr(k), 1) == abi.ERR_INVALID_ARG
        assert abi.lib.rlb_engine_set_hparams(eng.h, None, 0, None) == abi.ERR_UNSUPPORTED             # counts in force
        arr = eng.hparams_array([as_set(h)] * 2)
        grp = np.zeros(32, np.uint32)
        assert abi.lib.rlb_engine_set_hparams(eng.h, abi.ptr(arr), 2, abi.ptr(grp)) == abi.ERR_UNSUPPORTED   # model attached
        assert abi.lib.rlb_agent_set_model(eng.h, 5) == abi.ERR_UNSUPPORTED
        assert eng.hparam_sets() == 2 and abi.lib.rlb_model_capacity(eng.h) > 0
        after = (eng.download_tables()[0], eng.states(), eng.download_model())
        assert P.bits_equal(before[0], after[0]) and np.array_equal(before[1], after[1])
        assert np.array_equal(before[2][0], after[2][0]) and np.array_equal(before[2][1], after[2][1])
        eng.set_model(0)                                                                               # drops the counts too
        assert eng.planning is None and abi.lib.rlb_model_capacity(eng.h) == 0
        eng.set_hparams(None, None)
    cl = dict(c, agent=1)
    with P.make_engine(cl, h, 32, store_kind=2) as eng:                                                  # a shared-memory store
        eng.set_hparams([as_set(h)], np.zeros(32, np.uint32))
        with pytest.raises(abi.RlbError) as ei:
            eng.set_planning_steps(np.array([2], np.uint32))
        assert ei.value.status == abi.ERR_UNSUPPORTED and abi.lib.rlb_model_capacity(eng.h) == 0


def test_snapshot_with_counts_and_a_mask_resumes_bit_identically(tmp_path):
    c = dict(env=2, agent=0, selector=1, policy=0, target=1, real=1)
    h = P.hyper(30)
    sets = [dict(h, **s) for s in SEP_SETS]
    group = (np.arange(90) % 3).astype(np.uint32)
    path = str(tmp_path / "snap.npz")
    with engine_with_counts(c, h, group, sets, [5, 0, 2]) as a:
        a.train(10, 5)
        a.set_active_sets([True, False, True])
        snapshot.save_snapshot(a, path)
        with P.make_engine(c, h, 90) as b:
            snapshot.load_snapshot(b, path)
            assert list(b.planning) == [5, 0, 2] and list(b.active_sets) == [True, False, True]
            same_run(a, b, 10, 20, 5)
        with P.make_engine(c, dict(h, planning_steps=3), 90) as b:      # an engine that has a model of its own
            snapshot.load_snapshot(b, path)
            assert list(b.planning) == [5, 0, 2]


def test_sweep_with_a_planning_axis_equals_separate_engines():
    grid = {"planning_steps": [0, 3], "learning_rate": [0.1, 0.5]}
    per, n = 128, 40
    res = driver.run_sweep("cliffwalking", grid, target="qlearning", agents_per_point=per, n_episodes=n, real="f32", verbose=False)
    assert [p["params"]["planning_steps"] for p in res["points"]] == [0, 0, 3, 3]
    for g, pt in enumerate(res["points"]):
        env = driver.make_env("cliffwalking", **dict(driver.DEFAULTS, n_episodes=n))
        with abi.Engine(env.kind, n_agents=per, selector=abi.SEL_EPS_GREEDY, target=abi.TARGET_QLEARNING, real=abi.REAL_F32,
                        decay_kind=abi.DECAY_SUB, first_agent_id=g * per, planning_steps=pt["params"]["planning_steps"],
                        **pt["hparams"], **env._cfg()) as eng:
            r = eng.train(n, n // 10, sums=True)
            ev = eng.evaluate(n, sums=True)["sums"]
        window = max(1, n // driver.DEFAULTS["moving_average_window"])
        assert pt["train_rewards"] == driver.moving_average(window, r["sums"][:, 1] / per), g
        assert pt["eval_mean_return"] == float(ev[:, 1].sum()) / (per * n), g


def test_halving_and_pbt_run_end_to_end():
    grid = {"planning_steps": [0, 2, 5], "learning_rate": [0.1, 0.5]}
    kw = dict(target="qlearning", agents_per_point=64, n_episodes=60, real="f32", verbose=False)
    hv = driver.run_halving("cliffwalking", grid, min_episodes=10, eta=3, **kw)
    assert len(hv["rungs"]) >= 2 and len(hv["rungs"][-1]["active"]) >= 1
    a = driver.run_pbt("cliffwalking", grid, interval=20, fraction=0.34, pbt_seed=5, **kw)
    b = driver.run_pbt("cliffwalking", grid, interval=20, fraction=0.34, pbt_seed=5, **kw)
    a.pop("seconds"), b.pop("seconds")
    assert json.dumps(a) == json.dumps(b)
    moved = [p["flags"]["planning_steps"] for step in a["lineage"] for p in step["pairs"]]
    assert moved and all(isinstance(k, int) and k >= 0 for k in moved)
    assert all(isinstance(p["final_params"]["planning_steps"], int) for p in a["points"])
    with pytest.raises(ValueError):
        driver.run_pbt("cliffwalking", grid, interval=20, agent="traces", **kw)
