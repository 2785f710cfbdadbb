"""The action selector per hyper-parameter set (rlb_engine_set_selectors) on the GPU.  Agent i of an engine with sets and
per-set selectors gives, bit for bit, agent 0 of an engine built with sets[group[i]] and selector selectors[group[i]] —
checked against the CPU oracle agent by agent on every env x agent x policy and every store the case fits (neighbouring
lanes on different selectors, per-set targets mixed in), against engines that hold every set on one selector on four
call paths, under masks and at the step level, through selector changes, Dyna counts, clones, snapshots, errors and the
sweep drivers."""
import importlib
import json

import numpy as np
import pytest

import parity as P
from oracle import oracle_py as O
from test_gpu_dyna import CELLS
from test_gpu_hparams import CASES, agent_slice, as_set, draw_set
from test_gpu_targets import SEP_SETS, fields_equal, same_run

pytestmark = pytest.mark.gpu

abi = importlib.import_module("rl-rust_b200._abi")
snapshot = importlib.import_module("rl-rust_b200.snapshot")
driver = importlib.import_module("rl-rust_b200.driver")

# CASES without the selector (it is per set here): env x agent x policy
SEL_CASES = [c for c in CASES if c["selector"] == 0]
F64_CASES = (0, 3, 5, 6, 9, 15)
SEP_SEL = [abi.SEL_UCB, abi.SEL_EPS_GREEDY, abi.SEL_UCB]


def engine_with_selectors(c, h, group, sets, selectors, first=0, store_kind=0, targets=None):
    eng = P.make_engine(c, h, len(group), first, store_kind=store_kind)
    try:
        eng.set_hparams([as_set(s) for s in sets], group)
        if targets is not None:
            eng.set_targets(np.asarray(targets, np.int32))
        eng.set_selectors(np.asarray(selectors, np.int32))
    except BaseException:
        eng.close()
        raise
    return eng


@pytest.mark.parametrize("k,real", [(k, 0) for k in range(len(SEL_CASES))] + [(k, 1) for k in F64_CASES], ids=lambda v: str(v))
def test_selectors_match_the_oracle_agent_by_agent(k, real):
    rng = np.random.default_rng(14000 + 2 * k + real)
    selectors = [0, 1]
    targets = [int(x) for x in rng.choice(3, 2, replace=False)]
    c = dict(SEL_CASES[k], selector=int(rng.integers(0, 2)), target=int(rng.integers(0, 3)), real=real)   # engine-wide, overridden per set
    n_ep, eval_at = int(rng.integers(3, 7)), int(rng.integers(2, 4))
    n_agents, first = int(rng.integers(40, 71)), int(rng.integers(0, 2 ** 40))
    base = P.hyper(n_ep, map_id=int(rng.integers(0, 2)), slippery=bool(rng.integers(0, 2)), max_steps=int(rng.choice([17, 64, 100])),
                   decay_kind=int(rng.integers(0, 2)), seed=int(rng.integers(0, 2 ** 63)))
    sets = [dict(base, **draw_set(rng, base["decay_kind"], n_ep)) for _ in range(2)]
    group = np.arange(n_agents, dtype=np.uint32) % 2          # neighbouring lanes hold different selectors
    per_agent = [dict(c, selector=selectors[group[i]], target=targets[group[i]]) for i in range(n_agents)]
    oracle = [O.batch_train(P.oracle_config(per_agent[i], sets[group[i]]), first + i, 1, n_ep, eval_at, n_threads=1) for i in range(n_agents)]
    ran = set()
    for store in ((1, 2, 3) if c["env"] in (1, 2) else (1,)) + ((4,) if c["agent"] == 1 else ()):
        try:
            eng = P.make_engine(c, base, n_agents, first, store_kind=store)
        except abi.RlbError as exc:
            if store != 1 and exc.status == abi.ERR_UNSUPPORTED:   # the engine's own selector does not fit that store
                continue
            raise
        with eng:
            eng.set_hparams([as_set(s) for s in sets], group)
            eng.set_targets(np.asarray(targets, np.int32))
            try:
                eng.set_selectors(np.asarray(selectors, np.int32))
            except abi.RlbError as exc:
                # the store cannot run one of the selectors: refused, the engine untouched
                assert store in (2, 3) and exc.status == abi.ERR_UNSUPPORTED, (store, exc)
                assert eng.selectors is None
                with P.make_engine(c, base, n_agents, first, store_kind=store) as ref:
                    ref.set_hparams([as_set(s) for s in sets], group)
                    ref.set_targets(np.asarray(targets, np.int32))
                    same_run(eng, ref, 0, 2, eval_at)
                continue
            store_ran = eng.store_kind()
            res = eng.train(n_ep, eval_at, sums=True, episodes=True)
            q, counts = eng.download_tables()
            st = eng.states()
        eps = res["episodes"]
        g = dict(ret=eps["ret"].T.astype(np.float64), len=eps["length"].T.astype(np.uint64), tdsum=eps["td_sum"].T.astype(np.float64),
                 tdabs=eps["td_abs_sum"].T.astype(np.float64), q=q.astype(np.float64), counts=counts.astype(np.uint64), state=st,
                 train_steps=res["train_steps"], eval_steps=res["eval_steps"])
        ran.add(store_ran)
        for i in range(n_agents):
            o = oracle[i]
            P.compare(agent_slice(g, i), dict(o, train_steps=res["train_steps"], eval_steps=res["eval_steps"]), per_agent[i])
            if selectors[group[i]] == 0:
                assert not counts[i].any()                       # an eps-greedy agent's counts are zero
        assert res["train_steps"] == sum(o["train_steps"] for o in oracle)
        assert res["eval_steps"] == sum(o["eval_steps"] for o in oracle)
    assert 1 in ran
    if c["env"] == 3 and c["agent"] == 1:
        assert 4 in ran                                          # Taxi traces: the lazy store ran
    if c["env"] == 1 and c["agent"] == 1:
        try:                                                     # does the UCB variant fit the hybrid store?
            with P.make_engine(dict(c, selector=1), base, n_agents, first, store_kind=3) as probe:
                fits = probe.store_kind() == 3
        except abi.RlbError as exc:
            assert exc.status == abi.ERR_UNSUPPORTED
            fits = False
        assert (3 in ran) == fits


def uniform_twins(c, h, group, sets, selectors, first=0, store_kind=0, mask=None):
    """Two engines with the same sets and groups, every set on eps-greedy in one and on UCB in the other: agent i of the
    engine with per-set selectors must equal agent i of the twin of its set's selector."""
    out = []
    for k in (0, 1):
        e = engine_with_selectors(c, h, group, sets, [k] * len(sets), first, store_kind)
        if mask is not None:
            e.set_active_sets(mask)
        out.append(e)
    return out


def check_against_twins(sums, eps, q, counts, st, twin_res, selectors, group, tag):
    for g, k in enumerate(selectors):
        tr = twin_res[k]
        assert P.bits_equal(sums[:, g], tr["sums"][:, g]), (tag, g, P.first_diff(sums[:, g], tr["sums"][:, g]))
        mine = group == g
        assert fields_equal(eps[:, mine], tr["episodes"][:, mine]), (tag, g)
        assert P.bits_equal(q[mine], tr["q"][mine]), (tag, g)
        assert np.array_equal(counts[mine], tr["counts"][mine] if k == 1 else np.zeros_like(counts[mine])), (tag, g)
        assert fields_equal(st[mine], tr["state"][mine]), (tag, g)


def train_path(eng, path, n_ep, eval_at):
    if path == "blocking":
        r = eng.train(n_ep, eval_at, sums=True, episodes=True)
        return r["sums"], r["episodes"], r["train_steps"]
    if path == "chunked":
        parts = [eng.train(e, eval_at, ep_begin=b, sums=True, episodes=True) for b, e in ((0, 6), (6, 13), (13, n_ep))]
    elif path == "async":
        eng.train(9, eval_at, sums=True, episodes=True, wait=False)
        eng.train(n_ep, eval_at, ep_begin=9, sums=True, episodes=True, wait=False)
        parts = eng.train_wait()
    else:   # the record pipeline: the host buffer is filled chunk by chunk while the next chunk runs
        out = np.zeros((n_ep, eng.N), eng.episode_dtype)
        r = eng.train(n_ep, eval_at, sums=True, episodes_out=out)
        return r["sums"], out, r["train_steps"]
    return (np.concatenate([p["sums"] for p in parts]), np.concatenate([p["episodes"] for p in parts]),
            sum(p["train_steps"] for p in parts))


def finish(eng, r):
    q, counts = eng.download_tables()
    return dict(sums=r[0], episodes=r[1], steps=r[2], q=q, counts=counts, state=eng.states())


@pytest.mark.parametrize("layout", ["contiguous", "interleaved"])
@pytest.mark.parametrize("path", ["blocking", "chunked", "async", "pipelined"])
@pytest.mark.parametrize("wl", ["c2", "c4"])
def test_one_engine_equals_one_engine_per_selector(wl, path, layout):
    w = P._W.WORKLOADS[wl]
    c, h = P._W.combo(w, 0), P._W.workload_hyper(w)
    per, n_ep, eval_at = 300, 20, 7                             # 300: the UCB launch does not start on a warp boundary
    group = np.repeat(np.arange(3, dtype=np.uint32), per) if layout == "contiguous" else (np.arange(3 * per) % 3).astype(np.uint32)
    sets = [dict(h, **s) for s in SEP_SETS]
    with engine_with_selectors(c, h, group, sets, SEP_SEL) as eng:
        if wl == "c2":
            assert eng.store_kind() == 3                         # the hybrid store: two launches share its scratch
        got = finish(eng, train_path(eng, path, n_ep, eval_at))
    twins = uniform_twins(c, h, group, sets, SEP_SEL)
    try:
        twin_res = [finish(t, train_path(t, "blocking", n_ep, eval_at)) for t in twins]
    finally:
        for t in twins:
            t.close()
    assert got["steps"] == sum(int(twin_res[k]["episodes"]["length"][:, group == g].sum()) for g, k in enumerate(SEP_SEL))
    check_against_twins(got["sums"], got["episodes"], got["q"], got["counts"], got["state"], twin_res, SEP_SEL, group, (wl, path, layout))


@pytest.mark.parametrize("mask", [[True, False, True], [False, True, True], [False, True, False], [True, False, False], [False] * 3],
                         ids=lambda m: "".join("1" if x else "0" for x in m))
def test_masks(mask):
    w = P._W.WORKLOADS["c2"]
    c, h = P._W.combo(w, 0), P._W.workload_hyper(w)
    sets = [dict(h, **s) for s in SEP_SETS] + [dict(h, **SEP_SETS[0])]
    selectors = SEP_SEL + [abi.SEL_EPS_GREEDY]                 # [ucb, eps, ucb, eps]; mask[3] = True always
    mask = list(mask) + [mask != [False] * 3]
    group = (np.arange(4 * 200) % 4).astype(np.uint32)
    with engine_with_selectors(c, h, group, sets, selectors) as eng:
        eng.set_active_sets(mask)
        got = finish(eng, train_path(eng, "blocking", 12, 5))
        ev = eng.evaluate(6, sums=True, episodes=True)
    twins = uniform_twins(c, h, group, sets, selectors, mask=mask)
    try:
        twin_res = [finish(t, train_path(t, "blocking", 12, 5)) for t in twins]
        twin_ev = [t.evaluate(6, sums=True, episodes=True) for t in twins]
    finally:
        for t in twins:
            t.close()
    check_against_twins(got["sums"], got["episodes"], got["q"], got["counts"], got["state"], twin_res, selectors, group, mask)
    for g, k in enumerate(selectors):
        assert P.bits_equal(ev["sums"][:, g], twin_ev[k]["sums"][:, g]), (mask, g)
    if not any(mask):
        assert got["steps"] == 0 and not got["sums"].any()


def test_step_level_calls_and_resets():
    c = dict(env=2, agent=0, selector=0, policy=1, target=2, real=1)
    h = P.hyper(50)
    sets = [dict(h, **s) for s in SEP_SETS]
    group = (np.arange(48) % 3).astype(np.uint32)
    rng = np.random.default_rng(31)
    eng = engine_with_selectors(c, h, group, sets, SEP_SEL)
    twins = uniform_twins(c, h, group, sets, SEP_SEL)
    which = np.array([SEP_SEL[g] for g in group])               # agent -> the twin that holds its selector

    def pick(outs):
        return np.where(which.reshape((-1,) + (1,) * (np.asarray(outs[0]).ndim - 1)) == 1, outs[1], outs[0])

    try:
        n = len(group)
        for it in range(30):
            s = rng.integers(0, 37, n).astype(np.uint32)
            a = rng.integers(0, 4, n).astype(np.uint32)
            s2 = rng.integers(0, 48, n).astype(np.uint32)
            r = rng.choice([-1.0, -100.0], n)
            term = (rng.random(n) < 0.2).astype(np.uint8)
            a2 = eng.get_action(s2)
            assert np.array_equal(a2, pick([t.get_action(s2) for t in twins])), it
            td = eng.update(s, a, r, term, s2, a2)
            assert P.bits_equal(td, pick([t.update(s, a, r, term, s2, a2) for t in twins])), it
            vals = rng.standard_normal((n, 4))
            assert np.array_equal(eng.selector_get_action(s, vals), pick([t.selector_get_action(s, vals) for t in twins])), it
            pr = eng.selector_get_exploration_probs(s, vals)
            assert P.bits_equal(pr, pick([t.selector_get_exploration_probs(s, vals) for t in twins])), it
            eng.selector_update()
            for t in twins:
                t.selector_update()
        for it in range(40):
            got = eng.agent_step()
            want = [t.agent_step() for t in twins]
            for key in ("kind", "obs", "action", "reward", "terminated", "td"):
                assert P.bits_equal(np.asarray(got[key]).astype(np.float64), pick([np.asarray(x[key]).astype(np.float64) for x in want])), (it, key)
        for name, act in (("selector_reset", lambda e: e.selector_reset()), ("agent_reset", lambda e: e.agent_reset())):
            eng.train(3, 2)
            for t in twins:
                t.train(3, 2)
            act(eng)
            for t in twins:
                act(t)
            st, tw = eng.states(), [t.states() for t in twins]
            for g, k in enumerate(SEP_SEL):
                assert fields_equal(st[group == g], tw[k][group == g]), (name, g)
        q, counts = eng.download_tables()
        tq = [t.download_tables() for t in twins]
        for g, k in enumerate(SEP_SEL):
            mine = group == g
            assert P.bits_equal(q[mine], tq[k][0][mine]) and np.array_equal(counts[mine], tq[k][1][mine] if k else 0 * counts[mine]), g
    finally:
        eng.close()
        for t in twins:
            t.close()


def copy_with_selectors(a, c, h, selectors):
    """An engine B with a's config and sets, given `selectors` from the start and then a's tables and states."""
    sets, group = a.hparams
    b = P.make_engine(dict(c, agent=int(a.cfg.agent_kind)), h, len(group))
    b.set_hparams(sets, group)
    b.set_selectors(np.asarray(selectors, np.int32))
    q, counts = a.download_tables()
    b.upload_tables(q, counts)
    b.set_states(a.states())
    return b


@pytest.mark.parametrize("c", [dict(env=3, agent=0, selector=0, policy=0, target=1, real=0),
                               dict(env=2, agent=1, selector=1, policy=1, target=0, real=1)], ids=P.combo_id)
def test_changing_selectors_and_lifecycle(c):
    h = P.hyper(40)
    sets = [dict(h, **s) for s in SEP_SETS]
    group = (np.arange(96) % 3).astype(np.uint32)
    with engine_with_selectors(c, h, group, sets, SEP_SEL) as a:
        a.train(10, 5)
        q0, c0 = a.download_tables()
        st0 = a.states()
        new = [abi.SEL_UCB, abi.SEL_UCB, abi.SEL_EPS_GREEDY]          # set 0 unchanged, 1: eps -> UCB, 2: UCB -> eps
        a.set_selectors(np.asarray(new, np.int32))
        q1, c1 = a.download_tables()
        st1 = a.states()
        assert P.bits_equal(q0, q1)
        same = group == 0
        assert fields_equal(st1[same], st0[same]) and np.array_equal(c1[same], c0[same])   # unchanged: its selector state kept
        for g in (1, 2):
            m = group == g
            assert (st1["epsilon"][m] == sets[g]["eps0"]).all() and (st1["ucb_t"][m] == 1).all() and not c1[m].any(), g
        a.set_selectors(np.asarray(new, np.int32))                      # the same array again: nothing
        assert fields_equal(a.states(), st1) and np.array_equal(a.download_tables()[1], c1)
        with copy_with_selectors(a, c, h, new) as b:
            same_run(a, b, 10, 16, 5)
        ep = 16
        for name, act in (("retune", lambda e: e.retune_hparams([as_set(dict(s, lr=s["lr"] * 1.2)) for s in sets])),
                          ("mask", lambda e: e.set_active_sets([True, False, True])),
                          ("unmask", lambda e: e.set_active_sets(None)),
                          ("targets", lambda e: e.set_targets(np.array([2, 0, 1], np.int32))),
                          ("agent_reset", lambda e: e.agent_reset()),
                          ("selector_reset", lambda e: e.selector_reset()),
                          ("set_kind", lambda e: e.set_agent_kind(1 - int(c["agent"])))):
            act(a)
            assert list(a.selectors) == new, name                          # kept
            with copy_with_selectors(a, c, h, new) as b:
                if a.targets is not None:
                    b.set_targets(a.targets)
                if name == "mask":
                    b.set_active_sets([True, False, True])
                same_run(a, b, ep, ep + 3, 5)
            ep += 3
        # a clone across the selectors: set 1 (UCB) -> set 2 (eps-greedy) and set 2 -> set 0 (UCB); destinations keep
        # their set's selector, the counts reach only the UCB ones
        src, dst = np.concatenate([np.arange(1, 96, 3)[:16], np.arange(2, 96, 3)[16:]]), np.concatenate([np.arange(2, 96, 3)[:16], np.arange(0, 96, 3)[16:]])
        q, counts = a.download_tables()
        st = a.states()
        a.clone_agents(src, dst)
        q[dst] = q[src]
        counts[dst] = np.where((group[dst] == 2)[:, None, None], 0, counts[src])
        for f in ("epsilon", "ucb_t", "policy_flag"):
            st[f][dst] = st[f][src]
        qa, ca = a.download_tables()
        assert P.bits_equal(qa, q) and np.array_equal(ca, counts) and fields_equal(a.states(), st)
        with copy_with_selectors(a, c, h, new) as b:
            b.set_targets(a.targets)
            same_run(a, b, ep, ep + 5, 5)
        a.set_selector(abi.SEL_EPS_GREEDY)                                 # every set on one selector, fresh
        assert a.selectors is None and not a.download_tables()[1].any()
        a.set_selectors(np.asarray(new, np.int32))
        a.set_hparams(*a.hparams)                                          # back to the engine-wide selector
        assert a.selectors is None and not a.download_tables()[1].any()


@pytest.mark.parametrize("k", range(len(CELLS)), ids=lambda v: P.combo_id(dict(CELLS[v][0], real=0)))
def test_selectors_with_planning_counts_match_the_oracle(k):
    rng = np.random.default_rng(15000 + k)
    c = dict(CELLS[k][0], real=int(rng.integers(0, 2)))
    n_ep, eval_at = int(rng.integers(3, 6)), 100
    n_agents, first = int(rng.integers(24, 41)), int(rng.integers(0, 2 ** 40))
    base = P.hyper(n_ep, max_steps=int(rng.choice([40, 100])), decay_kind=int(rng.integers(0, 2)), seed=int(rng.integers(0, 2 ** 63)))
    sets = [dict(base, **draw_set(rng, base["decay_kind"], n_ep)) for _ in range(3)]
    selectors = [1 - int(c["selector"]), int(c["selector"]), 1 - int(c["selector"])]
    steps = [int(x) for x in rng.permutation([0, 2, 5])]
    group = np.arange(n_agents, dtype=np.uint32) % 3
    with engine_with_selectors(c, base, group, sets, selectors, first) as eng:
        eng.set_planning_steps(np.asarray(steps, np.uint32))
        assert list(eng.selectors) == selectors
        res = eng.train(n_ep, eval_at, sums=True, episodes=True)
        q, counts = eng.download_tables()
        st = eng.states()
    eps = res["episodes"]
    g = dict(ret=eps["ret"].T.astype(np.float64), len=eps["length"].T.astype(np.uint64), tdsum=eps["td_sum"].T.astype(np.float64),
             tdabs=eps["td_abs_sum"].T.astype(np.float64), q=q.astype(np.float64), counts=counts.astype(np.uint64), state=st)
    for i in range(n_agents):
        ci = dict(c, selector=selectors[group[i]])
        o = O.batch_train(P.oracle_config(ci, dict(sets[group[i]], planning_steps=steps[group[i]])), first + i, 1, n_ep, eval_at, n_threads=1)
        P.compare(dict(agent_slice(g, i), train_steps=o["train_steps"], eval_steps=o["eval_steps"]), o, ci)


def test_errors_leave_the_engine_untouched():
    c = dict(env=3, agent=0, selector=0, policy=0, target=1, real=0)
    h = P.hyper(10)
    with P.make_engine(c, h, 60) as eng:
        s = np.array([1, 0], np.int32)
        assert abi.lib.rlb_engine_set_selectors(eng.h, abi.ptr(s), 2) == abi.ERR_INVALID_ARG           # no sets
        eng.set_hparams([as_set(dict(h, **x)) for x in SEP_SETS[:2]], (np.arange(60) % 2).astype(np.uint32))
        eng.set_selectors(s)
        eng.train(4, 2)
        before = (eng.download_tables(), eng.states())
        for bad, n in ((s, 3), (s, 1), (None, 2), (s, 0), (None, 0), (np.array([0, 2], np.int32), 2),
                       (np.array([-1, 1], np.int32), 2), (np.array([1, 7], np.int32), 2)):
            assert abi.lib.rlb_engine_set_selectors(eng.h, abi.ptr(bad), n) == abi.ERR_INVALID_ARG, (bad, n)
        for bad in (np.array([0, 2]), np.array([0, 1, 1]), np.array([0.0, 1.0])):
            with pytest.raises(ValueError):
                eng.set_selectors(bad)
        after = (eng.download_tables(), eng.states())
        assert P.bits_equal(after[0][0], before[0][0]) and np.array_equal(after[0][1], before[0][1]) and fields_equal(after[1], before[1])
        assert list(eng.selectors) == [1, 0]
        with copy_with_selectors(eng, c, h, [1, 0]) as b:                         # the selectors in force are still [1, 0]
            same_run(eng, b, 4, 10, 2)


def test_snapshot_with_selectors_resumes_bit_identically(tmp_path):
    c = dict(env=2, agent=0, selector=0, policy=0, target=1, real=1)
    h = P.hyper(30)
    sets = [dict(h, **s) for s in SEP_SETS]
    group = (np.arange(90) % 3).astype(np.uint32)
    path = str(tmp_path / "snap.npz")
    with engine_with_selectors(c, h, group, sets, SEP_SEL, targets=[2, 0, 1]) as a:
        a.train(10, 5)
        a.set_active_sets([True, False, True])
        snapshot.save_snapshot(a, path)
        assert list(np.load(path)["hp_selector"]) == SEP_SEL
        with P.make_engine(c, h, 90) as b:
            snapshot.load_snapshot(b, path)
            assert list(b.selectors) == SEP_SEL and list(b.targets) == [2, 0, 1] and list(b.active_sets) == [True, False, True]
            same_run(a, b, 10, 20, 5)
            assert np.array_equal(a.download_tables()[1], b.download_tables()[1])


def sweep_kw(**kw):
    return dict(dict(agents_per_point=128, n_episodes=40, real="f32", verbose=False), **kw)


def test_sweep_with_a_selector_axis_equals_one_sweep_per_selector():
    grid = {"selector": ["eps", "ucb"], "learning_rate": [0.1, 0.5], "confidence_level": [0.5, 2.0]}
    res = driver.run_sweep("taxi", grid, **sweep_kw())
    assert res["selector"] is None and [p["params"]["selector"] for p in res["points"]] == ["eps"] * 4 + ["ucb"] * 4
    per = res["agents_per_point"]
    sub = {"learning_rate": [0.1, 0.5], "confidence_level": [0.5, 2.0]}
    for si, name in enumerate(grid["selector"]):
        one = driver.run_sweep("taxi", sub, selector=name, **sweep_kw())
        for j, pt in enumerate(one["points"]):
            g = 4 * si + j
            env = driver.make_env("taxi", **dict(driver.DEFAULTS, n_episodes=40))
            # the same point alone, with the agent ids it has in the grid (first_agent_id shifts by the points before)
            with abi.Engine(env.kind, n_agents=per, selector=driver.SELECTOR_NAMES[name], target=abi.TARGET_QLEARNING, real=abi.REAL_F32,
                            decay_kind=abi.DECAY_SUB, first_agent_id=g * per, **pt["hparams"], **env._cfg()) as eng:
                r = eng.train(40, 4, sums=True)
                ev = eng.evaluate(40, sums=True)["sums"]
            window = max(1, 40 // driver.DEFAULTS["moving_average_window"])
            assert res["points"][g]["train_rewards"] == driver.moving_average(window, r["sums"][:, 1] / per), (name, j)
            assert res["points"][g]["eval_mean_return"] == float(ev[:, 1].sum()) / (per * 40), (name, j)
            if si == 0:
                for key in ("train_rewards", "train_episodes_length", "test_rewards", "test_episodes_length", "eval_mean_return"):
                    assert res["points"][g][key] == pt[key], (name, j, key)


def test_pbt_and_halving_with_a_selector_axis():
    grid = {"selector": ["eps", "ucb"], "target": ["sarsa", "qlearning"], "learning_rate": [0.1, 0.5]}
    kw = sweep_kw(agents_per_point=64, n_episodes=60)
    a = driver.run_pbt("cliffwalking", grid, interval=20, fraction=0.25, pbt_seed=5, resample_probability=0.5, **kw)
    b = driver.run_pbt("cliffwalking", grid, interval=20, fraction=0.25, pbt_seed=5, resample_probability=0.5, **kw)
    a.pop("seconds"), b.pop("seconds")
    assert json.dumps(a) == json.dumps(b) and a["selector"] is None
    moved = [p["flags"]["selector"] for step in a["lineage"] for p in step["pairs"]]
    assert moved and all(s in driver.SELECTOR_NAMES for s in moved)
    hv = driver.run_halving("cliffwalking", grid, min_episodes=10, eta=3, **kw)
    sw = driver.run_sweep("cliffwalking", grid, **kw)
    survivors = hv["rungs"][-1]["active"]
    assert survivors
    for g in survivors:                                                        # a survivor is its sweep point, bit for bit
        for key in ("train_rewards", "test_rewards", "test_episodes_length", "eval_mean_return"):
            assert hv["points"][g][key] == sw["points"][g][key], (g, key)
