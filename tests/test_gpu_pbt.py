"""Population-based training on the GPU: rlb_agent_clone against the host round trip it stands for (download, copy the
fields from src[j] to dst[j], upload), rlb_engine_retune_hparams against an engine built with the new sets and given the
same learned state, their error cases, snapshots after a retune, and driver.run_pbt end to end.  Every comparison is
bit for bit."""
import importlib
import json

import numpy as np
import pytest

import parity as P

pytestmark = pytest.mark.gpu

abi = importlib.import_module("rl-rust_b200._abi")
snapshot = importlib.import_module("rl-rust_b200.snapshot")
driver = importlib.import_module("rl-rust_b200.driver")

N = 64


def raw_equal(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


def random_pairs(rng, n, n_pairs=20, n_sources=6):
    """Destinations distinct and disjoint from the sources; sources repeated."""
    perm = rng.permutation(n)
    pool, dst = perm[:n_sources], perm[n_sources:n_sources + n_pairs]
    return rng.choice(pool, n_pairs).astype(np.uint32), dst.astype(np.uint32)


def round_trip_clone(eng, src, dst, ucb, model):
    """What rlb_agent_clone stands for: the snapshot downloads, a copy of the learned fields on the host, the uploads."""
    q, counts = eng.download_tables()
    st = eng.states()
    q[dst] = q[src]
    counts[dst] = counts[src]
    for f in ("epsilon", "ucb_t", "policy_flag"):
        st[f][dst] = st[f][src]
    eng.upload_tables(q, counts if ucb else None)
    eng.set_states(st)
    if model:
        ln, ent = eng.download_model()
        ln[dst] = ln[src]
        ent[dst] = ent[src]
        eng.upload_model(ln, ent)


def learned_state(eng, model=False):
    q, counts = eng.download_tables()
    st = eng.states()
    out = dict(q=q, counts=counts, state=st)
    if model:
        out["model_len"], out["model"] = eng.download_model()
    return out


def assert_same_state(a, b, tag):
    for k in a:
        assert raw_equal(a[k], b[k]), (tag, k)


def continue_both(a, b, k, m, tag, model=False):
    """Train m more episodes and evaluate on both engines; records, sums, tables and states must be equal."""
    ra = a.train(k + m, 3, ep_begin=k, episodes=True)
    rb = b.train(k + m, 3, ep_begin=k, episodes=True)
    for key in ("sums", "episodes"):
        assert raw_equal(ra[key], rb[key]), (tag, "train", key)
    for key in ("train_steps", "eval_steps", "eval_return_sum"):
        assert ra[key] == rb[key], (tag, key)
    ea, eb = a.evaluate(5, episodes=True), b.evaluate(5, episodes=True)
    for key in ("sums", "episodes"):
        assert raw_equal(ea[key], eb[key]), (tag, "evaluate", key)
    assert_same_state(learned_state(a, model), learned_state(b, model), tag)


def interleaved_sets(rng, n):
    sets = [dict(learning_rate=float(rng.choice([0.05, 0.3, 0.9])), discount_factor=float(rng.choice([0.9, 0.99, 0.5])),
                 lambda_factor=float(rng.choice([0.3, 0.8])), initial_epsilon=float(rng.choice([1.0, 0.4])),
                 epsilon_decay=float(rng.choice([0.01, 0.1])), final_epsilon=float(rng.choice([0.0, 0.05])),
                 confidence_level=float(rng.choice([0.5, 2.0])), default_value=float(rng.choice([0.0, -1.0, 2.5])))
            for _ in range(3)]
    return sets, np.arange(n, dtype=np.uint32) % 3


CASES = [dict(env=env, agent=agent, selector=sel, policy=pol) for env in range(4) for agent in (0, 1) for sel in (0, 1) for pol in (0, 1)]


@pytest.mark.parametrize("with_sets", [False, True], ids=["config", "sets"])
@pytest.mark.parametrize("k", range(len(CASES)), ids=["%s-%s-%s-%s" % (P.ENV_NAMES[c["env"]], "traces" if c["agent"] else "onestep",
                                                                     "ucb" if c["selector"] else "eps", "double" if c["policy"] else "basic") for c in CASES])
def test_clone_equals_the_host_round_trip(k, with_sets):
    rng = np.random.default_rng(9100 + 2 * k + with_sets)
    reals = (0, 1) if k % 4 == 0 else (0,)
    ran = 0
    for real in reals:
        c = dict(CASES[k], target=int(rng.integers(0, 3)), real=real)
        h = P.hyper(12, max_steps=int(rng.choice([30, 100])), seed=int(rng.integers(0, 2 ** 63)))
        sets, group = interleaved_sets(rng, N)
        for store in ((1, 2, 3) if c["env"] in (1, 2) else (1,)) + ((4,) if c["agent"] == 1 else ()):
            try:
                a = P.make_engine(c, h, N, 1000, store_kind=store)
            except abi.RlbError as exc:
                if store != 1 and exc.status == abi.ERR_UNSUPPORTED:   # this configuration does not fit that store
                    continue
                raise
            b = P.make_engine(c, h, N, 1000, store_kind=store)
            tag = (P.combo_id(c), store, with_sets)
            if with_sets:
                a.set_hparams(sets, group)
                b.set_hparams(sets, group)
            a.train(4, 3, sums=False)
            b.train(4, 3, sums=False)
            src, dst = random_pairs(rng, N)
            a.clone_agents(src, dst)
            round_trip_clone(b, src, dst, c["selector"] == 1, False)
            sa = learned_state(a)
            assert_same_state(sa, learned_state(b), tag)
            assert raw_equal(sa["q"][dst], sa["q"][src]), tag          # and the clone did copy
            continue_both(a, b, 4, 5, tag)
            a.close()
            b.close()
            ran += 1
    assert ran >= 1


def test_clone_with_a_dyna_model_equals_the_round_trip():
    c = dict(env=2, agent=0, selector=0, policy=0, target=1, real=0)
    h = P.hyper(20, planning_steps=5)
    rng = np.random.default_rng(17)
    a, b = P.make_engine(c, h, N), P.make_engine(c, h, N)
    a.train(6, 3, sums=False)
    b.train(6, 3, sums=False)
    src, dst = random_pairs(rng, N)
    a.clone_agents(src, dst)
    round_trip_clone(b, src, dst, False, True)
    sa = learned_state(a, True)
    assert_same_state(sa, learned_state(b, True), "dyna")
    assert sa["model_len"][dst].any()
    continue_both(a, b, 6, 6, "dyna", model=True)
    a.close()
    b.close()
    with P.make_engine(dict(c, agent=1), h, N) as t:                   # a trace agent under a model
        src, dst = np.array([1], np.uint32), np.array([2], np.uint32)
        assert abi.lib.rlb_agent_clone(t.h, abi.ptr(src), abi.ptr(dst), 1) == abi.ERR_UNSUPPORTED


RETUNE_CASES = [(dict(env=3, agent=0, selector=0, policy=0, target=1), 0),
                (dict(env=1, agent=1, selector=0, policy=0, target=0), 3),
                (dict(env=2, agent=0, selector=1, policy=1, target=2), 0),
                (dict(env=3, agent=1, selector=1, policy=0, target=1), 4),
                (dict(env=0, agent=1, selector=0, policy=1, target=0), 0)]


@pytest.mark.parametrize("real", [0, 1], ids=["f32", "f64"])
@pytest.mark.parametrize("i", range(len(RETUNE_CASES)))
def test_retune_equals_an_engine_built_with_the_new_sets(i, real):
    c, store = dict(RETUNE_CASES[i][0], real=real), RETUNE_CASES[i][1]
    rng = np.random.default_rng(300 + i)
    h = P.hyper(12)
    sets, group = interleaved_sets(rng, N)
    new, _ = interleaved_sets(rng, N)
    a = P.make_engine(c, h, N, 77, store_kind=store)
    a.set_hparams(sets, group)
    a.train(5, 3, sums=False)
    a.retune_hparams(new)
    assert a.hparam_sets() == 3 and raw_equal(a.hparams[0], a.hparams_array(new))
    b = P.make_engine(c, h, N, 77, store_kind=store)
    b.set_hparams(new, group)
    s = learned_state(a)
    b.upload_tables(s["q"], s["counts"] if c["selector"] == 1 else None)
    b.set_states(s["state"])
    tag = (P.combo_id(c), store)
    continue_both(a, b, 5, 4, tag)
    a.agent_reset()                                                      # the new initial_epsilon and default_value
    b.agent_reset()
    sa = learned_state(a)
    assert_same_state(sa, learned_state(b), tag)
    for g, hs in enumerate(new):
        assert np.all(sa["q"][group == g] == a.rdtype(hs["default_value"])), (tag, g)
        if c["selector"] == 0:
            assert np.all(sa["state"]["epsilon"][group == g] == hs["initial_epsilon"]), (tag, g)
        else:                                                            # UCB: the reset clears counts and t instead
            assert not sa["counts"][group == g].any() and np.all(sa["state"]["ucb_t"][group == g] == 1), (tag, g)
    continue_both(a, b, 0, 6, tag)
    a.close()
    b.close()


def test_errors_leave_the_engine_untouched():
    w = P._W.WORKLOADS["c4"]
    c, h = P._W.combo(w, 0), P._W.workload_hyper(w)
    L = abi.lib
    with P.make_engine(c, h, 100) as eng:
        sets = eng.hparams_array([dict(default_value=3.0), dict(learning_rate=0.3)])
        eng.set_hparams(sets, np.arange(100) % 2)
        eng.train(4, 2, sums=False)
        before = learned_state(eng)

        def clone(src, dst, n=None):
            src = None if src is None else np.asarray(src, np.uint32)
            dst = None if dst is None else np.asarray(dst, np.uint32)
            return L.rlb_agent_clone(eng.h, abi.ptr(src), abi.ptr(dst), len(dst if dst is not None else src) if n is None else n)
        assert clone([100], [0]) == abi.ERR_INVALID_ARG                   # id >= N
        assert clone([0], [100]) == abi.ERR_INVALID_ARG
        assert clone([1, 2], [3, 3]) == abi.ERR_INVALID_ARG               # a destination twice
        assert clone([1, 2], [2, 4]) == abi.ERR_INVALID_ARG               # an id both a source and a destination
        assert clone([1, 5], [4, 1]) == abi.ERR_INVALID_ARG
        assert clone(None, [3, 4]) == abi.ERR_INVALID_ARG                 # NULL pointers
        assert clone([3, 4], None) == abi.ERR_INVALID_ARG
        assert clone(None, None, 0) == abi.OK                             # n_pairs == 0: nothing to do
        three = np.zeros(3, abi.HPARAMS_DTYPE)
        assert L.rlb_engine_retune_hparams(eng.h, abi.ptr(three), 3) == abi.ERR_INVALID_ARG   # wrong count
        assert L.rlb_engine_retune_hparams(eng.h, abi.ptr(three), 1) == abi.ERR_INVALID_ARG
        assert L.rlb_engine_retune_hparams(eng.h, None, 2) == abi.ERR_INVALID_ARG             # NULL sets
        assert_same_state(learned_state(eng), before, "errors")
        assert eng.hparam_sets() == 2 and eng.train(6, 2, ep_begin=4)["sums"].shape == (2, 2, 4)
    with P.make_engine(c, h, 100) as eng:                                 # retune without sets
        before = learned_state(eng)
        assert L.rlb_engine_retune_hparams(eng.h, abi.ptr(np.zeros(1, abi.HPARAMS_DTYPE)), 1) == abi.ERR_INVALID_ARG
        assert_same_state(learned_state(eng), before, "no sets")


def test_clone_and_retune_take_device_buffers():
    import torch
    c = dict(env=1, agent=1, selector=1, policy=0, target=0, real=0)
    h = P.hyper(12)
    rng = np.random.default_rng(23)
    sets, group = interleaved_sets(rng, N)
    new, _ = interleaved_sets(rng, N)
    src, dst = random_pairs(rng, N)
    with P.make_engine(c, h, N) as a, P.make_engine(c, h, N) as b:
        for e in (a, b):
            e.set_hparams(sets, group)
            e.train(4, 3, sums=False)
        d_src = torch.from_numpy(src.astype(np.int32)).cuda()          # the same bits as u32 for ids < 2**31
        d_dst = torch.from_numpy(dst.astype(np.int32)).cuda()
        d_sets = torch.from_numpy(a.hparams_array(new).view(np.float64).copy()).cuda()
        torch.cuda.synchronize()
        bad = torch.from_numpy(np.array([N], np.int32)).cuda()
        before = learned_state(a)
        assert abi.lib.rlb_agent_clone(a.h, bad.data_ptr(), d_dst.data_ptr(), 1) == abi.ERR_INVALID_ARG
        assert_same_state(learned_state(a), before, "device ids, id >= N")
        abi.check(abi.lib.rlb_agent_clone(a.h, d_src.data_ptr(), d_dst.data_ptr(), len(src)))
        abi.check(abi.lib.rlb_engine_retune_hparams(a.h, d_sets.data_ptr(), 3))
        b.clone_agents(src, dst)
        b.retune_hparams(new)
        assert_same_state(learned_state(a), learned_state(b), "device buffers")
        continue_both(a, b, 4, 5, "device buffers")


def test_clone_while_an_asynchronous_train_call_is_pending():
    w = P._W.WORKLOADS["c4"]
    c, h = P._W.combo(w, 0), P._W.workload_hyper(w)
    src, dst = random_pairs(np.random.default_rng(5), 2048, n_pairs=600, n_sources=40)
    with P.make_engine(c, h, 2048) as a, P.make_engine(c, h, 2048) as b:
        a.train(8, 4, wait=False)
        a.clone_agents(src, dst)                                          # waits for the pending call first
        ra = a.train_wait()
        rb = b.train(8, 4)
        b.clone_agents(src, dst)
        assert len(ra) == 1 and raw_equal(ra[0]["sums"], rb["sums"])
        assert_same_state(learned_state(a), learned_state(b), "async")


def test_snapshot_after_a_retune_resumes_bit_identically(tmp_path):
    path = str(tmp_path / "snap.npz")
    w = P._W.WORKLOADS["c4"]
    c, h = P._W.combo(w, 0), P._W.workload_hyper(w)
    sets = [dict(learning_rate=0.05 * (g + 1), initial_epsilon=1.0 - 0.2 * g, epsilon_decay=0.02 * (g + 1)) for g in range(3)]
    new = [dict(learning_rate=0.3 - 0.05 * g, discount_factor=0.9, epsilon_decay=0.05, default_value=1.0 * g) for g in range(3)]
    group = np.arange(900, dtype=np.uint32) % 3
    eng = P.make_engine(c, h, 900)
    eng.set_hparams(sets, group)
    eng.train(10, 5, sums=False)
    eng.clone_agents(np.arange(0, 300, dtype=np.uint32), np.arange(600, 900, dtype=np.uint32))
    eng.retune_hparams(new)
    snapshot.save_snapshot(eng, path)
    want = eng.train(20, 5, ep_begin=10, episodes=True)
    q_want = eng.download_tables()[0]
    eng.close()
    assert raw_equal(np.load(path)["hp_sets"], eng.hparams_array(new))
    with P.make_engine(c, h, 900) as eng2:
        snapshot.load_snapshot(eng2, path)
        assert eng2.hparam_sets() == 3
        got = eng2.train(20, 5, ep_begin=10, episodes=True)
        assert raw_equal(got["sums"], want["sums"])
        assert raw_equal(got["episodes"], want["episodes"])
        assert raw_equal(eng2.download_tables()[0], q_want)


GRID = {"learning_rate": [0.05, 0.1, 0.2, 0.4], "exploration_time": [0.25, 0.5]}


def test_run_pbt_end_to_end():
    kw = dict(agents_per_point=32, n_episodes=200, real="f32", verbose=False)
    a = driver.run_pbt("taxi", GRID, interval=50, pbt_seed=3, **kw)
    b = driver.run_pbt("taxi", GRID, interval=50, pbt_seed=3, **kw)
    a.pop("seconds"), b.pop("seconds")
    assert json.dumps(a) == json.dumps(b)
    assert len(a["lineage"]) == 3 and all(len(s["pairs"]) == 2 for s in a["lineage"])
    # fraction 0: chunking the run changes nothing, the per-set curves are the sweep's
    z = driver.run_pbt("taxi", GRID, interval=50, fraction=0.0, **kw)
    s = driver.run_sweep("taxi", GRID, **kw)
    assert z["ranking"] == s["ranking"]
    for pz, ps in zip(z["points"], s["points"]):
        for key in ("train_rewards", "train_episodes_length", "test_rewards", "test_episodes_length", "eval_mean_return", "hparams"):
            assert pz[key] == ps[key], key
