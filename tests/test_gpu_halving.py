"""Successive halving on the GPU: rlb_engine_set_active_sets against the same engine with every set active (active agents
bit-equal, inactive agents untouched, their records, counts and sums rows zero), against an engine holding just the
active agents, pause and resume against an engine that made only the active calls, every call path under a mask, the
mask's lifecycle and error cases, snapshots, and driver.run_halving end to end against driver.run_sweep."""
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
G = 4


def raw_equal(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


def rand_sets(rng, n_sets=G):
    return [dict(learning_rate=float(rng.choice([0.05, 0.3, 0.9])), discount_factor=float(rng.choice([0.9, 0.99, 0.5])),
                 lambda_factor=float(rng.choice([0.3, 0.8])), initial_epsilon=float(rng.choice([1.0, 0.4])),
                 epsilon_decay=float(rng.choice([0.01, 0.1])), final_epsilon=float(rng.choice([0.0, 0.05])),
                 confidence_level=float(rng.choice([0.5, 2.0])), default_value=float(rng.choice([0.0, -1.0, 2.5])))
            for _ in range(n_sets)]


def groups(layout, n=N):
    return (np.repeat(np.arange(G), n // G) if layout == "contiguous" else np.arange(n) % G).astype(np.uint32)


def full_state(eng):
    q, counts = eng.download_tables()
    return dict(q=q, counts=counts, state=eng.states())


def agents_equal(a, b, ids, tag):
    for k in a:
        assert raw_equal(a[k][ids], b[k][ids]), (tag, k)


def check_call(ra, rb, mask, group, tag, records="episodes"):
    """ra: the masked engine's result, rb: the all-active engine's: active records and sums rows equal, the others 0."""
    act = mask[group]
    sa, sb = ra["sums"], rb["sums"]
    assert raw_equal(sa[:, mask], sb[:, mask]), (tag, "sums")
    assert not sa[:, ~mask].any() and not np.signbit(sa[:, ~mask]).any(), (tag, "inactive sums rows are +0.0")
    if records in ra and ra[records] is not None:
        ea, eb = ra[records], rb[records]
        assert raw_equal(ea[:, act], eb[:, act]), (tag, "records")
        assert not np.ascontiguousarray(ea[:, ~act]).view(np.uint8).any(), (tag, "inactive records are zero")


def stores_for(c):
    return ((1, 2, 3) if c["env"] in (1, 2) else (1,)) + ((4,) if c["agent"] == 1 else ())


def engines(c, h, store, n=N, first=500, count=2):
    try:
        return [P.make_engine(c, h, n, first, store_kind=store) for _ in range(count)]
    except abi.RlbError as exc:
        if store != 1 and exc.status == abi.ERR_UNSUPPORTED:   # this configuration does not fit that store
            return None
        raise


CASES = [dict(env=env, agent=agent, selector=sel, policy=pol) for env in range(4) for agent in (0, 1) for sel in (0, 1) for pol in (0, 1)]


@pytest.mark.parametrize("layout", ["contiguous", "interleaved"])
@pytest.mark.parametrize("k", range(len(CASES)), ids=["%s-%s-%s-%s" % (P.ENV_NAMES[c["env"]], "traces" if c["agent"] else "onestep",
                                                                     "ucb" if c["selector"] else "eps", "double" if c["policy"] else "basic") for c in CASES])
def test_a_subset_equals_the_same_engine_with_every_set_active(k, layout):
    rng = np.random.default_rng(7100 + 2 * k + (layout == "interleaved"))
    ran = 0
    for real in ((0, 1) if k % 4 == 0 else (0,)):
        c = dict(CASES[k], target=int(rng.integers(0, 3)), real=real)
        h = P.hyper(12, max_steps=int(rng.choice([30, 100])), seed=int(rng.integers(0, 2 ** 63)))
        sets, group = rand_sets(rng), groups(layout)
        mask = np.zeros(G, bool)
        mask[rng.choice(G, int(rng.integers(1, G)), replace=False)] = True    # a strict, non-empty subset
        act = mask[group]
        for store in stores_for(c):
            pair = engines(c, h, store)
            if pair is None:
                continue
            a, b = pair
            tag = (P.combo_id(c), store, layout, tuple(mask))
            for e in (a, b):
                e.set_hparams(sets, group)
                e.train(3, 3, sums=False)                                  # every set has learned something
            a.set_active_sets(mask)
            assert raw_equal(a.active_sets, mask)
            before = full_state(a)
            ra = a.train(9, 3, ep_begin=3, episodes=True)
            rb = b.train(9, 3, ep_begin=3, episodes=True)
            check_call(ra, rb, mask, group, tag)
            sa, sb = full_state(a), full_state(b)
            agents_equal(sa, sb, act, tag)
            agents_equal(sa, before, ~act, tag)                            # inactive agents untouched
            ea, eb = a.evaluate(4, episodes=True), b.evaluate(4, episodes=True)
            check_call(ea, eb, mask, group, tag)
            agents_equal(full_state(a), full_state(b), act, tag)
            agents_equal(full_state(a), before, ~act, tag)
            a.close()
            b.close()
            ran += 1
    assert ran >= 1


def test_totals_equal_an_engine_holding_just_the_active_agents():
    w = P._W.WORKLOADS["c4"]
    c, h = P._W.combo(w, 0), P._W.workload_hyper(w)
    rng = np.random.default_rng(41)
    sets, group = rand_sets(rng), groups("contiguous", 1024)
    mask = np.array([False, True, True, False])                            # agents 256 .. 767: one contiguous id range
    with P.make_engine(c, h, 1024, 100) as a, P.make_engine(c, h, 512, 100 + 256) as d:
        a.set_hparams(sets, group)
        a.set_active_sets(mask)
        d.set_hparams(sets[1:3], np.repeat(np.arange(2), 256))
        ra, rd = a.train(12, 4), d.train(12, 4)
        for key in ("train_steps", "eval_steps", "eval_return_sum", "eval_episodes"):
            assert ra[key] == rd[key], key
        assert ra["train_steps"] > 0 and raw_equal(ra["sums"][:, 1:3], rd["sums"])
        ea, ed = a.evaluate(6), d.evaluate(6)
        assert ea["steps"] == ed["steps"] and raw_equal(ea["sums"][:, 1:3], ed["sums"])
        sa, sd = full_state(a), full_state(d)
        for key in sa:
            assert raw_equal(sa[key][256:768], sd[key]), key


@pytest.mark.parametrize("case", [(dict(env=3, agent=0, selector=0, policy=0, target=1, real=0), 1, "contiguous"),
                                  (dict(env=1, agent=1, selector=0, policy=0, target=0, real=0), 3, "interleaved"),
                                  (dict(env=2, agent=1, selector=1, policy=1, target=2, real=1), 2, "contiguous"),
                                  (dict(env=3, agent=1, selector=0, policy=1, target=1, real=0), 4, "interleaved"),
                                  (dict(env=0, agent=1, selector=1, policy=0, target=0, real=0), 1, "interleaved")],
                         ids=["taxi-hbm", "frozen-hybrid", "cliff-groups-f64", "taxi-lazy", "blackjack-traces"])
def test_pause_and_resume_equals_an_engine_that_made_only_the_active_calls(case):
    c, store, layout = case
    h = P.hyper(12, max_steps=40)
    rng = np.random.default_rng(store * 13 + c["env"])
    sets, group = rand_sets(rng), groups(layout)
    mask = np.array([True, False, True, False])
    a, b, only = (P.make_engine(c, h, N, 9, store_kind=store) for _ in range(3))
    for e in (a, b, only):
        e.set_hparams(sets, group)
    # a: all, then sets 1 and 3 paused, then all again.  b: the three calls.  only: the first and the last call.
    ra = [a.train(4, 3, episodes=True)]
    a.set_active_sets(mask)
    ra.append(a.train(8, 3, ep_begin=4, episodes=True))
    a.set_active_sets(None)
    assert a.active_sets is None
    ra.append(a.train(12, 3, ep_begin=8, episodes=True))
    rb = [b.train(4, 3, episodes=True), b.train(8, 3, ep_begin=4, episodes=True), b.train(12, 3, ep_begin=8, episodes=True)]
    ro = [only.train(4, 3, episodes=True), None, only.train(12, 3, ep_begin=8, episodes=True)]
    act, paused = mask[group], ~mask[group]
    for r in (0, 2):
        assert raw_equal(ra[r]["sums"][:, mask], rb[r]["sums"][:, mask]), r
        assert raw_equal(ra[r]["episodes"][:, act], rb[r]["episodes"][:, act]), r
        assert raw_equal(ra[r]["sums"][:, ~mask], ro[r]["sums"][:, ~mask]), r
        assert raw_equal(ra[r]["episodes"][:, paused], ro[r]["episodes"][:, paused]), r
    check_call(ra[1], rb[1], mask, group, "paused call")
    sa = full_state(a)
    agents_equal(sa, full_state(b), act, "resumed, always active")
    agents_equal(sa, full_state(only), paused, "resumed, paused sets")
    ea, eb, eo = a.evaluate(3, episodes=True), b.evaluate(3, episodes=True), only.evaluate(3, episodes=True)
    assert raw_equal(ea["episodes"][:, act], eb["episodes"][:, act])
    assert raw_equal(ea["episodes"][:, paused], eo["episodes"][:, paused])
    for e in (a, b, only):
        e.close()


def masked_pair(n=N, c=None, store=0):
    c = c or dict(env=1, agent=1, selector=0, policy=0, target=1, real=0)
    h = P.hyper(40, max_steps=30)
    rng = np.random.default_rng(77)
    sets, group = rand_sets(rng), groups("interleaved", n)
    a, b = P.make_engine(c, h, n, 3, store_kind=store), P.make_engine(c, h, n, 3, store_kind=store)
    for e in (a, b):
        e.set_hparams(sets, group)
    mask = np.array([False, True, True, False])
    a.set_active_sets(mask)
    return a, b, mask, group, sets


def test_call_paths_under_a_mask():
    import torch
    a, b, mask, group, _ = masked_pair(n=256, store=3)
    act = mask[group]
    # blocking call with host records: the pipelined path (>= 8 episodes, four launches over the two scratch halves)
    ra, rb = a.train(16, 5, episodes=True), b.train(16, 5, episodes=True)
    assert ra["kernel_launches"] >= 4
    check_call(ra, rb, mask, group, "pipelined")
    # asynchronous calls, the second pipelined behind the first
    a.train(24, 5, ep_begin=16, episodes=True, wait=False)
    a.train(32, 5, ep_begin=24, episodes=True, wait=False)
    ra2 = a.train_wait()
    rb2 = [b.train(24, 5, ep_begin=16, episodes=True), b.train(32, 5, ep_begin=24, episodes=True)]
    assert len(ra2) == 2
    for x, y in zip(ra2, rb2):
        check_call(x, y, mask, group, "async")
    # one asynchronous call without records
    a.train(36, 5, ep_begin=32, wait=False)
    check_call(a.train_wait()[0], b.train(36, 5, ep_begin=32), mask, group, "async, sums only")
    # trajectory and TD taps
    ra = a.train(40, 5, ep_begin=36, traj_capacity=64, td_capacity=200)
    rb = b.train(40, 5, ep_begin=36, traj_capacity=64, td_capacity=200)
    check_call(ra, rb, mask, group, "taps")
    assert not ra["traj_count"][~act].any() and not ra["td_count"][~act].any()
    assert raw_equal(ra["traj_count"][act], rb["traj_count"][act]) and raw_equal(ra["td_count"][act], rb["td_count"][act])
    assert ra["td_count"][act].all()
    for i in np.flatnonzero(act):
        assert raw_equal(ra["traj"][i, :int(min(64, ra["traj_count"][i]))], rb["traj"][i, :int(min(64, rb["traj_count"][i]))])
        assert raw_equal(ra["td_steps"][i, :int(ra["td_count"][i])], rb["td_steps"][i, :int(rb["td_count"][i])])
    # device buffers: the caller's records are zero for the inactive agents
    rec_a = torch.full((4, 256 * a.episode_dtype.itemsize), 0x5A, dtype=torch.uint8, device="cuda")
    sums_a = torch.full((4, G, 4), 7.0, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    a.train(44, 5, ep_begin=40, episodes_out=rec_a, sums_out=sums_a)
    rb = b.train(44, 5, ep_begin=40, episodes=True)
    got = dict(episodes=rec_a.cpu().numpy().view(a.episode_dtype).reshape(4, 256), sums=sums_a.cpu().numpy())
    check_call(got, rb, mask, group, "device buffers")
    # evaluate with host and device outputs
    ea, eb = a.evaluate(5, episodes=True), b.evaluate(5, episodes=True)
    check_call(ea, eb, mask, group, "evaluate")
    agents_equal(full_state(a), full_state(b), act, "after the calls")
    a.close()
    b.close()


def test_lifecycle_clone_and_step_level_calls():
    a, b, mask, group, sets = masked_pair()
    act = mask[group]
    a.train(4, 2, sums=False)
    b.set_active_sets(mask)
    b.train(4, 2, sums=False)
    # retune keeps the mask
    new = rand_sets(np.random.default_rng(5))
    a.retune_hparams(new)
    assert raw_equal(a.active_sets, mask)
    r = a.train(6, 2, ep_begin=4)
    assert not r["sums"][:, ~mask].any() and r["sums"][:, mask, 0].all()
    b.retune_hparams(new)
    b.train(6, 2, ep_begin=4)
    # clone into and out of paused sets: the mask does not touch clone
    ids = np.arange(N)
    paused_ids, active_ids = ids[~act], ids[act]
    src = np.concatenate([paused_ids[:4], active_ids[:4]]).astype(np.uint32)
    dst = np.concatenate([active_ids[-4:], paused_ids[-4:]]).astype(np.uint32)
    for e in (a, b):
        e.clone_agents(src, dst)
    sa = full_state(a)
    assert raw_equal(sa["q"][dst], sa["q"][src])
    agents_equal(sa, full_state(b), slice(None), "clone under a mask")
    ra, rb = a.train(9, 2, ep_begin=6, episodes=True), b.train(9, 2, ep_begin=6, episodes=True)
    assert raw_equal(ra["episodes"], rb["episodes"]) and raw_equal(ra["sums"], rb["sums"])
    # step-level calls still act on every agent
    b.set_active_sets(None)
    for e in (a, b):
        e.agent_reset()
    assert raw_equal(a.env_reset(), b.env_reset())
    for _ in range(5):
        sa_, sb_ = a.agent_step(), b.agent_step()
        for key in sa_:
            assert raw_equal(sa_[key], sb_[key]), key
    agents_equal(full_state(a), full_state(b), slice(None), "step-level calls")
    # set_hparams makes every set active again
    a.set_hparams(sets, group)
    assert a.active_sets is None
    r = a.train(2, 2)
    assert r["sums"][:, :, 0].all()
    a.close()
    b.close()


def test_errors_and_every_set_inactive():
    L = abi.lib
    w = P._W.WORKLOADS["c4"]
    c, h = P._W.combo(w, 0), P._W.workload_hyper(w)
    with P.make_engine(c, h, 100) as eng:
        assert L.rlb_engine_set_active_sets(eng.h, None, 0) == abi.ERR_INVALID_ARG            # no sets installed
        eng.set_hparams([dict(learning_rate=0.1), dict(learning_rate=0.4)], np.arange(100) % 2)
        eng.train(4, 2, sums=False)
        before = full_state(eng)
        m = np.array([1, 0], np.uint8)
        assert L.rlb_engine_set_active_sets(eng.h, abi.ptr(np.ones(3, np.uint8)), 3) == abi.ERR_INVALID_ARG   # wrong count
        assert L.rlb_engine_set_active_sets(eng.h, abi.ptr(m), 1) == abi.ERR_INVALID_ARG
        assert L.rlb_engine_set_active_sets(eng.h, abi.ptr(m), 0) == abi.ERR_INVALID_ARG      # non-NULL with 0
        assert L.rlb_engine_set_active_sets(eng.h, None, 2) == abi.ERR_INVALID_ARG            # NULL with 2
        r = eng.train(6, 2, ep_begin=4)
        assert r["sums"][:, :, 0].all()                                                      # the errors left every set active
        eng.set_active_sets([False, False])
        after = full_state(eng)
        r = eng.train(10, 2, ep_begin=6, episodes=True, td_capacity=8)
        assert r["train_steps"] == r["eval_steps"] == r["eval_episodes"] == 0 and r["eval_return_sum"] == 0.0
        assert r["kernel_launches"] >= 1 and not r["sums"].any() and not r["episodes"].view(np.uint8).any()
        assert not r["td_count"].any()
        e = eng.evaluate(3, episodes=True)
        assert e["steps"] == 0 and not e["sums"].any() and not e["episodes"].view(np.uint8).any()
        agents_equal(full_state(eng), after, slice(None), "all inactive")
        assert not raw_equal(before["q"], after["q"])
        eng.set_active_sets(np.array([True, True]))                                          # all ones: the same as None
        assert eng.active_sets is None
        eng.set_hparams(None, None)                                                          # uninstalling clears the mask too
        assert eng.active_sets is None and eng.train(2, 2)["sums"].shape == (2, 4)
        assert L.rlb_engine_set_active_sets(eng.h, abi.ptr(m), 2) == abi.ERR_INVALID_ARG


def test_mask_from_a_device_buffer_and_a_snapshot_round_trip(tmp_path):
    import torch
    path = str(tmp_path / "snap.npz")
    a, b, mask, group, _ = masked_pair()
    a.set_active_sets(None)
    d_mask = torch.from_numpy(mask.astype(np.uint8)).cuda()
    torch.cuda.synchronize()
    abi.check(abi.lib.rlb_engine_set_active_sets(a.h, d_mask.data_ptr(), G))
    a.active_sets = mask.copy()
    a.train(5, 2, sums=False)
    snapshot.save_snapshot(a, path)
    assert raw_equal(np.load(path)["hp_active"], mask.astype(np.uint8))
    want = a.train(10, 2, ep_begin=5, episodes=True)
    q_want = a.download_tables()[0]
    a.close()
    snapshot.load_snapshot(b, path)
    assert raw_equal(b.active_sets, mask)
    got = b.train(10, 2, ep_begin=5, episodes=True)
    assert raw_equal(got["sums"], want["sums"]) and raw_equal(got["episodes"], want["episodes"])
    assert raw_equal(b.download_tables()[0], q_want)
    b.close()


GRID = {"learning_rate": [0.05, 0.1, 0.2, 0.4], "exploration_time": [0.25, 0.5]}
KW = dict(agents_per_point=32, n_episodes=200, real="f32", verbose=False)


def test_run_halving_end_to_end():
    s = driver.run_sweep("taxi", GRID, **KW)
    a = driver.run_halving("taxi", GRID, min_episodes=20, eta=2, **KW)
    b = driver.run_halving("taxi", GRID, min_episodes=20, eta=2, **KW)
    a.pop("seconds"), b.pop("seconds")
    assert json.dumps(a) == json.dumps(b)
    assert [r["budget"] for r in a["rungs"]] == [20, 40, 80, 160, 200]
    assert [len(r["active"]) for r in a["rungs"]] == [8, 4, 2, 1, 1]
    survivors = a["rungs"][-1]["active"]
    for g in survivors:
        for key in ("train_rewards", "train_episodes_length", "test_rewards", "test_episodes_length", "eval_mean_return", "hparams"):
            assert a["points"][g][key] == s["points"][g][key], (g, key)
    assert a["ranking"][:len(survivors)] == sorted(survivors, key=lambda g: (-s["points"][g]["eval_mean_return"], g))
    # engine level: every set's per-episode training sums over the episodes it trained are the sweep's
    eng, n, *_ = driver.grid_engine("taxi", GRID, agent="onestep", selector="eps", target="qlearning", policy="basic",
                                    agents_per_point=32, seed=0x5EED0001, real="f32", device=0, n_episodes=200)
    full = eng.train(n, n // 10)["sums"]
    eng.close()
    eng, *_ = driver.grid_engine("taxi", GRID, agent="onestep", selector="eps", target="qlearning", policy="basic",
                                 agents_per_point=32, seed=0x5EED0001, real="f32", device=0, n_episodes=200)
    for r in a["rungs"]:
        m = np.zeros(8, bool)
        m[r["active"]] = True
        eng.set_active_sets(m)
        b0, b1 = r["episodes"]
        part = eng.train(b1, n // 10, ep_begin=b0)["sums"]
        assert raw_equal(part[:, m], full[b0:b1, m]), r
        assert not part[:, ~m].any()
    eng.close()
    for g, pt in enumerate(a["points"]):
        assert pt["train_rewards"] == s["points"][g]["train_rewards"][:len(pt["train_rewards"])]
    # min_episodes >= n: run_sweep's output
    one = driver.run_halving("taxi", GRID, min_episodes=500, eta=3, **KW)
    assert one["ranking"] == s["ranking"] and one["train_steps"] == s["train_steps"]
    for p1, ps in zip(one["points"], s["points"]):
        for key in ps:
            assert p1[key] == ps[key], key
