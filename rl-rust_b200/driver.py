"""Host experiment driver — the reference's per-env bins over the engine ("next" row N1/N2 of SURVEY.md §8f).

`run_model_experiment()` is `main()` of src/bin/cliffwalking_model.rs (Q-learning against Dyna-Q).
`run_experiment()` is `main()` of src/bin/{taxi,frozen_lake,cliffwalking,blackjack}.rs with the same flags and
defaults (bin/taxi.rs:22-68): two agents (OneStepAgent, ElegibilityTracesAgent) x two selectors (eps-greedy, UCB) x
three bootstrap targets = 12 runs, each `train(n, n/10)` -> `evaluate(n)` -> `agent.reset()` (bin/taxi.rs:158-203), the
env shared and never re-created, Blackjack followed by its win / loss / draw tally (bin/blackjack.rs:179-207).  The
curves are `moving_average` (utils.rs:78-93, quirk included) of the per-episode MEAN over the batch's agents; they are
returned / written as JSON and, with `--plots DIR`, drawn as the bins' five PNG charts (charts.py; utils.rs:97-157).

With n_agents = 1 every curve is the reference's, value for value (same Philox stream) — including "Training Error",
which the bins window over the raw per-STEP temporal differences with a window of `training_error.len() / window`
(bin/taxi.rs:170-174): the engine streams them (rlb_train_out.td_steps) whenever n_agents x n_episodes x (max_steps+1)
values fit TD_STREAM_BYTES; with more agents each agent's own curve is formed that way and the chart shows their mean.
Past that budget the curve falls back to windows over episodes (mean TD per step of each episode) and says so in
`train_errors_kind`.

`gpus=G` (CLI `--gpus G`) shards the agents over G GPUs of the box by global agent id — one engine per device, driven
from this one process through the asynchronous train call — and gathers the per-episode sums to GPU 0 with the library's
NCCL gather (rlb_comm_init_all / rlb_comm_gather_episode_sums).
"""
import json
import time

import numpy as np

from . import _abi as abi
from . import api

LEGENDS = ["ε-Greedy One-Step Sarsa", "ε-Greedy One-Step Qlearning", "ε-Greedy One-Step Expected Sarsa", "UCB One-Step Sarsa",
           "UCB One-Step Qlearning", "UCB One-Step Expected Sarsa", "ε-Greedy Trace Sarsa", "ε-Greedy Trace Qlearning",
           "ε-Greedy Trace Expected Sarsa", "UCB Trace Sarsa", "UCB Trace Qlearning", "UCB Trace Expected Sarsa"]   # bin/taxi.rs:96-110

DEFAULTS = dict(n_episodes=100000, max_steps=100, learning_rate=0.05, initial_epsilon=1.0, exploration_time=0.5, final_epsilon=0.0,
                confidence_level=0.5, discount_factor=0.95, lambda_factor=0.5, moving_average_window=100, stochastic_env=False,
                map="4x4")


def moving_average(window, vector):
    """utils.rs:78-93: sums of consecutive `window`-long slices, each divided by `window` — including the last,
    possibly shorter, slice (the reference's quirk); when len % window == 0 there is no short slice.  The sums are
    sequential left-to-right f64 additions like `slice.iter().sum()` (np.cumsum; np.sum would add pairwise)."""
    vector = np.asarray(vector, np.float64)
    out = []
    aux = 0
    if window <= 0:
        return out
    while aux < len(vector):
        end = aux + window if aux + window < len(vector) else len(vector)
        out.append(float(np.cumsum(vector[aux:end])[-1]) / float(window))
        aux = end
    return out


TD_STREAM_BYTES = 1 << 31   # host + device budget for the exact per-step TD stream of one train() call


def training_error_curve(res, n_agents, ma_window, window_episodes):
    """The bins' "Training Error" series (bin/taxi.rs:170-174): moving_average(training_error.len() / ma_window,
    &training_error) per agent from the per-step TD stream, averaged over agents point by point (an agent contributes
    to the points it has); without the stream, windows over episodes of the mean TD per step."""
    if "td_steps" in res and int(res["td_count"].max()) <= res["td_steps"].shape[1]:
        curves = []
        for i in range(n_agents):
            n = int(res["td_count"][i])
            curves.append(moving_average(n // ma_window, res["td_steps"][i, :n].astype(np.float64)))
        if n_agents == 1:
            return curves[0], "per-step (exact: bin/taxi.rs:170-174)"
        width = max(len(c) for c in curves)
        acc, cnt = np.zeros(width), np.zeros(width)
        for c in curves:
            acc[:len(c)] += c
            cnt[:len(c)] += 1
        return (acc / np.maximum(cnt, 1)).tolist(), "per-step, mean over agents of each agent's own curve"
    s_ = res["sums"]
    with np.errstate(invalid="ignore", divide="ignore"):
        mean_td = s_[:, 2] / s_[:, 0]
    return moving_average(window_episodes, mean_td), "per-episode windows of the mean TD per step (the per-step stream exceeds TD_STREAM_BYTES)"


class EngineGroup:
    """The engines of one experiment: one per GPU, agents sharded by global id; a single engine when gpus == 1.
    Forwards the agent / selector / target switches to every engine, trains them concurrently (asynchronous train
    call) and gathers the per-episode sums to GPU 0 with the library's NCCL gather."""

    def __init__(self, gpus, n_agents, **kw):
        self.gpus = gpus
        base, extra = divmod(n_agents, gpus)
        self.sizes = [base + (1 if r < extra else 0) for r in range(gpus)]
        if min(self.sizes) < 1:
            raise ValueError("n_agents must be >= gpus")
        first = 0
        self.engines = []
        dev0 = kw.pop("device", 0)
        for r, n in enumerate(self.sizes):
            self.engines.append(abi.Engine(n_agents=n, first_agent_id=first, device=dev0 + r, **kw))
            first += n
        self.comms = abi.Comm.init_all([dev0 + r for r in range(gpus)]) if gpus > 1 else None
        self.dev0 = dev0

    def __getattr__(self, name):   # set_agent_kind, set_selector, set_target, agent_reset, set_model: applied to every engine
        def call(*a, **k):
            out = [getattr(e, name)(*a, **k) for e in self.engines]
            return out[0]
        return call

    def train(self, n, eval_at, td_capacity=0):
        if self.gpus == 1:
            return self.engines[0].train(n, eval_at, td_capacity=td_capacity)
        import torch
        sums = [torch.zeros((n, 4), dtype=torch.float64, device="cuda:%d" % (self.dev0 + r)) for r in range(self.gpus)]
        gathered = torch.zeros((self.gpus, n, 4), dtype=torch.float64, device="cuda:%d" % self.dev0)
        for r, e in enumerate(self.engines):
            torch.cuda.synchronize(self.dev0 + r)
            e.train(n, eval_at, sums_out=sums[r], td_capacity=td_capacity, wait=False)
        parts = [e.train_wait()[0] for e in self.engines]
        abi.check(abi.lib.rlb_comm_group_begin())
        for r, cm in enumerate(self.comms):
            cm.gather_episode_sums(sums[r], gathered if r == 0 else None, root=0, stream=torch.cuda.current_stream(self.dev0 + r).cuda_stream)
        abi.check(abi.lib.rlb_comm_group_end())
        for r in range(self.gpus):
            torch.cuda.synchronize(self.dev0 + r)
        res = dict(sums=gathered.sum(0).cpu().numpy(), train_steps=sum(p["train_steps"] for p in parts), eval_steps=sum(p["eval_steps"] for p in parts))
        if td_capacity:
            res["td_steps"] = np.concatenate([p["td_steps"] for p in parts], 0)
            res["td_count"] = np.concatenate([p["td_count"] for p in parts], 0)
        return res

    def evaluate(self, n, sums=True, episodes=False):
        parts = [e.evaluate(n, sums=sums, episodes=episodes) for e in self.engines]
        out = dict(steps=sum(p["steps"] for p in parts))
        out["sums"] = sum(p["sums"] for p in parts) if sums else None
        out["episodes"] = np.concatenate([p["episodes"] for p in parts], 1) if episodes else None
        return out

    def get_action(self, obs):
        return self.engines[0].get_action(obs)

    def states(self):
        return np.concatenate([e.states() for e in self.engines])

    def close(self):
        for e in self.engines:
            e.close()
        for c in self.comms or []:
            c.close()


def make_env(name, **flags):
    if name == "blackjack":
        return api.BlackJackEnv()                                                                    # bin/blackjack.rs:78
    if name == "frozen_lake":
        m = api.FrozenLakeEnv.MAP_4X4 if flags.get("map", "4x4") == "4x4" else api.FrozenLakeEnv.MAP_8X8   # bin/frozen_lake.rs:93-97
        return api.FrozenLakeEnv(m, flags.get("stochastic_env", False), flags["max_steps"])
    if name in ("cliffwalking", "cliff_walking"):
        return api.CliffWalkingEnv(flags["max_steps"])
    if name == "taxi":
        return api.TaxiEnv(flags["max_steps"])
    raise ValueError("unknown env %r" % name)


def run_experiment(env_name, *, n_agents=1, seed=0x5EED0001, real="f64", device=0, tally_games=1000000, policy="basic",
                   verbose=True, show_example=False, gpus=1, **flags):
    """Returns {'legends', 'train_rewards', 'train_episodes_length', 'train_errors', 'test_rewards',
    'test_episodes_length', 'seconds', ['blackjack_rates']} — the five chart series of bin/taxi.rs:205-223."""
    f = dict(DEFAULTS)
    f.update(flags)
    n = int(f["n_episodes"])
    epsilon_decay = f["initial_epsilon"] / (f["exploration_time"] * n)                               # bin/taxi.rs:78
    window = max(1, n // int(f["moving_average_window"]))                                            # first argument at every call site
    env = make_env(env_name, **f)
    # ONE engine = the bins' one env + one RNG stream per agent slot; the two agent objects of bin/taxi.rs:138-156 take
    # turns on it (rlb_agent_set_kind), so run 7 continues the stream where run 6 left it, as in the reference.
    eng = EngineGroup(gpus, n_agents, env_kind=env.kind, policy=abi.POLICY_BASIC if policy == "basic" else abi.POLICY_DOUBLE,   # bins: Basic (bin/taxi.rs:126)
                      selector=abi.SEL_EPS_GREEDY, target=abi.TARGET_SARSA, agent=abi.AGENT_ONE_STEP,
                      real=abi.REAL_F32 if real == "f32" else abi.REAL_F64, learning_rate=f["learning_rate"],
                      discount_factor=f["discount_factor"], lambda_factor=f["lambda_factor"], initial_epsilon=f["initial_epsilon"],
                      decay_kind=abi.DECAY_SUB, epsilon_decay=epsilon_decay, final_epsilon=f["final_epsilon"],
                      confidence_level=f["confidence_level"], default_value=0.0, seed=seed, device=device, **env._cfg())
    env.bind(eng.engines[0])
    # per-step TD stream: at most max_steps + 1 steps per episode (Blackjack: a hand holds 16 cards, blackjack.rs:32-35)
    td_cap = n * (32 if env_name == "blackjack" else int(f["max_steps"]) + 1)
    if n_agents * td_cap * 8 > TD_STREAM_BYTES:
        td_cap = 0
    out = dict(legends=LEGENDS, train_rewards=[], train_episodes_length=[], train_errors=[], test_rewards=[],
               test_episodes_length=[], seconds=[], train_steps=[], gpus=gpus)
    if env_name == "blackjack":
        out["blackjack_rates"] = []
    i = 0
    for agent_kind in (abi.AGENT_ONE_STEP, abi.AGENT_TRACES):                                        # bin/taxi.rs:154-159
        eng.set_agent_kind(agent_kind)
        for sel in (abi.SEL_EPS_GREEDY, abi.SEL_UCB):
            eng.set_selector(sel)                                                                    # bin/taxi.rs:161 (a fresh clone)
            for func in (api.sarsa, api.qlearning, api.expected_sarsa):
                eng.set_target(func)                                                                 # bin/taxi.rs:163
                t0 = time.perf_counter()
                res = eng.train(n, max(1, n // 10), td_capacity=td_cap)                              # bin/taxi.rs:165-166
                dt = time.perf_counter() - t0
                if verbose:
                    print("%s %.2fs (%d agents, %.3g train steps/s)" % (LEGENDS[i], dt, n_agents, res["train_steps"] / dt))
                s_ = res["sums"]                                                                     # [n,4]: sum len, ret, td, |td|
                mean_len, mean_ret = s_[:, 0] / n_agents, s_[:, 1] / n_agents
                curve, kind = training_error_curve(res, n_agents, int(f["moving_average_window"]), window)   # bin/taxi.rs:170-174
                out["train_errors"].append(curve)
                out["train_errors_kind"] = kind
                out["train_rewards"].append(moving_average(window, mean_ret))
                out["train_episodes_length"].append(moving_average(window, mean_len))
                out["seconds"].append(dt)
                out["train_steps"].append(int(res["train_steps"]))
                if env_name == "blackjack" and tally_games:                                          # bin/blackjack.rs:179-207
                    ev = eng.evaluate(int(tally_games), sums=False, episodes=True)["episodes"]["ret"]
                    tot = float(ev.size)
                    rates = (float((ev == 1.0).sum()) / tot, float((ev == -1.0).sum()) / tot, float(((ev != 1.0) & (ev != -1.0)).sum()) / tot)
                    out["blackjack_rates"].append(rates)
                    if verbose:
                        print("%s has win-rate of %s%%, loss-rate of %s%% and draw-rate %s%%" % ((LEGENDS[i],) + rates))
                if show_example:                                                                     # bin/taxi.rs:184-186
                    out.setdefault("examples", []).append(api.example_episode(env, eng.get_action, out=print if verbose else (lambda _: None)))
                ev = eng.evaluate(n, sums=True)["sums"]                                              # bin/taxi.rs:188
                out["test_rewards"].append(moving_average(window, ev[:, 1] / n_agents))
                out["test_episodes_length"].append(moving_average(window, ev[:, 0] / n_agents))
                i += 1
                eng.agent_reset()                                                                    # bin/taxi.rs:200
    out["final_rng_n"] = [int(x) for x in eng.states()["rng_n"][:8]]
    eng.close()
    return out


LEGENDS_MODEL = ["ε-Greedy One-Step Qlearning", "ε-Greedy One-Step Dyna-Qlearning"]   # bin/cliffwalking_model.rs:96-111


def run_model_experiment(*, n_agents=1, seed=0x5EED0001, real="f64", device=0, planning_steps=10, verbose=True, **flags):
    """`main()` of src/bin/cliffwalking_model.rs: CliffWalking, a OneStepAgent with qlearning and then an
    InternalModelAgent (RandomModel, 10 planning steps) around a second such agent, eps-greedy, Basic policy; each
    `train(n, n/10)` -> `evaluate(n)` -> `reset()` on the one shared env (:158-203).  Same output dict as run_experiment."""
    f = dict(DEFAULTS)
    f.update(flags)
    n = int(f["n_episodes"])
    epsilon_decay = f["initial_epsilon"] / (f["exploration_time"] * n)                               # :77
    window = max(1, n // int(f["moving_average_window"]))
    env = api.CliffWalkingEnv(f["max_steps"])                                                        # :86
    eng = abi.Engine(env.kind, n_agents=n_agents, policy=abi.POLICY_BASIC, selector=abi.SEL_EPS_GREEDY, target=abi.TARGET_QLEARNING,
                     agent=abi.AGENT_ONE_STEP, real=abi.REAL_F32 if real == "f32" else abi.REAL_F64, learning_rate=f["learning_rate"],
                     discount_factor=f["discount_factor"], lambda_factor=f["lambda_factor"], initial_epsilon=f["initial_epsilon"],
                     decay_kind=abi.DECAY_SUB, epsilon_decay=epsilon_decay, final_epsilon=f["final_epsilon"],
                     confidence_level=f["confidence_level"], default_value=0.0, seed=seed, device=device, **env._cfg())
    env.bind(eng)
    out = dict(legends=LEGENDS_MODEL, train_rewards=[], train_episodes_length=[], train_errors=[], test_rewards=[],
               test_episodes_length=[], seconds=[], train_steps=[])
    for i, planning in enumerate((0, int(planning_steps))):                                          # :158-160
        eng.set_agent_kind(abi.AGENT_ONE_STEP)                                                       # `one_step_agent` / `other` (:136-148): a fresh agent
        if planning:
            eng.set_model(planning)                                                                  # :150-156
        eng.set_selector(abi.SEL_EPS_GREEDY)                                                         # :164
        t0 = time.perf_counter()
        td_cap = n * (int(f["max_steps"]) + 1)
        res = eng.train(n, max(1, n // 10), td_capacity=td_cap if n_agents * td_cap * 8 <= TD_STREAM_BYTES else 0)   # :166-167
        dt = time.perf_counter() - t0
        if verbose:
            print("%s %.2fs (%d agents, %.3g train steps/s)" % (LEGENDS_MODEL[i], dt, n_agents, res["train_steps"] / dt))
        s_ = res["sums"]
        curve, kind = training_error_curve(res, n_agents, int(f["moving_average_window"]), window)   # :171-175; the model agent returns the wrapped agent's TD (internal_model_agent.rs:78)
        out["train_errors"].append(curve)
        out["train_errors_kind"] = kind
        out["train_rewards"].append(moving_average(window, s_[:, 1] / n_agents))
        out["train_episodes_length"].append(moving_average(window, s_[:, 0] / n_agents))
        out["seconds"].append(dt)
        out["train_steps"].append(int(res["train_steps"]))
        ev = eng.evaluate(n, sums=True)["sums"]                                                      # :189
        out["test_rewards"].append(moving_average(window, ev[:, 1] / n_agents))
        out["test_episodes_length"].append(moving_average(window, ev[:, 0] / n_agents))
        eng.agent_reset()                                                                            # :201
    out["final_rng_n"] = [int(x) for x in eng.states()["rng_n"][:8]]
    eng.close()
    return out


def main(argv=None):
    import argparse
    ap = argparse.ArgumentParser(description="RL-Rust bins over the B200 engine: blackjack | frozen_lake | cliffwalking | taxi | cliffwalking_model")
    ap.add_argument("env", choices=["blackjack", "frozen_lake", "cliffwalking", "taxi", "cliffwalking_model"])
    ap.add_argument("--n_episodes", "-n", type=int, default=DEFAULTS["n_episodes"])
    for name in ("max_steps", "moving_average_window"):
        ap.add_argument("--" + name, type=int, default=DEFAULTS[name])
    for name in ("learning_rate", "initial_epsilon", "exploration_time", "final_epsilon", "confidence_level", "discount_factor",
                 "lambda_factor"):
        ap.add_argument("--" + name, type=float, default=DEFAULTS[name])
    ap.add_argument("--stochastic_env", action="store_true")
    ap.add_argument("--map", default="4x4")
    ap.add_argument("--show_example", action="store_true", help="print one rendered episode after each training run (needs --n_agents 1)")
    ap.add_argument("--n_agents", type=int, default=1)
    ap.add_argument("--gpus", type=int, default=1, help="shard the agents over this many GPUs of the box (NCCL gather of the curves)")
    ap.add_argument("--seed", type=lambda x: int(x, 0), default=0x5EED0001)
    ap.add_argument("--real", choices=["f32", "f64"], default="f64")
    ap.add_argument("--tally_games", type=int, default=1000000)
    ap.add_argument("--out", default=None, help="write the chart series as JSON here")
    ap.add_argument("--plots", default=None, help="directory for the five PNG charts of the bins (utils.rs:97-157)")
    a = vars(ap.parse_args(argv))
    env_name, outp, plots = a.pop("env"), a.pop("out"), a.pop("plots")
    if env_name == "cliffwalking_model":
        for k in ("tally_games", "stochastic_env", "map", "show_example", "gpus"):
            a.pop(k)
        res = run_model_experiment(**a)
    else:
        res = run_experiment(env_name, **a)
    if outp:
        with open(outp, "w") as fh:
            json.dump(res, fh)
    if plots:
        from . import charts
        charts.plot_experiment(res, plots)
    return res


# ---- hyper-parameter sweeps: the bins' flags as grids, every grid point a group of agents of ONE engine ------------------
SWEEP_FLAGS = ("learning_rate", "discount_factor", "lambda_factor", "initial_epsilon", "exploration_time", "final_epsilon",
               "confidence_level")   # the bin flags that are agent constructor arguments (bin/taxi.rs:22-68, :78)
AGENT_NAMES = {"onestep": abi.AGENT_ONE_STEP, "traces": abi.AGENT_TRACES}
SELECTOR_NAMES = {"eps": abi.SEL_EPS_GREEDY, "ucb": abi.SEL_UCB}
TARGET_KINDS = {"sarsa": abi.TARGET_SARSA, "qlearning": abi.TARGET_QLEARNING, "expected_sarsa": abi.TARGET_EXPECTED_SARSA}
# Dyna-Q's planning replays per real update (InternalModelAgent::new's third argument, bin/cliffwalking_model.rs): an
# integer axis of its own, kept beside rlb_hparams (rlb_engine_set_planning_steps); 0 is the plain agent
PLANNING_AXIS = "planning_steps"
# the bootstrap target (Agent::set_future_q_value_func, agent.rs:48) as a categorical axis: names of TARGET_KINDS, kept
# beside rlb_hparams (rlb_engine_set_targets)
TARGET_AXIS = "target"


def planning_value(v):
    """A planning-steps grid value as an int; anything but a non-negative integer is a ValueError."""
    if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, np.integer)) or v < 0:
        raise ValueError("planning_steps values must be non-negative integers, got %r" % (v,))
    return int(v)


def expand_grid(grid):
    """{flag: [values]} -> the cartesian product as a list of {flag: value}, the first flag varying slowest."""
    import itertools
    grid = dict(grid)
    for k in grid:
        if k == PLANNING_AXIS:
            grid[k] = [planning_value(v) for v in grid[k]]
        elif k == TARGET_AXIS:
            bad = [v for v in grid[k] if not isinstance(v, str) or v not in TARGET_KINDS]
            if bad:
                raise ValueError("target values must be among %s, got %r" % (", ".join(sorted(TARGET_KINDS)), bad))
        elif k not in SWEEP_FLAGS:
            raise ValueError("%r cannot be swept; the agent constructor flags are %s, %s and %s"
                             % (k, ", ".join(SWEEP_FLAGS), PLANNING_AXIS, TARGET_AXIS))
    keys = list(grid)
    return [dict(zip(keys, vals)) for vals in itertools.product(*(grid[k] for k in keys))]


def point_hparams(flags, n_episodes):
    """One grid point's rlb_hparams, the decay derived as run_experiment derives it (bin/taxi.rs:78)."""
    return dict(learning_rate=flags["learning_rate"], discount_factor=flags["discount_factor"], lambda_factor=flags["lambda_factor"],
                initial_epsilon=flags["initial_epsilon"], epsilon_decay=flags["initial_epsilon"] / (flags["exploration_time"] * n_episodes),
                final_epsilon=flags["final_epsilon"], confidence_level=flags["confidence_level"], default_value=0.0)


def grid_engine(env_name, grid, *, agent, selector, target, policy, agents_per_point, seed, real, device, **flags):
    """The grid as one engine: every point of the cartesian grid of `grid` a set, its agents a contiguous group of
    `agents_per_point` constructed with the point's values (rlb_engine_set_hparams).  Returns (engine, n_episodes,
    moving-average window, points, every point's flags, every point's rlb_hparams).  With a planning_steps axis every set
    is also a Dyna-Q agent with its point's planning count (rlb_engine_set_planning_steps), and with a target axis every
    set bootstraps with its point's target (rlb_engine_set_targets); `target` is then only the engine's configured one."""
    f = dict(DEFAULTS)
    f.update(flags)
    n = int(f["n_episodes"])
    window = max(1, n // int(f["moving_average_window"]))
    points = expand_grid(grid)
    point_flags = []
    for pt in points:
        pf = dict(f)
        pf.update(pt)
        point_flags.append(pf)
    sets = [point_hparams(pf, n) for pf in point_flags]
    if len(sets) > abi.MAX_HPARAM_SETS:
        raise ValueError("%d grid points; an engine holds at most %d sets" % (len(sets), abi.MAX_HPARAM_SETS))
    env = make_env(env_name, **f)
    eng = abi.Engine(env.kind, n_agents=len(points) * int(agents_per_point), policy=abi.POLICY_BASIC if policy == "basic" else abi.POLICY_DOUBLE,
                     selector=SELECTOR_NAMES[selector], target=TARGET_KINDS[target], agent=AGENT_NAMES[agent],
                     real=abi.REAL_F32 if real == "f32" else abi.REAL_F64, decay_kind=abi.DECAY_SUB, seed=seed, device=device,
                     **sets[0], **env._cfg())
    try:
        eng.set_hparams(sets, np.repeat(np.arange(len(points), dtype=np.uint32), int(agents_per_point)))
        if PLANNING_AXIS in grid:
            eng.set_planning_steps(np.array([pf[PLANNING_AXIS] for pf in point_flags], np.uint32))
        if TARGET_AXIS in grid:
            eng.set_targets(point_targets(point_flags))
    except BaseException:
        eng.close()
        raise
    return eng, n, window, points, point_flags, sets


def point_targets(point_flags):
    """Every point's target name as the RLB_TARGET_* array rlb_engine_set_targets takes."""
    return np.array([TARGET_KINDS[pf[TARGET_AXIS]] for pf in point_flags], np.int32)


def engine_target(grid, target):
    """The `target` of a result: the engine-wide name, or None where a target axis gives each point its own."""
    return None if TARGET_AXIS in grid else target


def point_results(points, sets, train_sums, eval_sums, agents_per_point, n, window):
    """Per point: the bins' moving averages of return and episode length (train and evaluate) and the evaluate mean
    return, from the grouped sums [n, G, 4]; and the points ranked by that return."""
    per = float(agents_per_point)
    out_points = []
    for g, pt in enumerate(points):
        s_, e_ = train_sums[:, g], eval_sums[:, g]
        out_points.append(dict(params=pt, hparams=sets[g],
                               train_rewards=moving_average(window, s_[:, 1] / per),
                               train_episodes_length=moving_average(window, s_[:, 0] / per),
                               test_rewards=moving_average(window, e_[:, 1] / per),
                               test_episodes_length=moving_average(window, e_[:, 0] / per),
                               eval_mean_return=float(e_[:, 1].sum()) / (per * n)))
    ranking = sorted(range(len(points)), key=lambda g: -out_points[g]["eval_mean_return"])
    return out_points, ranking


def run_sweep(env_name, grid, *, agent="onestep", selector="eps", target="qlearning", policy="basic", agents_per_point=1024,
              seed=0x5EED0001, real="f64", device=0, verbose=True, **flags):
    """One run of the bin (`train(n, n/10)` -> `evaluate(n)`, bin/taxi.rs:165-188) for every point of the cartesian grid
    of `grid` ({flag: [values]}, flags otherwise as in run_experiment), all points at once: ONE engine, the points'
    agents in contiguous groups of `agents_per_point`, each group constructed with its point's values
    (rlb_engine_set_hparams); the grouped per-episode sums give every point its own curves.  Returns the bins' moving
    averages of return and episode length per point, the evaluate mean return, and the points ranked by it."""
    eng, n, window, points, _, sets = grid_engine(env_name, grid, agent=agent, selector=selector, target=target, policy=policy,
                                                  agents_per_point=agents_per_point, seed=seed, real=real, device=device, **flags)
    try:
        t0 = time.perf_counter()
        res = eng.train(n, max(1, n // 10))                                                          # [n, G, 4]
        ev = eng.evaluate(n, sums=True)["sums"]                                                      # [n, G, 4]
        dt = time.perf_counter() - t0
    finally:
        eng.close()
    out_points, ranking = point_results(points, sets, res["sums"], ev, agents_per_point, n, window)
    if verbose:
        print("%d points x %d agents, %d episodes: %.2fs (%.3g train steps/s)" % (len(points), agents_per_point, n, dt,
                                                                                  res["train_steps"] / dt if dt > 0 else 0.0))
        for g in ranking[:10]:
            print("  %-60s evaluate mean return %.4f" % (points[g], out_points[g]["eval_mean_return"]))
    return dict(env=env_name, agent=agent, selector=selector, target=engine_target(grid, target), policy=policy, real=real, n_episodes=n,
                agents_per_point=int(agents_per_point), grid={k: list(v) for k, v in grid.items()}, points=out_points,
                ranking=ranking, seconds=dt, train_steps=int(res["train_steps"]))


def parse_list(text):
    return [float(x) for x in text.split(",") if x.strip()]


def parse_names(text):
    return [x.strip() for x in text.split(",") if x.strip()]


def sweep_parser(description):
    """The flags of tools/rl_sweep.py (and, with their own additions, tools/rl_pbt.py)."""
    import argparse
    ap = argparse.ArgumentParser(description=description)
    ap.add_argument("env", choices=["blackjack", "frozen_lake", "cliffwalking", "taxi"])
    ap.add_argument("--grid", action="append", default=[], metavar="FLAG=V1,V2,...",
                    help="a bin flag and its values (repeatable; one of %s, %s, %s)" % (", ".join(SWEEP_FLAGS), PLANNING_AXIS, TARGET_AXIS))
    for name in SWEEP_FLAGS:
        ap.add_argument("--" + name, default=None, metavar="V1,V2,...", help="values of this flag (a comma list: a grid axis)")
    ap.add_argument("--" + PLANNING_AXIS, default=None, metavar="K1,K2,...",
                    help="Dyna-Q planning replays per update (non-negative integers: a grid axis; 0 is the plain agent)")
    ap.add_argument("--n_episodes", "-n", type=int, default=DEFAULTS["n_episodes"])
    for name in ("max_steps", "moving_average_window"):
        ap.add_argument("--" + name, type=int, default=DEFAULTS[name])
    ap.add_argument("--stochastic_env", action="store_true")
    ap.add_argument("--map", default="4x4")
    ap.add_argument("--agent", choices=sorted(AGENT_NAMES), default="onestep")
    ap.add_argument("--selector", choices=sorted(SELECTOR_NAMES), default="eps")
    ap.add_argument("--target", default="qlearning", metavar="NAME[,NAME...]",
                    help="bootstrap target, one of %s: one name for every agent, or a comma list (a grid axis)" % ", ".join(sorted(TARGET_KINDS)))
    ap.add_argument("--policy", choices=["basic", "double"], default="basic")
    ap.add_argument("--agents_per_point", type=int, default=1024)
    ap.add_argument("--seed", type=lambda x: int(x, 0), default=0x5EED0001)
    ap.add_argument("--real", choices=["f32", "f64"], default="f64")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None, help="write the result as JSON here")
    return ap


def parse_sweep_args(ap, argv):
    """(env name, grid, output path, the other flags as keyword arguments)"""
    a = vars(ap.parse_args(argv))

    def planning_list(text):
        try:
            return [planning_value(int(x)) for x in text.split(",") if x.strip()]
        except ValueError:
            ap.error("--%s takes non-negative integers, got %r" % (PLANNING_AXIS, text))

    def target_list(text):
        names = parse_names(text)
        if not names or any(x not in TARGET_KINDS for x in names):
            ap.error("--%s takes names among %s, got %r" % (TARGET_AXIS, ", ".join(sorted(TARGET_KINDS)), text))
        return names

    grid = {}
    targets = target_list(a["target"])
    if len(targets) > 1:   # a comma list is an axis; a single name stays engine-wide
        grid[TARGET_AXIS] = targets
        a["target"] = targets[0]
    for name in SWEEP_FLAGS:
        v = a.pop(name)
        if v is not None:
            grid[name] = parse_list(v)
    v = a.pop(PLANNING_AXIS)
    if v is not None:
        grid[PLANNING_AXIS] = planning_list(v)
    for item in a.pop("grid"):
        if "=" not in item:
            ap.error("--grid takes FLAG=V1,V2,...")
        k, v = item.split("=", 1)
        if k == PLANNING_AXIS:
            grid[k] = planning_list(v)
            continue
        if k == TARGET_AXIS:
            grid[k] = target_list(v)
            a["target"] = grid[k][0]
            continue
        if k not in SWEEP_FLAGS:
            ap.error("--grid %s: not a sweepable flag (%s, %s, %s)" % (k, ", ".join(SWEEP_FLAGS), PLANNING_AXIS, TARGET_AXIS))
        grid[k] = parse_list(v)
    if not grid:
        ap.error("nothing to sweep: give at least one --grid FLAG=V1,V2,...")
    return a.pop("env"), grid, a.pop("out"), a


def write_json(res, path):
    if path:
        with open(path, "w") as fh:
            json.dump(res, fh)


def main_sweep(argv=None):
    ap = sweep_parser("Hyper-parameter sweep of one RL-Rust bin run over the B200 engine: every point of the grid is a "
                      "group of agents of one engine")
    env_name, grid, outp, kw = parse_sweep_args(ap, argv)
    res = run_sweep(env_name, grid, **kw)
    write_json(res, outp)
    return res


# ---- population-based training (Jaderberg et al., 2017): the sweep's grid as the initial population ----------------------
PBT_FACTORS = (0.8, 1.2)
_TINY = float(np.nextafter(0.0, 1.0))
PBT_BOUNDS = dict(learning_rate=(_TINY, 1.0), discount_factor=(0.0, 1.0), lambda_factor=(0.0, 1.0), initial_epsilon=(0.0, 1.0),
                  final_epsilon=(0.0, 1.0), exploration_time=(_TINY, np.inf), confidence_level=(0.0, np.inf))   # (0, 1], [0, 1], > 0, >= 0


def pbt_exploit(chunk_sums, fraction, rng):
    """Ranks the sets by their mean training return over a chunk (chunk_sums [episodes, G, 4]; every set holds the same
    number of agents) and pairs each of the bottom floor(fraction * G) sets with a set drawn uniformly from the top as many.
    Returns [(loser, winner)], losers from the weakest up."""
    n_sets = chunk_sums.shape[1]
    mean_ret = chunk_sums[:, :, 1].sum(0)
    order = sorted(range(n_sets), key=lambda g: (-mean_ret[g], g))   # best first; ties by set index
    k = int(np.floor(fraction * n_sets))
    top, bottom = order[:k], order[n_sets - k:][::-1]
    return [(loser, top[int(rng.integers(k))]) for loser in bottom]


def pbt_perturb_planning(k, f):
    """A planning count perturbed by the factor f (0.8 or 1.2) as an integer in [0, inf): round(k * f), and where that
    leaves k as it is, k + 1 for f > 1 and max(0, k - 1) for f < 1."""
    out = int(round(k * f))
    if out == k:
        out = k + 1 if f > 1.0 else max(0, k - 1)
    return out


def pbt_explore(flags, axes, rng, targets=None, resample_probability=0.25):
    """The winner's flags with every numeric grid axis multiplied by 0.8 or 1.2 at random and clamped into its range (the
    planning count as an integer: pbt_perturb_planning).  A target axis is inherited, and with probability
    `resample_probability` redrawn uniformly from `targets` (the axis values).  Without a target axis the draws are
    those of the numeric axes alone."""
    out = dict(flags)
    for k in axes:
        if k == TARGET_AXIS:
            if targets is None:
                raise ValueError("a target axis needs its values (targets=) to resample from")
            if rng.random() < resample_probability:
                out[k] = targets[int(rng.integers(len(targets)))]
            continue
        f = PBT_FACTORS[int(rng.integers(2))]
        if k == PLANNING_AXIS:
            out[k] = pbt_perturb_planning(int(flags[k]), f)
            continue
        lo, hi = PBT_BOUNDS[k]
        out[k] = float(min(max(flags[k] * f, lo), hi))
    return out


def run_pbt(env_name, grid, *, interval, fraction=0.25, pbt_seed=0x9B7, resample_probability=0.25, agent="onestep", selector="eps",
            target="qlearning", policy="basic", agents_per_point=1024, seed=0x5EED0001, real="f64", device=0, verbose=True, **flags):
    """Population-based training over the grid of `grid`: the initial population is run_sweep's (one set per point,
    contiguous groups of `agents_per_point`), and its one `train(n, n/10)` is driven in chunks of `interval` episodes.
    After every chunk but the last the sets are ranked by their mean training return over the chunk; each of the bottom
    floor(fraction * G) sets takes over the learned state of a set drawn from the top as many (agent j of the winner ->
    agent j of the loser, one rlb_agent_clone) and continues with the winner's flags, every numeric grid axis perturbed
    (rlb_engine_retune_hparams) and a target axis inherited, or with probability `resample_probability` redrawn from the
    axis values (rlb_engine_set_targets).  `pbt_seed` seeds those draws.  Returns run_sweep's output plus every set's final flags
    and the lineage: per chunk boundary, the list of (loser, winner, new flags)."""
    if not 0.0 <= fraction <= 0.5:
        raise ValueError("fraction must be in [0, 0.5]: the top and bottom sets may not overlap")
    interval = int(interval)
    if interval < 1:
        raise ValueError("interval must be >= 1")
    if not 0.0 <= resample_probability <= 1.0:
        raise ValueError("resample_probability must be in [0, 1]")
    if PLANNING_AXIS in grid and agent == "traces":
        raise ValueError("PBT with a planning_steps axis clones Dyna agents, and cloning a trace agent under a model is not supported")
    axes = list(grid)
    per = int(agents_per_point)
    eng, n, window, points, cur, sets = grid_engine(env_name, grid, agent=agent, selector=selector, target=target, policy=policy,
                                                    agents_per_point=per, seed=seed, real=real, device=device, **flags)
    rng = np.random.default_rng(pbt_seed)
    lineage, parts, train_steps = [], [], 0          # cur: every set's flags in force
    try:
        t0 = time.perf_counter()
        for begin in range(0, n, interval):
            end = min(begin + interval, n)
            res = eng.train(end, max(1, n // 10), ep_begin=begin)                                    # [end - begin, G, 4]
            parts.append(res["sums"])
            train_steps += int(res["train_steps"])
            if end == n:
                break
            pairs = pbt_exploit(res["sums"], fraction, rng)
            step = []
            for loser, winner in pairs:
                cur[loser] = pbt_explore(cur[winner], axes, rng, grid.get(TARGET_AXIS), resample_probability)
                sets[loser] = point_hparams(cur[loser], n)
                step.append(dict(loser=loser, winner=winner, flags={k: cur[loser][k] for k in axes}))
            if pairs:
                j = np.arange(per, dtype=np.int64)
                eng.clone_agents(np.concatenate([w * per + j for _, w in pairs]), np.concatenate([l * per + j for l, _ in pairs]))
                eng.retune_hparams(sets)
                if PLANNING_AXIS in axes:
                    eng.set_planning_steps(np.array([c[PLANNING_AXIS] for c in cur], np.uint32))
                if TARGET_AXIS in axes:
                    eng.set_targets(point_targets(cur))
            lineage.append(dict(episode=end, pairs=step))
        ev = eng.evaluate(n, sums=True)["sums"]                                                      # [n, G, 4]
        dt = time.perf_counter() - t0
    finally:
        eng.close()
    out_points, ranking = point_results(points, sets, np.concatenate(parts), ev, per, n, window)
    for g, pt in enumerate(out_points):
        pt["final_params"] = {k: cur[g][k] for k in axes}
    if verbose:
        print("PBT: %d sets x %d agents, %d episodes in chunks of %d, fraction %.3g: %.2fs" % (len(points), per, n, interval, fraction, dt))
        for g in ranking[:10]:
            print("  set %-4d %-60s evaluate mean return %.4f" % (g, out_points[g]["final_params"], out_points[g]["eval_mean_return"]))
    return dict(env=env_name, agent=agent, selector=selector, target=engine_target(grid, target), policy=policy, real=real, n_episodes=n,
                agents_per_point=per, grid={k: list(v) for k, v in grid.items()}, interval=interval, fraction=fraction,
                pbt_seed=int(pbt_seed), **({"resample_probability": resample_probability} if TARGET_AXIS in grid else {}), points=out_points, ranking=ranking, lineage=lineage, seconds=dt, train_steps=train_steps)


def main_pbt(argv=None):
    ap = sweep_parser("Population-based training over one RL-Rust bin run on the B200 engine: the grid is the initial "
                      "population, and between chunks the weakest sets take over the state of strong ones and perturb their flags")
    ap.add_argument("--interval", type=int, required=True, help="episodes per chunk between exploit / explore steps")
    ap.add_argument("--fraction", type=float, default=0.25, help="share of the sets replaced after each chunk (and drawn from)")
    ap.add_argument("--pbt_seed", type=lambda x: int(x, 0), default=0x9B7, help="seed of the winner draws and perturbations")
    ap.add_argument("--resample_probability", type=float, default=0.25,
                    help="with a target axis: chance that a loser's inherited target is redrawn from the axis values")
    env_name, grid, outp, kw = parse_sweep_args(ap, argv)
    res = run_pbt(env_name, grid, **kw)
    write_json(res, outp)
    return res


# ---- successive halving (Jamieson & Talwalkar, 2016): train the grid on growing budgets, keep the best 1/eta each time ----
def halving_rungs(n, min_episodes, eta):
    """The rung budgets b_k = min(n, min_episodes * eta**k), k = 0, 1, ... up to the first that reaches n."""
    if int(min_episodes) < 1 or int(eta) < 2:
        raise ValueError("min_episodes must be >= 1 and eta >= 2")
    out, b = [], int(min_episodes)
    while True:
        out.append(min(int(n), b))
        if out[-1] >= n:
            return out
        b *= int(eta)


def halving_select(rung_sums, active, eta):
    """Ranks the active sets by their mean training return over a rung (rung_sums [episodes, G, 4]; every set holds the
    same number of agents), ties by set index, and keeps the best max(1, floor(len(active) / eta)).  Returns (kept,
    dropped): kept in ascending set index, dropped from the strongest down."""
    ret = rung_sums[:, :, 1].sum(0)
    order = sorted(active, key=lambda g: (-ret[g], g))
    keep = max(1, len(active) // int(eta))
    return sorted(order[:keep]), order[keep:]


def run_halving(env_name, grid, *, min_episodes, eta=3, agent="onestep", selector="eps", target="qlearning", policy="basic",
                agents_per_point=1024, seed=0x5EED0001, real="f64", device=0, verbose=True, **flags):
    """Successive halving over the grid of `grid`: run_sweep's engine (one set per point, contiguous groups of
    `agents_per_point`) and its one `train(n, n/10)`, driven in rungs that end at the budgets min(n, min_episodes * eta**k).
    After every rung but the last the active sets are ranked by their mean training return over that rung, and all but
    the best max(1, floor(active / eta)) are paused (rlb_engine_set_active_sets): they train no further, and the engine's
    launches cover only the sets still running.  `evaluate(n)` then runs over the survivors.  A survivor's curves and
    evaluate return are exactly run_sweep's for its point.  Returns run_sweep's output, where a dropped set's training
    curves cover the episodes it trained and its test curves and evaluate return are None, plus per set
    `episodes_trained`, `rung` (the rung it stopped at) and `last_rung_mean_return`, and `rungs`: each rung's budget and
    its active and dropped sets.  The ranking lists the survivors by evaluate return, then the dropped sets by episodes
    trained and by their last rung's return."""
    per = int(agents_per_point)
    eng, n, window, points, _, sets = grid_engine(env_name, grid, agent=agent, selector=selector, target=target, policy=policy,
                                                  agents_per_point=per, seed=seed, real=real, device=device, **flags)
    n_sets = len(points)
    try:
        budgets = halving_rungs(n, min_episodes, eta)
        train_sums = np.zeros((n, n_sets, 4))
        trained, stopped, last_ret = [0] * n_sets, [0] * n_sets, [0.0] * n_sets
        active, rungs, train_steps, begin = list(range(n_sets)), [], 0, 0
        t0 = time.perf_counter()
        for k, end in enumerate(budgets):
            res = eng.train(end, max(1, n // 10), ep_begin=begin)                                    # [end - begin, G, 4]
            train_sums[begin:end] = res["sums"]                                                      # paused sets' rows: 0.0
            train_steps += int(res["train_steps"])
            rung_ret = res["sums"][:, :, 1].sum(0)
            for g in active:
                trained[g], stopped[g], last_ret[g] = end, k, float(rung_ret[g]) / (per * (end - begin))
            kept, dropped = (halving_select(res["sums"], active, eta) if end < n else (active, []))
            rungs.append(dict(rung=k, budget=end, episodes=[begin, end], active=list(active), dropped=sorted(dropped)))
            if dropped:
                mask = np.zeros(n_sets, bool)
                mask[kept] = True
                eng.set_active_sets(mask)
            active, begin = kept, end
        ev = eng.evaluate(n, sums=True)["sums"]                                                      # [n, G, 4]; dropped sets 0.0
        dt = time.perf_counter() - t0
    finally:
        eng.close()
    out_points, _ = point_results(points, sets, train_sums, ev, per, n, window)
    survivors = set(active)
    for g, pt in enumerate(out_points):
        pt.update(episodes_trained=trained[g], rung=stopped[g], last_rung_mean_return=last_ret[g])
        if g not in survivors:
            s_ = train_sums[:trained[g], g]
            pt.update(train_rewards=moving_average(window, s_[:, 1] / per), train_episodes_length=moving_average(window, s_[:, 0] / per),
                      test_rewards=None, test_episodes_length=None, eval_mean_return=None)
    ranking = sorted(survivors, key=lambda g: (-out_points[g]["eval_mean_return"], g))
    ranking += sorted(set(range(n_sets)) - survivors, key=lambda g: (-trained[g], -last_ret[g], g))
    if verbose:
        print("successive halving: %d sets x %d agents, %d episodes, rungs %s (eta %d): %.2fs, %d train steps"
              % (n_sets, per, n, budgets, int(eta), dt, train_steps))
        for g in ranking[:min(10, len(survivors))]:
            print("  set %-4d %-60s evaluate mean return %.4f" % (g, points[g], out_points[g]["eval_mean_return"]))
    return dict(env=env_name, agent=agent, selector=selector, target=engine_target(grid, target), policy=policy, real=real, n_episodes=n,
                agents_per_point=per, grid={k: list(v) for k, v in grid.items()}, min_episodes=int(min_episodes), eta=int(eta),
                points=out_points, ranking=ranking, rungs=rungs, seconds=dt, train_steps=train_steps)


def main_halving(argv=None):
    ap = sweep_parser("Successive halving over one RL-Rust bin run on the B200 engine: every grid point trains for "
                      "min_episodes, the best 1/eta go on for eta times as many, and so on up to n_episodes")
    ap.add_argument("--min_episodes", type=int, required=True, help="the first rung's budget in episodes")
    ap.add_argument("--eta", type=int, default=3, help="keep the best 1/eta of the sets after each rung; budgets grow eta-fold")
    env_name, grid, outp, kw = parse_sweep_args(ap, argv)
    res = run_halving(env_name, grid, **kw)
    write_json(res, outp)
    return res
