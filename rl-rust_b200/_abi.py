"""ctypes binding of librlb.so — the C ABI declared in include/rlb.h.

The shared library holds the hand-written sm_100a kernels; there is no CPU fallback and no
other backend.  Importing this module without the built library raises ImportError: build
it first with `python -c "import __graft_entry__ as g; g.build()"` (or `make -C
rl-rust_b200/csrc`).
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RLB_LIB", os.path.join(_HERE, "librlb.so"))   # RLB_LIB: A/B a differently built library

OK, ERR_ENV_NOT_READY, ERR_INVALID_ARG, ERR_CUDA, ERR_OOM, ERR_UNSUPPORTED, ERR_NCCL = range(7)
MAP_4X4, MAP_8X8, MAP_CUSTOM = 0, 1, 2
COMM_ID_BYTES = 128
ENV_BLACKJACK, ENV_FROZEN_LAKE, ENV_CLIFF_WALKING, ENV_TAXI = range(4)
POLICY_BASIC, POLICY_DOUBLE = 0, 1
SEL_EPS_GREEDY, SEL_UCB = 0, 1
TARGET_SARSA, TARGET_QLEARNING, TARGET_EXPECTED_SARSA = 0, 1, 2
AGENT_ONE_STEP, AGENT_TRACES = 0, 1
REAL_F32, REAL_F64 = 0, 1
DECAY_SUB, DECAY_MUL = 0, 1


class RlbConfig(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("env_kind", C.c_int32), ("map_id", C.c_int32), ("slippery", C.c_int32),
        ("max_steps", C.c_uint32), ("policy_kind", C.c_int32), ("selector_kind", C.c_int32),
        ("target_kind", C.c_int32), ("agent_kind", C.c_int32), ("real_kind", C.c_int32), ("decay_kind", C.c_int32),
        ("device", C.c_int32),
        ("learning_rate", C.c_double), ("discount_factor", C.c_double), ("lambda_factor", C.c_double),
        ("initial_epsilon", C.c_double), ("epsilon_decay", C.c_double), ("final_epsilon", C.c_double),
        ("confidence_level", C.c_double), ("default_value", C.c_double),
        ("seed", C.c_uint64), ("n_agents", C.c_uint64), ("first_agent_id", C.c_uint64),
        ("store_kind", C.c_uint32), ("planning_steps", C.c_uint32),
        ("map_rows", C.c_uint32), ("map_cols", C.c_uint32), ("map", C.c_char_p),
    ]


class RlbTrainOut(C.Structure):
    _fields_ = [
        ("episode_sums", C.c_void_p), ("episodes", C.c_void_p), ("traj", C.c_void_p), ("traj_capacity", C.c_uint64),
        ("traj_count", C.c_void_p), ("train_steps", C.c_uint64), ("eval_steps", C.c_uint64),
        ("eval_return_sum", C.c_double), ("eval_episodes", C.c_uint64), ("kernel_ms", C.c_float),
        ("kernel_launches", C.c_uint32), ("trace_rows", C.c_uint64),
        ("td_steps", C.c_void_p), ("td_capacity", C.c_uint64), ("td_count", C.c_void_p),
    ]


EPISODE_F32 = np.dtype([("length", "<u4"), ("ret", "<f4"), ("td_sum", "<f4"), ("td_abs_sum", "<f4")])
EPISODE_F64 = np.dtype([("ret", "<f8"), ("td_sum", "<f8"), ("td_abs_sum", "<f8"), ("length", "<u4"), ("pad", "<u4")])
TRAJ_DTYPE = np.dtype([("kind", "u1"), ("action", "u1"), ("terminated", "u1"), ("pad", "u1"), ("obs", "<u4"),
                       ("reward", "<f8"), ("td", "<f8")])
STATE_DTYPE = np.dtype([("epsilon", "<f8"), ("ucb_t", "<u8"), ("rng_n", "<u8"), ("policy_flag", "<i4"),
                        ("env_ready", "<i4")])
MODEL_ENTRY = np.dtype([("obs", "<u4"), ("action", "<u4"), ("next_obs", "<u4"), ("reward", "<f4")])
# rlb_hparams: one per-agent hyper-parameter set (rlb_engine_set_hparams), field for field rlb_config's
HPARAM_FIELDS = ("learning_rate", "discount_factor", "lambda_factor", "initial_epsilon", "epsilon_decay", "final_epsilon",
                 "confidence_level", "default_value")
HPARAMS_DTYPE = np.dtype([(f, "<f8") for f in HPARAM_FIELDS])
MAX_HPARAM_SETS = 65536


class RlbHparams(C.Structure):
    _fields_ = [(f, C.c_double) for f in HPARAM_FIELDS]

# every symbol include/rlb.h declares
EXPORTS = [
    "rlb_abi_version", "rlb_last_error_string", "rlb_device_count", "rlb_engine_create", "rlb_engine_destroy",
    "rlb_engine_set_stream", "rlb_engine_synchronize", "rlb_engine_dims", "rlb_engine_store_kind", "rlb_env_reset",
    "rlb_env_step", "rlb_agent_get_action", "rlb_agent_update", "rlb_agent_set_future_q_value_func",
    "rlb_agent_set_action_selector", "rlb_agent_set_kind", "rlb_agent_set_model", "rlb_agent_reset", "rlb_agent_train", "rlb_agent_train_range",
    "rlb_agent_evaluate", "rlb_policy_predict", "rlb_policy_get_values", "rlb_policy_update",
    "rlb_policy_after_update", "rlb_policy_reset", "rlb_selector_get_action", "rlb_selector_get_exploration_probs",
    "rlb_selector_update", "rlb_selector_reset", "rlb_download_tables", "rlb_upload_tables", "rlb_get_agent_states",
    "rlb_set_agent_states", "rlb_philox4x32_10", "rlb_rng_words", "rlb_rng_uniform_f64", "rlb_rng_uniform_usize",
    "rlb_rng_card", "rlb_rng_gen_range", "rlb_model_add_info", "rlb_model_get_info", "rlb_model_reset", "rlb_model_capacity",
    "rlb_download_model", "rlb_upload_model", "rlb_blackjack_obs_id", "rlb_blackjack_dense_index", "rlb_blackjack_decode",
    "rlb_agent_train_range_async", "rlb_agent_train_wait", "rlb_agent_step",
    "rlb_comm_unique_id", "rlb_comm_init_rank", "rlb_comm_init_all", "rlb_comm_destroy", "rlb_comm_rank", "rlb_comm_world_size",
    "rlb_comm_gather_episode_sums", "rlb_comm_allreduce_sum", "rlb_comm_group_begin", "rlb_comm_group_end",
    "rlb_selftest_ucb_math", "rlb_engine_set_hparams", "rlb_engine_hparam_sets", "rlb_engine_retune_hparams", "rlb_agent_clone",
    "rlb_engine_set_active_sets", "rlb_engine_set_planning_steps", "rlb_engine_set_targets",
]


class RlbError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("librlb status %d: %s" % (status, message))
        self.status = status


class EnvNotReady(RlbError):
    """reference src/env.rs:16-17"""


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "rl-rust_b200: %s is missing — the CUDA extension is the product and there is no fallback; "
            "build it with `make -C rl-rust_b200/csrc` or __graft_entry__.build()" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, u64, u32, i32, dbl = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32, C.c_double
    P = C.POINTER
    L.rlb_abi_version.restype = C.c_int
    L.rlb_last_error_string.restype = C.c_char_p
    L.rlb_device_count.restype = C.c_int
    L.rlb_engine_create.restype = C.c_int
    L.rlb_engine_create.argtypes = [P(RlbConfig), P(vp)]
    L.rlb_engine_destroy.restype = None
    L.rlb_engine_destroy.argtypes = [vp]
    L.rlb_engine_set_stream.argtypes = [vp, vp]
    L.rlb_engine_synchronize.argtypes = [vp]
    L.rlb_engine_dims.argtypes = [vp, P(u32), P(u32), P(u32)]
    L.rlb_engine_store_kind.restype = u32
    L.rlb_engine_store_kind.argtypes = [vp]
    L.rlb_engine_set_hparams.argtypes = [vp, vp, u32, vp]
    L.rlb_engine_hparam_sets.restype = u32
    L.rlb_engine_hparam_sets.argtypes = [vp]
    L.rlb_engine_retune_hparams.argtypes = [vp, vp, u32]
    L.rlb_agent_clone.argtypes = [vp, vp, vp, u64]
    L.rlb_engine_set_active_sets.argtypes = [vp, vp, u32]
    L.rlb_engine_set_planning_steps.argtypes = [vp, vp, u32]
    L.rlb_engine_set_targets.argtypes = [vp, vp, u32]
    L.rlb_env_reset.argtypes = [vp, vp]
    L.rlb_env_step.argtypes = [vp, vp, vp, vp, vp, vp]
    L.rlb_agent_get_action.argtypes = [vp, vp, vp]
    L.rlb_agent_update.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.rlb_agent_set_future_q_value_func.argtypes = [vp, i32]
    L.rlb_agent_set_action_selector.argtypes = [vp, i32]
    L.rlb_agent_set_kind.argtypes = [vp, i32]
    L.rlb_agent_reset.argtypes = [vp]
    L.rlb_agent_set_model.argtypes = [vp, u32]
    L.rlb_model_add_info.argtypes = [vp, vp, vp, vp, vp]
    L.rlb_model_get_info.argtypes = [vp, vp, vp, vp, vp]
    L.rlb_model_reset.argtypes = [vp]
    L.rlb_model_capacity.restype = u32
    L.rlb_model_capacity.argtypes = [vp]
    L.rlb_download_model.argtypes = [vp, vp, vp]
    L.rlb_upload_model.argtypes = [vp, vp, vp]
    L.rlb_rng_gen_range.restype = u64
    L.rlb_rng_gen_range.argtypes = [u64, u64, P(u64), u64]
    L.rlb_agent_train.argtypes = [vp, u64, u64, P(RlbTrainOut)]
    L.rlb_agent_train_range.argtypes = [vp, u64, u64, u64, P(RlbTrainOut)]
    L.rlb_agent_evaluate.argtypes = [vp, u64, vp, vp, P(u64)]
    L.rlb_agent_train_range_async.argtypes = [vp, u64, u64, u64, P(RlbTrainOut)]
    L.rlb_agent_train_wait.argtypes = [vp]
    L.rlb_agent_step.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.rlb_comm_unique_id.argtypes = [vp]
    L.rlb_comm_init_rank.argtypes = [vp, i32, i32, i32, P(vp)]
    L.rlb_comm_init_all.argtypes = [P(i32), i32, P(vp)]
    L.rlb_comm_destroy.restype = None
    L.rlb_comm_destroy.argtypes = [vp]
    L.rlb_comm_rank.restype = i32
    L.rlb_comm_rank.argtypes = [vp]
    L.rlb_comm_world_size.restype = i32
    L.rlb_comm_world_size.argtypes = [vp]
    L.rlb_comm_gather_episode_sums.argtypes = [vp, vp, u64, vp, i32, vp]
    L.rlb_comm_allreduce_sum.argtypes = [vp, vp, u64, vp]
    L.rlb_comm_group_begin.argtypes = []
    L.rlb_comm_group_end.argtypes = []
    L.rlb_selftest_ucb_math.argtypes = [i32, u64, u64, u64, u64, P(u64)]
    L.rlb_policy_predict.argtypes = [vp, vp, vp]
    L.rlb_policy_get_values.argtypes = [vp, vp, vp]
    L.rlb_policy_update.argtypes = [vp, vp, vp, vp, vp]
    L.rlb_policy_after_update.argtypes = [vp]
    L.rlb_policy_reset.argtypes = [vp]
    L.rlb_selector_get_action.argtypes = [vp, vp, vp, vp]
    L.rlb_selector_get_exploration_probs.argtypes = [vp, vp, vp, vp]
    L.rlb_selector_update.argtypes = [vp]
    L.rlb_selector_reset.argtypes = [vp]
    L.rlb_download_tables.argtypes = [vp, vp, vp]
    L.rlb_upload_tables.argtypes = [vp, vp, vp]
    L.rlb_get_agent_states.argtypes = [vp, vp]
    L.rlb_set_agent_states.argtypes = [vp, vp]
    L.rlb_philox4x32_10.restype = None
    L.rlb_philox4x32_10.argtypes = [vp, vp, vp]
    L.rlb_rng_words.restype = None
    L.rlb_rng_words.argtypes = [u64, u64, u64, u64, vp]
    L.rlb_rng_uniform_f64.restype = dbl
    L.rlb_rng_uniform_f64.argtypes = [u64, u64, P(u64)]
    L.rlb_rng_uniform_usize.restype = u64
    L.rlb_rng_uniform_usize.argtypes = [u64, u64, P(u64), u64]
    L.rlb_rng_card.restype = u32
    L.rlb_rng_card.argtypes = [u64, u64, P(u64)]
    L.rlb_blackjack_obs_id.restype = u64
    L.rlb_blackjack_obs_id.argtypes = [u32]
    L.rlb_blackjack_dense_index.restype = u32
    L.rlb_blackjack_dense_index.argtypes = [u64]
    L.rlb_blackjack_decode.restype = None
    L.rlb_blackjack_decode.argtypes = [u32, P(u32), P(u32), P(u32)]
    return L


lib = _load()


def check(status):
    if status != OK:
        msg = lib.rlb_last_error_string().decode("utf-8", "replace")
        raise (EnvNotReady if status == ERR_ENV_NOT_READY else RlbError)(status, msg)


def ptr(buf):
    """Raw address of a numpy array, a torch tensor (host or CUDA) or None."""
    if buf is None:
        return None
    if isinstance(buf, np.ndarray):
        assert buf.flags["C_CONTIGUOUS"]
        return buf.ctypes.data
    if hasattr(buf, "data_ptr"):
        assert buf.is_contiguous()
        return buf.data_ptr()
    raise TypeError("expected numpy array or torch tensor, got %r" % type(buf))


class Engine:
    """N agent+environment pairs on one GPU: a thin object over the C ABI.

    Keyword arguments are the reference constructors' arguments (see rlb_config in
    include/rlb.h); defaults are the reference CLI's (src/bin/taxi.rs:22-68 with
    n_episodes = 100000, i.e. epsilon_decay = 1.0 / (0.5 * 100000)).
    """

    def __init__(self, env_kind, *, n_agents=1, map_id=1, slippery=False, max_steps=100, policy=POLICY_BASIC,
                 selector=SEL_EPS_GREEDY, target=TARGET_QLEARNING, agent=AGENT_ONE_STEP, real=REAL_F32,
                 decay_kind=DECAY_SUB, learning_rate=0.05, discount_factor=0.95, lambda_factor=0.5,
                 initial_epsilon=1.0, epsilon_decay=2e-5, final_epsilon=0.0, confidence_level=0.5, default_value=0.0,
                 seed=0x5EED0001, first_agent_id=0, device=0, store_kind=0, planning_steps=0, map_rows=None):
        # map_rows: FrozenLakeEnv::new's `map: &[&str]` (frozen_lake.rs:48) — a list of equally long strings of S/F/H/G
        rows, cols, flat = 0, 0, None
        if map_rows is not None:
            map_rows = [str(r) for r in map_rows]
            if not map_rows or any(len(r) != len(map_rows[0]) for r in map_rows):
                raise ValueError("map rows must be non-empty and equally long")
            rows, cols, flat, map_id = len(map_rows), len(map_rows[0]), "".join(map_rows).encode("ascii"), MAP_CUSTOM
        self.cfg = RlbConfig(C.sizeof(RlbConfig), env_kind, map_id, int(bool(slippery)), max_steps, policy, selector,
                             target, agent, real, decay_kind, device, learning_rate, discount_factor, lambda_factor,
                             initial_epsilon, epsilon_decay, final_epsilon, confidence_level, default_value, seed,
                             n_agents, first_agent_id, store_kind, planning_steps, rows, cols, flat)
        self.h = C.c_void_p()
        check(lib.rlb_engine_create(C.byref(self.cfg), C.byref(self.h)))
        s, a, t = C.c_uint32(), C.c_uint32(), C.c_uint32()
        check(lib.rlb_engine_dims(self.h, C.byref(s), C.byref(a), C.byref(t)))
        self.S, self.A, self.T, self.N = s.value, a.value, t.value, n_agents
        self.seed, self.first_agent_id = int(seed), int(first_agent_id)
        self.real = real
        self.rdtype = np.float32 if real == REAL_F32 else np.float64
        self.episode_dtype = EPISODE_F32 if real == REAL_F32 else EPISODE_F64
        self.G = 0                  # hyper-parameter sets installed (set_hparams); per-episode sums are (E, G, 4) while G > 0
        self.hparams = None         # (sets, group) as installed
        self.active_sets = None     # bool (G,) while some set is paused (set_active_sets), else None
        self.planning = None        # uint32 (G,) per-set Dyna planning counts (set_planning_steps), else None
        self.targets = None         # int32 (G,) per-set targets while they differ from cfg.target_kind (set_targets), else None

    def close(self):
        if getattr(self, "h", None):
            lib.rlb_engine_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- plumbing
    def set_stream(self, cuda_stream):
        check(lib.rlb_engine_set_stream(self.h, C.c_void_p(cuda_stream)))

    def synchronize(self):
        check(lib.rlb_engine_synchronize(self.h))

    def store_kind(self):
        """Which table store the fused kernel runs with: 1 HBM, 2 shared-memory thread groups, 3 hybrid, 4 HBM with a trace
        agent's sweeps applied lazily (rlb.h: rlb_config.store_kind)."""
        return lib.rlb_engine_store_kind(self.h)

    # ---- per-agent hyper-parameter sets
    def hparams_array(self, sets):
        """`sets` as an HPARAMS_DTYPE array: an array of that dtype as it is, or a list of dicts whose missing fields take
        this engine's rlb_config values."""
        if isinstance(sets, np.ndarray) and sets.dtype == HPARAMS_DTYPE:
            return np.ascontiguousarray(sets)
        arr = np.zeros(len(sets), HPARAMS_DTYPE)
        for g, d in enumerate(sets):
            unknown = set(d) - set(HPARAM_FIELDS)
            if unknown:
                raise ValueError("unknown hyper-parameter(s) %s; known: %s" % (sorted(unknown), ", ".join(HPARAM_FIELDS)))
            for f in HPARAM_FIELDS:
                arr[g][f] = float(d.get(f, getattr(self.cfg, f)))
        return arr

    def set_hparams(self, sets, group):
        """rlb_engine_set_hparams: agent i is constructed with sets[group[i]] (fresh tables, epsilon and UCB state; see
        include/rlb.h).  `sets`: a list of dicts (fields missing from a dict take the engine's configured value) or an
        HPARAMS_DTYPE array; `group`: (N,) integers.  set_hparams(None, None) goes back to the configured values.
        While sets are installed, train() and evaluate() return per-episode sums shaped (E, G, 4)."""
        if sets is None and group is None:
            check(lib.rlb_engine_set_hparams(self.h, None, 0, None))
            self.G, self.hparams, self.active_sets, self.planning, self.targets = 0, None, None, None, None
            return
        arr = self.hparams_array(sets)
        grp = np.asarray(group)
        if grp.shape != (self.N,):
            raise ValueError("group must have shape (%d,), got %r" % (self.N, grp.shape))
        if grp.size and (grp.min() < 0 or grp.max() >= 2 ** 32):
            raise ValueError("group ids must be in [0, 2**32)")
        grp = np.ascontiguousarray(grp, np.uint32)
        check(lib.rlb_engine_set_hparams(self.h, ptr(arr) if len(arr) else None, len(arr), ptr(grp) if len(arr) else None))
        self.G, self.hparams, self.active_sets, self.planning, self.targets = len(arr), (arr.copy(), grp.copy()), None, None, None

    def hparam_sets(self):
        """rlb_engine_hparam_sets: the number of sets installed, 0 while the configured values apply."""
        return lib.rlb_engine_hparam_sets(self.h)

    def retune_hparams(self, sets):
        """rlb_engine_retune_hparams: sets[g] becomes the values of installed set g from the next call on, the learned
        state left alone (initial_epsilon and default_value take effect at the next reset; see include/rlb.h).  `sets` as
        for set_hparams, one per installed set.  `hparams` then holds the new values, so snapshots record them."""
        arr = self.hparams_array(sets)
        check(lib.rlb_engine_retune_hparams(self.h, ptr(arr) if len(arr) else None, len(arr)))
        self.hparams = (arr.copy(), self.hparams[1])

    def set_active_sets(self, mask):
        """rlb_engine_set_active_sets: only the sets whose entry of `mask` ((G,) bools) is true take part in later train()
        and evaluate() calls; the other sets' agents are left exactly as they are, and their rows of the sums are 0.
        mask=None makes every set active.  Every other call still acts on all agents (see include/rlb.h).
        `active_sets` then holds the mask, or None while every set is active."""
        if mask is None:
            check(lib.rlb_engine_set_active_sets(self.h, None, 0))
            self.active_sets = None
            return
        m = np.asarray(mask)
        if m.shape != (self.G,):
            raise ValueError("mask must have shape (%d,), got %r" % (self.G, m.shape))
        m = np.ascontiguousarray(m != 0, np.uint8)
        check(lib.rlb_engine_set_active_sets(self.h, ptr(m) if len(m) else None, len(m)))
        self.active_sets = None if m.all() else m.astype(bool)

    def set_planning_steps(self, steps):
        """rlb_engine_set_planning_steps: the agents of set g become Dyna-Q agents making steps[g] planning replays per real
        update ((G,) non-negative integers; 0 allowed).  The first call wraps every agent as it is around an empty model; a
        later one changes only the counts.  steps=None drops the model (as set_model(0)).  `planning` then holds the
        counts, or None (see include/rlb.h)."""
        if steps is None:
            check(lib.rlb_engine_set_planning_steps(self.h, None, 0))
            self.cfg.planning_steps, self.planning = 0, None
            return
        k = np.asarray(steps)
        if k.shape != (self.G,):
            raise ValueError("steps must have shape (%d,), got %r" % (self.G, k.shape))
        if k.size and (k.dtype.kind not in "iu" or k.min() < 0 or k.max() >= 2 ** 32):
            raise ValueError("planning steps must be integers in [0, 2**32)")
        k = np.ascontiguousarray(k, np.uint32)
        check(lib.rlb_engine_set_planning_steps(self.h, ptr(k) if len(k) else None, len(k)))
        self.cfg.planning_steps, self.planning = max(1, int(k.max())), k.copy()

    def set_targets(self, kinds):
        """rlb_engine_set_targets: the agents of set g bootstrap with target kinds[g] ((G,) TARGET_* integers) in every
        later update; tables and agent states stay as they are.  `targets` then holds the targets, or None while every
        set has cfg.target_kind (see include/rlb.h).  set_hparams and set_target put every set back on the engine's."""
        k = np.asarray(kinds)
        if k.shape != (self.G,):
            raise ValueError("targets must have shape (%d,), got %r" % (self.G, k.shape))
        if k.size and (k.dtype.kind not in "iu" or k.min() < TARGET_SARSA or k.max() > TARGET_EXPECTED_SARSA):
            raise ValueError("targets must be integers in [%d, %d]" % (TARGET_SARSA, TARGET_EXPECTED_SARSA))
        k = np.ascontiguousarray(k, np.int32)
        check(lib.rlb_engine_set_targets(self.h, ptr(k) if len(k) else None, len(k)))
        self.targets = None if (k == self.cfg.target_kind).all() else k.copy()

    # ---- population-based training: the exploit step
    def clone_agents(self, src, dst):
        """rlb_agent_clone: agent dst[j] takes the learned state (tables, counts, epsilon, UCB t, Double flag, model) of
        agent src[j]; it keeps its RNG stream, env and hyper-parameter set.  Complete at an episode boundary.  No id may be
        both a source and a destination, and no destination may appear twice."""
        ids = []
        for a in (src, dst):
            a = np.asarray(a)
            if a.ndim != 1 or (a.size and (a.min() < 0 or a.max() >= 2 ** 32)):
                raise ValueError("agent ids must be a 1-d array of integers in [0, 2**32)")
            ids.append(np.ascontiguousarray(a, np.uint32))
        if len(ids[0]) != len(ids[1]):
            raise ValueError("src and dst must have the same length")
        check(lib.rlb_agent_clone(self.h, ptr(ids[0]), ptr(ids[1]), len(ids[0])))

    def _sums_shape(self, n):
        return (n, self.G, 4) if self.G else (n, 4)

    # ---- Agent::train / evaluate
    def train(self, n_episodes, eval_at, *, ep_begin=0, sums=True, episodes=False, traj_capacity=0, sums_out=None,
              episodes_out=None, td_capacity=0, wait=True):
        """Agent::train (agent.rs:66-118), episodes [ep_begin, n_episodes).  Returns a dict.
        td_capacity > 0 also returns `training_error` (agent.rs:98,117): res["td_steps"] [N, td_capacity] and
        res["td_count"] [N] (steps taken; the first min(count, capacity) TDs of each agent are stored).
        wait=False enqueues the call and returns (rlb_agent_train_range_async); the scalar results are filled in
        by train_wait(), which returns the same dict."""
        n = n_episodes - ep_begin
        out = RlbTrainOut()
        res = {}
        if sums_out is not None:
            out.episode_sums = ptr(sums_out)
            res["sums"] = sums_out
        elif sums:
            res["sums"] = np.zeros(self._sums_shape(n), np.float64)
            out.episode_sums = ptr(res["sums"])
        if episodes_out is not None:
            out.episodes = ptr(episodes_out)
            res["episodes"] = episodes_out
        elif episodes:
            res["episodes"] = np.zeros((n, self.N), self.episode_dtype)
            out.episodes = ptr(res["episodes"])
        if traj_capacity:
            res["traj"] = np.zeros((self.N, traj_capacity), TRAJ_DTYPE)
            res["traj_count"] = np.zeros(self.N, np.uint64)
            out.traj = ptr(res["traj"])
            out.traj_capacity = traj_capacity
            out.traj_count = ptr(res["traj_count"])
        if td_capacity:
            res["td_steps"] = np.zeros((self.N, td_capacity), self.rdtype)
            res["td_count"] = np.zeros(self.N, np.uint64)
            out.td_steps = ptr(res["td_steps"])
            out.td_capacity = td_capacity
            out.td_count = ptr(res["td_count"])
        if not wait:
            self._pending = getattr(self, "_pending", [])
            self._pending.append((out, res))       # keeps `out` and the buffers alive until train_wait()
            check(lib.rlb_agent_train_range_async(self.h, ep_begin, n_episodes, eval_at, C.byref(out)))
            return res
        check(lib.rlb_agent_train_range(self.h, ep_begin, n_episodes, eval_at, C.byref(out)))
        self._fill(out, res)
        return res

    @staticmethod
    def _fill(out, res):
        res.update(train_steps=out.train_steps, eval_steps=out.eval_steps, eval_return_sum=out.eval_return_sum,
                   eval_episodes=out.eval_episodes, kernel_ms=out.kernel_ms, kernel_launches=out.kernel_launches,
                   trace_rows=out.trace_rows)

    def train_wait(self):
        """rlb_agent_train_wait: complete every train(wait=False) call; returns their result dicts, oldest first."""
        check(lib.rlb_agent_train_wait(self.h))
        done = []
        for out, res in getattr(self, "_pending", []):
            self._fill(out, res)
            done.append(res)
        self._pending = []
        return done

    def agent_step(self):
        """rlb_agent_step: one iteration of the loop at agent.rs:83-106 for every agent, one launch."""
        kind, term = np.zeros(self.N, np.uint8), np.zeros(self.N, np.uint8)
        obs, act = np.zeros(self.N, np.uint32), np.zeros(self.N, np.uint32)
        rew, td = np.zeros(self.N, np.float64), np.zeros(self.N, self.rdtype)
        check(lib.rlb_agent_step(self.h, ptr(kind), ptr(obs), ptr(act), ptr(rew), ptr(term), ptr(td)))
        return dict(kind=kind, obs=obs, action=act, reward=rew, terminated=term.astype(bool), td=td)

    def evaluate(self, n_episodes, *, sums=True, episodes=False):
        """Agent::evaluate (agent.rs:120-141)."""
        res = {}
        sums_buf = np.zeros(self._sums_shape(n_episodes), np.float64) if sums else None
        eps_buf = np.zeros((n_episodes, self.N), self.episode_dtype) if episodes else None
        steps = C.c_uint64()
        check(lib.rlb_agent_evaluate(self.h, n_episodes, ptr(eps_buf), ptr(sums_buf), C.byref(steps)))
        res["sums"], res["episodes"], res["steps"] = sums_buf, eps_buf, steps.value
        return res

    def set_target(self, kind):
        check(lib.rlb_agent_set_future_q_value_func(self.h, kind))
        self.cfg.target_kind = kind
        self.targets = None

    def set_selector(self, kind):
        check(lib.rlb_agent_set_action_selector(self.h, kind))
        self.cfg.selector_kind = kind

    def set_agent_kind(self, kind):
        check(lib.rlb_agent_set_kind(self.h, kind))
        self.cfg.agent_kind = kind

    def agent_reset(self):
        check(lib.rlb_agent_reset(self.h))

    # ---- InternalModelAgent / Model (agent/internal_model_agent.rs, model/random_model.rs)
    def set_model(self, planning_steps):
        check(lib.rlb_agent_set_model(self.h, planning_steps))
        self.cfg.planning_steps = planning_steps
        if not planning_steps:
            self.planning = None

    def model_add_info(self, obs, action, reward, next_obs):
        obs, action, next_obs = (np.ascontiguousarray(x, np.uint32) for x in (obs, action, next_obs))
        reward = np.ascontiguousarray(reward, np.float64)
        check(lib.rlb_model_add_info(self.h, ptr(obs), ptr(action), ptr(reward), ptr(next_obs)))

    def model_get_info(self):
        obs, action, next_obs = (np.zeros(self.N, np.uint32) for _ in range(3))
        reward = np.zeros(self.N, np.float64)
        check(lib.rlb_model_get_info(self.h, ptr(obs), ptr(action), ptr(next_obs), ptr(reward)))
        return obs, action, next_obs, reward

    def model_reset(self):
        check(lib.rlb_model_reset(self.h))

    def download_model(self):
        """(len [N], entries [N][capacity]) — each agent's remembered transitions in insertion order."""
        cap = lib.rlb_model_capacity(self.h)
        ln = np.zeros(self.N, np.uint32)
        ent = np.zeros((self.N, cap), MODEL_ENTRY)
        check(lib.rlb_download_model(self.h, ptr(ln), ptr(ent)))
        return ln, ent

    def upload_model(self, ln, ent):
        ln = np.ascontiguousarray(ln, np.uint32)
        ent = np.ascontiguousarray(ent, MODEL_ENTRY)
        check(lib.rlb_upload_model(self.h, ptr(ln), ptr(ent)))

    # ---- snapshots
    def download_tables(self, counts=True):
        q = np.zeros((self.N, self.T, self.S, self.A), self.rdtype)
        c = np.zeros((self.N, self.S, self.A), np.uint32) if counts else None
        check(lib.rlb_download_tables(self.h, ptr(q), ptr(c)))
        return q, c

    def upload_tables(self, q=None, counts=None):
        if q is not None:
            q = np.ascontiguousarray(q, self.rdtype)
        if counts is not None:
            counts = np.ascontiguousarray(counts, np.uint32)
        check(lib.rlb_upload_tables(self.h, ptr(q), ptr(counts)))

    def states(self):
        st = np.zeros(self.N, STATE_DTYPE)
        check(lib.rlb_get_agent_states(self.h, ptr(st)))
        return st

    def set_states(self, st):
        st = np.ascontiguousarray(st, STATE_DTYPE)
        check(lib.rlb_set_agent_states(self.h, ptr(st)))

    # ---- step-level trait methods
    def env_reset(self):
        obs = np.zeros(self.N, np.uint32)
        check(lib.rlb_env_reset(self.h, ptr(obs)))
        return obs

    def env_step(self, actions):
        actions = np.ascontiguousarray(actions, np.uint32)
        obs = np.zeros(self.N, np.uint32)
        rew = np.zeros(self.N, np.float64)
        term = np.zeros(self.N, np.uint8)
        nr = np.zeros(self.N, np.uint8)
        st = lib.rlb_env_step(self.h, ptr(actions), ptr(obs), ptr(rew), ptr(term), ptr(nr))
        if st == ERR_ENV_NOT_READY:
            raise EnvNotReady(st, lib.rlb_last_error_string().decode())
        check(st)
        return obs, rew, term.astype(bool)

    def get_action(self, obs):
        obs = np.ascontiguousarray(obs, np.uint32)
        act = np.zeros(self.N, np.uint32)
        check(lib.rlb_agent_get_action(self.h, ptr(obs), ptr(act)))
        return act

    def update(self, curr_obs, curr_action, reward, terminated, next_obs, next_action):
        a = [np.ascontiguousarray(curr_obs, np.uint32), np.ascontiguousarray(curr_action, np.uint32),
             np.ascontiguousarray(reward, np.float64), np.ascontiguousarray(terminated, np.uint8),
             np.ascontiguousarray(next_obs, np.uint32), np.ascontiguousarray(next_action, np.uint32)]
        td = np.zeros(self.N, self.rdtype)
        check(lib.rlb_agent_update(self.h, *[ptr(x) for x in a], ptr(td)))
        return td

    def policy_predict(self, obs):
        obs = np.ascontiguousarray(obs, np.uint32)
        v = np.zeros((self.N, self.A), self.rdtype)
        check(lib.rlb_policy_predict(self.h, ptr(obs), ptr(v)))
        return v

    def policy_get_values(self, obs):
        obs = np.ascontiguousarray(obs, np.uint32)
        v = np.zeros((self.N, self.A), self.rdtype)
        check(lib.rlb_policy_get_values(self.h, ptr(obs), ptr(v)))
        return v

    def policy_update(self, obs, action, next_obs, td):
        a = [np.ascontiguousarray(obs, np.uint32), np.ascontiguousarray(action, np.uint32),
             np.ascontiguousarray(next_obs, np.uint32), np.ascontiguousarray(td, self.rdtype)]
        check(lib.rlb_policy_update(self.h, *[ptr(x) for x in a]))

    def policy_after_update(self):
        check(lib.rlb_policy_after_update(self.h))

    def policy_reset(self):
        check(lib.rlb_policy_reset(self.h))

    def selector_get_action(self, obs, values):
        obs = np.ascontiguousarray(obs, np.uint32)
        values = np.ascontiguousarray(values, self.rdtype)
        act = np.zeros(self.N, np.uint32)
        check(lib.rlb_selector_get_action(self.h, ptr(obs), ptr(values), ptr(act)))
        return act

    def selector_get_exploration_probs(self, obs, values):
        obs = np.ascontiguousarray(obs, np.uint32)
        values = np.ascontiguousarray(values, self.rdtype)
        pr = np.zeros((self.N, self.A), self.rdtype)
        check(lib.rlb_selector_get_exploration_probs(self.h, ptr(obs), ptr(values), ptr(pr)))
        return pr

    def selector_update(self):
        check(lib.rlb_selector_update(self.h))

    def selector_reset(self):
        check(lib.rlb_selector_reset(self.h))


# ---- host-callable RNG contract and Blackjack ids (no device needed)
def philox4x32_10(ctr, key):
    c = np.ascontiguousarray(ctr, np.uint32)
    k = np.ascontiguousarray(key, np.uint32)
    out = np.zeros(4, np.uint32)
    lib.rlb_philox4x32_10(ptr(c), ptr(k), ptr(out))
    return out


def rng_words(seed, agent_id, first_word, count):
    out = np.zeros(count, np.uint32)
    lib.rlb_rng_words(seed, agent_id, first_word, count, ptr(out))
    return out


def blackjack_obs_id(dense_index):
    return lib.rlb_blackjack_obs_id(dense_index)


def blackjack_dense_index(obs_id):
    return lib.rlb_blackjack_dense_index(obs_id)


def _nccl_load_order():
    """librlb resolves NCCL at run time with dlopen("libnccl.so.2").  PyTorch links a NEWER NCCL under the same soname:
    if librlb's copy (the system's) is loaded first, a later `import torch` binds to it and fails on the symbols it lacks.
    So, where PyTorch is installed, import it BEFORE the first rlb_comm_* call — the loader then hands librlb the copy
    PyTorch brought.  A host without PyTorch (a Rust binary) has a single NCCL and no ordering to mind."""
    try:
        import torch  # noqa: F401
    except ImportError:
        pass


class Comm:
    """rlb_comm: the path's one multi-GPU exchange (NCCL send/recv gather of the per-episode metric sums)."""

    def __init__(self, handle):
        self.h = handle

    @staticmethod
    def unique_id():
        _nccl_load_order()
        buf = (C.c_uint8 * COMM_ID_BYTES)()
        check(lib.rlb_comm_unique_id(buf))
        return bytes(buf)

    @classmethod
    def init_rank(cls, unique_id, world_size, rank, device):
        _nccl_load_order()
        buf = (C.c_uint8 * COMM_ID_BYTES).from_buffer_copy(unique_id)
        h = C.c_void_p()
        check(lib.rlb_comm_init_rank(buf, world_size, rank, device, C.byref(h)))
        return cls(h)

    @classmethod
    def init_all(cls, devices):
        _nccl_load_order()
        devs = (C.c_int32 * len(devices))(*devices)
        hs = (C.c_void_p * len(devices))()
        check(lib.rlb_comm_init_all(devs, len(devices), hs))
        return [cls(C.c_void_p(h)) for h in hs]

    @property
    def rank(self):
        return lib.rlb_comm_rank(self.h)

    @property
    def world_size(self):
        return lib.rlb_comm_world_size(self.h)

    def gather_episode_sums(self, local_sums, gathered=None, root=0, stream=None):
        """local_sums: CUDA f64 [E,4]; gathered: CUDA f64 [world,E,4] on the root."""
        check(lib.rlb_comm_gather_episode_sums(self.h, ptr(local_sums), local_sums.shape[0], ptr(gathered), root,
                                               C.c_void_p(stream) if stream else None))
        return gathered

    def allreduce_sum(self, values, stream=None):
        check(lib.rlb_comm_allreduce_sum(self.h, ptr(values), values.numel(), C.c_void_p(stream) if stream else None))
        return values

    def close(self):
        if getattr(self, "h", None):
            lib.rlb_comm_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()
