"""Snapshot / resume of an engine at an episode boundary ("next" row N3; the reference has no checkpointing at all).
The complete state is: Q tables, UCB counts, and per agent the RNG word index, epsilon, UCB t and Double flag
(rlb_download_tables / rlb_get_agent_states), plus the Dyna model when one is attached (rlb_download_model) and the
per-agent hyper-parameter sets when they are installed (rlb_engine_set_hparams), with the active-set mask while some
set is paused (rlb_engine_set_active_sets), the per-set planning counts while they are in force
(rlb_engine_set_planning_steps) and the per-set targets while they are (rlb_engine_set_targets).  Stored as one .npz; the configuration
is stored beside it and checked."""
import ctypes as C

import numpy as np

_CFG_FIELDS = ("env_kind", "map_id", "slippery", "max_steps", "policy_kind", "real_kind", "n_agents", "first_agent_id", "seed")


def save_snapshot(engine, path):
    planning = int(engine.cfg.planning_steps)
    if planning and int(engine.cfg.agent_kind) == 1:
        # planning updates run with terminated = false and leave eligibility rows behind at episode boundaries
        raise NotImplementedError("snapshots of an eligibility-trace agent under a Dyna model are not supported")
    extra = {}
    if planning:
        extra["model_len"], extra["model"] = engine.download_model()
        if engine.planning is not None:
            extra["hp_planning"] = np.asarray(engine.planning, np.uint32)
    if engine.hparams is not None:
        extra["hp_sets"], extra["hp_group"] = engine.hparams
        if engine.active_sets is not None:
            extra["hp_active"] = np.asarray(engine.active_sets, np.uint8)
        if engine.targets is not None:
            extra["hp_target"] = np.asarray(engine.targets, np.int32)
    q, counts = engine.download_tables()
    cfg = {k: int(getattr(engine.cfg, k)) for k in _CFG_FIELDS}
    np.savez_compressed(path, q=q, counts=counts, states=engine.states(), selector_kind=np.int64(engine.cfg.selector_kind),
                        planning_steps=np.int64(planning), **extra,
                        **{"cfg_" + k: np.int64(v) if k != "seed" else np.uint64(v) for k, v in cfg.items()})


def load_snapshot(engine, path):
    z = np.load(path)
    for k in _CFG_FIELDS:
        if int(z["cfg_" + k]) != int(getattr(engine.cfg, k)):
            raise ValueError("snapshot was taken with %s = %d, engine has %d" % (k, int(z["cfg_" + k]), int(getattr(engine.cfg, k))))
    if int(z["selector_kind"]) != int(engine.cfg.selector_kind):
        engine.set_selector(int(z["selector_kind"]))
    # the sets before the tables and states: installing them refills both with each agent's constructor values
    if "hp_sets" in z.files:
        if "hp_planning" in z.files and int(engine.cfg.planning_steps):
            engine.set_model(0)   # sets are installed without a model; the counts attach it again below
        engine.set_hparams(z["hp_sets"], z["hp_group"])
    elif engine.G:
        engine.set_hparams(None, None)
    has_counts = int(z["selector_kind"]) == 1
    engine.upload_tables(z["q"], z["counts"] if has_counts else None)
    engine.set_states(z["states"])
    planning = int(z["planning_steps"]) if "planning_steps" in z.files else 0
    if "hp_planning" in z.files:
        engine.set_planning_steps(z["hp_planning"])
    elif planning != int(engine.cfg.planning_steps):
        engine.set_model(planning)
    if planning:
        engine.upload_model(z["model_len"], z["model"])
    if "hp_target" in z.files:
        engine.set_targets(z["hp_target"])
    if "hp_active" in z.files:
        engine.set_active_sets(z["hp_active"])
