/* include/rlb.h — C ABI of the B200 batched tabular-RL engine (librlb.so).
 *
 * This is the drop-in boundary for the hot path of JohnVithor/RL-Rust: the body of
 * `Agent::train` (src/agent.rs:66-118) and everything it calls — `Env::{reset,step}`,
 * `Agent::{get_action,update}`, `Policy::{predict,get_values,update,after_update}`,
 * `ActionSelection::{get_action,get_exploration_probs,update}` — for N independent
 * agent+environment pairs at once.  The reference has no FFI of its own; its boundary is
 * the Rust trait surface, so there is one C entry point per trait method, batched over the
 * engine's N agents (N = 1 reproduces the reference's single trait object).  Each function
 * below cites the reference item it replaces (paths under the reference's `src/`).
 * INTEGRATION.md shows the Rust `extern "C"` shim that binds these.
 *
 * Conventions
 *  - Every call returns rlb_status; nothing aborts.  rlb_last_error_string() describes
 *    the last failure on the calling thread.
 *  - Observations are dense u32 state indices on this side of the ABI.  For Blackjack the
 *    reference's ids are fxhash values (env/blackjack.rs:25-27); rlb_blackjack_obs_id()
 *    / rlb_blackjack_dense_index() convert.
 *  - `Real` is the engine's arithmetic type, chosen in rlb_config.real: f64 is the
 *    reference's own type (bit-faithful mode), f32 the fast mode.  Buffers typed `void*`
 *    below hold `Real` elements.
 *  - Buffer arguments may be HOST or DEVICE pointers (detected with
 *    cudaPointerGetAttributes); host buffers are staged through pinned memory.
 *  - One engine = one CUDA device + one stream.  Calls on one engine are not re-entrant;
 *    different engines may be driven from different host threads.
 *  - No CPU fallback exists: without a CUDA device every compute entry point fails with
 *    RLB_ERR_CUDA.
 */
#ifndef RLB_H
#define RLB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RLB_ABI_VERSION 2

typedef struct rlb_engine rlb_engine;

typedef enum rlb_status {
    RLB_OK = 0,
    RLB_ERR_ENV_NOT_READY = 1, /* env.rs:16-17 EnvNotReady: step before reset / after termination */
    RLB_ERR_INVALID_ARG = 2,   /* includes eval_at == 0 (agent.rs:107 divides by it) */
    RLB_ERR_CUDA = 3,
    RLB_ERR_OOM = 4,
    RLB_ERR_UNSUPPORTED = 5,
    RLB_ERR_NCCL = 6           /* a NCCL call failed, or libnccl.so.2 could not be loaded (rlb_comm_*) */
} rlb_status;

typedef enum rlb_env_kind {      /* env.rs:9-14 */
    RLB_ENV_BLACKJACK = 0,       /* env/blackjack.rs  Env<usize,2>, 1456 dense obs */
    RLB_ENV_FROZEN_LAKE = 1,     /* env/frozen_lake.rs Env<usize,4>, 16 or 64 states */
    RLB_ENV_CLIFF_WALKING = 2,   /* env/cliff_walking.rs Env<usize,4>, 48 states */
    RLB_ENV_TAXI = 3             /* env/taxi.rs Env<usize,6>, 500 states */
} rlb_env_kind;

typedef enum rlb_policy_kind {   /* policy.rs:27-33 EnumPolicy */
    RLB_POLICY_BASIC = 0,        /* policy/tabular_policy.rs TabularPolicy */
    RLB_POLICY_DOUBLE = 1        /* policy/double_tabular_policy.rs DoubleTabularPolicy */
} rlb_policy_kind;

typedef enum rlb_selector_kind { /* action_selection.rs:17-22 EnumActionSelection */
    RLB_SEL_EPS_GREEDY = 0,      /* action_selection/uniform_epsilon_greed.rs */
    RLB_SEL_UCB = 1              /* action_selection/upper_confidence_bound.rs */
} rlb_selector_kind;

typedef enum rlb_target_kind {   /* agent.rs:17 GetNextQValue */
    RLB_TARGET_SARSA = 0,            /* agent.rs:19-25 */
    RLB_TARGET_QLEARNING = 1,        /* agent.rs:27-33 */
    RLB_TARGET_EXPECTED_SARSA = 2    /* agent.rs:35-45 */
} rlb_target_kind;

typedef enum rlb_agent_kind {
    RLB_AGENT_ONE_STEP = 0,      /* agent/one_step_agent.rs OneStepAgent */
    RLB_AGENT_TRACES = 1         /* agent/elegibility_traces_agent.rs ElegibilityTracesAgent */
} rlb_agent_kind;

typedef enum rlb_real_kind { RLB_REAL_F32 = 0, RLB_REAL_F64 = 1 } rlb_real_kind;

/* The `Rc<dyn Fn(f64)->f64>` epsilon_decay closure (uniform_epsilon_greed.rs:14,31) cannot
 * cross to the device; the bins only ever pass `a - k` (bin/taxi.rs:132) or `a * k`
 * (bin/frozen_lake_neural.rs:181). */
typedef enum rlb_decay_kind { RLB_DECAY_SUB = 0, RLB_DECAY_MUL = 1 } rlb_decay_kind;

/* Constructor arguments of the reference objects, gathered in one struct:
 *   env:      BlackJackEnv::new() blackjack.rs:45 | FrozenLakeEnv::new(map,is_slippery,max_steps)
 *             frozen_lake.rs:48 | CliffWalkingEnv::new(max_steps) cliff_walking.rs:31 |
 *             TaxiEnv::new(max_steps) taxi.rs:57
 *   policy:   TabularPolicy::new(lr, default) tabular_policy.rs:15 |
 *             DoubleTabularPolicy::new(lr, default) double_tabular_policy.rs:17
 *   selector: UniformEpsilonGreed::new(eps, decay, final) uniform_epsilon_greed.rs:31 |
 *             UpperConfidenceBound::new(c) upper_confidence_bound.rs:17
 *   agent:    OneStepAgent::new(policy, gamma, selector, f) one_step_agent.rs:16 |
 *             ElegibilityTracesAgent::new(policy, gamma, selector, lambda, f)
 *             elegibility_traces_agent.rs:21 | InternalModelAgent::new(agent, model, planning_length)
 *             internal_model_agent.rs:17
 * plus the RNG injection contract (seed, global agent ids) and the device placement. */
typedef struct rlb_config {
    uint32_t struct_size;        /* = sizeof(rlb_config) */
    int32_t env_kind;            /* rlb_env_kind */
    int32_t map_id;              /* FrozenLake: 0 = MAP_4X4 (frozen_lake.rs:23), 1 = MAP_8X8 (:25-28) */
    int32_t slippery;            /* FrozenLake is_slippery */
    uint32_t max_steps;          /* ignored by Blackjack */
    int32_t policy_kind;         /* rlb_policy_kind */
    int32_t selector_kind;       /* rlb_selector_kind */
    int32_t target_kind;         /* rlb_target_kind */
    int32_t agent_kind;          /* rlb_agent_kind */
    int32_t real_kind;           /* rlb_real_kind */
    int32_t decay_kind;          /* rlb_decay_kind */
    int32_t device;              /* CUDA device ordinal */
    double learning_rate;
    double discount_factor;
    double lambda_factor;
    double initial_epsilon;
    double epsilon_decay;        /* the k of `a - k` / `a * k` */
    double final_epsilon;
    double confidence_level;     /* UCB c */
    double default_value;        /* Q default (bin/taxi.rs:126 passes 0.0) */
    uint64_t seed;               /* Philox key */
    uint64_t n_agents;           /* agents held by this engine */
    uint64_t first_agent_id;     /* global id of local agent 0 (Philox counter high words) */
    uint32_t store_kind;         /* where the fused kernel keeps the tables: 0 = auto, 1 = HBM, 2 = shared memory (one agent per
                                    4-lane thread group), 3 = hybrid (Q in shared memory, eligibility rows streamed through L2),
                                    4 = HBM with a trace agent's sweeps applied lazily (same results, row by row on demand) */
    uint32_t planning_steps;     /* > 0: the agent is wrapped as InternalModelAgent::new(agent, RandomModel::default(), planning_steps)
                                    (agent/internal_model_agent.rs:17-29; bin/cliffwalking_model.rs:150-156 passes 10).  Needs the HBM store. */
    /* FrozenLakeEnv::new(map: &[&str], ..) (frozen_lake.rs:48) with a caller-supplied map: map_id = RLB_MAP_CUSTOM and
     * `map` = the rows joined without separators (map_rows * map_cols chars of 'S' 'F' 'H' 'G', row-major; read during
     * rlb_engine_create only).  Every 'S' cell is a start cell: reset() draws among them with `categorical_sample` over
     * the 1/count distribution (:54-66,106-109); a map without 'S' starts at cell 0, as the reference's all-zero
     * distribution does.  At most 1024 cells. */
    uint32_t map_rows, map_cols;
    const char* map;
} rlb_config;
#define RLB_MAP_4X4 0
#define RLB_MAP_8X8 1
#define RLB_MAP_CUSTOM 2

/* Per-training-episode record streamed by the fused kernel (agent.rs:72-75,98,103,115):
 * episode length, episode return, and the episode's sum / sum of |.| of the per-step
 * temporal differences (accumulated in Real, in step order, from 0). */
typedef struct rlb_episode_f32 { uint32_t length; float ret; float td_sum; float td_abs_sum; } rlb_episode_f32;
typedef struct rlb_episode_f64 { double ret; double td_sum; double td_abs_sum; uint32_t length; uint32_t pad; } rlb_episode_f64;

/* One record per env transition, for step-level parity / `training_error` (agent.rs:98). */
typedef struct rlb_traj_record {
    uint8_t kind;        /* 0 = reset + first get_action, 1 = train step, 2 = evaluate step */
    uint8_t action;      /* action chosen on `obs` */
    uint8_t terminated;
    uint8_t pad;
    uint32_t obs;        /* dense observation returned by reset / step */
    double reward;
    double td;           /* temporal difference (train steps) */
} rlb_traj_record;

/* Outputs of rlb_agent_train / rlb_agent_train_range.  Any pointer may be NULL. */
typedef struct rlb_train_out {
    /* [n_episodes][4] f64, reduced over this engine's agents per episode index:
     * sum(length), sum(return), sum(td_sum), sum(td_abs_sum).  Divide by n_agents for the
     * reference's per-run curves.  This is what multi-GPU runs gather.  [n_episodes][n_sets][4], one reduction
     * per set, while rlb_engine_set_hparams sets are installed. */
    double* episode_sums;
    /* [n_episodes][n_agents] rlb_episode_f32 / rlb_episode_f64 (by rlb_config.real): the
     * raw per-agent stream (reward_history, episode_length of agent.rs:117). */
    void* episodes;
    /* per-agent step trajectory, [n_agents][traj_capacity] rlb_traj_record, and the number
     * of records written per agent [n_agents] (u64).  For parity tests and small runs. */
    rlb_traj_record* traj;
    uint64_t traj_capacity;
    uint64_t* traj_count;
    /* totals over all agents */
    uint64_t train_steps;        /* out: sum of training episode lengths */
    uint64_t eval_steps;         /* out: steps executed inside the injected evaluate(100) calls */
    double eval_return_sum;      /* out: sum of returns of those evaluate episodes */
    uint64_t eval_episodes;      /* out */
    float kernel_ms;             /* out: device time of the kernel launches (CUDA events): k_run, and the k_eval launches
                                    of the evaluate blocks of the thread-group and hybrid stores */
    uint32_t kernel_launches;    /* out: kernel launches (with per-set selectors: launch pairs); an on-chip store's
                                    engine of >= 2^17 agents makes one k_run launch per training segment and one k_eval
                                    launch per evaluate block */
    uint64_t trace_rows;         /* out: eligibility rows swept (elegibility_traces_agent.rs:86), for the roofline */
    /* `training_error` (agent.rs:73,98,117): the temporal difference of EVERY training step, in step order, episodes
     * concatenated — [n_agents][td_capacity] Real; td_count [n_agents] u64 receives the number of training steps each
     * agent took in this call (the first min(count, capacity) values are stored).  Optional (NULL / 0): at scale the
     * per-episode td_sum / td_abs_sum of the episode records are the stream; this is the exact per-step vector the
     * bins window for their "Training Error" chart (bin/taxi.rs:170-174).  Host or device buffers. */
    void* td_steps;
    uint64_t td_capacity;
    uint64_t* td_count;
} rlb_train_out;

/* Per-agent resumable state besides the tables — complete AT AN EPISODE BOUNDARY, which is where rlb_agent_train /
 * rlb_agent_evaluate leave every agent.  Not part of it: the env state inside an episode (position, step counter,
 * Blackjack hands; rlb_set_agent_states leaves env_ready alone) and a non-empty eligibility trace — a snapshot taken in
 * the middle of an episode driven through the step-level calls does not resume that episode.  rlb_set_agent_states
 * refuses an odd rng_n on the envs that only draw 64-bit values (every env but Blackjack). */
typedef struct rlb_agent_state {
    double epsilon;              /* uniform_epsilon_greed.rs:13 */
    uint64_t ucb_t;              /* upper_confidence_bound.rs:12 */
    uint64_t rng_n;              /* index of the next 32-bit word of the agent's Philox stream */
    int32_t policy_flag;         /* double_tabular_policy.rs:14 */
    int32_t env_ready;           /* env `ready` flag */
} rlb_agent_state;

/* One remembered transition of the Dyna model: `(obs, action) -> (next_obs, reward)` (model/random_model.rs:11). */
typedef struct rlb_model_entry { uint32_t obs; uint32_t action; uint32_t next_obs; float reward; } rlb_model_entry;

/* ---- library ------------------------------------------------------------------------- */
int rlb_abi_version(void);
const char* rlb_last_error_string(void);
/* number of CUDA devices visible (0 without a driver) */
int rlb_device_count(void);

/* ---- engine lifecycle: the constructors listed at rlb_config ---------------------------- */
rlb_status rlb_engine_create(const rlb_config* cfg, rlb_engine** out);
void rlb_engine_destroy(rlb_engine* e);
/* Run on an external CUDA stream (cudaStream_t as void*; e.g. torch's current stream). */
rlb_status rlb_engine_set_stream(rlb_engine* e, void* cuda_stream);
rlb_status rlb_engine_synchronize(rlb_engine* e);
/* Env::action_size (env.rs:20-22) and the dense observation count */
rlb_status rlb_engine_dims(const rlb_engine* e, uint32_t* n_states, uint32_t* n_actions, uint32_t* n_tables);
/* which table store the engine picked (1 HBM, 2 shared memory thread groups, 3 hybrid, 4 HBM + lazy trace sweeps) */
uint32_t rlb_engine_store_kind(const rlb_engine* e);

/* ---- per-agent hyper-parameter sets (no reference equivalent: the bins build one agent per run and sweep the
 * constructor arguments by hand, bin/taxi.rs:22-68) ------------------------------------------------------------------
 * The constructor arguments the bins vary, per agent:
 *   TabularPolicy::new(lr, default) tabular_policy.rs:15 / DoubleTabularPolicy::new(lr, default) double_tabular_policy.rs:17,
 *   UniformEpsilonGreed::new(eps, decay, final) uniform_epsilon_greed.rs:31, UpperConfidenceBound::new(c)
 *   upper_confidence_bound.rs:17, OneStepAgent::new(.., gamma, ..) one_step_agent.rs:16 /
 *   ElegibilityTracesAgent::new(.., gamma, .., lambda, ..) elegibility_traces_agent.rs:21.
 * Field for field the hyper-parameters of rlb_config. */
typedef struct rlb_hparams {
    double learning_rate, discount_factor, lambda_factor;
    double initial_epsilon, epsilon_decay, final_epsilon;   /* epsilon_decay: the k of rlb_config.decay_kind */
    double confidence_level, default_value;
} rlb_hparams;                                             /* 64 bytes */
#define RLB_MAX_HPARAM_SETS 65536
/* sets [n_sets]; group [N] u32: agent i is constructed with sets[group[i]].  Host or device buffers.
 * sets = NULL, n_sets = 0, group = NULL: back to rlb_config's values.
 * Constructor equivalence: after this call every call gives agent i the results, bit for bit, of agent 0 of an engine
 * created with rlb_config's eight hyper-parameters replaced by sets[group[i]], n_agents = 1 and first_agent_id + i.  So
 * the call acts as the constructor of the agents: their tables are refilled with their own default_value, epsilon set to
 * their initial_epsilon, UCB counts and t reset, policy_flag set (as rlb_agent_set_kind does; the env and the RNG
 * stream carry on).  Every later reset (rlb_selector_reset, rlb_policy_reset, rlb_agent_reset, rlb_agent_set_kind,
 * rlb_agent_set_action_selector) and compute call uses each agent's own set; decay_kind, agent kind, selector,
 * policy, real type and env stay engine-wide, and the target too unless rlb_engine_set_targets gives each set its own.
 * While sets are installed every per-episode sums output is [n_episodes][n_sets][4] (rlb_train_out.episode_sums,
 * rlb_agent_evaluate's sums_out): entry (e, g) is the rlb_train_out reduction, in the same order, over the agents of
 * set g in ascending local index — one set of all agents gives the [n_episodes][4] of an engine without sets, and a set
 * of a contiguous id range the sums of an engine holding just those agents.  Gather them with
 * rlb_comm_gather_episode_sums(.., n_episodes * n_sets, ..).
 * RLB_ERR_INVALID_ARG, the engine untouched: n_sets == 0 with a non-NULL pointer, n_sets > 0 with a NULL one,
 * n_sets > RLB_MAX_HPARAM_SETS, any group[i] >= n_sets.  Values are not checked.  RLB_ERR_UNSUPPORTED: a Dyna model
 * (rlb_agent_set_model / rlb_config.planning_steps) together with sets, whichever comes second (per-set planning counts
 * attach one: rlb_engine_set_planning_steps), and uninstalling the sets while such counts are in force. */
rlb_status rlb_engine_set_hparams(rlb_engine* e, const rlb_hparams* sets, uint32_t n_sets, const uint32_t* group);
uint32_t rlb_engine_hparam_sets(const rlb_engine* e);    /* 0 while rlb_config's values apply */
/* Replace the values of the installed hyper-parameter sets without reconstructing any agent (the explore step of
 * population-based training; no reference equivalent).  sets [n_sets], host or device: sets[g] becomes the values of
 * installed set g.  The groups, the grouped-reduction order and everything stored per agent (tables, epsilon, UCB state,
 * flags, model, RNG position) stay as they are.  From the next call on every kernel uses the new learning_rate,
 * discount_factor, lambda_factor, confidence_level, epsilon_decay and final_epsilon; initial_epsilon and default_value
 * take effect at the next reset (rlb_agent_reset, rlb_selector_reset, rlb_policy_reset, rlb_agent_set_kind,
 * rlb_agent_set_action_selector).
 * Equivalence: from here on every call gives the bits of an engine B created with the same rlb_config, then
 * rlb_engine_set_hparams(sets, n_sets, the same group), then given this engine's tables, agent states and model
 * (rlb_upload_tables, rlb_set_agent_states, rlb_upload_model).
 * RLB_ERR_INVALID_ARG, the engine untouched: sets == NULL, no sets installed, n_sets != rlb_engine_hparam_sets(e).
 * Values are not checked. */
rlb_status rlb_engine_retune_hparams(rlb_engine* e, const rlb_hparams* sets, uint32_t n_sets);
/* Pause and resume hyper-parameter sets (successive halving; no reference equivalent).  active [n_sets] u8, host or
 * device: nonzero = set g takes part in later train / evaluate calls.  active = NULL, n_sets = 0: every set active (also
 * the state after rlb_engine_set_hparams); an all-ones mask is the same.
 * Which calls: rlb_agent_train, rlb_agent_train_range, rlb_agent_train_range_async and rlb_agent_evaluate run only the
 * agents of active sets, in a launch sized to them.  Every other call (the step-level calls, rlb_agent_step, resets,
 * rlb_agent_set_kind, rlb_agent_clone, snapshots, uploads and downloads) still acts on all N agents.
 * Active agents get, bit for bit, what they would get with every set active: tables, counts, epsilon, UCB t, the Double
 * flag, RNG position, env state, their episode records and their set's row of the per-episode sums.
 * Inactive agents keep their whole state bit for bit (tables, counts, epsilon, t, flag, RNG position, env, eligibility
 * rows, lazy-sweep bookkeeping, rlb_agent_step state).  Their records in a returned episodes buffer are zero, their
 * td_count and traj_count 0, and their set's row of episode_sums / sums_out 0.0.  train_steps, eval_steps,
 * eval_return_sum and eval_episodes count active agents only.  A set paused for some calls and then resumed continues
 * from where it stopped: its agents equal those of an engine that made only the calls during which the set was active.
 * Every set inactive is allowed: the compute calls then launch nothing and return zero sums and totals.
 * rlb_engine_set_hparams makes every set active again (also when it uninstalls them); rlb_engine_retune_hparams keeps
 * the mask.
 * RLB_ERR_INVALID_ARG, the engine untouched: no sets installed, n_sets != rlb_engine_hparam_sets(e), or a NULL /
 * non-NULL mismatch between active and n_sets. */
rlb_status rlb_engine_set_active_sets(rlb_engine* e, const uint8_t* active, uint32_t n_sets);
/* Dyna-Q under hyper-parameter sets: a planning count per set (no reference equivalent; rlb_hparams' layout is ABI, so
 * the count is kept beside it).  steps [n_sets] u32, host or device: the agents of set g are
 * InternalModelAgent::new(agent, RandomModel::default(), steps[g]) (agent/internal_model_agent.rs:17-29), i.e. they make
 * steps[g] planning replays per real update.  The sets-aware way to attach a model: rlb_agent_set_model(k > 0) after
 * rlb_engine_set_hparams, and rlb_engine_set_hparams(n_sets > 0) with a model attached, still return RLB_ERR_UNSUPPORTED.
 * The first call on an engine without a model wraps every agent as it is (tables, epsilon, counts, flag and RNG stay; the
 * model starts empty), as rlb_agent_set_model does; it needs the HBM store and re-picks the store.  A later call changes
 * only the counts, models, tables and states left as they are: every later call then gives the bits of an engine B with
 * the same rlb_config and rlb_engine_set_hparams, given this engine's tables, agent states and model (rlb_upload_tables,
 * rlb_set_agent_states, rlb_upload_model) and then the same counts.  A count of 0 is allowed: those agents train as
 * the plain agent does (tables, states, records and sums), while their model still records every first-seen
 * transition.  rlb_model_capacity stays nonzero while the model is attached, every count 0 included.
 * steps = NULL, n_sets = 0: drop the model and the counts (as rlb_agent_set_model(e, 0), which does the same).
 * The counts are kept by rlb_agent_set_kind (which re-wraps around an empty model), rlb_agent_reset (which empties the
 * model), rlb_engine_retune_hparams and rlb_agent_clone (the destination keeps its set, so its count); the active-set
 * mask applies to the model launches as to every train launch.  Uninstalling the sets (rlb_engine_set_hparams(e, NULL,
 * 0, NULL)) while counts are in force returns RLB_ERR_UNSUPPORTED.
 * RLB_ERR_INVALID_ARG, the engine untouched: no sets installed, n_sets != rlb_engine_hparam_sets(e), or a NULL /
 * non-NULL mismatch between steps and n_sets.  RLB_ERR_UNSUPPORTED: store_kind names a store other than HBM.  Values
 * are not checked. */
rlb_status rlb_engine_set_planning_steps(rlb_engine* e, const uint32_t* steps, uint32_t n_sets);
/* The bootstrap target per hyper-parameter set (rlb_hparams' layout is ABI, so the target is kept beside it, as the
 * planning counts are).  targets [n_sets] i32 RLB_TARGET_*, host or device: the agents of set g use targets[g] as
 * Agent::set_future_q_value_func(targets[g]) would (agent.rs:19-48), in every update: the fused train calls, the
 * step-level rlb_agent_update and rlb_agent_step, and the Dyna planning replays under rlb_engine_set_planning_steps; for
 * one-step and eligibility-trace agents in every store.
 * Equivalence: from this call on every call gives agent i the bits of agent 0 of an engine created with target_kind =
 * targets[group[i]] and the rest as rlb_engine_set_hparams states it.  Nothing stored per agent changes (tables, epsilon,
 * UCB state, flag, model, RNG position): a call between chunks equals an engine B given this engine's tables, agent
 * states and model (rlb_upload_tables, rlb_set_agent_states, rlb_upload_model) and then the same targets.
 * rlb_engine_set_hparams (installing or uninstalling) sets every set's target to rlb_config.target_kind, and
 * rlb_agent_set_future_q_value_func(k) keeps its meaning, every agent now uses k: it sets every set's target to k.
 * rlb_engine_retune_hparams, rlb_engine_set_active_sets, rlb_agent_set_kind, the resets and
 * rlb_engine_set_planning_steps keep the targets; rlb_agent_clone's destination keeps its set, so its set's target.
 * RLB_ERR_INVALID_ARG, the engine untouched: no sets installed, n_sets != rlb_engine_hparam_sets(e), targets NULL, or a
 * value outside RLB_TARGET_SARSA .. RLB_TARGET_EXPECTED_SARSA.  Unlike rlb_hparams the values are checked: an
 * unknown target would otherwise run as Expected Sarsa. */
rlb_status rlb_engine_set_targets(rlb_engine* e, const int32_t* targets, uint32_t n_sets);
/* The action selector per hyper-parameter set (kept beside rlb_hparams, as the targets are).  selectors [n_sets] i32
 * RLB_SEL_*, host or device: the agents of set g select actions as rlb_agent_set_action_selector(selectors[g]) would
 * make them, in every call: the fused train and evaluate calls, rlb_agent_get_action, rlb_agent_update, rlb_agent_step,
 * rlb_selector_get_action, rlb_selector_get_exploration_probs, rlb_selector_update and the resets.
 * Equivalence: from this call on every call gives agent i the bits of agent 0 of an engine created with selector_kind =
 * selectors[group[i]], its set's values, target and planning count, n_agents = 1 and first_agent_id + i, given this
 * engine's tables and this agent's state.
 * A set whose selector changes gets a fresh selector of its new kind, as rlb_agent_set_action_selector gives every agent:
 * epsilon = its set's initial_epsilon, UCB t = 1, its agents' counts rows zero.  This holds in both directions, so an
 * eps-greedy agent's counts are always zero.  A set whose selector is unchanged keeps its selector state: a second call
 * with the same array does nothing.
 * rlb_engine_set_hparams (installing or uninstalling) and rlb_agent_set_action_selector(k) put every set on the
 * engine-wide selector, with a fresh selector everywhere.  rlb_engine_retune_hparams, rlb_engine_set_active_sets,
 * rlb_engine_set_planning_steps, rlb_engine_set_targets and rlb_agent_set_kind keep the per-set selectors
 * (rlb_agent_set_kind gives each agent a fresh selector of its set's kind); rlb_agent_reset and rlb_selector_reset reset
 * each agent's selector as its set's kind does, and rlb_selector_update decays epsilon only in eps-greedy sets.
 * rlb_agent_clone's destination keeps its set, so its set's selector: the counts segment is copied to destinations of
 * UCB sets and left zero in those of eps-greedy sets.  rlb_download_tables / rlb_upload_tables carry counts while any
 * set uses UCB.  Record, sums and totals layouts do not change.
 * The fused calls launch once per selector: the agents of the eps-greedy sets and those of the UCB sets (restricted to
 * the active sets) run as two concurrent launches, one launch where only one of them has agents.
 * RLB_ERR_INVALID_ARG, the engine untouched: no sets installed, n_sets != rlb_engine_hparam_sets(e), selectors NULL, or
 * a value outside RLB_SEL_EPS_GREEDY .. RLB_SEL_UCB.  RLB_ERR_UNSUPPORTED, the engine untouched: the engine's table
 * store cannot run a requested selector (the thread-group or hybrid store when that selector's on-chip bytes exceed
 * the per-block limit); the store is not re-picked. */
rlb_status rlb_engine_set_selectors(rlb_engine* e, const int32_t* selectors, uint32_t n_sets);

/* ---- Env<T,COUNT> (env.rs:19-49), batched ------------------------------------------------ */
/* Env::reset (blackjack.rs:105, frozen_lake.rs:106, cliff_walking.rs:67, taxi.rs:135).  obs_out [N] u32 */
rlb_status rlb_env_reset(rlb_engine* e, uint32_t* obs_out);
/* Env::step (blackjack.rs:118, frozen_lake.rs:115, cliff_walking.rs:74, taxi.rs:144).
 * actions [N] u32; obs_out [N] u32; reward_out [N] f64; terminated_out [N] u8.
 * Returns RLB_ERR_ENV_NOT_READY if any agent's env was not ready (those agents are left
 * untouched and flagged in not_ready_out [N] u8 when given). */
rlb_status rlb_env_step(rlb_engine* e, const uint32_t* actions, uint32_t* obs_out, double* reward_out,
                        uint8_t* terminated_out, uint8_t* not_ready_out);

/* ---- Agent<T,COUNT> (agent.rs:47-164), batched -------------------------------------------- */
/* Agent::get_action (one_step_agent.rs:48-51, elegibility_traces_agent.rs:56-59) */
rlb_status rlb_agent_get_action(rlb_engine* e, const uint32_t* obs, uint32_t* action_out);
/* Agent::update (one_step_agent.rs:53-86, elegibility_traces_agent.rs:61-104); td_out [N] Real */
rlb_status rlb_agent_update(rlb_engine* e, const uint32_t* curr_obs, const uint32_t* curr_action, const double* reward,
                            const uint8_t* terminated, const uint32_t* next_obs, const uint32_t* next_action,
                            void* td_out);
/* Agent::set_future_q_value_func (agent.rs:48) */
rlb_status rlb_agent_set_future_q_value_func(rlb_engine* e, int32_t target_kind);
/* Agent::set_action_selector (agent.rs:50): installs a fresh selector built from cfg's
 * parameters (the reference clones a never-used selector, bin/taxi.rs:161). */
rlb_status rlb_agent_set_action_selector(rlb_engine* e, int32_t selector_kind);
/* A second agent object on the SAME env and RNG stream, as the bins build (bin/taxi.rs:138-156: a OneStepAgent and an
 * ElegibilityTracesAgent, each with its own fresh policy, driven one after the other over one env).  Replaces the
 * engine's agent by a freshly constructed one of `agent_kind`: default tables, policy_flag = true, a fresh selector of
 * the current selector kind, no traces; the env state and the stream position carry on. */
rlb_status rlb_agent_set_kind(rlb_engine* e, int32_t agent_kind);
/* InternalModelAgent::new(agent, RandomModel::default(), planning_steps) (agent/internal_model_agent.rs:17-29) around the
 * engine's CURRENT agent, which keeps its tables and selector state (the wrapper only borrows it); the model starts
 * empty.  planning_steps = 0 drops the wrapper and its model.  From then on rlb_agent_update and rlb_agent_train run
 * InternalModelAgent::update (:46-79): the wrapped update, Model::add_info, then `planning_steps` replays of sampled
 * transitions (get_action on the remembered next_obs + update with terminated = false).  Needs the HBM store. */
rlb_status rlb_agent_set_model(rlb_engine* e, uint32_t planning_steps);
/* Agent::reset (one_step_agent.rs:43-46): selector.reset() + policy.reset(); with a model also Model::reset
 * (internal_model_agent.rs:81-84) */
rlb_status rlb_agent_reset(rlb_engine* e);
/* Agent::train (agent.rs:66-118): the fused hot path.  All N agents run episodes
 * [0, n_episodes) with evaluate(100) injected after every episode with
 * episode % eval_at == 0. */
rlb_status rlb_agent_train(rlb_engine* e, uint64_t n_episodes, uint64_t eval_at, rlb_train_out* out);
/* Episodes [ep_begin, ep_end) of the same train() call, so a run can be driven in chunks
 * (outputs are indexed from ep_begin). */
rlb_status rlb_agent_train_range(rlb_engine* e, uint64_t ep_begin, uint64_t ep_end, uint64_t eval_at, rlb_train_out* out);
/* The same call without the final wait: everything (kernels, the reduction, the device->host copies of records and
 * sums) is enqueued on the engine's streams and the call returns.  The buffers named in `out` — and `out` itself —
 * must stay valid until rlb_agent_train_wait(), which blocks until the work is done and fills out's scalar fields
 * (train_steps ... trace_rows).  One call may be pending per engine; any other compute call on the engine waits for it
 * first.  This is how a host thread keeps several engines (the cells of a sweep, bin/taxi.rs:158-203, or the GPUs of a
 * box) busy at once, and how the record copy of call i hides behind the kernels of call i + 1.  Host record / td
 * buffers should be pinned (cudaHostAlloc / cudaHostRegister) for the copies to be asynchronous. */
rlb_status rlb_agent_train_range_async(rlb_engine* e, uint64_t ep_begin, uint64_t ep_end, uint64_t eval_at, rlb_train_out* out);
rlb_status rlb_agent_train_wait(rlb_engine* e);
/* One iteration of the loop at agent.rs:83-106 for every agent, fused into ONE launch: an agent whose episode is over
 * (or not begun) does `curr_obs = env.reset(); curr_action = get_action(curr_obs)` (agent.rs:83-84; kind 0), any other
 * agent does `env.step(curr_action)`, `get_action(next_obs)`, `update(..)` and the bookkeeping of :88-105 (kind 1), the
 * engine keeping curr_obs / curr_action on the device.  A host loop over this call reproduces rlb_agent_train's
 * trajectory (without the injected evaluate); it is the low-latency form of the three step-level calls
 * rlb_env_step + rlb_agent_get_action + rlb_agent_update for trait-object style drivers.  Outputs [N], any may be
 * NULL: kind u8, obs u32 (the observation returned by reset / step), action u32 (chosen on it), reward f64,
 * terminated u8, td Real. */
rlb_status rlb_agent_step(rlb_engine* e, uint8_t* kind_out, uint32_t* obs_out, uint32_t* action_out, double* reward_out,
                          uint8_t* terminated_out, void* td_out);
/* Agent::evaluate (agent.rs:120-141).  episodes_out: [n_episodes][N] episode records
 * (td fields zero); sums_out [n_episodes][4] ([n_episodes][n_sets][4] with hyper-parameter sets) as in rlb_train_out.
 * Either may be NULL. */
rlb_status rlb_agent_evaluate(rlb_engine* e, uint64_t n_episodes, void* episodes_out, double* sums_out,
                              uint64_t* total_steps_out);

/* ---- Policy<T,COUNT> (policy.rs:15-25), batched -------------------------------------------- */
/* Policy::predict (tabular_policy.rs:27-29, double_tabular_policy.rs:31-39); values_out [N][A] Real */
rlb_status rlb_policy_predict(rlb_engine* e, const uint32_t* obs, void* values_out);
/* Policy::get_values (tabular_policy.rs:31-33, double_tabular_policy.rs:41-48) */
rlb_status rlb_policy_get_values(rlb_engine* e, const uint32_t* obs, void* values_out);
/* Policy::update (tabular_policy.rs:35-38, double_tabular_policy.rs:50-58); td [N] Real */
rlb_status rlb_policy_update(rlb_engine* e, const uint32_t* obs, const uint32_t* action, const uint32_t* next_obs,
                             const void* temporal_difference);
/* Policy::after_update (double_tabular_policy.rs:65-67) */
rlb_status rlb_policy_after_update(rlb_engine* e);
/* Policy::reset (tabular_policy.rs:40-42, double_tabular_policy.rs:60-63) */
rlb_status rlb_policy_reset(rlb_engine* e);

/* ---- ActionSelection<T,COUNT> (action_selection.rs:10-15), batched -------------------------- */
/* ActionSelection::get_action (uniform_epsilon_greed.rs:60-66, upper_confidence_bound.rs:29-42); values [N][A] Real */
rlb_status rlb_selector_get_action(rlb_engine* e, const uint32_t* obs, const void* values, uint32_t* action_out);
/* ActionSelection::get_exploration_probs (uniform_epsilon_greed.rs:72-76, upper_confidence_bound.rs:48-63); probs_out [N][A] Real */
rlb_status rlb_selector_get_exploration_probs(rlb_engine* e, const uint32_t* obs, const void* values, void* probs_out);
/* ActionSelection::update (uniform_epsilon_greed.rs:68-70, upper_confidence_bound.rs:44-46) */
rlb_status rlb_selector_update(rlb_engine* e);
/* ActionSelection::reset (uniform_epsilon_greed.rs:78-80, upper_confidence_bound.rs:65-68) */
rlb_status rlb_selector_reset(rlb_engine* e);

/* ---- Model<T,COUNT> (model.rs:12-16; RandomModel, model/random_model.rs), batched -------------- */
/* Model::add_info (random_model.rs:37-41): first-seen (obs, action) only, in insertion order.  reward [N] f64 */
rlb_status rlb_model_add_info(rlb_engine* e, const uint32_t* obs, const uint32_t* action, const double* reward, const uint32_t* next_obs);
/* Model::get_info (random_model.rs:27-35): entry number gen_range(0..len) of each agent's model, drawn from the agent's
 * stream.  RLB_ERR_INVALID_ARG if any agent's model is empty (the reference panics); those agents draw nothing. */
rlb_status rlb_model_get_info(rlb_engine* e, uint32_t* obs_out, uint32_t* action_out, uint32_t* next_obs_out, double* reward_out);
/* Model::reset (random_model.rs:43-45) */
rlb_status rlb_model_reset(rlb_engine* e);
/* entries one agent's model can hold (= S * A); 0 while no model is attached */
uint32_t rlb_model_capacity(const rlb_engine* e);
/* snapshot of the models: len [N] u32, entries [N][capacity] in insertion order (host or device buffers) */
rlb_status rlb_download_model(rlb_engine* e, uint32_t* len_out, rlb_model_entry* entries_out);
rlb_status rlb_upload_model(rlb_engine* e, const uint32_t* len, const rlb_model_entry* entries);

/* ---- state snapshot (no reference equivalent: the crate has no checkpointing) --------------- */
/* q: [N][n_tables][S][A] Real (alpha then beta for Double); counts: [N][S][A] u32 (UCB). */
rlb_status rlb_download_tables(rlb_engine* e, void* q_out, uint32_t* counts_out);
rlb_status rlb_upload_tables(rlb_engine* e, const void* q, const uint32_t* counts);
rlb_status rlb_get_agent_states(rlb_engine* e, rlb_agent_state* states_out /* [N] */);
rlb_status rlb_set_agent_states(rlb_engine* e, const rlb_agent_state* states /* [N] */);
/* Agent dst[j] takes the learned state of agent src[j], for j < n_pairs (the exploit step of population-based training;
 * no reference equivalent), in one device launch: its Q table(s) (both for Double), its UCB counts when the selector is
 * UCB (under rlb_engine_set_selectors: when dst[j]'s set is UCB), epsilon, ucb_t and policy_flag, and its Dyna model when one is attached (entries, membership bits, length).
 * dst[j] keeps its RNG stream position rng_n (its Philox stream stays keyed by its own global id, so a clone does not
 * replay the source's draws), its env state, its eligibility rows and lazy-sweep bookkeeping, its rlb_agent_step state
 * and its hyper-parameter set.  src, dst [n_pairs] u32, host or device.
 * Equivalence: the result is bit for bit what rlb_download_tables + rlb_get_agent_states (+ rlb_download_model), a copy
 * of those fields from src[j] to dst[j] on the host, and the matching uploads give.  So, like rlb_agent_state, the call
 * is complete AT AN EPISODE BOUNDARY, which is where rlb_agent_train / rlb_agent_evaluate leave every agent.
 * A source may appear any number of times (one winner, many losers).  n_pairs == 0 does nothing.
 * RLB_ERR_INVALID_ARG, the engine untouched: a NULL src or dst with n_pairs > 0, an id >= N, a dst that appears twice,
 * an id that is both a source and a destination anywhere in the call (so no pair writes what another reads, and the
 * result does not depend on the order of the pairs).  RLB_ERR_UNSUPPORTED: an eligibility-trace agent under a Dyna model
 * (its rows survive episode boundaries there). */
rlb_status rlb_agent_clone(rlb_engine* e, const uint32_t* src, const uint32_t* dst, uint64_t n_pairs);

/* ---- multi-GPU: the path's one exchange (no reference equivalent: the crate is single-threaded) ----------------
 * Agents are independent, so a job shards by contiguous ranges of GLOBAL agent id (rlb_config.first_agent_id) with no
 * data-path collective.  The only exchange is one gather per run (or per chunk) of the per-episode metric sums —
 * rlb_train_out.episode_sums, [n_episodes][4] f64 per engine — to the root rank for the training charts
 * (bin/taxi.rs:170-223), done here with grouped ncclSend / ncclRecv over NVLink (libnccl.so.2 is loaded on first use;
 * the system library 2.27 has no ncclGather).  Two ways to build the communicator:
 *   - one process per GPU (torchrun, MPI, a Rust launcher ...): rank 0 calls rlb_comm_unique_id(), the host side
 *     passes the 128 bytes to the other ranks by any means, every rank calls rlb_comm_init_rank();
 *   - one process driving several GPUs (one engine per device, e.g. from Rust threads): rlb_comm_init_all().
 * NCCL failures return RLB_ERR_NCCL with the NCCL error string in rlb_last_error_string().
 * Load order: a process that also loads a library linked against a NEWER NCCL under the same soname (PyTorch) must
 * load that library before the first rlb_comm_* call, so that the loader hands librlb the newer copy. */
typedef struct rlb_comm rlb_comm;
#define RLB_COMM_ID_BYTES 128
rlb_status rlb_comm_unique_id(uint8_t id_out[RLB_COMM_ID_BYTES]);
rlb_status rlb_comm_init_rank(const uint8_t id[RLB_COMM_ID_BYTES], int32_t world_size, int32_t rank, int32_t device, rlb_comm** out);
/* comms_out [n_devices]: one communicator per listed device, ranks 0 .. n_devices-1 in list order */
rlb_status rlb_comm_init_all(const int32_t* devices, int32_t n_devices, rlb_comm** comms_out);
void rlb_comm_destroy(rlb_comm* c);
int32_t rlb_comm_rank(const rlb_comm* c);
int32_t rlb_comm_world_size(const rlb_comm* c);
/* Every rank contributes local_sums [n_episodes][4] f64; rank `root` receives gathered_out [world][n_episodes][4]
 * (ignored elsewhere; may be NULL there).  DEVICE buffers, enqueued on `cuda_stream` (cudaStream_t as void*, NULL =
 * the communicator's own stream, synchronised before returning).  With rlb_comm_init_all the calls of the
 * communicators must be issued between rlb_comm_group_begin / rlb_comm_group_end or from one thread per rank. */
rlb_status rlb_comm_gather_episode_sums(rlb_comm* c, const double* local_sums, uint64_t n_episodes, double* gathered_out,
                                        int32_t root, void* cuda_stream);
/* sum over ranks of `count` f64 values, in place, on every rank (job totals: steps, max-reduced times travel as sums
 * of one-hot vectors).  DEVICE buffer. */
rlb_status rlb_comm_allreduce_sum(rlb_comm* c, double* values, uint64_t count, void* cuda_stream);
rlb_status rlb_comm_group_begin(void);
rlb_status rlb_comm_group_end(void);

/* ---- self test ---------------------------------------------------------------------------------------------------
 * The UCB bonus sqrt(ln t / n) (upper_confidence_bound.rs:33-37) is computed with hand-scheduled copies of the
 * compiler's own division / square-root sequences; this compares them with the compiler's, bit for bit, on `samples`
 * pseudo-random (t in [2, t_max], n in [1, n_max]) pairs and reports the number of differing results (expected: 0). */
rlb_status rlb_selftest_ucb_math(int32_t device, uint64_t samples, uint64_t t_max, uint64_t n_max, uint64_t seed, uint64_t* mismatches_out);

/* ---- RNG injection contract, host-callable (no device needed) -------------------------------
 * Replaces rand::thread_rng() at blackjack.rs:54,76; taxi.rs:136-137; frozen_lake.rs:107-108,126;
 * uniform_epsilon_greed.rs:53,62; random_model.rs:30.  Stream of agent g: 32-bit words
 * w[n] = Philox4x32-10(key = seed, ctr = (n>>2, g))[n & 3]. */
void rlb_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
void rlb_rng_words(uint64_t seed, uint64_t agent_id, uint64_t first_word, uint64_t count, uint32_t* out);
/* rand 0.8.5 samplers over that stream; *word_index is advanced. */
double rlb_rng_uniform_f64(uint64_t seed, uint64_t agent_id, uint64_t* word_index);
uint64_t rlb_rng_uniform_usize(uint64_t seed, uint64_t agent_id, uint64_t* word_index, uint64_t range);
uint32_t rlb_rng_card(uint64_t seed, uint64_t agent_id, uint64_t* word_index);
/* `Rng::gen_range(0..range)` on usize (the one-shot sampler with the conservative zone, random_model.rs:30) */
uint64_t rlb_rng_gen_range(uint64_t seed, uint64_t agent_id, uint64_t* word_index, uint64_t range);

/* ---- Blackjack observation ids (blackjack.rs:10-28) ------------------------------------------ */
uint64_t rlb_blackjack_obs_id(uint32_t dense_index);
uint32_t rlb_blackjack_dense_index(uint64_t obs_id);   /* 0xffffffff if not a Blackjack id */
void rlb_blackjack_decode(uint32_t dense_index, uint32_t* p_score, uint32_t* d_score, uint32_t* p_ace);

#ifdef __cplusplus
}
#endif
#endif /* RLB_H */
