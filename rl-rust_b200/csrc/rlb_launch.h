// rlb_launch.h — per-env launch entry points.  Each env's kernels are instantiated in its
// own translation unit (rlb_inst_<env>.cu) so the 16 (Real, Policy, Selector, Trace)
// variants of every kernel compile in parallel.
#pragma once
#include <cuda_runtime.h>

#include "rlb_device.cuh"

namespace rlb {

struct Variant {
    int real;     // rlb_real_kind
    int policy;   // rlb_policy_kind
    int sel;      // rlb_selector_kind
    int trace;    // 0 one-step, 1 eligibility traces
};

struct StepArgs {   // device pointers for the step-level kernels
    const uint32_t* obs = nullptr;
    const uint32_t* action = nullptr;
    const double* reward = nullptr;
    const uint8_t* term = nullptr;
    const uint32_t* obs2 = nullptr;
    const uint32_t* action2 = nullptr;
    const void* values = nullptr;
    const void* td_in = nullptr;
    void* real_out = nullptr;
    uint32_t* u32_out = nullptr;
    uint32_t* u32_out2 = nullptr;
    double* reward_out = nullptr;
    uint8_t* term_out = nullptr;
    uint8_t* kind_out = nullptr;
    uint8_t* not_ready_out = nullptr;
    uint32_t* any_not_ready = nullptr;   // the engine's flag word (FLAG_* bits, rlb_step_kernels.cuh)
    int which = 0;
    HpParams sets{};                     // launch_step<ENV, true>: every agent's hyper-parameter set
};

enum StepOp {
    OP_ENV_CONSTRUCT, OP_ENV_RESET, OP_ENV_STEP, OP_GET_ACTION, OP_UPDATE, OP_POLICY_ROWS, OP_POLICY_UPDATE,
    OP_SELECTOR_GET_ACTION, OP_SELECTOR_PROBS, OP_AGENT_STEP
};

// HP = true: the agents run with their own hyper-parameter sets `h` (k_run_hp); instantiated in rlb_inst_<env>_hp.cu
template <int ENV, bool HP = false> cudaError_t launch_run(const Variant& v, const DevParams& p, int store, cudaStream_t stream,
                                                          const HpParams& h = HpParams{});
// the same with the Dyna model attached (InternalModelAgent): HBM store only; instantiated in rlb_inst_<env>_model.cu, and
// with HP = true (k_run_hp, per-set planning counts h.planning) in rlb_inst_<env>_model_hp.cu
template <int ENV, bool HP = false> cudaError_t launch_run_model(const Variant& v, const DevParams& p, cudaStream_t stream,
                                                                const HpParams& h = HpParams{});
// bytes of dynamic shared memory one 1-warp CTA of the shared-memory / hybrid store needs (0: env not compiled for it)
template <int ENV> size_t smem_store_bytes(const Variant& v, int store, uint32_t rows, uint32_t S, uint32_t vmax);   // rows: table rows kept on chip
template <int ENV, bool HP = false> cudaError_t launch_step(StepOp op, const Variant& v, const DevParams& p, const StepArgs& a, cudaStream_t stream);
template <int ENV, bool HP = false> cudaError_t run_kernel_attributes(const Variant& v, int store, cudaFuncAttributes* attr);

// ---- per-agent hyper-parameter sets (rlb_hparams.cu) ----
// ptr[i * per_agent + k] = values[group[i]] for every agent i < n_agents and k < per_agent; elem_size 1, 4 or 8 bytes
cudaError_t launch_fill_grouped(void* ptr, size_t elem_size, uint64_t per_agent, uint64_t n_agents, const void* values,
                                const uint32_t* group, cudaStream_t stream);
// ActionSelection::update of every eps-greedy agent with its own set's decay k and floor
cudaError_t launch_eps_decay_grouped(double* eps, uint64_t n_agents, int kind, const rlb_hparams* sets, const uint32_t* group,
                                     cudaStream_t stream);
// out[e][g][4] for e < n_ep, g < n_sets: the k_episode_sums reduction over the agents order[offsets[g] .. offsets[g + 1])
cudaError_t launch_episode_sums_grouped(int real_kind, const void* records, uint64_t n_agents, const uint32_t* order,
                                        const uint32_t* offsets, uint32_t n_sets, uint64_t n_ep, double* out, cudaStream_t stream);

// ---- agent-to-agent copies of learned state (rlb_clone.cu, rlb_agent_clone) ----
constexpr int CLONE_MAX_SEGMENTS = 4;   // Q, UCB counts, model entries, model bits
struct CloneSegment {
    uint8_t* base;     // agent i's block is [base + i * stride, base + (i + 1) * stride)
    uint64_t stride;   // bytes, a multiple of 4
};
struct CloneArgs {
    CloneSegment seg[CLONE_MAX_SEGMENTS];
    uint32_t n_seg;
    const uint32_t* src;   // [n_pairs] device: no id in src is also in dst, no id appears twice in dst
    const uint32_t* dst;
    uint64_t n_pairs;
    double* eps;
    uint64_t* ucb_t;
    uint8_t* flag;
    uint32_t* model_len;   // nullptr without a model
};
// every segment's block, eps, ucb_t, flag and model_len of agent dst[j] = those of agent src[j]: one launch of k_clone_agents
cudaError_t launch_clone_agents(const CloneArgs& a, cudaStream_t stream);

}   // namespace rlb
