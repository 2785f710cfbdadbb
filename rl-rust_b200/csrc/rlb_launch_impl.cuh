// rlb_launch_impl.cuh — definitions behind rlb_launch.h; included by rlb_inst_<env>.cu only.
#pragma once
#include "rlb_launch.h"
#include "rlb_step_kernels.cuh"

namespace rlb {

#define RLB_VARIANT_SWITCH(v, CALL)                                                    \
    switch (((v).real << 3) | ((v).policy << 2) | ((v).sel << 1) | (v).trace) {        \
        case 0: CALL(float, 0, 0, false); break;                                       \
        case 1: CALL(float, 0, 0, true); break;                                        \
        case 2: CALL(float, 0, 1, false); break;                                       \
        case 3: CALL(float, 0, 1, true); break;                                        \
        case 4: CALL(float, 1, 0, false); break;                                       \
        case 5: CALL(float, 1, 0, true); break;                                        \
        case 6: CALL(float, 1, 1, false); break;                                       \
        case 7: CALL(float, 1, 1, true); break;                                        \
        case 8: CALL(double, 0, 0, false); break;                                      \
        case 9: CALL(double, 0, 0, true); break;                                       \
        case 10: CALL(double, 0, 1, false); break;                                     \
        case 11: CALL(double, 0, 1, true); break;                                      \
        case 12: CALL(double, 1, 0, false); break;                                     \
        case 13: CALL(double, 1, 0, true); break;                                      \
        case 14: CALL(double, 1, 1, false); break;                                     \
        case 15: CALL(double, 1, 1, true); break;                                      \
        default: break;                                                                \
    }

constexpr int kBlock = 128;
static inline unsigned grid_for(uint64_t n) { return (unsigned)((n + kBlock - 1) / kBlock); }

// HBM-store kernels read their Q rows through L1: ask for no more shared memory per SM than the resident CTAs use (the
// env table each, + 1 KB the system reserves per CTA), so that the rest of the 256 KB stays L1.  A hint; errors ignored.
#ifndef RLB_L1_CARVEOUT
#define RLB_L1_CARVEOUT 1
#endif
template <class K>
inline void prefer_l1(K kern, size_t smem) {
#if RLB_L1_CARVEOUT
    int blocks = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, kern, kBlock, smem) != cudaSuccess || blocks <= 0) { (void)cudaGetLastError(); return; }
    const size_t need = (size_t)blocks * (smem + 1024);
    int pct = (int)((need * 100 + 228 * 1024 - 1) / (228 * 1024));
    if (pct > 100) pct = 100;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, pct) != cudaSuccess) (void)cudaGetLastError();
#else
    (void)kern; (void)smem;
#endif
}

// shared-memory (thread-group) table store: compiled for the 4-action envs, whose whole per-agent working set is small
template <int ENV> struct SmemCapable { static constexpr bool value = (ENV == RLB_ENV_FROZEN_LAKE || ENV == RLB_ENV_CLIFF_WALKING); };

template <int ENV>
size_t smem_store_bytes(const Variant& v, int store, uint32_t rows, uint32_t S, uint32_t vmax) {
    if constexpr (!SmemCapable<ENV>::value) {
        return 0;
    } else {
        if (store == STORE_HYBRID) {
#define RLB_CALL(R, P, SL, T) return AgentCore<ENV, R, P, SL, T, STORE_HYBRID>::SStore::bytes(rows, vmax, SL == RLB_SEL_UCB, T) + EnvTab<ENV>::smem_bytes(S)
            RLB_VARIANT_SWITCH(v, RLB_CALL)
#undef RLB_CALL
        } else {
#define RLB_CALL(R, P, SL, T) return AgentCore<ENV, R, P, SL, T, STORE_SMEM>::SStore::bytes(rows, vmax, SL == RLB_SEL_UCB, T) + EnvTab<ENV>::smem_bytes(S)
            RLB_VARIANT_SWITCH(v, RLB_CALL)
#undef RLB_CALL
        }
        return 0;
    }
}

// k_run, or k_run_hp (one more parameter: the sets) when the agents hold their own hyper-parameter sets
template <bool HP, int ENV, typename R, int P, int SL, bool T, int STORE>
struct RunKernel {
    static auto ptr() {
        if constexpr (HP) return k_run_hp<ENV, R, P, SL, T, STORE>;
        else return k_run<ENV, R, P, SL, T, STORE>;
    }
    static void launch(unsigned grid, unsigned block, size_t smem, cudaStream_t stream, const DevParams& p, const HpParams& h) {
        if constexpr (HP) k_run_hp<ENV, R, P, SL, T, STORE><<<grid, block, smem, stream>>>(p, h);
        else k_run<ENV, R, P, SL, T, STORE><<<grid, block, smem, stream>>>(p);
    }
};

template <int ENV, bool HP>
cudaError_t launch_run(const Variant& v, const DevParams& p, int store, cudaStream_t stream, const HpParams& h) {
    // threads the grid covers: every agent, or with per-agent sets the launch positions of h (the active sets' agents)
    const uint64_t n = HP ? h.n_launch : p.n_agents;
    if (n == 0) return cudaSuccess;   // every set inactive: nothing to run, and a grid of zero CTAs is an error
    if (store == STORE_HYBRID) {
        if constexpr (SmemCapable<ENV>::value) {
            const unsigned grid = (unsigned)((n + 31) / 32);   // one warp per CTA: 32 agents, one per lane
            const size_t smem = smem_store_bytes<ENV>(v, store, p.n_live, p.S, p.vmax);
#define RLB_CALL(R, P, SL, T)                                                                                          \
    {                                                                                                                  \
        auto kern = RunKernel<HP, ENV, R, P, SL, T, STORE_HYBRID>::ptr();                                                          \
        cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);          \
        if (err != cudaSuccess) return err;                                                                            \
        RunKernel<HP, ENV, R, P, SL, T, STORE_HYBRID>::launch(grid, 32, smem, stream, p, h);                              \
    }
            RLB_VARIANT_SWITCH(v, RLB_CALL)
#undef RLB_CALL
            return cudaGetLastError();
        } else {
            return cudaErrorInvalidValue;
        }
    }
    if (store == STORE_SMEM) {
        if constexpr (SmemCapable<ENV>::value) {
            const unsigned grid = (unsigned)((n + 7) / 8);   // one warp per CTA: 8 agents x 4 lanes
            const size_t smem = smem_store_bytes<ENV>(v, store, p.S, p.S, p.vmax);
#define RLB_CALL(R, P, SL, T)                                                                                          \
    {                                                                                                                  \
        auto kern = RunKernel<HP, ENV, R, P, SL, T, STORE_SMEM>::ptr();                                                          \
        cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);          \
        if (err != cudaSuccess) return err;                                                                            \
        RunKernel<HP, ENV, R, P, SL, T, STORE_SMEM>::launch(grid, 32, smem, stream, p, h);                              \
    }
            RLB_VARIANT_SWITCH(v, RLB_CALL)
#undef RLB_CALL
            return cudaGetLastError();
        } else {
            return cudaErrorInvalidValue;
        }
    }
    const unsigned grid = grid_for(n);
    const size_t smem = EnvTab<ENV>::smem_bytes(p.S);
    if (store == STORE_LAZY) {   // trace agents, HBM tables, sweeps applied lazily: + the TD history in shared memory
        if (!v.trace) return cudaErrorInvalidValue;
        constexpr int kLazyBlock = RLB_LZ_BLOCK;
        const unsigned lz_grid = (unsigned)((n + kLazyBlock - 1) / kLazyBlock);
        const size_t hist = ((smem + 15) & ~(size_t)15) + (size_t)p.lz_cap * kLazyBlock * (v.real == RLB_REAL_F32 ? 4 : 8);
#define RLB_CALL(R, P, SL, T)                                                                                          \
    if constexpr (T) {                                                                                                 \
        auto kern = RunKernel<HP, ENV, R, P, SL, true, STORE_LAZY>::ptr();                                             \
        cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hist);          \
        if (err != cudaSuccess) return err;                                                                            \
        RunKernel<HP, ENV, R, P, SL, true, STORE_LAZY>::launch(lz_grid, kLazyBlock, hist, stream, p, h);               \
    }
        RLB_VARIANT_SWITCH(v, RLB_CALL)
#undef RLB_CALL
        return cudaGetLastError();
    }
#define RLB_CALL(R, P, SL, T)                                                   \
    {                                                                           \
        prefer_l1(RunKernel<HP, ENV, R, P, SL, T, STORE_GLOBAL>::ptr(), smem);                                  \
        RunKernel<HP, ENV, R, P, SL, T, STORE_GLOBAL>::launch(grid, kBlock, smem, stream, p, h);                \
    }
    RLB_VARIANT_SWITCH(v, RLB_CALL)
#undef RLB_CALL
    return cudaGetLastError();
}

template <int ENV, bool HP>
cudaError_t launch_run_model(const Variant& v, const DevParams& p, cudaStream_t stream, const HpParams& h) {
    // as launch_run: with per-agent sets the grid covers the launch positions of h (the active sets' agents)
    const uint64_t n = HP ? h.n_launch : p.n_agents;
    if (n == 0) return cudaSuccess;
    const unsigned grid = grid_for(n);
    const size_t smem = EnvTab<ENV>::smem_bytes(p.S);
#define RLB_CALL(R, P, SL, T)                                                                                          \
    {                                                                                                                  \
        if constexpr (HP) k_run_hp<ENV, R, P, SL, T, STORE_GLOBAL, true><<<grid, kBlock, smem, stream>>>(p, h);        \
        else k_run<ENV, R, P, SL, T, STORE_GLOBAL, true><<<grid, kBlock, smem, stream>>>(p);                           \
    }
    RLB_VARIANT_SWITCH(v, RLB_CALL)
#undef RLB_CALL
    return cudaGetLastError();
}

template <int ENV, bool HP>
cudaError_t run_kernel_attributes(const Variant& v, int store, cudaFuncAttributes* attr) {
    if (store == STORE_HYBRID) {
        if constexpr (SmemCapable<ENV>::value) {
#define RLB_CALL(R, P, SL, T) return cudaFuncGetAttributes(attr, RunKernel<HP, ENV, R, P, SL, T, STORE_HYBRID>::ptr())
            RLB_VARIANT_SWITCH(v, RLB_CALL)
#undef RLB_CALL
        }
        return cudaErrorInvalidValue;
    }
    if (store == STORE_SMEM) {
        if constexpr (SmemCapable<ENV>::value) {
#define RLB_CALL(R, P, SL, T) return cudaFuncGetAttributes(attr, RunKernel<HP, ENV, R, P, SL, T, STORE_SMEM>::ptr())
            RLB_VARIANT_SWITCH(v, RLB_CALL)
#undef RLB_CALL
        }
        return cudaErrorInvalidValue;
    }
    if (store == STORE_LAZY) {
#define RLB_CALL(R, P, SL, T) if constexpr (T) return cudaFuncGetAttributes(attr, RunKernel<HP, ENV, R, P, SL, true, STORE_LAZY>::ptr())
        RLB_VARIANT_SWITCH(v, RLB_CALL)
#undef RLB_CALL
        return cudaErrorInvalidValue;
    }
#define RLB_CALL(R, P, SL, T) return cudaFuncGetAttributes(attr, RunKernel<HP, ENV, R, P, SL, T, STORE_GLOBAL>::ptr())
    RLB_VARIANT_SWITCH(v, RLB_CALL)
#undef RLB_CALL
    return cudaSuccess;
}

// the step-level kernels that read hyper-parameters come in a plain and an _hp form (rlb_step_agent_kernels.inc); the
// _hp form takes the sets as its last parameter
#define RLB_STEP_LAUNCH(name, R, P, S, T, SMEM, ...)                                                               \
    do {                                                                                                           \
        if constexpr (HP) name##_hp<ENV, R, P, S, T><<<grid, kBlock, SMEM, stream>>>(__VA_ARGS__, a.sets);         \
        else name<ENV, R, P, S, T><<<grid, kBlock, SMEM, stream>>>(__VA_ARGS__);                                   \
    } while (0)

template <int ENV, bool HP>
cudaError_t launch_step(StepOp op, const Variant& v, const DevParams& p, const StepArgs& a, cudaStream_t stream) {
    const unsigned grid = grid_for(p.n_agents);
    const size_t smem = EnvTab<ENV>::smem_bytes(p.S);
    switch (op) {
        case OP_ENV_CONSTRUCT: k_env_construct<ENV><<<grid, kBlock, 0, stream>>>(p); break;
        case OP_ENV_RESET: k_env_reset<ENV><<<grid, kBlock, smem, stream>>>(p, a.u32_out); break;
        case OP_ENV_STEP:
            k_env_step<ENV><<<grid, kBlock, smem, stream>>>(p, a.action, a.u32_out, a.reward_out, a.term_out, a.not_ready_out, a.any_not_ready);
            break;
        case OP_GET_ACTION: {
#define RLB_CALL(R, P, S, T) RLB_STEP_LAUNCH(k_get_action, R, P, S, T, 0, p, a.obs, a.u32_out, a.any_not_ready)
            RLB_VARIANT_SWITCH(v, RLB_CALL)
#undef RLB_CALL
            break;
        }
        case OP_UPDATE: {
#define RLB_CALL(R, P, S, T) \
    RLB_STEP_LAUNCH(k_update, R, P, S, T, 0, p, a.obs, a.action, a.reward, a.term, a.obs2, a.action2, (R*)a.real_out, a.any_not_ready)
            RLB_VARIANT_SWITCH(v, RLB_CALL)
#undef RLB_CALL
            break;
        }
        case OP_POLICY_ROWS: {
#define RLB_CALL(R, P, S, T) k_policy_rows<ENV, R, P, S, T><<<grid, kBlock, 0, stream>>>(p, a.obs, (R*)a.real_out, a.which, a.any_not_ready)
            RLB_VARIANT_SWITCH(v, RLB_CALL)
#undef RLB_CALL
            break;
        }
        case OP_POLICY_UPDATE: {
#define RLB_CALL(R, P, S, T) RLB_STEP_LAUNCH(k_policy_update, R, P, S, T, 0, p, a.obs, a.action, (const R*)a.td_in, a.any_not_ready)
            RLB_VARIANT_SWITCH(v, RLB_CALL)
#undef RLB_CALL
            break;
        }
        case OP_SELECTOR_GET_ACTION: {
#define RLB_CALL(R, P, S, T) RLB_STEP_LAUNCH(k_selector_get_action, R, P, S, T, 0, p, a.obs, (const R*)a.values, a.u32_out, a.any_not_ready)
            RLB_VARIANT_SWITCH(v, RLB_CALL)
#undef RLB_CALL
            break;
        }
        case OP_SELECTOR_PROBS: {
#define RLB_CALL(R, P, S, T) RLB_STEP_LAUNCH(k_selector_probs, R, P, S, T, 0, p, a.obs, (const R*)a.values, (R*)a.real_out, a.any_not_ready)
            RLB_VARIANT_SWITCH(v, RLB_CALL)
#undef RLB_CALL
            break;
        }
        case OP_AGENT_STEP: {
#define RLB_CALL(R, P, S, T) \
    RLB_STEP_LAUNCH(k_agent_step, R, P, S, T, smem, p, a.kind_out, a.u32_out, a.u32_out2, a.reward_out, a.term_out, (R*)a.real_out)
            RLB_VARIANT_SWITCH(v, RLB_CALL)
#undef RLB_CALL
            break;
        }
    }
    return cudaGetLastError();
}

#define RLB_INSTANTIATE_ENV(ENV)                                                                         \
    template cudaError_t launch_run<ENV, false>(const Variant&, const DevParams&, int, cudaStream_t, const HpParams&); \
    template size_t smem_store_bytes<ENV>(const Variant&, int, uint32_t, uint32_t, uint32_t);                           \
    template cudaError_t launch_step<ENV, false>(StepOp, const Variant&, const DevParams&, const StepArgs&, cudaStream_t); \
    template cudaError_t run_kernel_attributes<ENV, false>(const Variant&, int, cudaFuncAttributes*);

// the same entry points with per-agent hyper-parameter sets (k_run_hp and the _hp step kernels); rlb_inst_<env>_hp.cu
#define RLB_INSTANTIATE_ENV_HP(ENV)                                                                      \
    template cudaError_t launch_run<ENV, true>(const Variant&, const DevParams&, int, cudaStream_t, const HpParams&);  \
    template cudaError_t launch_step<ENV, true>(StepOp, const Variant&, const DevParams&, const StepArgs&, cudaStream_t); \
    template cudaError_t run_kernel_attributes<ENV, true>(const Variant&, int, cudaFuncAttributes*);

#define RLB_INSTANTIATE_ENV_MODEL(ENV) template cudaError_t launch_run_model<ENV, false>(const Variant&, const DevParams&, cudaStream_t, const HpParams&);
// the same with per-agent hyper-parameter sets and per-set planning counts (k_run_hp with the model); rlb_inst_<env>_model_hp.cu
#define RLB_INSTANTIATE_ENV_MODEL_HP(ENV) template cudaError_t launch_run_model<ENV, true>(const Variant&, const DevParams&, cudaStream_t, const HpParams&);

}   // namespace rlb
