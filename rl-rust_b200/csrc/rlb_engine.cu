// rlb_engine.cu — engine lifecycle and the C ABI of include/rlb.h.
//
// The engine owns every device buffer: per-agent Q tables / UCB counts / eligibility rows
// in HBM (agent-major, one 32/64-byte-aligned row per state), per-agent scalars (RNG word
// index, epsilon, UCB t, Double flag, env state) as SoA arrays, the env transition tables,
// and a scratch ring for the per-episode record stream that k_run writes and
// k_episode_sums reduces.  There is no CPU path: every compute entry point needs a device.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <nvtx3/nvToolsExt.h>   // header-only NVTX v3: ranges show up in Nsight Systems / Compute timelines, no-ops otherwise

#include "rlb_host.h"
#include "rlb_launch.h"
#include "rlb_step_kernels.cuh"

using namespace rlb;

namespace {

rlb_status cuda_fail(cudaError_t err, const char* what) {
    set_error("%s: %s", what, cudaGetErrorString(err));
    return err == cudaErrorMemoryAllocation ? RLB_ERR_OOM : RLB_ERR_CUDA;
}

#define CK(call)                                                  \
    do {                                                          \
        cudaError_t err__ = (call);                               \
        if (err__ != cudaSuccess) return cuda_fail(err__, #call); \
    } while (0)


}   // namespace

struct rlb_engine {
    rlb_config cfg;
    uint32_t S = 0, A = 0, APAD = 0, T = 1;
    size_t real_size = 4;
    Variant variant{};
    int store = STORE_GLOBAL;          // where k_run keeps the tables: HBM or shared memory
    size_t smem_bytes = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    DevParams dp{};
    EnvTables tables;
    // owned device buffers
    void* d_q = nullptr; size_t q_bytes = 0;
    uint32_t* d_counts = nullptr; size_t counts_bytes = 0;
    void* d_etr = nullptr;
    void* d_etr_il = nullptr;   // warp-interleaved eligibility scratch of the hybrid store
    uint16_t* d_vis = nullptr;
    uint32_t* d_nvis = nullptr;
    uint64_t* d_rng_n = nullptr;
    double* d_eps = nullptr;
    uint64_t* d_ucb_t = nullptr;
    uint8_t* d_flag = nullptr;
    EnvState* d_env = nullptr;
    uint16_t* d_trans = nullptr;
    uint64_t* d_thr = nullptr;
    uint16_t* d_thr_state = nullptr;
    uint2* d_model_ent = nullptr;       // Dyna model (only while an InternalModelAgent wraps the agent)
    uint32_t* d_model_bits = nullptr;
    uint32_t* d_model_len = nullptr;
    unsigned long long* d_totals = nullptr;   // [3][8] (one block per call in flight): train steps, eval steps, eval episodes, (i64) eval return, trace rows
    uint64_t call_counter = 0;                // picks the totals block and the sums region of a call
    uint32_t* d_flagword = nullptr;
    // scratch
    void* d_episodes = nullptr; size_t episodes_cap = 0;
    double* d_sums = nullptr; size_t sums_cap = 0;
    void* d_stage[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    size_t stage_cap[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // device -> host pipeline of the episode records (run_range): a copy stream and, per half of the scratch, "launch
    // done" / "copy done" events
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_filled[2] = {nullptr, nullptr}, ev_drained[2] = {nullptr, nullptr};
    uint64_t last_pipeline_chunk = 0;  // episodes per scratch half of the last pipelined call
    uint64_t launch_counter = 0;       // k_run launches writing records for a host buffer, over all calls: picks the scratch half
    // rlb_agent_step: curr_obs / curr_action of every agent
    uint32_t* d_cur_obs = nullptr;
    uint32_t* d_cur_action = nullptr;
    void* h_step_stage = nullptr; size_t step_stage_cap = 0;   // rlb_agent_step: mapped pinned block for host outputs
    uint8_t* d_lz_slot = nullptr;      // lazy trace sweeps: row key -> slot candidate [N][S]
    uint8_t* d_lz_tmat = nullptr;      //                    sweeps applied per slot  [N][VMAX]
    uint32_t d_lz_tmat_rows = 0;
    double* d_log_table = nullptr;     // ln(t) for t < RLB_LOG_TABLE_N (UCB), filled on the device by portable_log
    // per-agent hyper-parameter sets (rlb_engine_set_hparams); hp_n = 0 while rlb_config's values apply
    uint32_t hp_n = 0;
    rlb_hparams* d_hp_sets = nullptr;  // [hp_n]
    uint32_t* d_hp_group = nullptr;    // [N] set of each agent
    uint32_t* d_hp_order = nullptr;    // [N] local agent indices, stably sorted by set: the grouped reduction's read order
    uint32_t* d_hp_offsets = nullptr;  // [hp_n + 1] where each set starts in d_hp_order
    void* d_hp_q0 = nullptr;           // [hp_n] default_value narrowed to Real, for the table fills
    double* d_hp_eps0 = nullptr;       // [hp_n] initial_epsilon
    std::vector<uint32_t> h_hp_order, h_hp_offsets;   // host copies of d_hp_order / d_hp_offsets
    // active sets (rlb_engine_set_active_sets); hp_active is empty while every set is active
    std::vector<uint8_t> hp_active;    // [hp_n] nonzero: the set takes part in train / evaluate calls
    uint32_t* d_hp_run = nullptr;      // [hp_n_run] d_hp_order restricted to the active sets: k_run_hp's agent list and the reduction's order
    uint32_t* d_hp_run_offsets = nullptr;   // [hp_n + 1] where each set starts in d_hp_run (an inactive set has length 0)
    uint64_t hp_n_run = 0;
    // per-set Dyna planning counts (rlb_engine_set_planning_steps); empty while no per-set model is attached
    std::vector<uint32_t> h_hp_planning;   // [hp_n]
    uint32_t* d_hp_planning = nullptr;     // [hp_n] device copy: HpParams::planning
    // per-set bootstrap targets (rlb_engine_set_targets); every entry cfg.target_kind until that call
    std::vector<int32_t> h_hp_targets;     // [hp_n]
    int32_t* d_hp_targets = nullptr;       // [hp_n] device copy: HpParams::targets
    // Calls whose work is enqueued but not yet waited for (rlb_agent_train_range_async): at most two, so that the
    // kernels of call i + 1 are in the queue before the host blocks on the copies of call i.
    struct Pending {
        int mode = 0;
        rlb_train_out* out = nullptr;
        uint64_t* eval_steps_out = nullptr;
        std::vector<cudaEvent_t> events;             // (start, stop) per k_run launch
        cudaEvent_t done = nullptr;                  // after everything the call enqueued on the main stream
        cudaEvent_t copies_done = nullptr;           // after its last record copy on the copy stream (pipelined calls)
        unsigned long long* h_totals = nullptr;      // pinned [8]
        bool pipelined = false;
        bool host_records = false;                   // the call copies per-agent records to a host buffer
        rlb_traj_record* d_traj = nullptr; uint64_t* d_traj_count = nullptr; bool own_traj = false, own_count = false;
        void* d_td = nullptr; uint64_t* d_td_count = nullptr; bool own_td = false, own_td_count = false;
    };
    std::vector<Pending> pending;
    std::vector<cudaEvent_t> event_pool;             // timing events not in use
    std::vector<unsigned long long*> totals_pool;    // pinned [8] blocks not in use
};

namespace {

bool is_device_ptr(const void* p) {
    cudaPointerAttributes attr;
    cudaError_t err = cudaPointerGetAttributes(&attr, p);
    if (err != cudaSuccess) { cudaGetLastError(); return false; }
    return attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged;
}

// copy device -> caller buffer (host or device)
cudaError_t copy_out(rlb_engine* e, void* dst, const void* src_dev, size_t bytes) {
    if (!dst || !bytes) return cudaSuccess;
    cudaError_t err = cudaMemcpyAsync(dst, src_dev, bytes, is_device_ptr(dst) ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, e->stream);
    if (err != cudaSuccess) return err;
    return is_device_ptr(dst) ? cudaSuccess : cudaStreamSynchronize(e->stream);
}

// the same without waiting: complete once the stream reaches it (immediately for pageable host memory)
cudaError_t copy_async(rlb_engine* e, void* dst, const void* src_dev, size_t bytes) {
    if (!dst || !bytes) return cudaSuccess;
    return cudaMemcpyAsync(dst, src_dev, bytes, is_device_ptr(dst) ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, e->stream);
}

// make caller data (host or device) readable on the device; returns a device pointer
cudaError_t stage_in(rlb_engine* e, int slot, const void* src, size_t bytes, const void** out) {
    if (!src) { *out = nullptr; return cudaSuccess; }
    if (is_device_ptr(src)) { *out = src; return cudaSuccess; }
    if (e->stage_cap[slot] < bytes) {
        if (e->d_stage[slot]) cudaFree(e->d_stage[slot]);
        e->d_stage[slot] = nullptr; e->stage_cap[slot] = 0;
        cudaError_t err = cudaMalloc(&e->d_stage[slot], bytes);
        if (err != cudaSuccess) return err;
        e->stage_cap[slot] = bytes;
    }
    cudaError_t err = cudaMemcpyAsync(e->d_stage[slot], src, bytes, cudaMemcpyHostToDevice, e->stream);
    *out = e->d_stage[slot];
    return err;
}
// device scratch to receive an output that the caller wants on the host (or the caller's own device buffer)
cudaError_t stage_out(rlb_engine* e, int slot, void* dst, size_t bytes, void** dev) {
    if (!dst) { *dev = nullptr; return cudaSuccess; }
    if (is_device_ptr(dst)) { *dev = dst; return cudaSuccess; }
    if (e->stage_cap[slot] < bytes) {
        if (e->d_stage[slot]) cudaFree(e->d_stage[slot]);
        e->d_stage[slot] = nullptr; e->stage_cap[slot] = 0;
        cudaError_t err = cudaMalloc(&e->d_stage[slot], bytes);
        if (err != cudaSuccess) return err;
        e->stage_cap[slot] = bytes;
    }
    *dev = e->d_stage[slot];
    return cudaSuccess;
}
cudaError_t finish_out(rlb_engine* e, void* dst, const void* dev, size_t bytes) {
    if (!dst || dst == dev) return cudaSuccess;
    return copy_out(e, dst, dev, bytes);
}

template <typename V>
cudaError_t fill(rlb_engine* e, V* ptr, uint64_t n, V value) {
    if (!n) return cudaSuccess;
    unsigned grid = (unsigned)std::min<uint64_t>((n + 255) / 256, 148u * 16u);
    k_fill<V><<<grid, 256, 0, e->stream>>>(ptr, n, value);
    return cudaGetLastError();
}

cudaError_t fill_q_default(rlb_engine* e) {
    const uint64_t n = e->q_bytes / e->real_size;
    if (e->hp_n) return launch_fill_grouped(e->d_q, e->real_size, n / e->cfg.n_agents, e->cfg.n_agents, e->d_hp_q0, e->d_hp_group, e->stream);
    if (e->cfg.real_kind == RLB_REAL_F32) return fill<float>(e, (float*)e->d_q, n, (float)e->cfg.default_value);
    return fill<double>(e, (double*)e->d_q, n, e->cfg.default_value);
}

// UniformEpsilonGreed::new / reset: epsilon = initial_epsilon (uniform_epsilon_greed.rs:31,78-80)
cudaError_t fill_eps_initial(rlb_engine* e) {
    if (e->hp_n) return launch_fill_grouped(e->d_eps, sizeof(double), 1, e->cfg.n_agents, e->d_hp_eps0, e->d_hp_group, e->stream);
    return fill<double>(e, e->d_eps, e->cfg.n_agents, e->cfg.initial_epsilon);
}

cudaError_t dispatch_run(rlb_engine* e, const DevParams& p) {
    const bool masked = !e->hp_active.empty();   // only the active sets' agents run: a launch sized to them
    const HpParams sets{e->d_hp_sets, e->d_hp_group, masked ? e->d_hp_run : nullptr, masked ? e->hp_n_run : e->cfg.n_agents, e->d_hp_planning,
                        e->d_hp_targets};
    if (p.planning_steps && p.mode == 0 && e->hp_n) {   // the model under sets: each set's own planning count
        switch (e->cfg.env_kind) {
            case RLB_ENV_BLACKJACK: return launch_run_model<RLB_ENV_BLACKJACK, true>(e->variant, p, e->stream, sets);
            case RLB_ENV_FROZEN_LAKE: return launch_run_model<RLB_ENV_FROZEN_LAKE, true>(e->variant, p, e->stream, sets);
            case RLB_ENV_CLIFF_WALKING: return launch_run_model<RLB_ENV_CLIFF_WALKING, true>(e->variant, p, e->stream, sets);
            default: return launch_run_model<RLB_ENV_TAXI, true>(e->variant, p, e->stream, sets);
        }
    }
    if (p.planning_steps && p.mode == 0) {   // InternalModelAgent::update on the training path; evaluate never touches the model
        switch (e->cfg.env_kind) {
            case RLB_ENV_BLACKJACK: return launch_run_model<RLB_ENV_BLACKJACK>(e->variant, p, e->stream);
            case RLB_ENV_FROZEN_LAKE: return launch_run_model<RLB_ENV_FROZEN_LAKE>(e->variant, p, e->stream);
            case RLB_ENV_CLIFF_WALKING: return launch_run_model<RLB_ENV_CLIFF_WALKING>(e->variant, p, e->stream);
            default: return launch_run_model<RLB_ENV_TAXI>(e->variant, p, e->stream);
        }
    }
    if (e->hp_n) {   // every agent with its own hyper-parameter set (with a model: evaluate, which never touches it)
        switch (e->cfg.env_kind) {
            case RLB_ENV_BLACKJACK: return launch_run<RLB_ENV_BLACKJACK, true>(e->variant, p, e->store, e->stream, sets);
            case RLB_ENV_FROZEN_LAKE: return launch_run<RLB_ENV_FROZEN_LAKE, true>(e->variant, p, e->store, e->stream, sets);
            case RLB_ENV_CLIFF_WALKING: return launch_run<RLB_ENV_CLIFF_WALKING, true>(e->variant, p, e->store, e->stream, sets);
            default: return launch_run<RLB_ENV_TAXI, true>(e->variant, p, e->store, e->stream, sets);
        }
    }
    switch (e->cfg.env_kind) {
        case RLB_ENV_BLACKJACK: return launch_run<RLB_ENV_BLACKJACK>(e->variant, p, e->store, e->stream);
        case RLB_ENV_FROZEN_LAKE: return launch_run<RLB_ENV_FROZEN_LAKE>(e->variant, p, e->store, e->stream);
        case RLB_ENV_CLIFF_WALKING: return launch_run<RLB_ENV_CLIFF_WALKING>(e->variant, p, e->store, e->stream);
        default: return launch_run<RLB_ENV_TAXI>(e->variant, p, e->store, e->stream);
    }
}

// Where k_run keeps the per-agent tables.  The shared-memory (thread-group) store pays when every step sweeps many
// rows, i.e. for the eligibility-trace agents of the 4-action envs; one-step updates touch two rows per step and run
// faster from HBM at full occupancy (measured, DESIGN.md §7).
size_t store_bytes(rlb_engine* e, int store) {
    switch (e->cfg.env_kind) {
        case RLB_ENV_BLACKJACK: return smem_store_bytes<RLB_ENV_BLACKJACK>(e->variant, store, e->S, e->S, e->dp.vmax);
        case RLB_ENV_FROZEN_LAKE: return smem_store_bytes<RLB_ENV_FROZEN_LAKE>(e->variant, store, store == STORE_HYBRID ? e->dp.n_live : e->S, e->S, e->dp.vmax);
        case RLB_ENV_CLIFF_WALKING: return smem_store_bytes<RLB_ENV_CLIFF_WALKING>(e->variant, store, store == STORE_HYBRID ? e->dp.n_live : e->S, e->S, e->dp.vmax);
        default: return smem_store_bytes<RLB_ENV_TAXI>(e->variant, store, e->S, e->S, e->dp.vmax);
    }
}

rlb_status pick_store(rlb_engine* e) {
    const size_t per_block_max = 227 * 1024, per_sm = 228 * 1024;
    const size_t b_group = store_bytes(e, STORE_SMEM), b_hybrid = store_bytes(e, STORE_HYBRID);
    const bool fits_group = b_group > 0 && b_group <= per_block_max && e->S <= 256;      // GroupStore keeps visited states in 8 bits
    const bool fits_hybrid = b_hybrid > 0 && b_hybrid <= per_block_max && e->S <= 64;   // DevParams::row_lut holds 64 states
    int want = e->cfg.store_kind;
    if (e->cfg.planning_steps) {
        // planning replays arbitrary remembered states, terminal ones included, and the model itself lives in HBM
        if (want != 0 && want != STORE_GLOBAL) { set_error("a Dyna model (planning_steps > 0) needs the HBM store"); return RLB_ERR_UNSUPPORTED; }
        want = STORE_GLOBAL;
    } else if (want == 0) {
        // measured (DESIGN.md §7): one-step updates touch two rows per step and run fastest from HBM at full occupancy;
        // trace sweeps want the tables on chip.  Hybrid when >= 3 warps per SM fit, else the thread-group store (>= 4).
        want = STORE_GLOBAL;
        if (e->variant.trace) {
            if (fits_hybrid && 3 * (b_hybrid + 1024) <= per_sm) want = STORE_HYBRID;   // f64 C2 at 3 CTAs/SM: 4.2e9 vs 3.4e9 (groups, HBM)
            else if (fits_group && 4 * (b_group + 1024) <= per_sm) want = STORE_SMEM;
            // tables too big for the chip: HBM, and the sweeps applied lazily where episodes are long (Taxi: 10-12 rows
            // swept per step; Blackjack's 1.5 rows per step are cheaper swept as they come — profiles/r02s_lazy_phase.txt)
            else if (e->dp.vmax <= 255 && e->cfg.env_kind != RLB_ENV_BLACKJACK) want = STORE_LAZY;
        }
    } else if (want == STORE_SMEM && !fits_group) {
        set_error("store_kind = shared memory (thread groups): needs %zu bytes per 8 agents (max %zu) or the env is not compiled for it", b_group, per_block_max);
        return RLB_ERR_UNSUPPORTED;
    } else if (want == STORE_HYBRID && !fits_hybrid) {
        set_error("store_kind = hybrid: needs %zu bytes per 32 agents (max %zu) or the env is not compiled for it", b_hybrid, per_block_max);
        return RLB_ERR_UNSUPPORTED;
    }
    if (want == STORE_LAZY) {
        if (!e->variant.trace) { set_error("store_kind = lazy sweeps is for eligibility-trace agents"); return RLB_ERR_UNSUPPORTED; }
        if (e->dp.vmax > 255) { set_error("store_kind = lazy sweeps: more than 255 eligibility rows per agent"); return RLB_ERR_UNSUPPORTED; }
        // TD history per agent: one value per sweep of an episode (max_steps + 1; Blackjack: a hand holds 16 cards), capped by
        // 64 KB of shared memory per 128-agent CTA — a longer episode brings every row up to date when the history is full
        const uint64_t by_steps = e->cfg.env_kind == RLB_ENV_BLACKJACK ? 32ull : (uint64_t)e->cfg.max_steps + 1ull;
        const uint64_t by_smem = (64u * 1024u) / (128u * e->real_size);
        e->dp.lz_cap = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(std::min<uint64_t>(by_steps, by_smem), 255));
        if (const char* t = getenv("RLB_LZ_CAP")) {   // tuning override (tools/lazy_phase.py): sweeps between two full updates of the rows
            const long v = atol(t);
            if (v >= 1) e->dp.lz_cap = (uint32_t)std::min<uint64_t>((uint64_t)v, e->dp.lz_cap);
        }
        const uint64_t N = e->cfg.n_agents;
        if (!e->d_lz_slot) {
            CK(cudaMalloc(&e->d_lz_slot, (size_t)N * e->S));
            CK(cudaMemsetAsync(e->d_lz_slot, 0, (size_t)N * e->S, e->stream));
        }
        if (e->d_lz_tmat_rows < e->dp.vmax) {
            if (e->d_lz_tmat) cudaFree(e->d_lz_tmat);
            CK(cudaMalloc(&e->d_lz_tmat, (size_t)N * e->dp.vmax));
            CK(cudaMemsetAsync(e->d_lz_tmat, 0, (size_t)N * e->dp.vmax, e->stream));
            e->d_lz_tmat_rows = e->dp.vmax;
        }
        e->dp.lz_slot = e->d_lz_slot; e->dp.lz_tmat = e->d_lz_tmat;
    }
    e->store = want;
    e->smem_bytes = want == STORE_SMEM ? b_group : (want == STORE_HYBRID ? b_hybrid : 0);
    if (want == STORE_HYBRID && e->variant.trace && !e->d_etr_il) {
        const uint64_t n32 = (e->cfg.n_agents + 31) / 32 * 32;
        CK(cudaMalloc(&e->d_etr_il, (size_t)n32 * e->dp.vmax * e->APAD * e->real_size));
        e->dp.etr_il = e->d_etr_il;
    }
    return RLB_OK;
}

cudaError_t dispatch_step(rlb_engine* e, StepOp op, const StepArgs& a) {
    if (e->hp_n) {
        StepArgs with_sets = a;
        with_sets.sets = HpParams{e->d_hp_sets, e->d_hp_group, nullptr, 0, e->d_hp_planning, e->d_hp_targets};
        switch (e->cfg.env_kind) {
            case RLB_ENV_BLACKJACK: return launch_step<RLB_ENV_BLACKJACK, true>(op, e->variant, e->dp, with_sets, e->stream);
            case RLB_ENV_FROZEN_LAKE: return launch_step<RLB_ENV_FROZEN_LAKE, true>(op, e->variant, e->dp, with_sets, e->stream);
            case RLB_ENV_CLIFF_WALKING: return launch_step<RLB_ENV_CLIFF_WALKING, true>(op, e->variant, e->dp, with_sets, e->stream);
            default: return launch_step<RLB_ENV_TAXI, true>(op, e->variant, e->dp, with_sets, e->stream);
        }
    }
    switch (e->cfg.env_kind) {
        case RLB_ENV_BLACKJACK: return launch_step<RLB_ENV_BLACKJACK>(op, e->variant, e->dp, a, e->stream);
        case RLB_ENV_FROZEN_LAKE: return launch_step<RLB_ENV_FROZEN_LAKE>(op, e->variant, e->dp, a, e->stream);
        case RLB_ENV_CLIFF_WALKING: return launch_step<RLB_ENV_CLIFF_WALKING>(op, e->variant, e->dp, a, e->stream);
        default: return launch_step<RLB_ENV_TAXI>(op, e->variant, e->dp, a, e->stream);
    }
}

// Eligibility rows an agent can hold.  Without a model: distinct states updated in one episode <= episode length <=
// max_steps + 1 (truncation pseudo-step), <= S; Blackjack has no step limit, a hand holds at most 16 cards
// (blackjack.rs:32-35).  With a Dyna model the planning updates (terminated = false, internal_model_agent.rs:68-75) put
// any remembered state into the trace map and nothing clears it before the next real termination: S rows.
uint32_t wanted_vmax(const rlb_engine* e) {
    if (e->cfg.planning_steps) return e->S;
    const uint64_t by_steps = e->cfg.env_kind == RLB_ENV_BLACKJACK ? 32ull : (uint64_t)e->cfg.max_steps + 1ull;
    return (uint32_t)std::min<uint64_t>(e->S, by_steps);
}
rlb_status ensure_trace_buffers(rlb_engine* e) {
    if (!e->variant.trace) return RLB_OK;
    const uint64_t N = e->cfg.n_agents;
    const uint32_t need = wanted_vmax(e);
    if (e->d_etr && e->dp.vmax >= need) return RLB_OK;
    void* etr = nullptr;
    uint16_t* vis = nullptr;
    const size_t row = (size_t)e->APAD * e->real_size;
    CK(cudaMalloc(&etr, (size_t)N * need * row));
    CK(cudaMalloc(&vis, (size_t)N * need * sizeof(uint16_t)));
    if (e->d_etr) {   // keep the live rows: same per-agent order, wider stride
        const size_t old_v = e->dp.vmax;
        CK(cudaMemcpy2DAsync(etr, need * row, e->d_etr, old_v * row, old_v * row, N, cudaMemcpyDeviceToDevice, e->stream));
        CK(cudaMemcpy2DAsync(vis, need * 2, e->d_vis, old_v * 2, old_v * 2, N, cudaMemcpyDeviceToDevice, e->stream));
        CK(cudaStreamSynchronize(e->stream));
        cudaFree(e->d_etr); cudaFree(e->d_vis);
        if (e->d_etr_il) { cudaFree(e->d_etr_il); e->d_etr_il = nullptr; e->dp.etr_il = nullptr; }
    }
    e->d_etr = etr; e->d_vis = vis;
    e->dp.etr = etr; e->dp.vis = vis; e->dp.vmax = need;
    return RLB_OK;
}

// InternalModelAgent::new(agent, RandomModel::default(), planning_steps) / unwrap when planning_steps == 0 (which also
// drops the per-set planning counts)
rlb_status attach_model(rlb_engine* e, uint32_t planning_steps) {
    const uint64_t N = e->cfg.n_agents;
    e->cfg.planning_steps = planning_steps;
    e->dp.planning_steps = planning_steps;
    if (!planning_steps) {
        void* bufs[] = {e->d_model_ent, e->d_model_bits, e->d_model_len, e->d_hp_planning};
        CK(cudaStreamSynchronize(e->stream));
        for (void* b : bufs) if (b) cudaFree(b);
        e->d_hp_planning = nullptr;
        e->h_hp_planning.clear();
        e->d_model_ent = nullptr; e->d_model_bits = nullptr; e->d_model_len = nullptr;
        e->dp.model_ent = nullptr; e->dp.model_bits = nullptr; e->dp.model_len = nullptr; e->dp.mcap = 0; e->dp.mwords = 0;
        return RLB_OK;
    }
    const uint32_t mcap = e->S * e->A, mwords = (mcap + 31u) / 32u;
    if (!e->d_model_ent) {
        CK(cudaMalloc(&e->d_model_ent, (size_t)N * mcap * sizeof(uint2)));
        CK(cudaMalloc(&e->d_model_bits, (size_t)N * mwords * sizeof(uint32_t)));
        CK(cudaMalloc(&e->d_model_len, N * sizeof(uint32_t)));
    }
    CK(cudaMemsetAsync(e->d_model_bits, 0, (size_t)N * mwords * sizeof(uint32_t), e->stream));
    CK(cudaMemsetAsync(e->d_model_len, 0, N * sizeof(uint32_t), e->stream));
    e->dp.model_ent = e->d_model_ent; e->dp.model_bits = e->d_model_bits; e->dp.model_len = e->d_model_len;
    e->dp.mcap = mcap; e->dp.mwords = mwords;
    return ensure_trace_buffers(e);
}

// (re)build the selector state: UniformEpsilonGreed::new / UpperConfidenceBound::new
rlb_status install_selector(rlb_engine* e, int kind) {
    const uint64_t N = e->cfg.n_agents;
    e->cfg.selector_kind = kind;
    e->variant.sel = kind;
    CK(fill_eps_initial(e));
    CK(fill<uint64_t>(e, e->d_ucb_t, N, 1ull));
    if (kind == RLB_SEL_UCB) {
        if (!e->d_counts) {
            e->counts_bytes = (size_t)N * e->S * e->APAD * sizeof(uint32_t);
            CK(cudaMalloc(&e->d_counts, e->counts_bytes));
        }
        CK(cudaMemsetAsync(e->d_counts, 0, e->counts_bytes, e->stream));
        if (!e->d_log_table) {   // ln(t) table of the UCB bonus
            CK(cudaMalloc(&e->d_log_table, (size_t)RLB_LOG_TABLE_N * sizeof(double)));
            k_fill_log_table<<<(RLB_LOG_TABLE_N + 255) / 256, 256, 0, e->stream>>>(e->d_log_table, RLB_LOG_TABLE_N);
            CK(cudaGetLastError());
            e->dp.log_table = e->d_log_table; e->dp.log_table_n = RLB_LOG_TABLE_N;
        }
    }
    e->dp.counts = e->d_counts;
    return RLB_OK;
}

size_t episode_rec_size(const rlb_engine* e) { return e->cfg.real_kind == RLB_REAL_F32 ? sizeof(rlb_episode_f32) : sizeof(rlb_episode_f64); }

rlb_status ensure_episode_scratch(rlb_engine* e, uint64_t episodes, uint64_t sums_values) {
    const size_t need = (size_t)episodes * e->cfg.n_agents * episode_rec_size(e);
    if (e->episodes_cap < need) {
        if (e->d_episodes) cudaFree(e->d_episodes);
        e->d_episodes = nullptr; e->episodes_cap = 0;
        CK(cudaMalloc(&e->d_episodes, need));
        e->episodes_cap = need;
    }
    const size_t need_s = (size_t)sums_values * sizeof(double);
    if (e->sums_cap < need_s) {
        if (e->d_sums) cudaFree(e->d_sums);
        e->d_sums = nullptr; e->sums_cap = 0;
        CK(cudaMalloc(&e->d_sums, need_s));
        e->sums_cap = need_s;
    }
    return RLB_OK;
}

// how many episode indices one launch may cover so that the record stream fits the scratch budget
uint64_t chunk_episodes(const rlb_engine* e, uint64_t want) {
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); free_b = 1ull << 30; }
    size_t budget = std::min<size_t>((size_t)16 << 30, (free_b + e->episodes_cap) / 3);
    const size_t per_ep = (size_t)e->cfg.n_agents * episode_rec_size(e);
    uint64_t chunk = std::max<uint64_t>(1, budget / std::max<size_t>(per_ep, 1));
    return std::min<uint64_t>(chunk, std::max<uint64_t>(want, 1));
}

// sums_out [n_ep][4], or [n_ep][hp_n][4] with hyper-parameter sets
rlb_status reduce_episodes(rlb_engine* e, uint64_t n_ep, const void* records, double* sums_out) {
    if (!n_ep) return RLB_OK;
    if (e->hp_n) {   // with inactive sets: only the active sets' agents are read, an inactive set's row is 0.0
        const bool masked = !e->hp_active.empty();
        CK(launch_episode_sums_grouped(e->cfg.real_kind, records, e->cfg.n_agents, masked ? e->d_hp_run : e->d_hp_order,
                                       masked ? e->d_hp_run_offsets : e->d_hp_offsets, e->hp_n, n_ep, sums_out, e->stream));
        return RLB_OK;
    }
    if (e->cfg.real_kind == RLB_REAL_F32) k_episode_sums<float><<<(unsigned)n_ep, 256, 0, e->stream>>>(records, e->cfg.n_agents, sums_out);
    else k_episode_sums<double><<<(unsigned)n_ep, 256, 0, e->stream>>>(records, e->cfg.n_agents, sums_out);
    CK(cudaGetLastError());
    return RLB_OK;
}

// The copy stream and the events of the record pipeline, created on first use.
rlb_status ensure_copy_pipeline(rlb_engine* e) {
    if (e->copy_stream) return RLB_OK;
    CK(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
    for (int b = 0; b < 2; ++b) {
        CK(cudaEventCreateWithFlags(&e->ev_filled[b], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&e->ev_drained[b], cudaEventDisableTiming));
    }
    return RLB_OK;
}

bool valid_cfg(const rlb_config* c) {
    if (!c || c->struct_size != sizeof(rlb_config)) { set_error("rlb_config.struct_size mismatch (got %u, want %zu)", c ? c->struct_size : 0u, sizeof(rlb_config)); return false; }
    if (c->env_kind < 0 || c->env_kind > 3) { set_error("env_kind out of range"); return false; }
    if (c->policy_kind < 0 || c->policy_kind > 1 || c->selector_kind < 0 || c->selector_kind > 1 || c->target_kind < 0 ||
        c->target_kind > 2 || c->agent_kind < 0 || c->agent_kind > 1 || c->real_kind < 0 || c->real_kind > 1 ||
        c->decay_kind < 0 || c->decay_kind > 1) { set_error("enum field out of range"); return false; }
    if (c->n_agents == 0) { set_error("n_agents must be > 0"); return false; }
    if (c->store_kind > 4) { set_error("store_kind out of range"); return false; }
    return true;
}

// The flag word the step-level kernels raise (FLAG_* in rlb_step_kernels.cuh): cleared before the launch, read after it.
cudaError_t flags_clear(rlb_engine* e) { return cudaMemsetAsync(e->d_flagword, 0, 4, e->stream); }
rlb_status flags_check(rlb_engine* e) {
    uint32_t any = 0;
    CK(cudaMemcpyAsync(&any, e->d_flagword, 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    if (any & FLAG_BAD_ARG) {
        set_error("observation, action or model entry out of range for this env (the reference would panic on the same index); the agents concerned were left untouched");
        return RLB_ERR_INVALID_ARG;
    }
    if (any & FLAG_TRACE_FULL) {
        set_error("update(): the eligibility trace would exceed the %u rows the engine holds per agent (episodes of its own env never do)", e->dp.vmax);
        return RLB_ERR_INVALID_ARG;
    }
    if (any & FLAG_DEAD_STATE) {
        set_error("update(): curr_obs is a terminal cell of the env (never an observation an action is taken from); unsupported by the trace agent's table stores");
        return RLB_ERR_UNSUPPORTED;
    }
    if (any & FLAG_NOT_READY) { set_error("EnvNotReady: step() before reset() or after termination"); return RLB_ERR_ENV_NOT_READY; }
    return RLB_OK;
}

// ---- the fused path: enqueue everything, wait later -------------------------------------------------------------
cudaEvent_t take_event(rlb_engine* e) {
    if (!e->event_pool.empty()) { cudaEvent_t ev = e->event_pool.back(); e->event_pool.pop_back(); return ev; }
    cudaEvent_t ev = nullptr;
    if (cudaEventCreate(&ev) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return ev;
}

// Block until the OLDEST pending call is complete and fill its outputs.
rlb_status finish_oldest(rlb_engine* e) {
    if (e->pending.empty()) return RLB_OK;
    rlb_engine::Pending pd = std::move(e->pending.front());
    e->pending.erase(e->pending.begin());
    rlb_status status = RLB_OK;
    auto note = [&](cudaError_t err, const char* what) { if (err != cudaSuccess && status == RLB_OK) status = cuda_fail(err, what); };
    note(cudaEventSynchronize(pd.done), "cudaEventSynchronize(done)");                  // kernels, reductions, sums and totals copies
    if (pd.copies_done) note(cudaEventSynchronize(pd.copies_done), "cudaEventSynchronize(copies)");   // this call's records are in host memory
    float ms_total = 0.f;
    for (size_t k = 0; k + 1 < pd.events.size(); k += 2) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, pd.events[k], pd.events[k + 1]) == cudaSuccess) ms_total += ms; else cudaGetLastError();
    }
    const uint32_t launches = (uint32_t)(pd.events.size() / 2);
    for (cudaEvent_t ev : pd.events) e->event_pool.push_back(ev);
    e->event_pool.push_back(pd.done);
    if (pd.copies_done) e->event_pool.push_back(pd.copies_done);
    unsigned long long totals[8];
    std::memcpy(totals, pd.h_totals, sizeof totals);
    e->totals_pool.push_back(pd.h_totals);
    const uint64_t N = e->cfg.n_agents;
    if (pd.d_traj) {
        if (pd.own_traj) { note(copy_out(e, pd.out->traj, pd.d_traj, N * pd.out->traj_capacity * sizeof(rlb_traj_record)), "copy traj"); cudaFree(pd.d_traj); }
        if (pd.own_count) { if (pd.out->traj_count) note(copy_out(e, pd.out->traj_count, pd.d_traj_count, N * sizeof(uint64_t)), "copy traj_count"); cudaFree(pd.d_traj_count); }
    }
    if (pd.d_td) {
        if (pd.own_td) { note(copy_out(e, pd.out->td_steps, pd.d_td, N * pd.out->td_capacity * e->real_size), "copy td_steps"); cudaFree(pd.d_td); }
        if (pd.own_td_count) { if (pd.out->td_count) note(copy_out(e, pd.out->td_count, pd.d_td_count, N * sizeof(uint64_t)), "copy td_count"); cudaFree(pd.d_td_count); }
    }
    if (pd.mode == 0 && pd.out) {
        pd.out->train_steps = totals[0]; pd.out->eval_steps = totals[1]; pd.out->eval_episodes = totals[2];
        pd.out->eval_return_sum = (double)(long long)totals[3];   // an exact integer (rlb_device.cuh, LaneTotals)
        pd.out->kernel_ms = ms_total; pd.out->kernel_launches = launches; pd.out->trace_rows = totals[4];
    }
    if (pd.mode == 1 && pd.eval_steps_out) *pd.eval_steps_out = totals[1];
    return status;
}
rlb_status finish_pending(rlb_engine* e) {
    rlb_status status = RLB_OK;
    while (!e->pending.empty()) {
        rlb_status st = finish_oldest(e);
        if (status == RLB_OK) status = st;
    }
    return status;
}
// every entry point but the asynchronous train call: select the device, complete what is pending
#define ENTER(e)                                           \
    do {                                                   \
        CK(cudaSetDevice((e)->cfg.device));                \
        rlb_status st__ = finish_pending(e);               \
        if (st__ != RLB_OK) return st__;                   \
    } while (0)

rlb_status enqueue_range(rlb_engine* e, int mode, uint64_t begin, uint64_t end, uint64_t eval_at, rlb_train_out* out,
                         void* eval_episodes_out, double* eval_sums_out, uint64_t* eval_steps_out, bool async_call = false) {
    const uint64_t N = e->cfg.n_agents;
    const size_t rec = episode_rec_size(e);
    const uint64_t total = end - begin;
    const uint64_t sums_per_ep = 4ull * (e->hp_n ? e->hp_n : 1u);   // [4] per episode, [n_sets][4] with hyper-parameter sets
    const bool want_records = mode == 0 ? (out && (out->episodes || out->episode_sums)) : (eval_episodes_out || eval_sums_out);
    uint64_t chunk = std::min<uint64_t>(total, 0xffffffffull);   // a launch counts its episodes in 32 bits
    // Records for a HOST buffer are pipelined: the range is cut into (at least) four launches writing alternately into
    // the two halves of the scratch, and while launch i + 1 runs the records of launch i travel to the host on a second
    // stream — the PCIe copy (1.7 GB per step on C2, 3.2 GB on C4) hides behind the kernels, the tail of the last copy
    // behind the NEXT call's kernels when the caller uses the asynchronous form.
    void* const rec_host = mode == 0 ? (out ? out->episodes : nullptr) : eval_episodes_out;
    const bool pipelined = rec_host && !is_device_ptr(rec_host) && total >= 8;
    if (want_records) {
        chunk = std::min<uint64_t>(chunk, chunk_episodes(e, total));
        // A blocking call hides its record copy behind its own kernels: at least four launches over the two halves.  An
        // asynchronous call hides it behind the NEXT call's kernel, so it stays ONE launch when its records fit a half
        // (each extra launch costs its tail: the last CTAs of a 32 768-CTA grid run on a mostly idle GPU).
        if (pipelined) chunk = std::max<uint64_t>(1, std::min<uint64_t>((chunk + 1) / 2, async_call ? total : (total + 3) / 4));
    }
    // A call may overlap the one before it when both stream records through the same two scratch halves — or when
    // neither sends records to the host at all: then everything either call does is in main-stream order (the record
    // scratch is written by call i + 1's kernel only after call i's reduction has read it), and the blocks of totals
    // and sums are per call.
    const bool sums_fit = 3 * total * sums_per_ep * sizeof(double) <= e->sums_cap && (size_t)chunk * N * rec <= e->episodes_cap;
    const bool both_pipelined = pipelined && !e->pending.empty() && e->pending.back().pipelined && chunk == e->last_pipeline_chunk;
    const bool host_rec = rec_host && !is_device_ptr(rec_host);
    const bool both_on_device = !host_rec && !e->pending.empty() && !e->pending.back().pipelined && !e->pending.back().host_records;
    if (!e->pending.empty() && !((both_pipelined || both_on_device) && (sums_fit || !want_records))) {
        rlb_status st = finish_pending(e);
        if (st != RLB_OK) return st;
    }
    // A call in flight owns one of three blocks of totals and of per-episode sums (at most two calls are pending while
    // a third is being enqueued), so that nothing of call i + 1 on the main stream has to wait for the small
    // device->host copies of call i: those ride the COPY stream behind call i's records.  (They used to sit on the main
    // stream, where the copy engine served them in issue order BEHIND the 1.7–3.4 GB record copy — and the next call's
    // kernel behind them: the whole record copy was serialised after all, profiles/r02e_e2e_probe_*.json.)
    const uint64_t slot = e->call_counter++ % 3;
    if (want_records) {
        rlb_status st = ensure_episode_scratch(e, pipelined ? 2 * chunk : chunk, 3 * total * sums_per_ep);
        if (st != RLB_OK) return st;
        if (pipelined) { st = ensure_copy_pipeline(e); if (st != RLB_OK) return st; e->last_pipeline_chunk = chunk; }
    }
    unsigned long long* const d_totals = e->d_totals + 8 * slot;
    double* const d_sums_call = e->d_sums + (want_records ? slot * total * sums_per_ep : 0);
    rlb_engine::Pending pd;
    pd.mode = mode; pd.out = out; pd.eval_steps_out = eval_steps_out; pd.pipelined = pipelined;
    pd.host_records = host_rec;
    if (e->totals_pool.empty()) {
        unsigned long long* h = nullptr;
        CK(cudaHostAlloc(&h, 8 * sizeof(unsigned long long), cudaHostAllocDefault));
        e->totals_pool.push_back(h);
    }
    pd.h_totals = e->totals_pool.back(); e->totals_pool.pop_back();
    // trajectory tap and per-step TD stream: device scratch when the caller's buffers are on the host
    if (mode == 0 && out && out->traj && out->traj_capacity) {
        if (is_device_ptr(out->traj)) pd.d_traj = out->traj;
        else { CK(cudaMalloc(&pd.d_traj, N * out->traj_capacity * sizeof(rlb_traj_record))); pd.own_traj = true; }
        if (out->traj_count && is_device_ptr(out->traj_count)) pd.d_traj_count = out->traj_count;
        else { CK(cudaMalloc(&pd.d_traj_count, N * sizeof(uint64_t))); pd.own_count = true; }
        CK(cudaMemsetAsync(pd.d_traj_count, 0, N * sizeof(uint64_t), e->stream));
    }
    if (mode == 0 && out && out->td_steps && out->td_capacity) {
        if (is_device_ptr(out->td_steps)) pd.d_td = out->td_steps;
        else { CK(cudaMalloc(&pd.d_td, N * out->td_capacity * e->real_size)); pd.own_td = true; }
        if (out->td_count && is_device_ptr(out->td_count)) pd.d_td_count = out->td_count;
        else { CK(cudaMalloc(&pd.d_td_count, N * sizeof(uint64_t))); pd.own_td_count = true; }
        CK(cudaMemsetAsync(pd.d_td_count, 0, N * sizeof(uint64_t), e->stream));
    }
    CK(cudaMemsetAsync(d_totals, 0, 8 * sizeof(unsigned long long), e->stream));
    double* const sums_dst = mode == 0 ? (out ? out->episode_sums : nullptr) : eval_sums_out;
    void* const rec_dst = mode == 0 ? (out ? out->episodes : nullptr) : eval_episodes_out;
    for (uint64_t c0 = begin; c0 < end; c0 += chunk) {
        const uint64_t c1 = std::min<uint64_t>(end, c0 + chunk);
        const int half = pipelined ? (int)(e->launch_counter & 1) : 0;
        if (pipelined) e->launch_counter += 1;
        char* const scratch = (char*)e->d_episodes + (pipelined ? (size_t)half * chunk * N * rec : 0);
        // this half's previous records — of this call or of the one before it — must have left
        if (pipelined) CK(cudaStreamWaitEvent(e->stream, e->ev_drained[half], 0));
        // inactive sets' agents write no records: the caller gets zeros for them
        if (rec_dst && !e->hp_active.empty()) CK(cudaMemsetAsync(scratch, 0, (c1 - c0) * N * rec, e->stream));
        DevParams p = e->dp;
        p.mode = mode;
        p.eval_at = eval_at;
        p.totals = d_totals;
        if (mode == 0) { p.ep0 = c0; p.ep1 = c1; p.n_eval = 0; }
        else { p.ep0 = p.ep1 = 0; p.n_eval = c1 - c0; }
        p.episodes = want_records ? scratch : nullptr;
        p.traj = pd.d_traj; p.traj_cap = pd.d_traj ? out->traj_capacity : 0; p.traj_count = pd.d_traj_count;
        p.td_steps = pd.d_td; p.td_cap = pd.d_td ? out->td_capacity : 0; p.td_count = pd.d_td_count;
        cudaEvent_t ev0 = take_event(e), ev1 = take_event(e);
        if (!ev0 || !ev1) { set_error("cudaEventCreate failed"); return RLB_ERR_CUDA; }
        pd.events.push_back(ev0); pd.events.push_back(ev1);
        CK(cudaEventRecord(ev0, e->stream));
        {
            char label[96];
            snprintf(label, sizeof label, "rlb %s env=%d agents=%llu episodes=[%llu,%llu)", mode == 0 ? "train" : "evaluate", e->cfg.env_kind,
                     (unsigned long long)N, (unsigned long long)c0, (unsigned long long)c1);
            nvtxRangePushA(label);
            cudaError_t lerr = dispatch_run(e, p);
            nvtxRangePop();
            if (lerr != cudaSuccess) return cuda_fail(lerr, "k_run launch");
        }
        CK(cudaEventRecord(ev1, e->stream));
        const uint64_t n_ep = c1 - c0;
        if (sums_dst) {   // reads the records on the main stream, before that scratch is written again
            rlb_status st = reduce_episodes(e, n_ep, scratch, d_sums_call + (c0 - begin) * sums_per_ep);
            if (st != RLB_OK) return st;
        }
        if (pipelined) {
            CK(cudaEventRecord(e->ev_filled[half], e->stream));
            CK(cudaStreamWaitEvent(e->copy_stream, e->ev_filled[half], 0));
            CK(cudaMemcpyAsync((char*)rec_dst + (c0 - begin) * N * rec, scratch, n_ep * N * rec, cudaMemcpyDeviceToHost, e->copy_stream));
            CK(cudaEventRecord(e->ev_drained[half], e->copy_stream));
        } else if (rec_dst) {
            CK(copy_async(e, (char*)rec_dst + (c0 - begin) * N * rec, scratch, n_ep * N * rec));
        }
    }
    pd.done = take_event(e);
    if (!pd.done) { set_error("cudaEventCreate failed"); return RLB_ERR_CUDA; }
    if (pipelined) {
        // kernels and reductions are in the main stream's queue; every device->host copy of this call goes to the copy stream
        const bool sums_on_device = sums_dst && is_device_ptr(sums_dst);   // e.g. about to be gathered on the caller's stream: stays in stream order
        if (sums_on_device && total) CK(cudaMemcpyAsync(sums_dst, d_sums_call, total * sums_per_ep * sizeof(double), cudaMemcpyDeviceToDevice, e->stream));
        CK(cudaEventRecord(pd.done, e->stream));
        CK(cudaStreamWaitEvent(e->copy_stream, pd.done, 0));
        if (sums_dst && !sums_on_device && total) CK(cudaMemcpyAsync(sums_dst, d_sums_call, total * sums_per_ep * sizeof(double), cudaMemcpyDeviceToHost, e->copy_stream));
        CK(cudaMemcpyAsync(pd.h_totals, d_totals, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, e->copy_stream));
        pd.copies_done = take_event(e);
        if (!pd.copies_done) { set_error("cudaEventCreate failed"); return RLB_ERR_CUDA; }
        CK(cudaEventRecord(pd.copies_done, e->copy_stream));
    } else {
        if (sums_dst && total) CK(copy_async(e, sums_dst, d_sums_call, total * sums_per_ep * sizeof(double)));
        CK(cudaMemcpyAsync(pd.h_totals, d_totals, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, e->stream));
        CK(cudaEventRecord(pd.done, e->stream));
    }
    e->pending.push_back(std::move(pd));
    return RLB_OK;
}

}   // namespace

extern "C" {

int rlb_abi_version(void) { return RLB_ABI_VERSION; }
const char* rlb_last_error_string(void) { return last_error_cstr(); }
int rlb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

rlb_status rlb_engine_create(const rlb_config* cfg, rlb_engine** out) {
    if (!out) { set_error("out is NULL"); return RLB_ERR_INVALID_ARG; }
    *out = nullptr;
    if (!valid_cfg(cfg)) return RLB_ERR_INVALID_ARG;
    int ndev = 0;
    cudaError_t derr = cudaGetDeviceCount(&ndev);
    if (derr != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error("no CUDA device available (%s); librlb has no CPU path", derr == cudaSuccess ? "0 devices" : cudaGetErrorString(derr));
        return RLB_ERR_CUDA;
    }
    if (cfg->device < 0 || cfg->device >= ndev) { set_error("device %d out of range (have %d)", cfg->device, ndev); return RLB_ERR_INVALID_ARG; }
    CK(cudaSetDevice(cfg->device));

    rlb_engine* e = new rlb_engine();
    e->cfg = *cfg;
    std::string err;
    if (!build_env_tables(e->cfg, e->tables, err)) { set_error("%s", err.c_str()); delete e; return RLB_ERR_INVALID_ARG; }
    e->S = e->tables.S;
    e->A = e->tables.A;
    e->APAD = e->A == 6 ? RLB_TAXI_APAD : e->A;   // EnvDims<ENV>::APAD
    e->T = cfg->policy_kind == RLB_POLICY_DOUBLE ? 2 : 1;
    e->real_size = cfg->real_kind == RLB_REAL_F32 ? 4 : 8;
    e->variant = Variant{cfg->real_kind, cfg->policy_kind, cfg->selector_kind, cfg->agent_kind == RLB_AGENT_TRACES ? 1 : 0};
    const uint64_t N = cfg->n_agents;

    auto fail = [&](rlb_status st) { rlb_engine_destroy(e); return st; };
#define CKE(call)                                                          \
    do {                                                                   \
        cudaError_t err__ = (call);                                        \
        if (err__ != cudaSuccess) return fail(cuda_fail(err__, #call));    \
    } while (0)

    CKE(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    e->own_stream = true;
    CKE(cudaEventCreate(&e->ev0));
    CKE(cudaEventCreate(&e->ev1));

    e->q_bytes = (size_t)N * e->S * e->T * e->APAD * e->real_size;
    CKE(cudaMalloc(&e->d_q, e->q_bytes));
    CKE(cudaMalloc(&e->d_nvis, N * sizeof(uint32_t)));
    CKE(cudaMalloc(&e->d_rng_n, N * sizeof(uint64_t)));
    CKE(cudaMalloc(&e->d_eps, N * sizeof(double)));
    CKE(cudaMalloc(&e->d_ucb_t, N * sizeof(uint64_t)));
    CKE(cudaMalloc(&e->d_flag, N * sizeof(uint8_t)));
    CKE(cudaMalloc(&e->d_env, N * sizeof(EnvState)));
    CKE(cudaMalloc(&e->d_totals, 3 * 8 * sizeof(unsigned long long)));
    CKE(cudaMalloc(&e->d_flagword, sizeof(uint32_t)));
    if (!e->tables.trans.empty()) {
        CKE(cudaMalloc(&e->d_trans, e->tables.trans.size() * sizeof(uint16_t)));
        CKE(cudaMemcpyAsync(e->d_trans, e->tables.trans.data(), e->tables.trans.size() * sizeof(uint16_t), cudaMemcpyHostToDevice, e->stream));
    }
    if (!e->tables.thr.empty()) {
        CKE(cudaMalloc(&e->d_thr, e->tables.thr.size() * sizeof(uint64_t)));
        CKE(cudaMalloc(&e->d_thr_state, e->tables.thr_state.size() * sizeof(uint16_t)));
        CKE(cudaMemcpyAsync(e->d_thr, e->tables.thr.data(), e->tables.thr.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, e->stream));
        CKE(cudaMemcpyAsync(e->d_thr_state, e->tables.thr_state.data(), e->tables.thr_state.size() * sizeof(uint16_t), cudaMemcpyHostToDevice, e->stream));
    }

    DevParams& p = e->dp;
    p.q = e->d_q; p.counts = nullptr; p.etr = e->d_etr; p.etr_il = nullptr; p.vis = e->d_vis; p.nvis = e->d_nvis;
    p.rng_n = e->d_rng_n; p.eps = e->d_eps; p.ucb_t = e->d_ucb_t; p.flag = e->d_flag; p.env = e->d_env;
    p.trans = e->d_trans; p.thr = e->d_thr; p.thr_state = e->d_thr_state; p.n_thr = (uint32_t)e->tables.thr.size(); p.thr_direct = e->tables.thr_direct;
    p.slip_thr0 = e->tables.slip_thr0; p.slip_thr1 = e->tables.slip_thr1; p.slippery = cfg->slippery;
    p.lr = cfg->learning_rate; p.gamma = cfg->discount_factor; p.lambda = cfg->lambda_factor;
    p.eps0 = cfg->initial_epsilon; p.eps_decay = cfg->epsilon_decay; p.eps_final = cfg->final_epsilon;
    p.ucb_c = cfg->confidence_level; p.default_q = cfg->default_value;
    p.decay_kind = cfg->decay_kind; p.target = cfg->target_kind;
    p.max_steps = cfg->max_steps; p.S = e->S; p.vmax = 0;
    p.n_live = e->tables.n_live;
    std::memcpy(p.row_lut, e->tables.row_lut, sizeof p.row_lut);
    p.seed = cfg->seed; p.first_agent = cfg->first_agent_id; p.n_agents = N;
    for (uint32_t r = 0; r < 10; ++r) {   // Philox4x32-10 key schedule, the same for every block of every agent
        p.rk[2 * r] = (uint32_t)cfg->seed + r * 0x9E3779B9u;
        p.rk[2 * r + 1] = (uint32_t)(cfg->seed >> 32) + r * 0xBB67AE85u;
    }
    p.mode = 0; p.eval_episodes = 100; p.ep0 = p.ep1 = 0; p.eval_at = 1; p.n_eval = 0;
    p.episodes = nullptr; p.traj = nullptr; p.traj_cap = 0; p.traj_count = nullptr;
    p.totals = e->d_totals;
    p.td_steps = nullptr; p.td_cap = 0; p.td_count = nullptr;
    p.cur_obs = nullptr; p.cur_action = nullptr;
    p.fl_start = e->tables.fl_start;
    p.log_table = nullptr; p.log_table_n = 0;
    p.lz_slot = nullptr; p.lz_tmat = nullptr; p.lz_cap = 0;
    p.model_ent = nullptr; p.model_bits = nullptr; p.model_len = nullptr; p.planning_steps = 0; p.mcap = 0; p.mwords = 0;

    CKE(fill_q_default(e));
    CKE(cudaMemsetAsync(e->d_nvis, 0, N * sizeof(uint32_t), e->stream));
    CKE(cudaMemsetAsync(e->d_rng_n, 0, N * sizeof(uint64_t), e->stream));
    CKE(fill<uint8_t>(e, e->d_flag, N, (uint8_t)1));   // policy_flag: true (double_tabular_policy.rs:23)
    rlb_status st = install_selector(e, cfg->selector_kind);
    if (st != RLB_OK) return fail(st);
    st = cfg->planning_steps ? attach_model(e, cfg->planning_steps) : ensure_trace_buffers(e);
    if (st != RLB_OK) return fail(st);
    st = pick_store(e);
    if (st != RLB_OK) return fail(st);
    CKE(dispatch_step(e, OP_ENV_CONSTRUCT, StepArgs()));   // Env::new(): Blackjack deals a hand
    CKE(cudaStreamSynchronize(e->stream));
#undef CKE
    *out = e;
    return RLB_OK;
}

void rlb_engine_destroy(rlb_engine* e) {
    if (!e) return;
    cudaSetDevice(e->cfg.device);
    finish_pending(e);
    if (e->stream) cudaStreamSynchronize(e->stream);
    for (cudaEvent_t ev : e->event_pool) cudaEventDestroy(ev);
    for (unsigned long long* h : e->totals_pool) cudaFreeHost(h);
    if (e->d_cur_obs) cudaFree(e->d_cur_obs);
    if (e->d_cur_action) cudaFree(e->d_cur_action);
    if (e->d_log_table) cudaFree(e->d_log_table);
    if (e->d_lz_slot) cudaFree(e->d_lz_slot);
    if (e->d_lz_tmat) cudaFree(e->d_lz_tmat);
    if (e->h_step_stage) cudaFreeHost(e->h_step_stage);
    void* bufs[] = {e->d_q, e->d_counts, e->d_etr, e->d_etr_il, e->d_vis, e->d_nvis, e->d_rng_n, e->d_eps, e->d_ucb_t, e->d_flag, e->d_env,
                    e->d_trans, e->d_thr, e->d_thr_state, e->d_totals, e->d_flagword, e->d_episodes, e->d_sums,
                    e->d_model_ent, e->d_model_bits, e->d_model_len, e->d_hp_sets, e->d_hp_group, e->d_hp_order, e->d_hp_offsets,
                    e->d_hp_q0, e->d_hp_eps0, e->d_hp_run, e->d_hp_run_offsets, e->d_hp_planning,
                    e->d_hp_targets};
    for (void* b : bufs) if (b) cudaFree(b);
    for (void* b : e->d_stage) if (b) cudaFree(b);
    if (e->ev0) cudaEventDestroy(e->ev0);
    if (e->ev1) cudaEventDestroy(e->ev1);
    if (e->copy_stream) { cudaStreamSynchronize(e->copy_stream); cudaStreamDestroy(e->copy_stream); }
    for (int b = 0; b < 2; ++b) {
        if (e->ev_filled[b]) cudaEventDestroy(e->ev_filled[b]);
        if (e->ev_drained[b]) cudaEventDestroy(e->ev_drained[b]);
    }
    if (e->own_stream && e->stream) cudaStreamDestroy(e->stream);
    cudaGetLastError();
    delete e;
}

rlb_status rlb_engine_set_stream(rlb_engine* e, void* cuda_stream) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    CK(cudaStreamSynchronize(e->stream));
    if (e->own_stream) { cudaStreamDestroy(e->stream); e->own_stream = false; }
    e->stream = (cudaStream_t)cuda_stream;
    return RLB_OK;
}
rlb_status rlb_engine_synchronize(rlb_engine* e) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    CK(cudaStreamSynchronize(e->stream));
    return RLB_OK;
}
rlb_status rlb_engine_dims(const rlb_engine* e, uint32_t* n_states, uint32_t* n_actions, uint32_t* n_tables) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    if (n_states) *n_states = e->S;
    if (n_actions) *n_actions = e->A;
    if (n_tables) *n_tables = e->T;
    return RLB_OK;
}
uint32_t rlb_engine_store_kind(const rlb_engine* e) { return e ? (uint32_t)e->store : 0u; }

// the installed sets' values (d_hp_sets) and, narrowed on the host exactly as the engine-wide fills narrow rlb_config's,
// the fills' values (d_hp_q0, d_hp_eps0); synchronous, so `h_sets` may go when it returns
static cudaError_t write_set_values(rlb_engine* e, const std::vector<rlb_hparams>& h_sets) {
    const size_t n_sets = h_sets.size();
    std::vector<double> eps0(n_sets), q0d(n_sets);
    std::vector<float> q0f(n_sets);
    for (size_t g = 0; g < n_sets; ++g) { eps0[g] = h_sets[g].initial_epsilon; q0d[g] = h_sets[g].default_value; q0f[g] = (float)h_sets[g].default_value; }
    cudaError_t err = cudaMemcpyAsync(e->d_hp_sets, h_sets.data(), n_sets * sizeof(rlb_hparams), cudaMemcpyHostToDevice, e->stream);
    if (err == cudaSuccess) {
        if (e->cfg.real_kind == RLB_REAL_F32) err = cudaMemcpyAsync(e->d_hp_q0, q0f.data(), n_sets * 4, cudaMemcpyHostToDevice, e->stream);
        else err = cudaMemcpyAsync(e->d_hp_q0, q0d.data(), n_sets * 8, cudaMemcpyHostToDevice, e->stream);
    }
    if (err == cudaSuccess) err = cudaMemcpyAsync(e->d_hp_eps0, eps0.data(), n_sets * sizeof(double), cudaMemcpyHostToDevice, e->stream);
    if (err == cudaSuccess) err = cudaStreamSynchronize(e->stream);
    return err;
}

rlb_status rlb_engine_set_hparams(rlb_engine* e, const rlb_hparams* sets, uint32_t n_sets, const uint32_t* group) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    if (n_sets == 0 && (sets || group)) { set_error("n_sets == 0 with a non-NULL sets or group"); return RLB_ERR_INVALID_ARG; }
    if (n_sets > 0 && (!sets || !group)) { set_error("n_sets > 0 needs both sets and group"); return RLB_ERR_INVALID_ARG; }
    if (n_sets > RLB_MAX_HPARAM_SETS) { set_error("n_sets = %u exceeds %d", n_sets, RLB_MAX_HPARAM_SETS); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    std::vector<rlb_hparams> h_sets(n_sets);
    std::vector<uint32_t> h_group(n_sets ? N : 0);
    if (n_sets) {
        CK(cudaMemcpy(h_sets.data(), sets, (size_t)n_sets * sizeof(rlb_hparams), is_device_ptr(sets) ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost));
        CK(cudaMemcpy(h_group.data(), group, N * sizeof(uint32_t), is_device_ptr(group) ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost));
        for (uint64_t i = 0; i < N; ++i)
            if (h_group[i] >= n_sets) { set_error("group[%llu] = %u >= n_sets = %u", (unsigned long long)i, h_group[i], n_sets); return RLB_ERR_INVALID_ARG; }
        if (e->cfg.planning_steps) { set_error("per-agent hyper-parameter sets together with a Dyna model are not supported"); return RLB_ERR_UNSUPPORTED; }
    } else if (!e->h_hp_planning.empty()) {
        set_error("the per-set planning counts need the sets: drop the model first (rlb_engine_set_planning_steps(e, NULL, 0))");
        return RLB_ERR_UNSUPPORTED;
    }
    // release the old sets (the kernels that read them have completed: ENTER waited for pending calls, and the stream
    // is drained before the buffers go)
    CK(cudaStreamSynchronize(e->stream));
    void* old[] = {e->d_hp_sets, e->d_hp_group, e->d_hp_order, e->d_hp_offsets, e->d_hp_q0, e->d_hp_eps0, e->d_hp_run, e->d_hp_run_offsets,
                   e->d_hp_targets};
    for (void* b : old) if (b) cudaFree(b);
    e->d_hp_sets = nullptr; e->d_hp_group = nullptr; e->d_hp_order = nullptr; e->d_hp_offsets = nullptr;
    e->d_hp_q0 = nullptr; e->d_hp_eps0 = nullptr; e->d_hp_targets = nullptr;
    e->h_hp_targets.clear();
    e->d_hp_run = nullptr; e->d_hp_run_offsets = nullptr; e->hp_n_run = 0;
    e->hp_active.clear();   // every set active again
    e->h_hp_order.clear(); e->h_hp_offsets.clear();
    e->hp_n = 0;
    if (n_sets) {
        // the grouped reduction's read order: agents by set, ascending local index within a set (a stable counting sort)
        std::vector<uint32_t> offsets(n_sets + 1, 0), order(N);
        for (uint64_t i = 0; i < N; ++i) offsets[h_group[i] + 1] += 1;
        for (uint32_t g = 0; g < n_sets; ++g) offsets[g + 1] += offsets[g];
        std::vector<uint32_t> next(offsets.begin(), offsets.end() - 1);
        for (uint64_t i = 0; i < N; ++i) order[next[h_group[i]]++] = (uint32_t)i;
        CK(cudaMalloc(&e->d_hp_sets, (size_t)n_sets * sizeof(rlb_hparams)));
        CK(cudaMalloc(&e->d_hp_group, N * sizeof(uint32_t)));
        CK(cudaMalloc(&e->d_hp_order, N * sizeof(uint32_t)));
        CK(cudaMalloc(&e->d_hp_offsets, (size_t)(n_sets + 1) * sizeof(uint32_t)));
        CK(cudaMalloc(&e->d_hp_q0, (size_t)n_sets * e->real_size));
        CK(cudaMalloc(&e->d_hp_eps0, (size_t)n_sets * sizeof(double)));
        CK(cudaMalloc(&e->d_hp_targets, (size_t)n_sets * sizeof(int32_t)));
        CK(cudaMemcpyAsync(e->d_hp_group, h_group.data(), N * sizeof(uint32_t), cudaMemcpyHostToDevice, e->stream));
        CK(cudaMemcpyAsync(e->d_hp_order, order.data(), N * sizeof(uint32_t), cudaMemcpyHostToDevice, e->stream));
        CK(cudaMemcpyAsync(e->d_hp_offsets, offsets.data(), (size_t)(n_sets + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, e->stream));
        // every set starts with the engine-wide target (rlb_engine_set_targets changes them)
        std::vector<int32_t> targets(n_sets, e->cfg.target_kind);
        CK(cudaMemcpyAsync(e->d_hp_targets, targets.data(), (size_t)n_sets * sizeof(int32_t), cudaMemcpyHostToDevice, e->stream));
        CK(write_set_values(e, h_sets));   // synchronous: `targets` may go
        e->h_hp_order = std::move(order); e->h_hp_offsets = std::move(offsets);
        e->h_hp_targets = std::move(targets);
        e->hp_n = n_sets;
    }
    // the constructors again, with each agent's own values: fresh tables, policy_flag = true, an empty trace, a fresh
    // selector (as rlb_agent_set_kind); the env and the RNG stream carry on
    CK(fill_q_default(e));
    CK(fill<uint8_t>(e, e->d_flag, N, (uint8_t)1));
    CK(cudaMemsetAsync(e->d_nvis, 0, N * sizeof(uint32_t), e->stream));
    rlb_status st = install_selector(e, e->cfg.selector_kind);
    if (st != RLB_OK) return st;
    CK(cudaStreamSynchronize(e->stream));
    return RLB_OK;
}
uint32_t rlb_engine_hparam_sets(const rlb_engine* e) { return e ? e->hp_n : 0u; }

rlb_status rlb_engine_retune_hparams(rlb_engine* e, const rlb_hparams* sets, uint32_t n_sets) {
    if (!e || !sets) { set_error("NULL argument"); return RLB_ERR_INVALID_ARG; }
    if (!e->hp_n) { set_error("no hyper-parameter sets are installed (rlb_engine_set_hparams)"); return RLB_ERR_INVALID_ARG; }
    if (n_sets != e->hp_n) { set_error("n_sets = %u, but %u sets are installed", n_sets, e->hp_n); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    std::vector<rlb_hparams> h_sets(n_sets);
    CK(cudaMemcpy(h_sets.data(), sets, (size_t)n_sets * sizeof(rlb_hparams), is_device_ptr(sets) ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost));
    CK(write_set_values(e, h_sets));
    return RLB_OK;
}

rlb_status rlb_engine_set_active_sets(rlb_engine* e, const uint8_t* active, uint32_t n_sets) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    if (!e->hp_n) { set_error("no hyper-parameter sets are installed (rlb_engine_set_hparams)"); return RLB_ERR_INVALID_ARG; }
    if ((n_sets == 0) != (active == nullptr)) { set_error("active and n_sets: NULL with 0, or a mask of rlb_engine_hparam_sets() entries"); return RLB_ERR_INVALID_ARG; }
    if (active && n_sets != e->hp_n) { set_error("n_sets = %u, but %u sets are installed", n_sets, e->hp_n); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    std::vector<uint8_t> mask(e->hp_n, 1);
    if (active) CK(cudaMemcpy(mask.data(), active, n_sets, is_device_ptr(active) ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost));
    bool all = true;
    for (uint8_t& m : mask) { m = m ? 1 : 0; all = all && m; }
    // the kernels that read the old list have completed (ENTER); drain the stream before it goes
    CK(cudaStreamSynchronize(e->stream));
    if (e->d_hp_run) cudaFree(e->d_hp_run);
    if (e->d_hp_run_offsets) cudaFree(e->d_hp_run_offsets);
    e->d_hp_run = nullptr; e->d_hp_run_offsets = nullptr; e->hp_n_run = 0;
    e->hp_active.clear();
    if (all) return RLB_OK;   // an all-ones mask is NULL: the identity launch
    // d_hp_order restricted to the active sets, in the same order: contiguous groups stay ascending id ranges
    std::vector<uint32_t> run, offsets(e->hp_n + 1, 0);
    for (uint32_t g = 0; g < e->hp_n; ++g) {
        if (mask[g]) run.insert(run.end(), e->h_hp_order.begin() + e->h_hp_offsets[g], e->h_hp_order.begin() + e->h_hp_offsets[g + 1]);
        offsets[g + 1] = (uint32_t)run.size();
    }
    CK(cudaMalloc(&e->d_hp_run, std::max<size_t>(run.size(), 1) * sizeof(uint32_t)));
    CK(cudaMalloc(&e->d_hp_run_offsets, offsets.size() * sizeof(uint32_t)));
    if (!run.empty()) CK(cudaMemcpyAsync(e->d_hp_run, run.data(), run.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, e->stream));
    CK(cudaMemcpyAsync(e->d_hp_run_offsets, offsets.data(), offsets.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    e->hp_n_run = run.size();
    e->hp_active = std::move(mask);
    return RLB_OK;
}

rlb_status rlb_engine_set_planning_steps(rlb_engine* e, const uint32_t* steps, uint32_t n_sets) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    if (!e->hp_n) { set_error("no hyper-parameter sets are installed (rlb_engine_set_hparams)"); return RLB_ERR_INVALID_ARG; }
    if ((n_sets == 0) != (steps == nullptr)) { set_error("steps and n_sets: NULL with 0, or rlb_engine_hparam_sets() counts"); return RLB_ERR_INVALID_ARG; }
    if (steps && n_sets != e->hp_n) { set_error("n_sets = %u, but %u sets are installed", n_sets, e->hp_n); return RLB_ERR_INVALID_ARG; }
    if (steps && e->cfg.store_kind != 0 && e->cfg.store_kind != STORE_GLOBAL) {
        set_error("a Dyna model (planning_steps > 0) needs the HBM store");
        return RLB_ERR_UNSUPPORTED;
    }
    ENTER(e);
    if (!steps) {   // unwrap: rlb_agent_set_model(e, 0)
        rlb_status st = attach_model(e, 0);
        if (st != RLB_OK) return st;
        return pick_store(e);
    }
    std::vector<uint32_t> h(n_sets);
    CK(cudaMemcpy(h.data(), steps, (size_t)n_sets * sizeof(uint32_t), is_device_ptr(steps) ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost));
    // DevParams::planning_steps stays nonzero while the model is attached, every count 0 included: it is what tells the
    // dispatch and the step kernels that a model is there, and what rlb_agent_set_kind wraps the new agent with
    const uint32_t wrap = std::max<uint32_t>(1u, *std::max_element(h.begin(), h.end()));
    const bool first = !e->cfg.planning_steps;
    if (first) {   // every agent wrapped as it is, around an empty model
        rlb_status st = attach_model(e, wrap);
        if (st != RLB_OK) return st;
    } else {       // a model is attached: only the counts change
        e->cfg.planning_steps = wrap;
        e->dp.planning_steps = wrap;
    }
    if (!e->d_hp_planning) CK(cudaMalloc(&e->d_hp_planning, (size_t)n_sets * sizeof(uint32_t)));
    // the kernels that read the old counts have completed (ENTER): the new ones go over them in stream order
    CK(cudaMemcpyAsync(e->d_hp_planning, h.data(), (size_t)n_sets * sizeof(uint32_t), cudaMemcpyHostToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    e->h_hp_planning = std::move(h);
    return first ? pick_store(e) : RLB_OK;
}

// the device copy of h_hp_targets, after the kernels that read the old one (ENTER waited for pending calls; the copy
// follows the rest in stream order)
static rlb_status write_targets(rlb_engine* e) {
    CK(cudaMemcpyAsync(e->d_hp_targets, e->h_hp_targets.data(), e->h_hp_targets.size() * sizeof(int32_t), cudaMemcpyHostToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return RLB_OK;
}

rlb_status rlb_engine_set_targets(rlb_engine* e, const int32_t* targets, uint32_t n_sets) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    if (!e->hp_n) { set_error("no hyper-parameter sets are installed (rlb_engine_set_hparams)"); return RLB_ERR_INVALID_ARG; }
    if (!targets || n_sets != e->hp_n) { set_error("targets: one RLB_TARGET_* per installed set (%u), got %u", e->hp_n, n_sets); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    std::vector<int32_t> h(n_sets);
    CK(cudaMemcpy(h.data(), targets, (size_t)n_sets * sizeof(int32_t), is_device_ptr(targets) ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost));
    for (uint32_t g = 0; g < n_sets; ++g)
        if (h[g] < RLB_TARGET_SARSA || h[g] > RLB_TARGET_EXPECTED_SARSA) { set_error("targets[%u] = %d is not an RLB_TARGET_*", g, h[g]); return RLB_ERR_INVALID_ARG; }
    e->h_hp_targets = std::move(h);
    return write_targets(e);
}

rlb_status rlb_agent_clone(rlb_engine* e, const uint32_t* src, const uint32_t* dst, uint64_t n_pairs) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    if (!n_pairs) return RLB_OK;
    if (!src || !dst) { set_error("NULL argument"); return RLB_ERR_INVALID_ARG; }
    const uint64_t N = e->cfg.n_agents;
    if (n_pairs > N) { set_error("n_pairs = %llu > n_agents: some destination appears twice", (unsigned long long)n_pairs); return RLB_ERR_INVALID_ARG; }
    if (e->cfg.planning_steps && e->cfg.agent_kind == RLB_AGENT_TRACES) {
        // planning updates run with terminated = false: the eligibility rows survive episode boundaries
        set_error("cloning an eligibility-trace agent under a Dyna model is not supported");
        return RLB_ERR_UNSUPPORTED;
    }
    ENTER(e);
    std::vector<uint32_t> ids(2 * n_pairs);   // src then dst
    CK(cudaMemcpy(ids.data(), src, n_pairs * 4, is_device_ptr(src) ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost));
    CK(cudaMemcpy(ids.data() + n_pairs, dst, n_pairs * 4, is_device_ptr(dst) ? cudaMemcpyDeviceToHost : cudaMemcpyHostToHost));
    for (uint64_t j = 0; j < 2 * n_pairs; ++j)
        if (ids[j] >= N) { set_error("%s[%llu] = %u >= n_agents", j < n_pairs ? "src" : "dst", (unsigned long long)(j % n_pairs), ids[j]); return RLB_ERR_INVALID_ARG; }
    // no destination twice, and no id both a source and a destination: then no pair writes what another reads
    std::vector<uint8_t> is_dst(N, 0);
    for (uint64_t j = 0; j < n_pairs; ++j) {
        if (is_dst[ids[n_pairs + j]]) { set_error("dst[%llu] = %u appears twice", (unsigned long long)j, ids[n_pairs + j]); return RLB_ERR_INVALID_ARG; }
        is_dst[ids[n_pairs + j]] = 1;
    }
    for (uint64_t j = 0; j < n_pairs; ++j)
        if (is_dst[ids[j]]) { set_error("agent %u is both a source and a destination", ids[j]); return RLB_ERR_INVALID_ARG; }
    const void* d_ids;
    CK(stage_in(e, 0, ids.data(), 2 * n_pairs * 4, &d_ids));
    CloneArgs a{};
    // whole padded rows: the round trip moves only the A real columns, but padding exists only under -DRLB_TAXI_APAD=8,
    // and load_row / store_row read and write the first A columns of a row alone, so what the padding holds is never used
    a.seg[a.n_seg++] = CloneSegment{(uint8_t*)e->d_q, e->q_bytes / N};
    if (e->cfg.selector_kind == RLB_SEL_UCB) a.seg[a.n_seg++] = CloneSegment{(uint8_t*)e->d_counts, e->counts_bytes / N};
    if (e->cfg.planning_steps) {
        a.seg[a.n_seg++] = CloneSegment{(uint8_t*)e->d_model_ent, (uint64_t)e->dp.mcap * sizeof(uint2)};
        a.seg[a.n_seg++] = CloneSegment{(uint8_t*)e->d_model_bits, (uint64_t)e->dp.mwords * sizeof(uint32_t)};
        a.model_len = e->d_model_len;
    }
    a.src = (const uint32_t*)d_ids; a.dst = a.src + n_pairs; a.n_pairs = n_pairs;
    a.eps = e->d_eps; a.ucb_t = e->d_ucb_t; a.flag = e->d_flag;
    CK(launch_clone_agents(a, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return RLB_OK;
}

// ------------------------------------------------------------------------------- Env
rlb_status rlb_env_reset(rlb_engine* e, uint32_t* obs_out) {
    if (!e || !obs_out) { set_error("NULL argument"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    StepArgs a;
    void* dev;
    CK(stage_out(e, 0, obs_out, N * 4, &dev));
    a.u32_out = (uint32_t*)dev;
    CK(dispatch_step(e, OP_ENV_RESET, a));
    CK(finish_out(e, obs_out, dev, N * 4));
    return RLB_OK;
}

rlb_status rlb_env_step(rlb_engine* e, const uint32_t* actions, uint32_t* obs_out, double* reward_out, uint8_t* terminated_out,
                        uint8_t* not_ready_out) {
    if (!e || !actions || !obs_out || !reward_out || !terminated_out) { set_error("NULL argument"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    StepArgs a;
    const void* in;
    void *d_obs, *d_rew, *d_term, *d_nr;
    CK(stage_in(e, 0, actions, N * 4, &in));
    a.action = (const uint32_t*)in;
    CK(stage_out(e, 1, obs_out, N * 4, &d_obs));
    CK(stage_out(e, 2, reward_out, N * 8, &d_rew));
    CK(stage_out(e, 3, terminated_out, N, &d_term));
    CK(stage_out(e, 4, not_ready_out, N, &d_nr));
    a.u32_out = (uint32_t*)d_obs; a.reward_out = (double*)d_rew; a.term_out = (uint8_t*)d_term; a.not_ready_out = (uint8_t*)d_nr;
    a.any_not_ready = e->d_flagword;
    CK(flags_clear(e));
    CK(dispatch_step(e, OP_ENV_STEP, a));
    CK(finish_out(e, obs_out, d_obs, N * 4));
    CK(finish_out(e, reward_out, d_rew, N * 8));
    CK(finish_out(e, terminated_out, d_term, N));
    CK(finish_out(e, not_ready_out, d_nr, N));
    return flags_check(e);
}

// ------------------------------------------------------------------------------- Agent
rlb_status rlb_agent_get_action(rlb_engine* e, const uint32_t* obs, uint32_t* action_out) {
    if (!e || !obs || !action_out) { set_error("NULL argument"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    StepArgs a;
    const void* in;
    void* dev;
    CK(stage_in(e, 0, obs, N * 4, &in));
    CK(stage_out(e, 1, action_out, N * 4, &dev));
    a.obs = (const uint32_t*)in; a.u32_out = (uint32_t*)dev; a.any_not_ready = e->d_flagword;
    CK(flags_clear(e));
    CK(dispatch_step(e, OP_GET_ACTION, a));
    CK(finish_out(e, action_out, dev, N * 4));
    return flags_check(e);
}

rlb_status rlb_agent_update(rlb_engine* e, const uint32_t* curr_obs, const uint32_t* curr_action, const double* reward,
                            const uint8_t* terminated, const uint32_t* next_obs, const uint32_t* next_action, void* td_out) {
    if (!e || !curr_obs || !curr_action || !reward || !terminated || !next_obs || !next_action) { set_error("NULL argument"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    StepArgs a;
    const void* in[6];
    void* dev;
    CK(stage_in(e, 0, curr_obs, N * 4, &in[0]));
    CK(stage_in(e, 1, curr_action, N * 4, &in[1]));
    CK(stage_in(e, 2, reward, N * 8, &in[2]));
    CK(stage_in(e, 3, terminated, N, &in[3]));
    CK(stage_in(e, 4, next_obs, N * 4, &in[4]));
    CK(stage_in(e, 5, next_action, N * 4, &in[5]));
    CK(stage_out(e, 6, td_out, N * e->real_size, &dev));
    a.obs = (const uint32_t*)in[0]; a.action = (const uint32_t*)in[1]; a.reward = (const double*)in[2];
    a.term = (const uint8_t*)in[3]; a.obs2 = (const uint32_t*)in[4]; a.action2 = (const uint32_t*)in[5];
    a.real_out = dev; a.any_not_ready = e->d_flagword;
    CK(flags_clear(e));
    CK(dispatch_step(e, OP_UPDATE, a));
    CK(finish_out(e, td_out, dev, N * e->real_size));
    return flags_check(e);
}

rlb_status rlb_agent_step(rlb_engine* e, uint8_t* kind_out, uint32_t* obs_out, uint32_t* action_out, double* reward_out,
                          uint8_t* terminated_out, void* td_out) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    if (!e->d_cur_obs) {
        CK(cudaMalloc(&e->d_cur_obs, N * 4));
        CK(cudaMalloc(&e->d_cur_action, N * 4));
        CK(cudaMemsetAsync(e->d_cur_obs, 0, N * 4, e->stream));
        CK(cudaMemsetAsync(e->d_cur_action, 0, N * 4, e->stream));
        e->dp.cur_obs = e->d_cur_obs; e->dp.cur_action = e->d_cur_action;
    }
    // Outputs for HOST buffers are written by the kernel straight into one block of mapped pinned memory (the device
    // sees it through unified addressing) and copied out by the CPU after the single wait: launch + wait is the whole
    // latency of a transition, with no per-array cudaMemcpy.  DEVICE buffers are written in place.
    const size_t sizes[6] = {(size_t)N * 8, (size_t)N * e->real_size, (size_t)N * 4, (size_t)N * 4, (size_t)N, (size_t)N};   // reward, td, obs, action, kind, terminated
    void* const user[6] = {reward_out, td_out, obs_out, action_out, kind_out, terminated_out};
    size_t need = 0;
    for (int k = 0; k < 6; ++k) if (user[k] && !is_device_ptr(user[k])) need += (sizes[k] + 15) & ~(size_t)15;
    if (need > e->step_stage_cap) {
        if (e->h_step_stage) cudaFreeHost(e->h_step_stage);
        e->h_step_stage = nullptr; e->step_stage_cap = 0;
        CK(cudaHostAlloc(&e->h_step_stage, need, cudaHostAllocMapped));
        e->step_stage_cap = need;
    }
    void* dev[6];
    size_t off = 0;
    for (int k = 0; k < 6; ++k) {
        if (!user[k]) dev[k] = nullptr;
        else if (is_device_ptr(user[k])) dev[k] = user[k];
        else { dev[k] = (char*)e->h_step_stage + off; off += (sizes[k] + 15) & ~(size_t)15; }
    }
    StepArgs a;
    a.reward_out = (double*)dev[0]; a.real_out = dev[1]; a.u32_out = (uint32_t*)dev[2]; a.u32_out2 = (uint32_t*)dev[3];
    a.kind_out = (uint8_t*)dev[4]; a.term_out = (uint8_t*)dev[5];
    CK(dispatch_step(e, OP_AGENT_STEP, a));
    CK(cudaStreamSynchronize(e->stream));
    for (int k = 0; k < 6; ++k) if (user[k] && dev[k] != user[k]) std::memcpy(user[k], dev[k], sizes[k]);
    return RLB_OK;
}

rlb_status rlb_agent_set_future_q_value_func(rlb_engine* e, int32_t target_kind) {
    if (!e || target_kind < 0 || target_kind > 2) { set_error("bad target_kind"); return RLB_ERR_INVALID_ARG; }
    if (e->hp_n) {   // every agent now uses target_kind: every set's target too
        ENTER(e);
        std::fill(e->h_hp_targets.begin(), e->h_hp_targets.end(), target_kind);
        rlb_status st = write_targets(e);
        if (st != RLB_OK) return st;
    }
    e->cfg.target_kind = target_kind;
    e->dp.target = target_kind;
    return RLB_OK;
}

rlb_status rlb_agent_set_action_selector(rlb_engine* e, int32_t selector_kind) {
    if (!e || selector_kind < 0 || selector_kind > 1) { set_error("bad selector_kind"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    rlb_status st = install_selector(e, selector_kind);
    if (st != RLB_OK) return st;
    return pick_store(e);
}

rlb_status rlb_agent_set_kind(rlb_engine* e, int32_t agent_kind) {
    if (!e || agent_kind < 0 || agent_kind > 1) { set_error("bad agent_kind"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    e->cfg.agent_kind = agent_kind;
    e->variant.trace = agent_kind == RLB_AGENT_TRACES ? 1 : 0;
    {
        rlb_status st0 = ensure_trace_buffers(e);
        if (st0 != RLB_OK) return st0;
        if (e->cfg.planning_steps) {   // the new agent is wrapped again, around an empty model
            st0 = attach_model(e, e->cfg.planning_steps);
            if (st0 != RLB_OK) return st0;
        }
    }
    CK(fill_q_default(e));
    CK(fill<uint8_t>(e, e->d_flag, N, (uint8_t)1));
    CK(cudaMemsetAsync(e->d_nvis, 0, N * sizeof(uint32_t), e->stream));
    rlb_status st = install_selector(e, e->cfg.selector_kind);
    if (st != RLB_OK) return st;
    return pick_store(e);
}

rlb_status rlb_selector_reset(rlb_engine* e) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    if (e->cfg.selector_kind == RLB_SEL_EPS_GREEDY) {
        CK(fill_eps_initial(e));                                                // uniform_epsilon_greed.rs:78-80
    } else {
        CK(cudaMemsetAsync(e->d_counts, 0, e->counts_bytes, e->stream));        // upper_confidence_bound.rs:65-68
        CK(fill<uint64_t>(e, e->d_ucb_t, N, 1ull));
    }
    return RLB_OK;
}

rlb_status rlb_policy_reset(rlb_engine* e) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    CK(fill_q_default(e));   // tables back to the default row; Double keeps its flag (double_tabular_policy.rs:60-63)
    return RLB_OK;
}

rlb_status rlb_agent_reset(rlb_engine* e) {   // one_step_agent.rs:43-46: action_selection.reset(); policy.reset()
    rlb_status st = rlb_selector_reset(e);
    if (st != RLB_OK) return st;
    st = rlb_policy_reset(e);
    if (st != RLB_OK) return st;
    return e->cfg.planning_steps ? rlb_model_reset(e) : RLB_OK;   // internal_model_agent.rs:81-84
}

rlb_status rlb_agent_set_model(rlb_engine* e, uint32_t planning_steps) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    if (planning_steps && e->cfg.store_kind != 0 && e->cfg.store_kind != STORE_GLOBAL) {
        set_error("a Dyna model (planning_steps > 0) needs the HBM store");
        return RLB_ERR_UNSUPPORTED;
    }
    if (planning_steps && e->hp_n) {
        set_error("a Dyna model together with per-agent hyper-parameter sets: use rlb_engine_set_planning_steps");
        return RLB_ERR_UNSUPPORTED;
    }
    rlb_status st = attach_model(e, planning_steps);
    if (st != RLB_OK) return st;
    return pick_store(e);
}

// ------------------------------------------------------------------------------- Model
rlb_status rlb_model_add_info(rlb_engine* e, const uint32_t* obs, const uint32_t* action, const double* reward, const uint32_t* next_obs) {
    if (!e || !obs || !action || !reward || !next_obs) { set_error("NULL argument"); return RLB_ERR_INVALID_ARG; }
    if (!e->cfg.planning_steps) { set_error("no model attached (rlb_agent_set_model)"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    const void* in[4];
    CK(stage_in(e, 0, obs, N * 4, &in[0]));
    CK(stage_in(e, 1, action, N * 4, &in[1]));
    CK(stage_in(e, 2, reward, N * 8, &in[2]));
    CK(stage_in(e, 3, next_obs, N * 4, &in[3]));
    CK(flags_clear(e));
    k_model_add_info<<<(unsigned)((N + 127) / 128), 128, 0, e->stream>>>(e->dp, e->A, (const uint32_t*)in[0], (const uint32_t*)in[1],
                                                                         (const double*)in[2], (const uint32_t*)in[3], e->d_flagword);
    CK(cudaGetLastError());
    return flags_check(e);
}
rlb_status rlb_model_get_info(rlb_engine* e, uint32_t* obs_out, uint32_t* action_out, uint32_t* next_obs_out, double* reward_out) {
    if (!e || !obs_out || !action_out || !next_obs_out || !reward_out) { set_error("NULL argument"); return RLB_ERR_INVALID_ARG; }
    if (!e->cfg.planning_steps) { set_error("no model attached (rlb_agent_set_model)"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    void* dev[4];
    CK(stage_out(e, 0, obs_out, N * 4, &dev[0]));
    CK(stage_out(e, 1, action_out, N * 4, &dev[1]));
    CK(stage_out(e, 2, next_obs_out, N * 4, &dev[2]));
    CK(stage_out(e, 3, reward_out, N * 8, &dev[3]));
    CK(cudaMemsetAsync(e->d_flagword, 0, 4, e->stream));
    k_model_get_info<<<(unsigned)((N + 127) / 128), 128, 0, e->stream>>>(e->dp, e->A, (uint32_t*)dev[0], (uint32_t*)dev[1], (uint32_t*)dev[2],
                                                                         (double*)dev[3], e->d_flagword);
    CK(cudaGetLastError());
    uint32_t any = 0;
    CK(cudaMemcpyAsync(&any, e->d_flagword, 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    CK(finish_out(e, obs_out, dev[0], N * 4));
    CK(finish_out(e, action_out, dev[1], N * 4));
    CK(finish_out(e, next_obs_out, dev[2], N * 4));
    CK(finish_out(e, reward_out, dev[3], N * 8));
    if (any) { set_error("RandomModel::get_info on an empty model (the reference panics: gen_range over an empty range)"); return RLB_ERR_INVALID_ARG; }
    return RLB_OK;
}
rlb_status rlb_model_reset(rlb_engine* e) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    if (!e->cfg.planning_steps) return RLB_OK;
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    CK(cudaMemsetAsync(e->d_model_bits, 0, (size_t)N * e->dp.mwords * sizeof(uint32_t), e->stream));
    CK(cudaMemsetAsync(e->d_model_len, 0, N * sizeof(uint32_t), e->stream));
    return RLB_OK;
}
uint32_t rlb_model_capacity(const rlb_engine* e) { return e ? e->dp.mcap : 0u; }
rlb_status rlb_download_model(rlb_engine* e, uint32_t* len_out, rlb_model_entry* entries_out) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    if (!e->cfg.planning_steps) { set_error("no model attached (rlb_agent_set_model)"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    if (len_out) CK(copy_out(e, len_out, e->d_model_len, N * 4));
    if (entries_out) {
        const size_t n_el = (size_t)N * e->dp.mcap;
        void* dev;
        CK(stage_out(e, 7, entries_out, n_el * sizeof(rlb_model_entry), &dev));
        k_model_export<<<(unsigned)((n_el + 255) / 256), 256, 0, e->stream>>>(e->dp, e->A, (rlb_model_entry*)dev);
        CK(cudaGetLastError());
        CK(finish_out(e, entries_out, dev, n_el * sizeof(rlb_model_entry)));
    }
    CK(cudaStreamSynchronize(e->stream));
    return RLB_OK;
}
rlb_status rlb_upload_model(rlb_engine* e, const uint32_t* len, const rlb_model_entry* entries) {
    if (!e || !len || !entries) { set_error("NULL argument"); return RLB_ERR_INVALID_ARG; }
    if (!e->cfg.planning_steps) { set_error("no model attached (rlb_agent_set_model)"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    const void* in[2];
    CK(stage_in(e, 0, len, N * 4, &in[0]));
    CK(stage_in(e, 7, entries, (size_t)N * e->dp.mcap * sizeof(rlb_model_entry), &in[1]));
    CK(flags_clear(e));
    k_model_import<<<(unsigned)((N + 127) / 128), 128, 0, e->stream>>>(e->dp, e->A, (const uint32_t*)in[0], (const rlb_model_entry*)in[1], e->d_flagword);
    CK(cudaGetLastError());
    return flags_check(e);
}

static rlb_status check_train_args(rlb_engine* e, uint64_t ep_begin, uint64_t ep_end, uint64_t eval_at) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    if (eval_at == 0) { set_error("eval_at == 0 (the reference divides by it, agent.rs:107)"); return RLB_ERR_INVALID_ARG; }
    if (ep_end < ep_begin) { set_error("ep_end < ep_begin"); return RLB_ERR_INVALID_ARG; }
    return RLB_OK;
}
rlb_status rlb_agent_train_range(rlb_engine* e, uint64_t ep_begin, uint64_t ep_end, uint64_t eval_at, rlb_train_out* out) {
    rlb_status st = check_train_args(e, ep_begin, ep_end, eval_at);
    if (st != RLB_OK) return st;
    ENTER(e);
    st = enqueue_range(e, 0, ep_begin, ep_end, eval_at, out, nullptr, nullptr, nullptr);
    rlb_status st2 = finish_pending(e);
    return st != RLB_OK ? st : st2;
}
rlb_status rlb_agent_train_range_async(rlb_engine* e, uint64_t ep_begin, uint64_t ep_end, uint64_t eval_at, rlb_train_out* out) {
    rlb_status st = check_train_args(e, ep_begin, ep_end, eval_at);
    if (st != RLB_OK) return st;
    CK(cudaSetDevice(e->cfg.device));
    st = enqueue_range(e, 0, ep_begin, ep_end, eval_at, out, nullptr, nullptr, nullptr, true);
    if (st != RLB_OK) { finish_pending(e); return st; }
    // the new call's kernels are in the queue: now the host may block on the call before it
    while (e->pending.size() > 1) {
        st = finish_oldest(e);
        if (st != RLB_OK) return st;
    }
    return RLB_OK;
}
rlb_status rlb_agent_train_wait(rlb_engine* e) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    CK(cudaSetDevice(e->cfg.device));
    return finish_pending(e);
}
rlb_status rlb_agent_train(rlb_engine* e, uint64_t n_episodes, uint64_t eval_at, rlb_train_out* out) {
    return rlb_agent_train_range(e, 0, n_episodes, eval_at, out);
}
rlb_status rlb_agent_evaluate(rlb_engine* e, uint64_t n_episodes, void* episodes_out, double* sums_out, uint64_t* total_steps_out) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    rlb_status st = enqueue_range(e, 1, 0, n_episodes, 1, nullptr, episodes_out, sums_out, total_steps_out);
    rlb_status st2 = finish_pending(e);
    return st != RLB_OK ? st : st2;
}

// ------------------------------------------------------------------------------- Policy
static rlb_status policy_rows(rlb_engine* e, const uint32_t* obs, void* values_out, int which) {
    if (!e || !obs || !values_out) { set_error("NULL argument"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    StepArgs a;
    const void* in;
    void* dev;
    CK(stage_in(e, 0, obs, N * 4, &in));
    CK(stage_out(e, 1, values_out, N * e->A * e->real_size, &dev));
    a.obs = (const uint32_t*)in; a.real_out = dev; a.which = which; a.any_not_ready = e->d_flagword;
    CK(flags_clear(e));
    CK(dispatch_step(e, OP_POLICY_ROWS, a));
    CK(finish_out(e, values_out, dev, N * e->A * e->real_size));
    return flags_check(e);
}
rlb_status rlb_policy_predict(rlb_engine* e, const uint32_t* obs, void* values_out) { return policy_rows(e, obs, values_out, 0); }
rlb_status rlb_policy_get_values(rlb_engine* e, const uint32_t* obs, void* values_out) { return policy_rows(e, obs, values_out, 1); }

rlb_status rlb_policy_update(rlb_engine* e, const uint32_t* obs, const uint32_t* action, const uint32_t* next_obs, const void* temporal_difference) {
    (void)next_obs;   // unused by both tabular policies (tabular_policy.rs:35 `_next_obs`)
    if (!e || !obs || !action || !temporal_difference) { set_error("NULL argument"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    StepArgs a;
    const void* in[3];
    CK(stage_in(e, 0, obs, N * 4, &in[0]));
    CK(stage_in(e, 1, action, N * 4, &in[1]));
    CK(stage_in(e, 2, temporal_difference, N * e->real_size, &in[2]));
    a.obs = (const uint32_t*)in[0]; a.action = (const uint32_t*)in[1]; a.td_in = in[2]; a.any_not_ready = e->d_flagword;
    CK(flags_clear(e));
    CK(dispatch_step(e, OP_POLICY_UPDATE, a));
    return flags_check(e);
}
rlb_status rlb_policy_after_update(rlb_engine* e) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    if (e->cfg.policy_kind == RLB_POLICY_DOUBLE) {
        const uint64_t N = e->cfg.n_agents;
        k_flag_flip<<<(unsigned)((N + 255) / 256), 256, 0, e->stream>>>(e->d_flag, N);
        CK(cudaGetLastError());
    }
    return RLB_OK;
}

// ------------------------------------------------------------------------------- ActionSelection
rlb_status rlb_selector_get_action(rlb_engine* e, const uint32_t* obs, const void* values, uint32_t* action_out) {
    if (!e || !obs || !values || !action_out) { set_error("NULL argument"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    StepArgs a;
    const void* in[2];
    void* dev;
    CK(stage_in(e, 0, obs, N * 4, &in[0]));
    CK(stage_in(e, 1, values, N * e->A * e->real_size, &in[1]));
    CK(stage_out(e, 2, action_out, N * 4, &dev));
    a.obs = (const uint32_t*)in[0]; a.values = in[1]; a.u32_out = (uint32_t*)dev; a.any_not_ready = e->d_flagword;
    CK(flags_clear(e));
    CK(dispatch_step(e, OP_SELECTOR_GET_ACTION, a));
    CK(finish_out(e, action_out, dev, N * 4));
    return flags_check(e);
}
rlb_status rlb_selector_get_exploration_probs(rlb_engine* e, const uint32_t* obs, const void* values, void* probs_out) {
    if (!e || !obs || !values || !probs_out) { set_error("NULL argument"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    StepArgs a;
    const void* in[2];
    void* dev;
    CK(stage_in(e, 0, obs, N * 4, &in[0]));
    CK(stage_in(e, 1, values, N * e->A * e->real_size, &in[1]));
    CK(stage_out(e, 2, probs_out, N * e->A * e->real_size, &dev));
    a.obs = (const uint32_t*)in[0]; a.values = in[1]; a.real_out = dev; a.any_not_ready = e->d_flagword;
    CK(flags_clear(e));
    CK(dispatch_step(e, OP_SELECTOR_PROBS, a));
    CK(finish_out(e, probs_out, dev, N * e->A * e->real_size));
    return flags_check(e);
}
rlb_status rlb_selector_update(rlb_engine* e) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    if (e->cfg.selector_kind == RLB_SEL_EPS_GREEDY && e->hp_n) {   // each agent with its own k and floor
        CK(launch_eps_decay_grouped(e->d_eps, e->cfg.n_agents, e->cfg.decay_kind, e->d_hp_sets, e->d_hp_group, e->stream));
    } else if (e->cfg.selector_kind == RLB_SEL_EPS_GREEDY) {
        const uint64_t N = e->cfg.n_agents;
        k_eps_decay<<<(unsigned)((N + 255) / 256), 256, 0, e->stream>>>(e->d_eps, N, e->cfg.decay_kind, e->cfg.epsilon_decay, e->cfg.final_epsilon);
        CK(cudaGetLastError());
    }
    return RLB_OK;
}

// ------------------------------------------------------------------------------- snapshots
rlb_status rlb_download_tables(rlb_engine* e, void* q_out, uint32_t* counts_out) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    if (q_out) {
        const size_t n_el = (size_t)N * e->T * e->S * e->A;
        void* dev;
        CK(stage_out(e, 7, q_out, n_el * e->real_size, &dev));
        unsigned grid = (unsigned)std::min<uint64_t>((n_el + 255) / 256, 148u * 32u);
        if (e->cfg.real_kind == RLB_REAL_F32) k_pack_q<float><<<grid, 256, 0, e->stream>>>((const float*)e->d_q, (float*)dev, N, e->S, e->T, e->A, e->APAD);
        else k_pack_q<double><<<grid, 256, 0, e->stream>>>((const double*)e->d_q, (double*)dev, N, e->S, e->T, e->A, e->APAD);
        CK(cudaGetLastError());
        CK(finish_out(e, q_out, dev, n_el * e->real_size));
    }
    if (counts_out) {
        const size_t n_el = (size_t)N * e->S * e->A;
        void* dev;
        CK(stage_out(e, 7, counts_out, n_el * 4, &dev));
        if (e->d_counts) {
            unsigned grid = (unsigned)std::min<uint64_t>((n_el + 255) / 256, 148u * 32u);
            k_pack_q<uint32_t><<<grid, 256, 0, e->stream>>>(e->d_counts, (uint32_t*)dev, N, e->S, 1, e->A, e->APAD);
            CK(cudaGetLastError());
        } else {
            CK(cudaMemsetAsync(dev, 0, n_el * 4, e->stream));
        }
        CK(finish_out(e, counts_out, dev, n_el * 4));
    }
    CK(cudaStreamSynchronize(e->stream));
    return RLB_OK;
}

rlb_status rlb_upload_tables(rlb_engine* e, const void* q, const uint32_t* counts) {
    if (!e) { set_error("engine is NULL"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    if (q) {
        const size_t n_el = (size_t)N * e->T * e->S * e->A;
        const void* dev;
        CK(stage_in(e, 7, q, n_el * e->real_size, &dev));
        unsigned grid = (unsigned)std::min<uint64_t>((n_el + 255) / 256, 148u * 32u);
        if (e->cfg.real_kind == RLB_REAL_F32) k_unpack_q<float><<<grid, 256, 0, e->stream>>>((float*)e->d_q, (const float*)dev, N, e->S, e->T, e->A, e->APAD);
        else k_unpack_q<double><<<grid, 256, 0, e->stream>>>((double*)e->d_q, (const double*)dev, N, e->S, e->T, e->A, e->APAD);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(e->stream));
    }
    if (counts) {
        if (!e->d_counts) { set_error("engine has no UCB counts (selector is eps-greedy)"); return RLB_ERR_INVALID_ARG; }
        const size_t n_el = (size_t)N * e->S * e->A;
        const void* dev;
        CK(stage_in(e, 7, counts, n_el * 4, &dev));
        unsigned grid = (unsigned)std::min<uint64_t>((n_el + 255) / 256, 148u * 32u);
        k_unpack_q<uint32_t><<<grid, 256, 0, e->stream>>>(e->d_counts, (const uint32_t*)dev, N, e->S, 1, e->A, e->APAD);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(e->stream));
    }
    return RLB_OK;
}

rlb_status rlb_get_agent_states(rlb_engine* e, rlb_agent_state* states_out) {
    if (!e || !states_out) { set_error("NULL argument"); return RLB_ERR_INVALID_ARG; }
    if (is_device_ptr(states_out)) { set_error("states_out must be a host pointer"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    std::vector<double> eps(N);
    std::vector<uint64_t> t(N), n(N);
    std::vector<uint8_t> flag(N);
    std::vector<EnvState> env(N);
    CK(cudaMemcpyAsync(eps.data(), e->d_eps, N * 8, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaMemcpyAsync(t.data(), e->d_ucb_t, N * 8, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaMemcpyAsync(n.data(), e->d_rng_n, N * 8, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaMemcpyAsync(flag.data(), e->d_flag, N, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaMemcpyAsync(env.data(), e->d_env, N * sizeof(EnvState), cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    for (uint64_t i = 0; i < N; ++i) states_out[i] = rlb_agent_state{eps[i], t[i], n[i], flag[i] ? 1 : 0, env[i].ready ? 1 : 0};
    return RLB_OK;
}

rlb_status rlb_set_agent_states(rlb_engine* e, const rlb_agent_state* states) {
    if (!e || !states) { set_error("NULL argument"); return RLB_ERR_INVALID_ARG; }
    if (is_device_ptr(states)) { set_error("states must be a host pointer"); return RLB_ERR_INVALID_ARG; }
    ENTER(e);
    const uint64_t N = e->cfg.n_agents;
    std::vector<double> eps(N);
    std::vector<uint64_t> t(N), n(N);
    std::vector<uint8_t> flag(N);
    for (uint64_t i = 0; i < N; ++i) {
        eps[i] = states[i].epsilon; t[i] = states[i].ucb_t; n[i] = states[i].rng_n; flag[i] = states[i].policy_flag ? 1 : 0;
        // every env but Blackjack draws 64-bit values only: its stream position is always even, and the fused kernel
        // reads aligned pairs (Rng::next_u64<EVEN>)
        if (e->cfg.env_kind != RLB_ENV_BLACKJACK && (n[i] & 1ull)) { set_error("agent %llu: odd rng_n %llu on an env that only draws 64-bit values", (unsigned long long)i, (unsigned long long)n[i]); return RLB_ERR_INVALID_ARG; }
    }
    CK(cudaMemcpyAsync(e->d_eps, eps.data(), N * 8, cudaMemcpyHostToDevice, e->stream));
    CK(cudaMemcpyAsync(e->d_ucb_t, t.data(), N * 8, cudaMemcpyHostToDevice, e->stream));
    CK(cudaMemcpyAsync(e->d_rng_n, n.data(), N * 8, cudaMemcpyHostToDevice, e->stream));
    CK(cudaMemcpyAsync(e->d_flag, flag.data(), N, cudaMemcpyHostToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return RLB_OK;
}

// ------------------------------------------------------------------------------- self tests
rlb_status rlb_selftest_ucb_math(int32_t device, uint64_t samples, uint64_t t_max, uint64_t n_max, uint64_t seed, uint64_t* mismatches_out) {
    if (!mismatches_out || t_max < 2 || n_max < 1 || n_max > 0xffffffffull) { set_error("bad arguments"); return RLB_ERR_INVALID_ARG; }
    CK(cudaSetDevice(device));
    unsigned long long* d = nullptr;
    CK(cudaMalloc(&d, 8));
    CK(cudaMemset(d, 0, 8));
    k_selftest_ucb_math<<<148 * 8, 256>>>(samples, t_max, n_max, seed, d);
    CK(cudaGetLastError());
    unsigned long long h = 0;
    CK(cudaMemcpy(&h, d, 8, cudaMemcpyDeviceToHost));
    cudaFree(d);
    *mismatches_out = h;
    return RLB_OK;
}

// ------------------------------------------------------------------------------- host RNG contract
void rlb_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) { host_philox(ctr, key, out); }
void rlb_rng_words(uint64_t seed, uint64_t agent_id, uint64_t first_word, uint64_t count, uint32_t* out) {
    for (uint64_t i = 0; i < count; ++i) out[i] = host_word(seed, agent_id, first_word + i);
}
static uint64_t host_u64(uint64_t seed, uint64_t agent, uint64_t* n) {
    uint64_t lo = host_word(seed, agent, (*n)++);
    uint64_t hi = host_word(seed, agent, (*n)++);
    return lo | (hi << 32);
}
double rlb_rng_uniform_f64(uint64_t seed, uint64_t agent_id, uint64_t* word_index) {
    return (double)(host_u64(seed, agent_id, word_index) >> 12) * 0x1p-52;
}
uint64_t rlb_rng_uniform_usize(uint64_t seed, uint64_t agent_id, uint64_t* word_index, uint64_t range) {
    if (range == 0) return host_u64(seed, agent_id, word_index);
    const uint64_t zone = UINT64_MAX - (UINT64_MAX - range + 1) % range;
    for (;;) {
        const uint64_t v = host_u64(seed, agent_id, word_index);
        const unsigned __int128 m = (unsigned __int128)v * range;
        if ((uint64_t)m <= zone) return (uint64_t)(m >> 64);
    }
}
uint64_t rlb_rng_gen_range(uint64_t seed, uint64_t agent_id, uint64_t* word_index, uint64_t range) {
    if (range == 0) return host_u64(seed, agent_id, word_index);
    const uint64_t zone = (range << __builtin_clzll(range)) - 1;
    for (;;) {
        const uint64_t v = host_u64(seed, agent_id, word_index);
        const unsigned __int128 m = (unsigned __int128)v * range;
        if ((uint64_t)m <= zone) return (uint64_t)(m >> 64);
    }
}
uint32_t rlb_rng_card(uint64_t seed, uint64_t agent_id, uint64_t* word_index) {
    for (;;) {
        const uint64_t m = (uint64_t)host_word(seed, agent_id, (*word_index)++) * 10u;
        if ((uint32_t)m <= 0xfffffff9u) return 1u + (uint32_t)(m >> 32);
    }
}

// ------------------------------------------------------------------------------- Blackjack ids
void rlb_blackjack_decode(uint32_t dense_index, uint32_t* p_score, uint32_t* d_score, uint32_t* p_ace) {
    if (p_ace) *p_ace = dense_index & 1u;
    if (d_score) *d_score = (dense_index >> 1) % 26u + 1u;
    if (p_score) *p_score = (dense_index >> 1) / 26u + 4u;
}
uint64_t rlb_blackjack_obs_id(uint32_t dense_index) {
    uint32_t p, d, a;
    rlb_blackjack_decode(dense_index, &p, &d, &a);
    return blackjack_id(p, d, a);
}
uint32_t rlb_blackjack_dense_index(uint64_t obs_id) {
    for (uint32_t i = 0; i < 1456; ++i) if (rlb_blackjack_obs_id(i) == obs_id) return i;
    return 0xffffffffu;
}

}   // extern "C"
