// rlb_step_kernels.cuh — the individual trait methods of the reference, batched over the
// engine's agents (one thread per agent).  They share AgentCore / EnvRegs with the fused
// kernel, so a host loop over these calls reproduces k_run bit for bit; they exist for the
// drop-in trait objects (N = 1 or a few) and for step-level parity tests.
#pragma once
#include "rlb_device.cuh"

namespace rlb {

// Bits of the engine's flag word (rlb_engine::d_flagword), raised by the step-level kernels and read back by the entry
// point: an agent whose arguments are out of range is left untouched (the reference would panic on the same input:
// an index past a `[f64; COUNT]` row or a table lookup that cannot exist).
constexpr uint32_t FLAG_NOT_READY = 1u;     // Env::step before reset / after termination (env.rs:16-17)
constexpr uint32_t FLAG_BAD_ARG = 2u;       // obs >= S, action >= A, model entry out of range
constexpr uint32_t FLAG_TRACE_FULL = 4u;    // the trace would need more rows than the engine holds (foreign transitions fed to update())
constexpr uint32_t FLAG_DEAD_STATE = 8u;    // trace update from a terminal cell (never a curr_obs of the env itself)

// Env::new() — only Blackjack's constructor touches the RNG (deals a hand, blackjack.rs:57).
template <int ENV>
__global__ void k_env_construct(const DevParams p) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n_agents) return;
    EnvState es;
    es.pos = 0; es.curr_step = 0; es.ready = 0;
    es.p_sum = es.d_sum = es.d_first = 0; es.p_ace = es.d_ace = 0; es.pad[0] = es.pad[1] = 0;
    if constexpr (ENV == RLB_ENV_BLACKJACK) {
        EnvRng<ENV> rng;
        rng.init(p, p.first_agent + i, p.rng_n[i]);
        EnvRegs<RLB_ENV_BLACKJACK> env;
        env.deal(rng, p);
        env.to_state(es, 0);
        p.rng_n[i] = rng.n();
    }
    p.env[i] = es;
}

// Env::reset
template <int ENV>
__global__ void __launch_bounds__(128) k_env_reset(const DevParams p, uint32_t* obs_out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    EnvTab<ENV> tab;
    tab.load(p, smem_raw);
    __syncthreads();
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n_agents) return;
    EnvRng<ENV> rng;
    rng.init(p, p.first_agent + i, p.rng_n[i]);
    EnvState es = p.env[i];
    EnvRegs<ENV> env;
    env.from_state(es);
    uint32_t o = env.reset(rng, tab, p);
    env.to_state(es, o);
    es.pos = o;
    es.ready = 1;
    p.env[i] = es;
    p.rng_n[i] = rng.n();
    obs_out[i] = o;
}

// Env::step.  Err(EnvNotReady) -> agent untouched, not_ready flag set.
template <int ENV>
__global__ void __launch_bounds__(128) k_env_step(const DevParams p, const uint32_t* actions, uint32_t* obs_out,
                                                   double* reward_out, uint8_t* term_out, uint8_t* not_ready_out,
                                                   uint32_t* any_not_ready) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    EnvTab<ENV> tab;
    tab.load(p, smem_raw);
    __syncthreads();
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n_agents) return;
    EnvState es = p.env[i];
    if (!es.ready) {
        if (not_ready_out) not_ready_out[i] = 1;
        atomicOr(any_not_ready, FLAG_NOT_READY);
        return;
    }
    if (not_ready_out) not_ready_out[i] = 0;
    if (actions[i] >= (uint32_t)EnvDims<ENV>::A) { atomicOr(any_not_ready, FLAG_BAD_ARG); return; }
    EnvRng<ENV> rng;
    rng.init(p, p.first_agent + i, p.rng_n[i]);
    EnvRegs<ENV> env;
    env.from_state(es);
    uint32_t o;
    double r;
    bool term;
    env.template step<double>(es.pos, actions[i], rng, tab, p, o, r, term);
    // a truncated step reports obs 0 but does not move the env (taxi.rs:148-151)
    const bool truncated = (ENV != RLB_ENV_BLACKJACK) && es.curr_step >= p.max_steps;
    env.to_state(es, truncated ? es.pos : o);
    if (term) es.ready = 0;
    p.env[i] = es;
    p.rng_n[i] = rng.n();
    obs_out[i] = o;
    reward_out[i] = r;
    term_out[i] = term ? 1 : 0;
}

// Policy::predict (which = 0) / Policy::get_values (which = 1)
template <int ENV, typename Real, int POLICY, int SEL, bool TRACE>
__global__ void __launch_bounds__(128) k_policy_rows(const DevParams p, const uint32_t* obs, Real* out, int which, uint32_t* flags) {
    using Core = AgentCore<ENV, Real, POLICY, SEL, TRACE>;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n_agents) return;
    if (obs[i] >= p.S) { atomicOr(flags, FLAG_BAD_ARG); return; }
    Core core;
    core.load(p, i);
    Real pred[Core::A], vals[Core::A];
    core.rows(obs[i], pred, vals);
#pragma unroll
    for (int k = 0; k < Core::A; ++k) out[i * Core::A + k] = which == 0 ? pred[k] : vals[k];
}

#define RLB_STEP_HP 0
#include "rlb_step_agent_kernels.inc"
#undef RLB_STEP_HP
#define RLB_STEP_HP 1
#include "rlb_step_agent_kernels.inc"
#undef RLB_STEP_HP

// Model::add_info (random_model.rs:37-41)
static __global__ void k_model_add_info(const DevParams p, uint32_t A, const uint32_t* s, const uint32_t* a, const double* reward, const uint32_t* s2, uint32_t* flags) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n_agents) return;
    if (s[i] >= p.S || s2[i] >= p.S || a[i] >= A) { atomicOr(flags, FLAG_BAD_ARG); return; }
    RandomModelDev model;
    model.load(p, i);
    model.add_info(s[i] * A + a[i], s2[i], (float)reward[i]);
    model.save(p, i);
}
// Model::get_info (random_model.rs:27-35); agents with an empty model are flagged and draw nothing
static __global__ void k_model_get_info(const DevParams p, uint32_t A, uint32_t* s, uint32_t* a, uint32_t* s2, double* reward, uint32_t* any_empty) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n_agents) return;
    RandomModelDev model;
    model.load(p, i);
    if (model.len == 0) { atomicOr(any_empty, 1u); return; }
    Rng rng;
    rng.init(p, p.first_agent + i, p.rng_n[i]);
    const uint2 info = model.get_info(rng, p);
    p.rng_n[i] = rng.n();
    const uint32_t key = info.x & 0xffffu;
    s[i] = key / A; a[i] = key % A; s2[i] = info.x >> 16; reward[i] = (double)__uint_as_float(info.y);
}
// model snapshots: device layout <-> rlb_model_entry [N][mcap]
static __global__ void k_model_export(const DevParams p, uint32_t A, rlb_model_entry* out) {
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= p.n_agents * p.mcap) return;
    const uint64_t i = idx / p.mcap;
    const uint32_t j = (uint32_t)(idx % p.mcap);
    rlb_model_entry en{0u, 0u, 0u, 0.0f};
    if (j < p.model_len[i]) {
        const uint2 info = p.model_ent[idx];
        const uint32_t key = info.x & 0xffffu;
        en = rlb_model_entry{key / A, key % A, info.x >> 16, __uint_as_float(info.y)};
    }
    out[idx] = en;
}
static __global__ void k_model_import(const DevParams p, uint32_t A, const uint32_t* len, const rlb_model_entry* in, uint32_t* flags) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n_agents) return;
    uint32_t* bits = p.model_bits + i * p.mwords;
    if (len[i] > p.mcap) { atomicOr(flags, FLAG_BAD_ARG); return; }
    const uint32_t n = len[i];
    for (uint32_t j = 0; j < n; ++j) {   // validate before touching the agent's model: a bad snapshot leaves it as it was
        const rlb_model_entry en = in[i * p.mcap + j];
        if (en.obs >= p.S || en.next_obs >= p.S || en.action >= A) { atomicOr(flags, FLAG_BAD_ARG); return; }
    }
    for (uint32_t w = 0; w < p.mwords; ++w) bits[w] = 0u;
    for (uint32_t j = 0; j < n; ++j) {
        const rlb_model_entry en = in[i * p.mcap + j];
        const uint32_t key = en.obs * A + en.action;
        bits[key >> 5] |= 1u << (key & 31u);
        p.model_ent[i * p.mcap + j] = make_uint2(key | (en.next_obs << 16), __float_as_uint(en.reward));
    }
    p.model_len[i] = n;
}

// ActionSelection::update for eps-greedy: decay_epsilon (uniform_epsilon_greed.rs:42-49)
static __global__ void k_eps_decay(double* eps, uint64_t n, int kind, double param, double final_eps) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) eps[i] = decay_epsilon(eps[i], kind, param, final_eps);
}
// Policy::after_update for Double
static __global__ void k_flag_flip(uint8_t* flag, uint64_t n) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[i] = flag[i] ? 0 : 1;
}

// ln(t) for t < n, by the engine's own portable_log (DevParams::log_table)
static __global__ void k_fill_log_table(double* tab, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) tab[i] = i == 0u ? 0.0 : portable_log((double)i);   // entry 0 is never read: t starts at 1
}

// Test hook (rlb_selftest_ucb_math): div_fast / sqrt_fast against the compiler's own division and square root over the
// UCB domain — ln(t) for t in [2, t_max], n in [1, n_max] — on a grid-stride sample; counts mismatching bit patterns.
static __global__ void k_selftest_ucb_math(uint64_t samples, uint64_t t_max, uint64_t n_max, uint64_t seed, unsigned long long* mismatches) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    unsigned long long bad = 0;
    for (; i < samples; i += stride) {
        uint64_t x = (i + seed) * 0x9E3779B97F4A7C15ull;   // splitmix-style scramble of the sample index
        x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 27; x *= 0x94D049BB133111EBull; x ^= x >> 31;
        const uint64_t t = 2u + (x % (t_max - 1u));
        const uint64_t n = 1u + ((x >> 32) % n_max);
        const double a = portable_log((double)(long long)t), b = (double)(long long)n;
        const double q_ref = a / b, q = div_fast(a, b);
        const double r_ref = sqrt(q_ref), r = sqrt_fast(q);
        bad += (__double_as_longlong(q_ref) != __double_as_longlong(q)) + (__double_as_longlong(r_ref) != __double_as_longlong(r));
    }
    if (bad) atomicAdd(mismatches, bad);
}

template <typename V>
__global__ void k_fill(V* ptr, uint64_t n, V value) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) ptr[i] = value;
}

// padded device layout [N][row_of(S)][T][APAD] <-> ABI layout [N][T][S][A]
template <typename V>
__global__ void k_pack_q(const V* padded, V* packed, uint64_t n_agents, uint32_t S, uint32_t T, uint32_t A, uint32_t APAD) {
    uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t total = n_agents * S * T * A;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (; idx < total; idx += stride) {
        uint32_t a = idx % A;
        uint64_t r = idx / A;
        uint32_t s = r % S; r /= S;
        uint32_t t = r % T;
        uint64_t n = r / T;
        packed[idx] = padded[((n * S + row_of_rt(A, s)) * T + t) * APAD + a];
    }
}
template <typename V>
__global__ void k_unpack_q(V* padded, const V* packed, uint64_t n_agents, uint32_t S, uint32_t T, uint32_t A, uint32_t APAD) {
    uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t total = n_agents * S * T * A;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (; idx < total; idx += stride) {
        uint32_t a = idx % A;
        uint64_t r = idx / A;
        uint32_t s = r % S; r /= S;
        uint32_t t = r % T;
        uint64_t n = r / T;
        padded[((n * S + row_of_rt(A, s)) * T + t) * APAD + a] = packed[idx];
    }
}

// Per-episode-index reduction over this engine's agents of the streamed episode records:
// out[e] = (sum length, sum return, sum td_sum, sum td_abs_sum) in f64, fixed tree order.
// One CTA per episode index; coalesced 16/32-byte record reads.
template <typename Real>
__global__ void __launch_bounds__(256) k_episode_sums(const void* episodes, uint64_t n_agents, double* out) {
    using Rec = typename EpisodeRec<Real>::type;
    const Rec* rec = reinterpret_cast<const Rec*>(episodes) + (uint64_t)blockIdx.x * n_agents;
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    for (uint64_t i = threadIdx.x; i < n_agents; i += blockDim.x) {
        Rec r = rec[i];
        acc[0] += (double)r.length;
        acc[1] += (double)r.ret;
        acc[2] += (double)r.td_sum;
        acc[3] += (double)r.td_abs_sum;
    }
    __shared__ double sm[4][256];
#pragma unroll
    for (int k = 0; k < 4; ++k) sm[k][threadIdx.x] = acc[k];
    __syncthreads();
    for (int off = 128; off > 0; off >>= 1) {
        if ((int)threadIdx.x < off) {
#pragma unroll
            for (int k = 0; k < 4; ++k) sm[k][threadIdx.x] += sm[k][threadIdx.x + off];
        }
        __syncthreads();
    }
    if (threadIdx.x < 4) out[(uint64_t)blockIdx.x * 4 + threadIdx.x] = sm[threadIdx.x][0];
}

}   // namespace rlb
