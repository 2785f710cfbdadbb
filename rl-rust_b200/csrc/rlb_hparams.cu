// rlb_hparams.cu — the engine-side kernels of per-agent hyper-parameter sets (rlb_engine_set_hparams): the per-agent
// fills that stand in for the constructors, the per-agent epsilon decay, and the per-set reduction of the episode records.
// The fused kernel and the step-level kernels with sets (k_run_hp, k_*_hp) are instantiated in rlb_inst_<env>_hp.cu.
#include "rlb_launch.h"

namespace rlb {

namespace {

// ptr[i * per_agent + k] = values[group[i]]: the values are narrowed to the table's type on the host, as the plain fill's are
template <typename V>
__global__ void k_fill_grouped(V* ptr, uint64_t per_agent, uint64_t n_agents, const V* values, const uint32_t* group) {
    uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (; idx < n_agents * per_agent; idx += stride) ptr[idx] = values[group[idx / per_agent]];
}

__global__ void k_eps_decay_grouped(double* eps, uint64_t n, int kind, const rlb_hparams* sets, const uint32_t* group) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const rlb_hparams& h = sets[group[i]];
    eps[i] = decay_epsilon(eps[i], kind, h.epsilon_decay, h.final_epsilon);
}

// k_episode_sums over the agents of one set: CTA (e, g) reduces records [e][order[offsets[g] .. offsets[g + 1])] with the
// same strided accumulation and tree, so one set of all agents gives k_episode_sums' bits.
template <typename Real>
__global__ void __launch_bounds__(256) k_episode_sums_grouped(const void* episodes, uint64_t n_agents, const uint32_t* order,
                                                              const uint32_t* offsets, uint32_t n_sets, uint64_t ep0, double* out) {
    using Rec = typename EpisodeRec<Real>::type;
    const uint64_t e = ep0 + blockIdx.x / n_sets;
    const uint32_t g = blockIdx.x % n_sets;
    const Rec* rec = reinterpret_cast<const Rec*>(episodes) + e * n_agents;
    const uint32_t* mine = order + offsets[g];
    const uint64_t count = offsets[g + 1] - offsets[g];
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    for (uint64_t k = threadIdx.x; k < count; k += blockDim.x) {
        Rec r = rec[mine[k]];
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
    if (threadIdx.x < 4) out[(e * n_sets + g) * 4 + threadIdx.x] = sm[threadIdx.x][0];
}

}   // namespace

cudaError_t launch_fill_grouped(void* ptr, size_t elem_size, uint64_t per_agent, uint64_t n_agents, const void* values,
                                const uint32_t* group, cudaStream_t stream) {
    const uint64_t n = per_agent * n_agents;
    if (!n) return cudaSuccess;
    const unsigned grid = (unsigned)std::min<uint64_t>((n + 255) / 256, 148u * 16u);
    switch (elem_size) {
        case 1: k_fill_grouped<uint8_t><<<grid, 256, 0, stream>>>((uint8_t*)ptr, per_agent, n_agents, (const uint8_t*)values, group); break;
        case 4: k_fill_grouped<uint32_t><<<grid, 256, 0, stream>>>((uint32_t*)ptr, per_agent, n_agents, (const uint32_t*)values, group); break;
        case 8: k_fill_grouped<uint64_t><<<grid, 256, 0, stream>>>((uint64_t*)ptr, per_agent, n_agents, (const uint64_t*)values, group); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

cudaError_t launch_eps_decay_grouped(double* eps, uint64_t n_agents, int kind, const rlb_hparams* sets, const uint32_t* group,
                                     cudaStream_t stream) {
    if (!n_agents) return cudaSuccess;
    k_eps_decay_grouped<<<(unsigned)((n_agents + 255) / 256), 256, 0, stream>>>(eps, n_agents, kind, sets, group);
    return cudaGetLastError();
}

cudaError_t launch_episode_sums_grouped(int real_kind, const void* records, uint64_t n_agents, const uint32_t* order,
                                        const uint32_t* offsets, uint32_t n_sets, uint64_t n_ep, double* out, cudaStream_t stream) {
    const uint64_t per_launch = std::max<uint64_t>(1, 0x7fffffffull / n_sets);   // episodes per launch: grid.x < 2^31
    for (uint64_t e0 = 0; e0 < n_ep; e0 += per_launch) {
        const unsigned grid = (unsigned)(std::min<uint64_t>(per_launch, n_ep - e0) * n_sets);
        if (real_kind == RLB_REAL_F32) k_episode_sums_grouped<float><<<grid, 256, 0, stream>>>(records, n_agents, order, offsets, n_sets, e0, out);
        else k_episode_sums_grouped<double><<<grid, 256, 0, stream>>>(records, n_agents, order, offsets, n_sets, e0, out);
        const cudaError_t err = cudaGetLastError();
        if (err != cudaSuccess) return err;
    }
    return cudaSuccess;
}

}   // namespace rlb
