// rlb_selectors.cu — the engine-side kernels of per-set action selectors (rlb_engine_set_selectors): a fresh selector for
// the sets whose kind changes (and the per-kind resets), and the epsilon decay restricted to the eps-greedy sets.  The
// fused and step-level kernels themselves stay one selector per launch (rlb_engine.cu launches one per selector).
#include "rlb_launch.h"

namespace rlb {

namespace {

// one thread per counts word (one per agent without counts): the words of one agent's row are adjacent, so the zeroing
// is coalesced; the row's first word's thread writes the scalars
__global__ void k_selector_fresh(const uint8_t* mode, const uint32_t* group, uint64_t n_agents, const double* eps0, double* eps,
                                 uint64_t* ucb_t, uint32_t* counts, uint64_t row_words) {
    const uint64_t words = counts ? row_words : 1;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n_agents * words; idx += stride) {
        const uint64_t i = idx / words, w = idx - i * words;
        const uint32_t g = __ldg(group + i);
        const uint8_t m = __ldg(mode + g);
        if (!m) continue;
        if ((m & 2) && counts) counts[idx] = 0u;                        // upper_confidence_bound.rs:65-68
        if (w == 0) {
            if (m & 1) eps[i] = __ldg(eps0 + g);                        // uniform_epsilon_greed.rs:78-80
            if (m & 2) ucb_t[i] = 1ull;
        }
    }
}

__global__ void k_eps_decay_selected(double* eps, uint64_t n, int kind, const rlb_hparams* sets, const uint32_t* group, const int32_t* sel) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t g = group[i];
    if (sel[g] != RLB_SEL_EPS_GREEDY) return;                          // UCB's update does nothing
    const rlb_hparams& h = sets[g];
    eps[i] = decay_epsilon(eps[i], kind, h.epsilon_decay, h.final_epsilon);
}

}   // namespace

cudaError_t launch_selector_fresh(const uint8_t* mode, const uint32_t* group, uint64_t n_agents, const double* eps0, double* eps,
                                  uint64_t* ucb_t, uint32_t* counts, uint64_t row_words, cudaStream_t stream) {
    const uint64_t n = n_agents * (counts ? row_words : 1);
    if (!n) return cudaSuccess;
    const unsigned grid = (unsigned)std::min<uint64_t>((n + 255) / 256, 148u * 16u);
    k_selector_fresh<<<grid, 256, 0, stream>>>(mode, group, n_agents, eps0, eps, ucb_t, counts, row_words);
    return cudaGetLastError();
}

cudaError_t launch_eps_decay_selected(double* eps, uint64_t n_agents, int kind, const rlb_hparams* sets, const uint32_t* group,
                                      const int32_t* sel, cudaStream_t stream) {
    if (!n_agents) return cudaSuccess;
    k_eps_decay_selected<<<(unsigned)((n_agents + 255) / 256), 256, 0, stream>>>(eps, n_agents, kind, sets, group, sel);
    return cudaGetLastError();
}

}   // namespace rlb
