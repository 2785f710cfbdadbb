// rlb_clone.cu — rlb_agent_clone: agent dst[j] takes the learned state of agent src[j] (the exploit step of
// population-based training).  One gather-scatter launch over the engine's agent-major buffers: every segment is a
// per-agent block of `stride` bytes, and each CTA copies one tile of one pair's block of one segment; a tail of CTAs
// copies the per-agent scalars, one thread per pair.  No source is a destination in the same call (checked on the host),
// so sources are read through the non-coherent path and the result does not depend on the order of the pairs.
#include "rlb_launch.h"

namespace rlb {

namespace {

constexpr int CLONE_THREADS = 256;
constexpr int CLONE_VECS = 4;   // vectors per thread per tile: the loads of a tile are all in flight before its stores

struct CloneTiling {
    uint32_t first[CLONE_MAX_SEGMENTS];   // tile index of a pair at which segment k starts
    uint32_t width[CLONE_MAX_SEGMENTS];   // bytes per vector access: 16, 8 or 4
    uint32_t per_pair;                    // tiles of one pair over all segments
};

template <typename V>
__device__ __forceinline__ void copy_tile(const uint8_t* from, uint8_t* to, uint64_t stride, uint32_t tile) {
    const uint64_t n = stride / sizeof(V);
    const uint64_t first = (uint64_t)tile * CLONE_THREADS * CLONE_VECS + threadIdx.x;
    const V* s = reinterpret_cast<const V*>(from);
    V* d = reinterpret_cast<V*>(to);
    V v[CLONE_VECS];
#pragma unroll
    for (int k = 0; k < CLONE_VECS; ++k) {
        const uint64_t idx = first + (uint64_t)k * CLONE_THREADS;
        if (idx < n) v[k] = __ldg(s + idx);
    }
#pragma unroll
    for (int k = 0; k < CLONE_VECS; ++k) {
        const uint64_t idx = first + (uint64_t)k * CLONE_THREADS;
        if (idx < n) d[idx] = v[k];
    }
}

// virtual blocks [0, n_pairs * per_pair): tile (vb % per_pair) of pair (vb / per_pair); the rest: scalars of 256 pairs each
__global__ void __launch_bounds__(CLONE_THREADS) k_clone_agents(const CloneArgs a, const CloneTiling t, uint64_t n_tile_blocks,
                                                                uint64_t n_blocks) {
    for (uint64_t vb = blockIdx.x; vb < n_blocks; vb += gridDim.x) {
        if (vb >= n_tile_blocks) {
            const uint64_t j = (vb - n_tile_blocks) * CLONE_THREADS + threadIdx.x;
            if (j >= a.n_pairs) continue;
            const uint32_t from = __ldg(a.src + j), to = __ldg(a.dst + j);
            a.eps[to] = __ldg(a.eps + from);
            a.ucb_t[to] = __ldg(reinterpret_cast<const unsigned long long*>(a.ucb_t) + from);
            a.flag[to] = __ldg(a.flag + from);
            if (a.model_len) a.model_len[to] = __ldg(a.model_len + from);
            continue;
        }
        const uint64_t pair = vb / t.per_pair;
        uint32_t tile = (uint32_t)(vb % t.per_pair);
        // the segment holding this tile (unrolled: constant indices keep the kernel parameters out of local memory)
        uint8_t* base = a.seg[0].base;
        uint64_t stride = a.seg[0].stride;
        uint32_t width = t.width[0], t0 = tile;
#pragma unroll
        for (int k = 1; k < CLONE_MAX_SEGMENTS; ++k) {
            if (k < (int)a.n_seg && tile >= t.first[k]) {
                base = a.seg[k].base; stride = a.seg[k].stride; width = t.width[k]; t0 = tile - t.first[k];
            }
        }
        const uint8_t* from = base + (uint64_t)__ldg(a.src + pair) * stride;
        uint8_t* to = base + (uint64_t)__ldg(a.dst + pair) * stride;
        if (width == 16) copy_tile<uint4>(from, to, stride, t0);
        else if (width == 8) copy_tile<uint2>(from, to, stride, t0);
        else copy_tile<unsigned int>(from, to, stride, t0);
    }
}

}   // namespace

cudaError_t launch_clone_agents(const CloneArgs& a, cudaStream_t stream) {
    if (!a.n_pairs) return cudaSuccess;
    if (a.n_seg < 1 || a.n_seg > (uint32_t)CLONE_MAX_SEGMENTS) return cudaErrorInvalidValue;
    CloneTiling t{};
    for (uint32_t k = 0; k < a.n_seg; ++k) {
        const uint64_t s = a.seg[k].stride;
        if (s == 0 || s % 4) return cudaErrorInvalidValue;
        const uint32_t w = s % 16 == 0 ? 16u : s % 8 == 0 ? 8u : 4u;   // the stride keeps every agent's block aligned to it
        t.first[k] = t.per_pair;
        t.width[k] = w;
        t.per_pair += (uint32_t)((s / w + CLONE_THREADS * CLONE_VECS - 1) / (CLONE_THREADS * CLONE_VECS));
    }
    const uint64_t n_tile_blocks = a.n_pairs * t.per_pair;
    const uint64_t n_blocks = n_tile_blocks + (a.n_pairs + CLONE_THREADS - 1) / CLONE_THREADS;
    const unsigned grid = (unsigned)std::min<uint64_t>(n_blocks, 148u * 16u);
    k_clone_agents<<<grid, CLONE_THREADS, 0, stream>>>(a, t, n_tile_blocks, n_blocks);
    return cudaGetLastError();
}

}   // namespace rlb
