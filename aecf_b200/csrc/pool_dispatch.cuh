// Explicit (M, J, DROP) dispatch of the pool kernels; one translation unit per
// (direction, dtype, dropout) so the instantiations compile in parallel.
#pragma once

#include "pool_core.cuh"

namespace aecf {

#define AECF_DISPATCH_M(M_, ...)                              \
    switch (M_) {                                             \
        case 1: { constexpr int kM = 1; __VA_ARGS__; } break; \
        case 2: { constexpr int kM = 2; __VA_ARGS__; } break; \
        case 3: { constexpr int kM = 3; __VA_ARGS__; } break; \
        case 4: { constexpr int kM = 4; __VA_ARGS__; } break; \
        case 5: { constexpr int kM = 5; __VA_ARGS__; } break; \
        case 6: { constexpr int kM = 6; __VA_ARGS__; } break; \
        case 7: { constexpr int kM = 7; __VA_ARGS__; } break; \
        case 8: { constexpr int kM = 8; __VA_ARGS__; } break; \
        default: return AECF_ERR_UNSUPPORTED;                 \
    }

#define AECF_DISPATCH_J(J_, ...)                              \
    switch (J_) {                                             \
        case 1: { constexpr int kJ = 1; __VA_ARGS__; } break; \
        case 2: { constexpr int kJ = 2; __VA_ARGS__; } break; \
        case 4: { constexpr int kJ = 4; __VA_ARGS__; } break; \
        default: return AECF_ERR_UNSUPPORTED;                 \
    }

// J = chunk columns per lane (1, 2, 4); DROP = attention dropout active; PAD = padded lane map (head_dim not a
// power-of-two number of chunks, pool_core.cuh).
// grid: CTAs of the slice kernel; sms: SM count (the streaming kernel sizes its persistent grid from it)
// fold: the folded-key-projection variants (values only in kv, precomputed scores)
template <typename T, bool DROP, bool PAD> int launch_pool_fwd(int M, int J, const PoolParams& p, int grid, int sms, bool fold, void* stream);
template <typename T, bool DROP, bool PAD> int launch_pool_bwd(int M, int J, const PoolParams& p, int grid, bool fold, void* stream);
template <typename T, bool DROP, bool PAD> int pool_bwd_blocks_per_sm(int M, int J, bool fold);
// several fusion queries per sample (pool_multi.cuh); the backward runs one CTA per SM
template <typename T, bool DROP, bool PAD> int launch_pool_fwd_multi(int M, int J, const PoolParams& p, const MultiQuery& mq, int grid, void* stream);
template <typename T, bool DROP, bool PAD> int launch_pool_bwd_multi(int M, int J, const PoolParams& p, const MultiQuery& mq, int grid, void* stream);

void note_pool_kernel(const char* fmt, ...);         // api.cu: records what aecf_pool_last_kernel() reports

}  // namespace aecf
