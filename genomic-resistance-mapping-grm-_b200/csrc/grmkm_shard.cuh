// grmkm_shard.cuh -- the device side of the sharded runs (grmkm_*_run_sharded): a rank packs the columns it owns of the
// rules a step chose, the splits a level chose or the models an evaluation scores, to send them to the other ranks.
// Every rank then runs the unchanged kernels on the compact matrix of those columns.
#pragma once
#include <cstdint>

namespace grmkm {

// out[w][i] = matrix[w][idx[i]], w < W, i < n: one warp per column, lanes over its word rows
__global__ void __launch_bounds__(256)
k_gather_columns(const unsigned long long* __restrict__ matrix, unsigned long long pitch, uint32_t W,
                 const unsigned long long* __restrict__ idx, uint32_t n, unsigned long long* __restrict__ out) {
    const uint32_t lane = threadIdx.x & 31u;
    for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += (gridDim.x * blockDim.x) >> 5) {
        const unsigned long long j = idx[i];
        for (uint32_t w = lane; w < W; w += 32) out[(unsigned long long)w * n + i] = matrix[(unsigned long long)w * pitch + j];
    }
}

}  // namespace grmkm
