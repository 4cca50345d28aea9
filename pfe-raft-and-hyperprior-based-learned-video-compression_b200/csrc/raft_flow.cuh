// raft_flow.cuh -- the one kernel of rdvc_raft_flow that is not a network layer: the refinement loop's starting
// state.  coords1 = coords0 = the 1/8-resolution pixel grid (TV:_utils.py:22-26: channel 0 = x, channel 1 = y) and
// flow = coords1 - coords0 = 0, both fp32 (B, 2, h, w).  The grid itself is never stored: FH_CONV2's coordinate-update
// epilogue subtracts each pixel's own (x, y).
#pragma once

namespace rdvc {

__global__ void raft_coords_init_kernel(float* __restrict__ coords, float* __restrict__ flow, int B, int h, int w) {
    const long long hw = static_cast<long long>(h) * w;
    const long long n = static_cast<long long>(B) * hw;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long b = i / hw, r = i - b * hw;
        const long long o = 2 * b * hw + r;
        coords[o] = static_cast<float>(r % w);
        coords[o + hw] = static_cast<float>(r / w);
        flow[o] = 0.f;
        flow[o + hw] = 0.f;
    }
}

}  // namespace rdvc
