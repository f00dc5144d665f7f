// dmma.cuh -- the fp64 tensor-core instruction shared by gp.cu and synlik.cu.
//
// tcgen05.mma has no f64 kind, so fp64 products on sm_100a go through mma.sync m8n8k4.f64
// (SASS DMMA).  Fragment layout per lane (g = lane / 4, t = lane % 4):
//   a = A[g][t] (8 x 4, row-major),  b = B[t][g] (4 x 8),  {c0, c1} = C[g][2t], C[g][2t + 1].
#pragma once

namespace elfi {

__device__ __forceinline__ void dmma_m8n8k4(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

}  // namespace elfi
