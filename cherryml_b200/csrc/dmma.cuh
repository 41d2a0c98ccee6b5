// FP64 tensor-core product shared by the fit kernels and the pair posterior pass.
#pragma once

// D += A B for one 8x8x4 step of mma.sync.m8n8k4.f64.  Fragments: A: lane -> (row = lane/4,
// k = lane%4); B: (k = lane%4, col = lane/4); D: (row = lane/4, cols = 2*(lane%4), +1).
__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}
