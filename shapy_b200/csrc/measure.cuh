// Capacities and hull predicates shared by the measurement forward (measure.cu) and its backward
// (measure_grad.cu).  The backward rebuilds the forward's point sets and hulls, so both must agree on
// these exactly.  Translation units including this header are compiled with -fmad=false.
#pragma once
#include <cuda_runtime.h>

namespace shapy {

// measure_kernel (v1, triangles entry and fallback)
constexpr int kMaxPts = 512;
constexpr int kMaxCand = 4096;  // (face, plane, query triangle) candidates that pass the AABB filter, per body

// measure_smem_kernel (v2, vertices staged in shared memory)
constexpr int kM2Threads = 1024;
constexpr int kM2MaxPts = 1024;
constexpr int kM2MaxCand = 8192;     // ints; the buffer is reused for the per-chain candidate lists (u16) in phase 3
constexpr int kM2ChainCap = 640;     // 24 chains x 640 x 2 B = 30 KB <= 32 KB

__device__ __forceinline__ bool better_next(double cx, double cz, float ax, float az, float bx, float bz) {
  // true when candidate b should replace a as the next hull vertex after c (counter-clockwise walk):
  // b is strictly to the right of c->a, or collinear and farther.
  double ux = (double)ax - cx, uz = (double)az - cz, wx = (double)bx - cx, wz = (double)bz - cz;
  double o = ux * wz - uz * wx;
  if (o < 0) return true;
  if (o > 0) return false;
  return (wx * wx + wz * wz) > (ux * ux + uz * uz);
}

struct M2Ext { float x, z; int idx; };

__device__ __forceinline__ void m2_key(float x, float z, int k, double &k1, double &k2) {
  // direction d_k = (dx, dz), k * 45 degrees (unnormalised, exact); tie-break direction = d_k rotated by +90 degrees
  const int dxs[8] = {1, 1, 0, -1, -1, -1, 0, 1}, dzs[8] = {0, 1, 1, 1, 0, -1, -1, -1};
  const double dx = dxs[k], dz = dzs[k];
  k1 = dx * (double)x + dz * (double)z;
  k2 = -dz * (double)x + dx * (double)z;
}

// dynamic shared memory of measure_smem_kernel: vertices (16-byte padded) + 3 point lists + candidate queue
size_t measure_smem_bytes(int V);

}  // namespace shapy
