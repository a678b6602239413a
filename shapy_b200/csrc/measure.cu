// Virtual measurements (mass, height, chest / waist / hip circumference) in ONE launch, one CTA per body.
//
// Replaces, for the fixed query the reference issues (a 2-triangle horizontal quad per measurement):
//   BodyMeasurements.forward           mesh-mesh-intersection/body_measurements/body_measurements.py:217-246
//   3 x (LBVH build + traversal)       mesh-mesh-intersection/src/mesh_mesh_intersect_cuda_op.cu:969-1079
//   3 x scipy.spatial.ConvexHull (CPU) body_measurements.py:160-173
// A plane touches O(sqrt(F)) triangles, so one streaming pass over the faces (read v_shaped once,
// 125 KB / body) beats building a 3 MB BVH three times: every face is tested against the query quad of
// each plane with exactly the reference's predicates (inclusive AABB test, 11-axis SAT with its
// fallback axes, "first ray hit" point selection -- see mmi_device.cuh), hits are appended to a
// shared-memory point list, and a warp per plane gift-wraps the 2-D hull (exact fp64 orientation
// predicate on the fp32 points, as qhull sees them) and sums the 3-D edge lengths in fp32.
// Compiled with -fmad=false (bit parity of the predicates with oracle/mmi_oracle.c).
#include <cstdlib>

#include "common.cuh"
#include "measure.cuh"
#include "mmi_device.cuh"

namespace shapy {

struct MeasureArgs {
  const float *verts;  // (B,V,3) or null
  const int *faces;    // (F,3)
  const float *tris;   // (B,F,3,3) or null
  int B, V, F;
  shapy_measure_landmarks_t lm;
  float *out;          // (B,5)
  float *pts_out;      // (B,3,maxp,3) or null
  int *cnt_out;        // (B,3) or null
  int maxp;
  int *status;
};

__device__ __forceinline__ mmi::Tri load_tri(const MeasureArgs &a, int b, int f) {
  mmi::Tri t;
  if (a.tris) {
    const float *p = a.tris + ((size_t)b * a.F + f) * 9;
    t.v0 = make_float3(p[0], p[1], p[2]);
    t.v1 = make_float3(p[3], p[4], p[5]);
    t.v2 = make_float3(p[6], p[7], p[8]);
  } else {
    const int *fi = a.faces + 3 * (size_t)f;
    const float *vb = a.verts + (size_t)b * a.V * 3;
    int i0 = fi[0], i1 = fi[1], i2 = fi[2];
    t.v0 = make_float3(vb[3 * i0], vb[3 * i0 + 1], vb[3 * i0 + 2]);
    t.v1 = make_float3(vb[3 * i1], vb[3 * i1 + 1], vb[3 * i1 + 2]);
    t.v2 = make_float3(vb[3 * i2], vb[3 * i2 + 1], vb[3 * i2 + 2]);
  }
  return t;
}

constexpr int kMeasThreads = 512;
__global__ void __launch_bounds__(kMeasThreads) measure_kernel(MeasureArgs a) {
  const int b = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  __shared__ float pts[3][kMaxPts][3];
  __shared__ int cnt[3];
  __shared__ float hs[3];
  __shared__ float lmy[2];
  __shared__ float red[kMeasThreads / 32];
  __shared__ int cand[kMaxCand];
  __shared__ int ncand;
  if (t < 3) cnt[t] = 0;
  if (t == 0) ncand = 0;
  if (t < 5) {
    mmi::Tri tr = load_tri(a, b, a.lm.face_idx[t]);
    // (tri * bc.reshape(3,1)).sum(0): v0*bc0 + v1*bc1 + v2*bc2, y component
    float y = tr.v0.y * a.lm.bc[t][0] + tr.v1.y * a.lm.bc[t][1] + tr.v2.y * a.lm.bc[t][2];
    if (t < 2) lmy[t] = y; else hs[t - 2] = y;
  }
  __syncthreads();
  const float h0 = hs[0], h1 = hs[1], h2 = hs[2];
  float vol = 0.f;
  // ---- phase 1: stream all faces once: signed volume + coarse (AABB) filter against the three planes.
  // Survivors go to a shared-memory queue so that the expensive exact predicates (phase 2) run with one
  // candidate per thread instead of one diverged lane per warp.
  for (int f = t; f < a.F; f += blockDim.x) {
    mmi::Tri T = load_tri(a, b, f);
    // compute_mass, body_measurements.py:207-214
    vol += -T.v2.x * T.v1.y * T.v0.z + T.v1.x * T.v2.y * T.v0.z + T.v2.x * T.v0.y * T.v1.z -
           T.v0.x * T.v2.y * T.v1.z - T.v1.x * T.v0.y * T.v2.z + T.v0.x * T.v1.y * T.v2.z;
    mmi::Box tb = mmi::tri_box(T);
    bool xz = (-1.f <= tb.hi.x) && (1.f >= tb.lo.x) && (-1.f <= tb.hi.z) && (1.f >= tb.lo.z);
    if (!xz || f == 0) continue;  // python keeps collision_faces > 0 only (body_measurements.py:161)
#pragma unroll
    for (int p = 0; p < 3; ++p) {
      float h = p == 0 ? h0 : (p == 1 ? h1 : h2);
      if (!((h <= tb.hi.y) && (h >= tb.lo.y))) continue;
      int slot = atomicAdd(&ncand, 2);
      if (slot + 1 < kMaxCand) { cand[slot] = (f << 3) | (p << 1); cand[slot + 1] = (f << 3) | (p << 1) | 1; }
    }
  }
  __syncthreads();
  // ---- phase 2: exact SAT + "first ray hit" point selection, one (face, plane, query triangle) per thread
  {
    const int n = min(ncand, kMaxCand);
    if (ncand > kMaxCand && t == 0 && a.status) atomicExch(a.status, 1);
    for (int i = t; i < n; i += blockDim.x) {
      const int c = cand[i], f = c >> 3, p = (c >> 1) & 3, q = c & 1;
      const float h = p == 0 ? h0 : (p == 1 ? h1 : h2);
      mmi::Tri T = load_tri(a, b, f);
      mmi::Tri Q;
      Q.v0 = make_float3(-1.f, h, -1.f);
      Q.v1 = q == 0 ? make_float3(1.f, h, -1.f) : make_float3(1.f, h, 1.f);
      Q.v2 = q == 0 ? make_float3(1.f, h, 1.f) : make_float3(-1.f, h, 1.f);
      if (!mmi::sat11(Q, T)) continue;
      float3 b1 = make_float3(0, 0, 0), b2 = b1;
      mmi::isect_points(Q, T, b1, b2);  // no hit -> barycentrics stay 0 (first-body semantics)
      int slot = atomicAdd(&cnt[p], 1);
      if (slot < kMaxPts) {
        pts[p][slot][0] = T.v0.x * b1.x + T.v1.x * b1.y + T.v2.x * b1.z;
        pts[p][slot][1] = T.v0.y * b1.x + T.v1.y * b1.y + T.v2.y * b1.z;
        pts[p][slot][2] = T.v0.z * b1.x + T.v1.z * b1.y + T.v2.z * b1.z;
      }
    }
  }
  for (int o = 16; o; o >>= 1) vol += __shfl_xor_sync(0xffffffffu, vol, o);
  if (lane == 0) red[warp] = vol;
  __syncthreads();
  if (t == 0) {
    float v = 0.f;
    for (int i = 0; i < kMeasThreads / 32; ++i) v += red[i];
    a.out[(size_t)b * 5 + 0] = fabsf(v) / 6.0f * 985.0f;
    a.out[(size_t)b * 5 + 1] = fabsf(lmy[0] - lmy[1]);
  }
  if (warp < 3) {
    const int p = warp;
    int n = cnt[p];
    bool truncated = ncand > kMaxCand;         // a truncated point set must not pass for a measurement: NaN below
    if (n > kMaxPts) {
      if (lane == 0 && a.status) atomicExch(a.status, 1);
      n = kMaxPts;
      truncated = true;
    }
    if (a.cnt_out && lane == 0) a.cnt_out[(size_t)b * 3 + p] = n;
    if (a.pts_out) {
      int m = min(n, a.maxp);
      for (int i = lane; i < m * 3; i += 32)
        a.pts_out[(((size_t)b * 3 + p) * a.maxp) * 3 + i] = pts[p][i / 3][i % 3];
      if (n > a.maxp && lane == 0 && a.status) atomicExch(a.status, 1);
    }
    float perim = 0.f;
    if (n < 3) {
      perim = __int_as_float(0x7fc00000);  // qhull would raise on a degenerate input
    } else {
      // start: lexicographic min (x, z)
      int best = -1;
      float bx = 0.f, bz = 0.f;
      for (int i = lane; i < n; i += 32) {
        float x = pts[p][i][0], z = pts[p][i][2];
        if (best < 0 || x < bx || (x == bx && z < bz)) { best = i; bx = x; bz = z; }
      }
      for (int o = 16; o; o >>= 1) {
        int ob = __shfl_xor_sync(0xffffffffu, best, o);
        float ox = __shfl_xor_sync(0xffffffffu, bx, o), oz = __shfl_xor_sync(0xffffffffu, bz, o);
        if (ob >= 0 && (best < 0 || ox < bx || (ox == bx && oz < bz) || (ox == bx && oz == bz && ob < best))) {
          best = ob; bx = ox; bz = oz;
        }
      }
      const int start = best;
      const float sx = bx, sz = bz;
      int cur = start;
      for (int it = 0; it < n + 1; ++it) {
        const float cx = pts[p][cur][0], cz = pts[p][cur][2];
        int nb = -1;
        float nx = 0.f, nz = 0.f;
        for (int i = lane; i < n; i += 32) {
          float x = pts[p][i][0], z = pts[p][i][2];
          if (x == cx && z == cz) continue;  // the point itself and its duplicates
          if (nb < 0 || better_next(cx, cz, nx, nz, x, z)) { nb = i; nx = x; nz = z; }
        }
        for (int o = 16; o; o >>= 1) {
          int ob = __shfl_xor_sync(0xffffffffu, nb, o);
          float ox = __shfl_xor_sync(0xffffffffu, nx, o), oz = __shfl_xor_sync(0xffffffffu, nz, o);
          if (ob >= 0) {
            bool take = nb < 0 || better_next(cx, cz, nx, nz, ox, oz) ||
                        (ox == nx && oz == nz && ob < nb);
            if (take) { nb = ob; nx = ox; nz = oz; }
          }
        }
        if (nb < 0) break;  // all points coincide
        float dx = pts[p][nb][0] - pts[p][cur][0], dy = pts[p][nb][1] - pts[p][cur][1],
              dz = pts[p][nb][2] - pts[p][cur][2];
        perim += sqrtf(dx * dx + dy * dy + dz * dz);
        cur = nb;
        if (nx == sx && nz == sz) break;
      }
    }
    if (lane == 0) a.out[(size_t)b * 5 + 2 + p] = truncated ? __int_as_float(0x7fc00000) : perim;
  }
}


// =================================================================================================================
// v2: the body's vertices are staged ONCE in shared memory (125.7 KB of the SM's 227 KB), every face then gathers its
// 9 coordinates from shared memory instead of through L1 / L2 (the gathers of v1 moved 752 KB per body for 125.7 KB
// of data and were latency bound), and the three hulls are wrapped by 24 warps instead of 3:
//   phase 0  coalesced copy of the body's vertices into shared memory (128-bit loads where the row is aligned)
//   phase 1  one pass over the faces: signed volume + AABB filter against the three planes -> candidate queue
//   phase 2  exact SAT + "first ray hit" point, one candidate per thread (as v1)
//   phase 3  per plane: the 8 extreme points in the directions k * 45 deg (exact: the keys x +- z are sums of two
//            floats in fp64) cut the hull into 8 chains; warp (plane, k) compacts the points on the outer side of the
//            chord E_k -> E_k+1 (exact fp64 orientation) and gift-wraps its chain from E_k to E_k+1.  The chain
//            lengths are summed in chain order, so the result does not depend on timing.
// Capacity overflows (candidates, points per plane) are reported through `status` AND poison the affected outputs
// with NaN: a truncated point set must never pass for a measurement.
__global__ void __launch_bounds__(kM2Threads, 1) measure_smem_kernel(MeasureArgs a) {
  extern __shared__ __align__(16) unsigned char m2_smem[];
  const int b = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int nvf = a.V * 3;
  float *vs = reinterpret_cast<float *>(m2_smem);                                   // [V * 3] (+ pad to 16 B)
  const size_t vs_bytes = ((size_t)nvf * 4 + 15) & ~(size_t)15;
  float *pts = reinterpret_cast<float *>(m2_smem + vs_bytes);                       // [3][kM2MaxPts][3]
  int *cand = reinterpret_cast<int *>(m2_smem + vs_bytes + 3 * kM2MaxPts * 12);     // [kM2MaxCand]
  unsigned short *clist = reinterpret_cast<unsigned short *>(cand);                // phase 3: [24][kM2ChainCap]
  __shared__ int cnt[3];
  __shared__ int ncand;
  __shared__ float hs[3], lmy[2];
  __shared__ float red[kM2Threads / 32];
  __shared__ M2Ext ext[3][8];
  __shared__ float chain_len[3][8];
  __shared__ int overflow;
  if (t < 3) cnt[t] = 0;
  if (t == 0) { ncand = 0; overflow = 0; }
  // ---- phase 0: vertices -> shared memory
  {
    const float *src = a.verts + (size_t)b * nvf;
    const int head = (int)((4 - (((size_t)b * nvf) & 3)) & 3);          // floats before the first 16-byte boundary
    const int nvec = nvf > head ? (nvf - head) / 4 : 0;
    for (int i = t; i < min(head, nvf); i += blockDim.x) vs[i] = src[i];
    const float4 *s4 = reinterpret_cast<const float4 *>(src + head);
    for (int i = t; i < nvec; i += blockDim.x) {
      const float4 q = __ldg(s4 + i);
      float *d = vs + head + 4 * i;
      d[0] = q.x; d[1] = q.y; d[2] = q.z; d[3] = q.w;
    }
    for (int i = head + 4 * nvec + t; i < nvf; i += blockDim.x) vs[i] = src[i];
  }
  __syncthreads();
  auto tri_of = [&](int f) {
    const int *fi = a.faces + 3 * (size_t)f;
    const int i0 = __ldg(fi), i1 = __ldg(fi + 1), i2 = __ldg(fi + 2);
    mmi::Tri T;
    T.v0 = make_float3(vs[3 * i0], vs[3 * i0 + 1], vs[3 * i0 + 2]);
    T.v1 = make_float3(vs[3 * i1], vs[3 * i1 + 1], vs[3 * i1 + 2]);
    T.v2 = make_float3(vs[3 * i2], vs[3 * i2 + 1], vs[3 * i2 + 2]);
    return T;
  };
  if (t < 5) {
    mmi::Tri tr = tri_of(a.lm.face_idx[t]);
    float y = tr.v0.y * a.lm.bc[t][0] + tr.v1.y * a.lm.bc[t][1] + tr.v2.y * a.lm.bc[t][2];
    if (t < 2) lmy[t] = y; else hs[t - 2] = y;
  }
  __syncthreads();
  const float h0 = hs[0], h1 = hs[1], h2 = hs[2];
  // ---- phase 1
  float vol = 0.f;
  for (int f = t; f < a.F; f += blockDim.x) {
    mmi::Tri T = tri_of(f);
    vol += -T.v2.x * T.v1.y * T.v0.z + T.v1.x * T.v2.y * T.v0.z + T.v2.x * T.v0.y * T.v1.z -
           T.v0.x * T.v2.y * T.v1.z - T.v1.x * T.v0.y * T.v2.z + T.v0.x * T.v1.y * T.v2.z;
    const float ylo = fminf(T.v0.y, fminf(T.v1.y, T.v2.y)), yhi = fmaxf(T.v0.y, fmaxf(T.v1.y, T.v2.y));
    const bool c0 = (h0 <= yhi) && (h0 >= ylo), c1 = (h1 <= yhi) && (h1 >= ylo), c2 = (h2 <= yhi) && (h2 >= ylo);
    if (!(c0 || c1 || c2) || f == 0) continue;   // python keeps collision_faces > 0 only (body_measurements.py:161)
    mmi::Box tb = mmi::tri_box(T);
    if (!((-1.f <= tb.hi.x) && (1.f >= tb.lo.x) && (-1.f <= tb.hi.z) && (1.f >= tb.lo.z))) continue;
#pragma unroll
    for (int p = 0; p < 3; ++p) {
      if (!(p == 0 ? c0 : (p == 1 ? c1 : c2))) continue;
      const int slot = atomicAdd(&ncand, 2);
      if (slot + 1 < kM2MaxCand) { cand[slot] = (f << 3) | (p << 1); cand[slot + 1] = (f << 3) | (p << 1) | 1; }
    }
  }
  for (int o = 16; o; o >>= 1) vol += __shfl_xor_sync(0xffffffffu, vol, o);
  if (lane == 0) red[warp] = vol;
  __syncthreads();
  // ---- phase 2
  {
    const int n = min(ncand, kM2MaxCand);
    if (ncand > kM2MaxCand && t == 0) overflow = 7;
    for (int i = t; i < n; i += blockDim.x) {
      const int c = cand[i], f = c >> 3, p = (c >> 1) & 3, q = c & 1;
      const float h = p == 0 ? h0 : (p == 1 ? h1 : h2);
      mmi::Tri T = tri_of(f);
      mmi::Tri Q;
      Q.v0 = make_float3(-1.f, h, -1.f);
      Q.v1 = q == 0 ? make_float3(1.f, h, -1.f) : make_float3(1.f, h, 1.f);
      Q.v2 = q == 0 ? make_float3(1.f, h, 1.f) : make_float3(-1.f, h, 1.f);
      if (!mmi::sat11(Q, T)) continue;
      float3 b1 = make_float3(0, 0, 0), b2 = b1;
      mmi::isect_points(Q, T, b1, b2);
      const int slot = atomicAdd(&cnt[p], 1);
      if (slot < kM2MaxPts) {
        float *o = pts + ((size_t)p * kM2MaxPts + slot) * 3;
        o[0] = T.v0.x * b1.x + T.v1.x * b1.y + T.v2.x * b1.z;
        o[1] = T.v0.y * b1.x + T.v1.y * b1.y + T.v2.y * b1.z;
        o[2] = T.v0.z * b1.x + T.v1.z * b1.y + T.v2.z * b1.z;
      }
    }
  }
  __syncthreads();     // the candidate queue is dead from here on: its storage becomes the chain lists
  if (t == 0) {
    float v = 0.f;
    for (int i = 0; i < kM2Threads / 32; ++i) v += red[i];
    a.out[(size_t)b * 5 + 0] = fabsf(v) / 6.0f * 985.0f;
    a.out[(size_t)b * 5 + 1] = fabsf(lmy[0] - lmy[1]);
  }
  // ---- phase 3a: extreme points
  const int hp = warp / 8, hk = warp % 8;          // warps 0..23: (plane, chain)
  int n = 0;
  if (warp < 24) {
    n = cnt[hp];
    if (n > kM2MaxPts) { if (lane == 0) atomicOr(&overflow, 1 << hp); n = kM2MaxPts; }
    const float *P = pts + (size_t)hp * kM2MaxPts * 3;
    int best = -1;
    double b1 = 0, b2 = 0;
    for (int i = lane; i < n; i += 32) {
      double k1, k2;
      m2_key(P[3 * i], P[3 * i + 2], hk, k1, k2);
      if (best < 0 || k1 > b1 || (k1 == b1 && k2 > b2)) { best = i; b1 = k1; b2 = k2; }
    }
    for (int o = 16; o; o >>= 1) {
      const int ob = __shfl_xor_sync(0xffffffffu, best, o);
      const double o1 = __shfl_xor_sync(0xffffffffu, b1, o), o2 = __shfl_xor_sync(0xffffffffu, b2, o);
      if (ob >= 0 && (best < 0 || o1 > b1 || (o1 == b1 && (o2 > b2 || (o2 == b2 && ob < best))))) { best = ob; b1 = o1; b2 = o2; }
    }
    if (lane == 0) {
      M2Ext e;
      e.idx = best;
      e.x = best >= 0 ? P[3 * best] : 0.f;
      e.z = best >= 0 ? P[3 * best + 2] : 0.f;
      ext[hp][hk] = e;
    }
  }
  __syncthreads();
  // ---- phase 3b: chain (plane hp, from E_hk to E_hk+1)
  if (warp < 24) {
    const float *P = pts + (size_t)hp * kM2MaxPts * 3;
    if (hk == 0) {
      if (a.cnt_out && lane == 0) a.cnt_out[(size_t)b * 3 + hp] = n;
      if (a.pts_out) {
        const int mcopy = min(n, a.maxp);
        for (int i = lane; i < mcopy * 3; i += 32) a.pts_out[(((size_t)b * 3 + hp) * a.maxp) * 3 + i] = P[i];
        if (n > a.maxp && lane == 0) atomicOr(&overflow, 8);
      }
    }
    float len = 0.f;
    const M2Ext e0 = ext[hp][hk], e1 = ext[hp][(hk + 1) & 7];
    if (n >= 3 && e0.idx >= 0 && !(e0.x == e1.x && e0.z == e1.z)) {
      // candidates of this chain: points on the outer side of (or on) the chord e0 -> e1
      unsigned short *L = clist + (size_t)warp * kM2ChainCap;
      int nl = 0;
      bool listed = true;
      {
        const double ux = (double)e1.x - (double)e0.x, uz = (double)e1.z - (double)e0.z;
        for (int base = 0; base < n; base += 32) {
          const int i = base + lane;
          bool keep = false;
          if (i < n) {
            const double wx = (double)P[3 * i] - (double)e0.x, wz = (double)P[3 * i + 2] - (double)e0.z;
            keep = (ux * wz - uz * wx) <= 0.0;
          }
          const unsigned m = __ballot_sync(0xffffffffu, keep);
          const int pos = nl + __popc(m & ((1u << lane) - 1));
          if (keep && pos < kM2ChainCap) L[pos] = (unsigned short)i;
          nl += __popc(m);
        }
        if (nl > kM2ChainCap) listed = false;     // degenerate distribution: scan every point instead
        __syncwarp();
      }
      const int nscan = listed ? nl : n;
      int cur = e0.idx;
      float cx = e0.x, cz = e0.z;
      for (int it = 0; it < n + 1; ++it) {
        int nb = -1;
        float nx = 0.f, nz = 0.f;
        for (int q = lane; q < nscan; q += 32) {
          const int i = listed ? (int)L[q] : q;
          const float x = P[3 * i], z = P[3 * i + 2];
          if (x == cx && z == cz) continue;
          if (nb < 0 || better_next(cx, cz, nx, nz, x, z)) { nb = i; nx = x; nz = z; }
        }
        for (int o = 16; o; o >>= 1) {
          const int ob = __shfl_xor_sync(0xffffffffu, nb, o);
          const float ox = __shfl_xor_sync(0xffffffffu, nx, o), oz = __shfl_xor_sync(0xffffffffu, nz, o);
          if (ob >= 0) {
            const bool take = nb < 0 || better_next(cx, cz, nx, nz, ox, oz) || (ox == nx && oz == nz && ob < nb);
            if (take) { nb = ob; nx = ox; nz = oz; }
          }
        }
        if (nb < 0) break;
        const float dx = P[3 * nb] - P[3 * cur], dy = P[3 * nb + 1] - P[3 * cur + 1], dz = P[3 * nb + 2] - P[3 * cur + 2];
        len += sqrtf(dx * dx + dy * dy + dz * dz);
        cur = nb; cx = nx; cz = nz;
        if (nx == e1.x && nz == e1.z) break;
      }
    }
    if (lane == 0) chain_len[hp][hk] = len;
  }
  __syncthreads();
  if (t < 3) {
    const int p = t;
    float perim = 0.f;
    for (int k = 0; k < 8; ++k) perim += chain_len[p][k];
    const int np = cnt[p];
    if (np < 3) perim = __int_as_float(0x7fc00000);                       // qhull would raise on a degenerate input
    if ((overflow & (1 << p))) perim = __int_as_float(0x7fc00000);   // truncated point set
    a.out[(size_t)b * 5 + 2 + p] = perim;
  }
  if (t == 0 && overflow && a.status) atomicExch(a.status, 1);
}

size_t measure_smem_bytes(int V) { return (((size_t)V * 12 + 15) & ~(size_t)15) + 3 * kM2MaxPts * 12 + kM2MaxCand * 4; }

}  // namespace shapy

using namespace shapy;

static int launch_measure(MeasureArgs a, void *stream) {
  SHAPY_REQUIRE(a.out && a.B > 0 && a.F > 0, "shapy_measure: bad argument");
  for (int i = 0; i < 5; ++i)
    SHAPY_REQUIRE(a.lm.face_idx[i] >= 0 && a.lm.face_idx[i] < a.F, "landmark face %d out of range", a.lm.face_idx[i]);
  if (a.status) SHAPY_CUDA_TRY(cudaMemsetAsync(a.status, 0, sizeof(int), (cudaStream_t)stream));
  static const bool v1_only = []() { const char *e = getenv("SHAPY_MEASURE_V1"); return e && e[0] == '1'; }();
  if (a.verts && !v1_only && a.V < 65536 && measure_smem_bytes(a.V) <= 220 * 1024) {
    static std::atomic<unsigned long long> attr_done{0};
    SHAPY_CUDA_TRY(set_max_dynamic_smem(measure_smem_kernel, 226 * 1024, attr_done));   // + 560 B static <= 227 KB
    measure_smem_kernel<<<a.B, kM2Threads, measure_smem_bytes(a.V), (cudaStream_t)stream>>>(a);
    SHAPY_LAUNCH_CHECK();
    return SHAPY_OK;
  }
  measure_kernel<<<a.B, kMeasThreads, 0, (cudaStream_t)stream>>>(a);
  SHAPY_LAUNCH_CHECK();
  return SHAPY_OK;
}

extern "C" int shapy_measure_forward(const float *v_shaped, const int32_t *faces, int batch, int num_verts,
                                     int num_faces, const shapy_measure_landmarks_t *lm, float *out,
                                     float *plane_points, int32_t *plane_counts, int max_points, int32_t *status,
                                     void *stream) {
  SHAPY_REQUIRE(v_shaped && faces && lm, "shapy_measure_forward: null argument");
  MeasureArgs a{v_shaped, faces, nullptr, batch, num_verts, num_faces, *lm, out, plane_points, plane_counts,
                max_points, status};
  return launch_measure(a, stream);
}

extern "C" int shapy_measure_forward_tris(const float *triangles, int batch, int num_faces,
                                          const shapy_measure_landmarks_t *lm, float *out, float *plane_points,
                                          int32_t *plane_counts, int max_points, int32_t *status, void *stream) {
  SHAPY_REQUIRE(triangles && lm, "shapy_measure_forward_tris: null argument");
  MeasureArgs a{nullptr, nullptr, triangles, batch, 0, num_faces, *lm, out, plane_points, plane_counts, max_points,
                status};
  return launch_measure(a, stream);
}
