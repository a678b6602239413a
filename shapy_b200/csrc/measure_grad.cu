// Backward of the virtual measurements (measure.cu): d(mass, height, chest, waist, hips) / d(vertices or triangles)
// for an upstream gradient g (B, 5), with the reference's autograd semantics
// (mesh-mesh-intersection/body_measurements/body_measurements.py:132-215):
//   mass    985 |sum_f det(T0, T1, T2)| / 6   -> corner k of face f gets s 985/6 (T_k+1 x T_k+2), s = sign(sum det)
//   height  |y_ht - y_hl|, y = sum_k bc_k T[f, k].y  -> only the y components of the two landmark faces
//   chest / waist / hips  sum over hull edges (a, b) of |p_b - p_a|, p = sum_k bc_k T[f, k] with the recorded
//           barycentric bc held constant (the collision query runs under no_grad, as does the slicing plane):
//           each edge adds -/+ (p_b - p_a) / |p_b - p_a| to its two points, each point bc_k times that to its corners.
// There is no tape: one CTA per body recomputes the forward's selection with the same predicates and capacities
// (candidate filter, exact SAT, "first ray hit" point, hull), so the forward kernels and their cost are untouched.
// The hull is one gift-wrap per plane whose ties (two points with the same (x, z)) go to the smaller candidate code
// f << 3 | p << 1 | q, not to the order in which atomics filled the point list: gradients are bit-reproducible.
// Every output element is a sum in a fixed order (vertex -> adjacent faces in face order -> mass, height, hull
// points in walk order), accumulated in fp64 and rounded once; there are no float atomics.  A circumference that the
// forward returns as NaN (capacity overflow, fewer than 3 points) makes the body's whole gradient NaN when its g entry
// is non-zero and contributes nothing when it is zero.  Compiled with -fmad=false like measure.cu: the recomputed points are bit-identical.
#include "common.cuh"
#include "measure.cuh"
#include "mmi_device.cuh"

namespace shapy {

struct GradArgs {
  const float *verts;    // (B,V,3) or null
  const int *faces;      // (F,3)
  const float *tris;     // (B,F,3,3) or null
  int B, V, F;
  shapy_measure_landmarks_t lm;
  const float *g;        // (B,5)
  const int *adj_off;    // (V+1) vertex -> range of adj          (vertices entry)
  const int *adj;        // (3F)  f << 2 | corner, sorted per vertex
  float *grad;           // (B,V,3) or (B,F,3,3)
  int maxpts, maxcand;   // the capacities of the forward kernel this entry mirrors
};

constexpr int kGThreads = kM2Threads;

__device__ __forceinline__ mmi::Tri plane_query(float h, int q) {
  mmi::Tri Q;
  Q.v0 = make_float3(-1.f, h, -1.f);
  Q.v1 = q == 0 ? make_float3(1.f, h, -1.f) : make_float3(1.f, h, 1.f);
  Q.v2 = q == 0 ? make_float3(1.f, h, 1.f) : make_float3(-1.f, h, 1.f);
  return Q;
}

__device__ __forceinline__ float3 corner(const mmi::Tri &T, int k) { return k == 0 ? T.v0 : (k == 1 ? T.v1 : T.v2); }

template <bool kTris>
__global__ void __launch_bounds__(kGThreads, 1) measure_grad_kernel(GradArgs a) {
  extern __shared__ __align__(16) unsigned char mg_smem[];
  const int b = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int nvf = kTris ? 0 : a.V * 3;
  const size_t vs_bytes = ((size_t)nvf * 4 + 15) & ~(size_t)15;
  float *vs = reinterpret_cast<float *>(mg_smem);                                             // [V * 3]
  float *pts = reinterpret_cast<float *>(mg_smem + vs_bytes);                                 // [3][kM2MaxPts][3]
  int *cand = reinterpret_cast<int *>(mg_smem + vs_bytes + 3 * kM2MaxPts * 12);               // [kM2MaxCand]
  int *codes = cand + kM2MaxCand;                                                             // [3][kM2MaxPts]
  int *hull = cand;                         // after phase 2: [3][kM2MaxPts] slots in walk order
  unsigned *fbits = reinterpret_cast<unsigned *>(cand + 3 * kM2MaxPts);   // faces carrying a hull point (bitset)
  __shared__ int cnt[3], nhull[3];
  __shared__ int ncand, overflow;
  __shared__ float hs[3], lmy[2];
  __shared__ float red[kGThreads / 32];
  if (t < 3) cnt[t] = 0;
  if (t == 0) { ncand = 0; overflow = 0; }
  if (!kTris) {
    const float *src = a.verts + (size_t)b * nvf;
    for (int i = t; i < nvf; i += blockDim.x) vs[i] = __ldg(src + i);
  }
  __syncthreads();
  auto tri_of = [&](int f) {
    mmi::Tri T;
    if (kTris) {
      const float *p = a.tris + ((size_t)b * a.F + f) * 9;
      T.v0 = make_float3(__ldg(p), __ldg(p + 1), __ldg(p + 2));
      T.v1 = make_float3(__ldg(p + 3), __ldg(p + 4), __ldg(p + 5));
      T.v2 = make_float3(__ldg(p + 6), __ldg(p + 7), __ldg(p + 8));
    } else {
      const int *fi = a.faces + 3 * (size_t)f;
      const int i0 = __ldg(fi), i1 = __ldg(fi + 1), i2 = __ldg(fi + 2);
      T.v0 = make_float3(vs[3 * i0], vs[3 * i0 + 1], vs[3 * i0 + 2]);
      T.v1 = make_float3(vs[3 * i1], vs[3 * i1 + 1], vs[3 * i1 + 2]);
      T.v2 = make_float3(vs[3 * i2], vs[3 * i2 + 1], vs[3 * i2 + 2]);
    }
    return T;
  };
  if (t < 5) {
    mmi::Tri tr = tri_of(a.lm.face_idx[t]);
    float y = tr.v0.y * a.lm.bc[t][0] + tr.v1.y * a.lm.bc[t][1] + tr.v2.y * a.lm.bc[t][2];
    if (t < 2) lmy[t] = y; else hs[t - 2] = y;
  }
  __syncthreads();
  const float h0 = hs[0], h1 = hs[1], h2 = hs[2];
  // ---- the forward's phase 1: signed volume + candidate filter
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
      if (slot + 1 < a.maxcand) { cand[slot] = (f << 3) | (p << 1); cand[slot + 1] = (f << 3) | (p << 1) | 1; }
    }
  }
  for (int o = 16; o; o >>= 1) vol += __shfl_xor_sync(0xffffffffu, vol, o);
  if (lane == 0) red[warp] = vol;
  __syncthreads();
  // ---- the forward's phase 2: exact SAT + first-hit point, recorded with its candidate code
  {
    const int n = min(ncand, a.maxcand);
    if (ncand > a.maxcand && t == 0) overflow = 7;
    for (int i = t; i < n; i += blockDim.x) {
      const int c = cand[i], f = c >> 3, p = (c >> 1) & 3, q = c & 1;
      const mmi::Tri T = tri_of(f), Q = plane_query(p == 0 ? h0 : (p == 1 ? h1 : h2), q);
      if (!mmi::sat11(Q, T)) continue;
      float3 b1 = make_float3(0, 0, 0), b2 = b1;
      mmi::isect_points(Q, T, b1, b2);
      const int slot = atomicAdd(&cnt[p], 1);
      if (slot < kM2MaxPts) {
        float *o = pts + ((size_t)p * kM2MaxPts + slot) * 3;
        o[0] = T.v0.x * b1.x + T.v1.x * b1.y + T.v2.x * b1.z;
        o[1] = T.v0.y * b1.x + T.v1.y * b1.y + T.v2.y * b1.z;
        o[2] = T.v0.z * b1.x + T.v1.z * b1.y + T.v2.z * b1.z;
        codes[p * kM2MaxPts + slot] = c;
      }
    }
  }
  __syncthreads();     // the candidate queue is dead: its storage becomes the hull lists and the face bitset
  for (int i = t; i < (a.F + 31) / 32; i += blockDim.x) fbits[i] = 0u;
  // ---- hull: one warp per plane, gift-wrap from the lexicographic (x, z) minimum, ties to the smaller code
  if (warp < 3) {
    const int p = warp;
    const int n = min(cnt[p], kM2MaxPts);
    if (cnt[p] > a.maxpts && lane == 0) atomicOr(&overflow, 1 << p);
    const float *P = pts + (size_t)p * kM2MaxPts * 3;
    const int *Cd = codes + p * kM2MaxPts;
    int *L = hull + p * kM2MaxPts;
    int nh = 0;
    if (n >= 3 && cnt[p] <= a.maxpts && ncand <= a.maxcand) {
      int best = -1, bc = 0;
      float bx = 0.f, bz = 0.f;
      for (int i = lane; i < n; i += 32) {
        const float x = P[3 * i], z = P[3 * i + 2];
        const int c = Cd[i];
        if (best < 0 || x < bx || (x == bx && (z < bz || (z == bz && c < bc)))) { best = i; bx = x; bz = z; bc = c; }
      }
      for (int o = 16; o; o >>= 1) {
        const int ob = __shfl_xor_sync(0xffffffffu, best, o), oc = __shfl_xor_sync(0xffffffffu, bc, o);
        const float ox = __shfl_xor_sync(0xffffffffu, bx, o), oz = __shfl_xor_sync(0xffffffffu, bz, o);
        if (ob >= 0 && (best < 0 || ox < bx || (ox == bx && (oz < bz || (oz == bz && oc < bc))))) {
          best = ob; bx = ox; bz = oz; bc = oc;
        }
      }
      const float sx = bx, sz = bz;
      int cur = best;
      for (int it = 0; it < n + 1 && nh < kM2MaxPts; ++it) {
        const float cx = P[3 * cur], cz = P[3 * cur + 2];
        int nb = -1, nc = 0;
        float nx = 0.f, nz = 0.f;
        for (int i = lane; i < n; i += 32) {
          const float x = P[3 * i], z = P[3 * i + 2];
          if (x == cx && z == cz) continue;
          const int c = Cd[i];
          if (nb < 0 || better_next(cx, cz, nx, nz, x, z) || (x == nx && z == nz && c < nc)) {
            nb = i; nx = x; nz = z; nc = c;
          }
        }
        for (int o = 16; o; o >>= 1) {
          const int ob = __shfl_xor_sync(0xffffffffu, nb, o), oc = __shfl_xor_sync(0xffffffffu, nc, o);
          const float ox = __shfl_xor_sync(0xffffffffu, nx, o), oz = __shfl_xor_sync(0xffffffffu, nz, o);
          if (ob >= 0 && (nb < 0 || better_next(cx, cz, nx, nz, ox, oz) || (ox == nx && oz == nz && oc < nc))) {
            nb = ob; nx = ox; nz = oz; nc = oc;
          }
        }
        if (nb < 0) break;  // all points coincide: no edge
        if (lane == 0) L[nh] = cur;
        ++nh;
        cur = nb;
        if (nx == sx && nz == sz) break;
      }
    }
    if (lane == 0) nhull[p] = nh;
  }
  __syncthreads();
  for (int i = t; i < 3 * kM2MaxPts; i += blockDim.x) {
    const int p = i / kM2MaxPts, j = i % kM2MaxPts;
    if (j < nhull[p]) {
      const int f = codes[p * kM2MaxPts + hull[i]] >> 3;
      atomicOr(&fbits[f >> 5], 1u << (f & 31));
    }
  }
  __syncthreads();
  // ---- scales of the five terms
  const float *gb = a.g + (size_t)b * 5;
  const float gm = gb[0], gh = gb[1];
  float gc[3];
  bool nan_body = false;
#pragma unroll
  for (int p = 0; p < 3; ++p) {
    gc[p] = gb[2 + p];
    const bool fwd_nan = cnt[p] < 3 || (overflow & (1 << p));
    if (gc[p] != 0.f && fwd_nan) nan_body = true;
    if (fwd_nan) gc[p] = 0.f;
  }
  float v = 0.f;
  for (int i = 0; i < kGThreads / 32; ++i) v += red[i];
  const float sm = (float)((v > 0.f) - (v < 0.f)), sh = (float)((lmy[0] > lmy[1]) - (lmy[0] < lmy[1]));
  const float cm = gm * sm * (985.0f / 6.0f), ch = gh * sh;
  const int fht = a.lm.face_idx[0], fhl = a.lm.face_idx[1];
  // adds d/dT[f, k] of the five terms to out[k - k0] for the corners k0 <= k < k1.  The mass term is formed in fp64:
  // the faces around a vertex cancel to ~1e-5 of their size, which fp32 products would not resolve.
  auto face_grad = [&](int f, const mmi::Tri &T, int k0, int k1, double3 *out) {
    for (int k = k0; k < k1; ++k) {
      double3 acc = out[k - k0];
      if (gm != 0.f) {
        const float3 u = corner(T, (k + 1) % 3), w = corner(T, (k + 2) % 3);
        const double ux = u.x, uy = u.y, uz = u.z, wx = w.x, wy = w.y, wz = w.z;
        acc.x += (double)cm * (uy * wz - uz * wy);
        acc.y += (double)cm * (uz * wx - ux * wz);
        acc.z += (double)cm * (ux * wy - uy * wx);
      }
      if (gh != 0.f) {
        if (f == fht) acc.y += ch * a.lm.bc[0][k];
        if (f == fhl) acc.y -= ch * a.lm.bc[1][k];
      }
      out[k - k0] = acc;
    }
    if (!(fbits[f >> 5] & (1u << (f & 31)))) return;
    for (int p = 0; p < 3; ++p) {
      if (gc[p] == 0.f) continue;
      const int H = nhull[p];
      const int *L = hull + p * kM2MaxPts, *Cd = codes + p * kM2MaxPts;
      const float *P = pts + (size_t)p * kM2MaxPts * 3;
      for (int i = 0; i < H; ++i) {
        const int s = L[i], c = Cd[s];
        if ((c >> 3) != f) continue;
        const int sp = L[(i + H - 1) % H], sn = L[(i + 1) % H];
        const float3 pi = make_float3(P[3 * s], P[3 * s + 1], P[3 * s + 2]);
        const float3 din = mmi::sub3(pi, make_float3(P[3 * sp], P[3 * sp + 1], P[3 * sp + 2]));
        const float3 dout = mmi::sub3(make_float3(P[3 * sn], P[3 * sn + 1], P[3 * sn + 2]), pi);
        const float lin = sqrtf(din.x * din.x + din.y * din.y + din.z * din.z);
        const float lout = sqrtf(dout.x * dout.x + dout.y * dout.y + dout.z * dout.z);
        const float3 gp = mmi::sub3(make_float3(din.x / lin, din.y / lin, din.z / lin),
                                    make_float3(dout.x / lout, dout.y / lout, dout.z / lout));
        float3 b1 = make_float3(0, 0, 0), b2 = b1;
        mmi::isect_points(plane_query(p == 0 ? h0 : (p == 1 ? h1 : h2), c & 1), T, b1, b2);
        for (int k = k0; k < k1; ++k) {
          const float w = gc[p] * (k == 0 ? b1.x : (k == 1 ? b1.y : b1.z));
          out[k - k0].x += w * gp.x;
          out[k - k0].y += w * gp.y;
          out[k - k0].z += w * gp.z;
        }
      }
    }
  };
  const float qnan = __int_as_float(0x7fc00000);
  if (kTris) {
    float *o = a.grad + (size_t)b * a.F * 9;
    for (int f = t; f < a.F; f += blockDim.x) {
      const mmi::Tri T = tri_of(f);
      double3 r[3];
      for (int k = 0; k < 3; ++k) r[k] = make_double3(0.0, 0.0, 0.0);
      face_grad(f, T, 0, 3, r);
      float *of = o + (size_t)f * 9;
      for (int k = 0; k < 3; ++k) {
        of[3 * k] = nan_body ? qnan : (float)r[k].x;
        of[3 * k + 1] = nan_body ? qnan : (float)r[k].y;
        of[3 * k + 2] = nan_body ? qnan : (float)r[k].z;
      }
    }
  } else {
    float *o = a.grad + (size_t)b * nvf;
    for (int vi = t; vi < a.V; vi += blockDim.x) {
      double3 acc = make_double3(0.0, 0.0, 0.0);
      const int e0 = __ldg(a.adj_off + vi), e1 = __ldg(a.adj_off + vi + 1);
      for (int e = e0; e < e1; ++e) {
        const int fk = __ldg(a.adj + e), f = fk >> 2, k = fk & 3;
        face_grad(f, tri_of(f), k, k + 1, &acc);
      }
      o[3 * vi] = nan_body ? qnan : (float)acc.x;
      o[3 * vi + 1] = nan_body ? qnan : (float)acc.y;
      o[3 * vi + 2] = nan_body ? qnan : (float)acc.z;
    }
  }
}

// vertex -> (face << 2 | corner) adjacency, each vertex's list in increasing order.  One CTA: counts in shared
// memory, one exclusive scan, an unordered fill, then a per-vertex insertion sort (lists are ~6 long).
constexpr int kAdjThreads = 1024;
__global__ void __launch_bounds__(kAdjThreads) measure_adjacency_kernel(const int *faces, int V, int F, int *off,
                                                                        int *adj) {
  extern __shared__ int cur[];   // [V]
  __shared__ int wsum[kAdjThreads / 32];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  for (int v = t; v < V; v += blockDim.x) cur[v] = 0;
  __syncthreads();
  for (int i = t; i < 3 * F; i += blockDim.x) {
    const int v = faces[i];
    if ((unsigned)v < (unsigned)V) atomicAdd(&cur[v], 1);
  }
  __syncthreads();
  const int chunk = (V + blockDim.x - 1) / blockDim.x, lo = min(V, t * chunk), hi = min(V, lo + chunk);
  int s = 0;
  for (int v = lo; v < hi; ++v) s += cur[v];
  int x = s;
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) wsum[warp] = x;
  __syncthreads();
  if (warp == 0) {
    int w = wsum[lane];
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += y;
    }
    wsum[lane] = w;
  }
  __syncthreads();
  int pre = x - s + (warp ? wsum[warp - 1] : 0);
  for (int v = lo; v < hi; ++v) {
    const int c = cur[v];
    off[v] = pre;
    cur[v] = pre;
    pre += c;
  }
  if (t == blockDim.x - 1) off[V] = wsum[31];
  __syncthreads();
  for (int i = t; i < 3 * F; i += blockDim.x) {
    const int v = faces[i];
    if ((unsigned)v < (unsigned)V) adj[atomicAdd(&cur[v], 1)] = ((i / 3) << 2) | (i % 3);
  }
  __syncthreads();
  for (int v = t; v < V; v += blockDim.x) {
    const int e0 = off[v], e1 = off[v + 1];
    for (int i = e0 + 1; i < e1; ++i) {
      const int key = adj[i];
      int j = i - 1;
      while (j >= e0 && adj[j] > key) { adj[j + 1] = adj[j]; --j; }
      adj[j + 1] = key;
    }
  }
}

static size_t grad_smem_bytes(int V) {
  return (((size_t)V * 12 + 15) & ~(size_t)15) + 3 * kM2MaxPts * 12 + kM2MaxCand * 4 + 3 * kM2MaxPts * 4;
}
constexpr size_t kGradSmemMax = 226 * 1024;   // + static shared memory <= 227 KB

}  // namespace shapy

using namespace shapy;

static int check_grad_args(const GradArgs &a) {
  SHAPY_REQUIRE(a.g && a.grad && a.B > 0 && a.F > 0, "shapy_measure_backward: bad argument");
  // the hull lists and the face bitset share the candidate queue's storage; codes hold f << 3
  SHAPY_REQUIRE(a.F <= (kM2MaxCand - 3 * kM2MaxPts) * 32 && a.F < (1 << 27),
                "shapy_measure_backward: %d faces exceed the kernel's face bitset", a.F);
  for (int i = 0; i < 5; ++i)
    SHAPY_REQUIRE(a.lm.face_idx[i] >= 0 && a.lm.face_idx[i] < a.F, "landmark face %d out of range", a.lm.face_idx[i]);
  return SHAPY_OK;
}

extern "C" size_t shapy_measure_backward_workspace_bytes(int num_verts, int num_faces) {
  if (num_verts <= 0 || num_faces <= 0) return 0;
  return align_up((size_t)(num_verts + 1) * sizeof(int), 256) + (size_t)3 * num_faces * sizeof(int);
}

extern "C" int shapy_measure_backward(const float *v_shaped, const int32_t *faces, int batch, int num_verts,
                                      int num_faces, const shapy_measure_landmarks_t *lm, const float *grad_out,
                                      float *grad_v, void *workspace, size_t workspace_bytes, void *stream) {
  SHAPY_REQUIRE(v_shaped && faces && lm, "shapy_measure_backward: null argument");
  SHAPY_REQUIRE(num_verts > 0 && grad_smem_bytes(num_verts) <= kGradSmemMax,
                "shapy_measure_backward: %d vertices do not fit the kernel's shared-memory staging (at most %d)",
                num_verts, (int)((kGradSmemMax - grad_smem_bytes(0)) / 12));
  SHAPY_REQUIRE(workspace && workspace_bytes >= shapy_measure_backward_workspace_bytes(num_verts, num_faces),
                "shapy_measure_backward: workspace too small");
  int *off = (int *)workspace;
  int *adj = (int *)((char *)workspace + align_up((size_t)(num_verts + 1) * sizeof(int), 256));
  GradArgs a{v_shaped, faces, nullptr, batch, num_verts, num_faces, *lm, grad_out, off, adj, grad_v,
             kM2MaxPts, kM2MaxCand};
  const int rc = check_grad_args(a);
  if (rc != SHAPY_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  static std::atomic<unsigned long long> adj_attr{0}, attr{0};
  SHAPY_CUDA_TRY(set_max_dynamic_smem(measure_adjacency_kernel, 200 * 1024, adj_attr));
  measure_adjacency_kernel<<<1, kAdjThreads, (size_t)num_verts * 4, st>>>(faces, num_verts, num_faces, off, adj);
  SHAPY_LAUNCH_CHECK();
  SHAPY_CUDA_TRY(set_max_dynamic_smem(measure_grad_kernel<false>, (int)kGradSmemMax, attr));
  measure_grad_kernel<false><<<batch, kGThreads, grad_smem_bytes(num_verts), st>>>(a);
  SHAPY_LAUNCH_CHECK();
  return SHAPY_OK;
}

extern "C" int shapy_measure_backward_tris(const float *triangles, int batch, int num_faces,
                                           const shapy_measure_landmarks_t *lm, const float *grad_out,
                                           float *grad_tris, void *stream) {
  SHAPY_REQUIRE(triangles && lm, "shapy_measure_backward_tris: null argument");
  // the triangles forward is measure_kernel: its capacities decide which circumferences are NaN
  GradArgs a{nullptr, nullptr, triangles, batch, 0, num_faces, *lm, grad_out, nullptr, nullptr, grad_tris,
             kMaxPts, kMaxCand};
  const int rc = check_grad_args(a);
  if (rc != SHAPY_OK) return rc;
  static std::atomic<unsigned long long> attr{0};
  SHAPY_CUDA_TRY(set_max_dynamic_smem(measure_grad_kernel<true>, (int)grad_smem_bytes(0), attr));
  measure_grad_kernel<true><<<batch, kGThreads, grad_smem_bytes(0), (cudaStream_t)stream>>>(a);
  SHAPY_LAUNCH_CHECK();
  return SHAPY_OK;
}
