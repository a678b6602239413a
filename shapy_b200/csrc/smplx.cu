// Fused SMPL-X body-model evaluation for sm_100a.
//
// Replaces the ~90-launch reference chain (blend_shapes -> vertices2joints -> pose blend ->
// batch_rigid_transform (54 serial bmm) -> skinning -> landmarks -> J14), reference
// regressor/human_shape/models/body_models/lbs.py:99-295 and body_models.py:628-767, by three
// launches:
//   smplx_pose_kernel    per body: joints from the (pre-contracted, exact) J_template + J_dirs . beta,
//                        level-parallel kinematic chain, A = G - [0 | G . J], pose feature, contour LUT row
//   smplx_vertex_kernel  tile of 32 vertices x 32 bodies: shape blend + pose blend (constants staged
//                        through shared memory once per tile, reused by all 32 bodies) + sparse skinning
//   smplx_joints_kernel  per body: landmarks, sparse J14 regressor + overwrite, weak-perspective camera
// plus smplx_shape_kernel for the T-pose path (SMPL.forward_shape, body_models.py:292-302).
//
// Exact structure that is exploited (changes summation order only):
//   * J = J_regressor . (T + S.beta) = J_regressor.T + (J_regressor.S).beta  (contracted once, in fp64)
//   * joints >= n_rot are identity => their pose-feature rows are exactly 0 and are skipped
//   * lbs_weights and the J14 regressor are stored sparse (ELL / CSR); zero entries contribute exactly 0
#include <algorithm>
#include <cmath>
#include <cstring>

#include "smplx.cuh"
#include "umma.cuh"

namespace shapy {

constexpr int TV = 32;  // vertices per tile (one per lane)
constexpr int TB = 32;  // bodies per tile (8 per warp, 4 warps)
constexpr int KC = 32;  // pose-feature rows staged per chunk

// ----------------------------------------------------------------------------------------------
__global__ void decode_rot6d_kernel(const float *__restrict__ raw, int n, float *__restrict__ rot) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float *x = raw + 6 * (size_t)i;
  // row-major 3x2: column 0 = x[0], x[2], x[4]; column 1 = x[1], x[3], x[5]  (pose_utils.py:138-153)
  float a0 = x[0], a1 = x[2], a2 = x[4], c0 = x[1], c1 = x[3], c2 = x[5];
  float n1 = fmaxf(sqrtf(a0 * a0 + a1 * a1 + a2 * a2), 1e-12f);
  float b10 = a0 / n1, b11 = a1 / n1, b12 = a2 / n1;
  float d = b10 * c0 + b11 * c1 + b12 * c2;
  float u0 = c0 - d * b10, u1 = c1 - d * b11, u2 = c2 - d * b12;
  float n2 = fmaxf(sqrtf(u0 * u0 + u1 * u1 + u2 * u2), 1e-12f);
  float b20 = u0 / n2, b21 = u1 / n2, b22 = u2 / n2;
  float b30 = b11 * b22 - b12 * b21, b31 = b12 * b20 - b10 * b22, b32 = b10 * b21 - b11 * b20;
  float *R = rot + 9 * (size_t)i;  // columns b1 b2 b3
  R[0] = b10; R[1] = b20; R[2] = b30;
  R[3] = b11; R[4] = b21; R[5] = b31;
  R[6] = b12; R[7] = b22; R[8] = b32;
}

// ----------------------------------------------------------------------------------------------
// Workspace layout (floats): A [B][J][12] | pfT [NC + Kp][Bpad] (blend coefficients, transposed) | lut [B] (int)
struct PoseArgs {
  SmplxDev m;
  const float *betas, *expr, *rot;
  int n_rot, B, Bpad, Kp;
  float *A, *pfT, *joints;  // joints may be null
  int *lut;
};

__global__ void __launch_bounds__(128) smplx_pose_kernel(PoseArgs a) {
  const SmplxDev &m = a.m;
  const int b = blockIdx.x, t = threadIdx.x;
  __shared__ float R[kMaxJoints][9];
  __shared__ float Jr[kMaxJoints][3];
  __shared__ float G[kMaxJoints][12];
  __shared__ float coef[kMaxCoef];
  const int J = m.J;
  if (t < m.NC) coef[t] = t < m.NB ? a.betas[(size_t)b * m.NB + t] : (a.expr ? a.expr[(size_t)b * m.NE + (t - m.NB)] : 0.f);
  for (int i = t; i < J * 9; i += blockDim.x) {
    int j = i / 9, e = i % 9;
    R[j][e] = j < a.n_rot ? a.rot[((size_t)b * a.n_rot + j) * 9 + e] : ((e == 0 || e == 4 || e == 8) ? 1.f : 0.f);
  }
  __syncthreads();
  for (int i = t; i < J * 3; i += blockDim.x) {
    float s = m.J_template[i];
    const float *jd = m.J_dirs + (size_t)i * m.NC;
    for (int l = 0; l < m.NC; ++l) s += jd[l] * coef[l];
    Jr[i / 3][i % 3] = s;
  }
  __syncthreads();
  if (t < 12) {
    int r = t / 4, c = t % 4;
    G[0][t] = c < 3 ? R[0][r * 3 + c] : Jr[0][r];
  }
  __syncthreads();
  for (int lv = 1; lv < m.n_levels; ++lv) {
    int off = m.level_off[lv], cnt = m.level_off[lv + 1] - off;
    for (int i = t; i < cnt * 12; i += blockDim.x) {
      int j = m.level_joints[off + i / 12], e = i % 12, r = e / 4, c = e % 4;
      int p = m.parents[j];
      float g0 = G[p][r * 4 + 0], g1 = G[p][r * 4 + 1], g2 = G[p][r * 4 + 2];
      float v;
      if (c < 3) {
        v = g0 * R[j][c] + g1 * R[j][3 + c] + g2 * R[j][6 + c];
      } else {
        float r0 = Jr[j][0] - Jr[p][0], r1 = Jr[j][1] - Jr[p][1], r2 = Jr[j][2] - Jr[p][2];
        v = g0 * r0 + g1 * r1 + g2 * r2 + G[p][r * 4 + 3];
      }
      G[j][e] = v;
    }
    __syncthreads();
  }
  // relative transforms A = G - [0 | G.R . J_rest]   (lbs.py:289-293)
  for (int i = t; i < J * 12; i += blockDim.x) {
    int j = i / 12, e = i % 12, r = e / 4, c = e % 4;
    float v = G[j][e];
    if (c == 3) v -= G[j][r * 4 + 0] * Jr[j][0] + G[j][r * 4 + 1] * Jr[j][1] + G[j][r * 4 + 2] * Jr[j][2];
    a.A[((size_t)b * J + j) * 12 + e] = v;
  }
  if (a.joints) {
    for (int i = t; i < J * 3; i += blockDim.x) a.joints[((size_t)b * m.K) * 3 + i] = G[i / 3][(i % 3) * 4 + 3];
  }
  // pose feature (R[1:] - I), transposed so that a body tile is contiguous
  // blend coefficients of this body, one row per basis row: [betas | expression | pose feature]
  if (t < m.NC) a.pfT[(size_t)t * a.Bpad + b] = coef[t];
  for (int k = t; k < a.Kp; k += blockDim.x) {
    int j = 1 + k / 9, e = k % 9;
    a.pfT[(size_t)(m.NC + k) * a.Bpad + b] = R[j][e] - ((e == 0 || e == 4 || e == 8) ? 1.f : 0.f);
  }
  // dynamic-contour LUT row (lbs.py:30-41, rotation_utils.py:86-92)
  if (t == 0 && m.D > 0) {
    float rel[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    for (int q = 0; q < m.n_chain; ++q) {
      const float *Rq = R[m.neck[q]];
      float o[9];
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) o[r * 3 + c] = Rq[r * 3] * rel[c] + Rq[r * 3 + 1] * rel[3 + c] + Rq[r * 3 + 2] * rel[6 + c];
      for (int e = 0; e < 9; ++e) rel[e] = o[e];
    }
    float sy = sqrtf(rel[0] * rel[0] + rel[3] * rel[3]);
    float ang = atan2f(-rel[6], sy);
    float deg = fminf(-ang * 180.0f / 3.14159265358979323846f, 39.0f);
    int y = (int)rintf(deg);  // torch.round == round-half-even
    int row = y < 0 ? (y < -39 ? 78 : 39 - y) : y;
    a.lut[b] = min(max(row, 0), m.rows - 1);
  }
}

// ----------------------------------------------------------------------------------------------
struct VertexArgs {
  SmplxDev m;
  const float *betas, *expr;
  const float *A, *pfT;
  int B, Bpad, Kp;
  float *vertices, *v_shaped;  // either may be null
};

__device__ __forceinline__ void cp_async16_zfill(void *smem_dst, const void *src, int src_bytes) {
  unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(src_bytes) : "memory");
}

// One tile = 32 vertices (one per lane) x 32 bodies (8 per warp).  All blend-shape rows (shape, expression, pose)
// are one [rows][V3p] basis; a chunk of 32 rows (96 floats each) and the matching [rows][32 bodies] coefficient
// block are staged in shared memory with 16-byte cp.async, double buffered, so every constant crosses L2 once
// per tile and the loads of chunk i+1 overlap the FMAs of chunk i.
__global__ void __launch_bounds__(128) smplx_vertex_kernel(VertexArgs a) {
  const SmplxDev &m = a.m;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, t = threadIdx.x;
  const int v0 = blockIdx.x * TV, b0 = blockIdx.y * TB;
  const int c0 = v0 * 3;
  __shared__ __align__(16) float Ps[2][KC][TV * 3];
  __shared__ __align__(16) float pfs[2][KC][TB];
  const int v = v0 + lane;
  const bool vok = v < m.V;
  float acc[8][3];
  {
    float tx = 0.f, ty = 0.f, tz = 0.f;
    if (vok) { tx = m.v_template[3 * v]; ty = m.v_template[3 * v + 1]; tz = m.v_template[3 * v + 2]; }
#pragma unroll
    for (int i = 0; i < 8; ++i) { acc[i][0] = tx; acc[i][1] = ty; acc[i][2] = tz; }
  }
  // row schedule: [0, NB) shape | [NB, NC) expression (only when given) | [NC, NC + Kp) pose (only for vertices)
  const bool posed = a.vertices != nullptr;
  const int n_expr = (a.expr && posed) ? m.NC - m.NB : 0;
  const int n_rows = m.NB + n_expr + (posed ? a.Kp : 0);
  auto row_of = [&](int i) { return i < m.NB + n_expr ? i : m.NC + (i - m.NB - n_expr); };
  // chunk boundaries: the first chunk ends exactly after the NB shape rows (v_shaped snapshot)
  auto chunk_begin = [&](int ch) { return ch == 0 ? 0 : m.NB + (ch - 1) * KC; };
  const int n_chunks = 1 + (n_rows > m.NB ? (n_rows - m.NB + KC - 1) / KC : 0);
  auto load_chunk = [&](int ch, int buf) {
    const int r0 = chunk_begin(ch), r1 = min(n_rows, ch == 0 ? m.NB : r0 + KC);
    const int nr = r1 - r0;
    for (int i = t; i < nr * 24; i += 128) {            // 96 floats = 24 x 16 bytes per row
      const int k = i / 24, q = i % 24;
      const int col = c0 + q * 4;
      const int nb = max(0, min(16, (m.V3p - col) * 4));
      const float *src = m.basis + (size_t)row_of(r0 + k) * m.V3p + (nb ? col : 0);
      cp_async16_zfill(&Ps[buf][k][q * 4], src, nb);
    }
    for (int i = t; i < nr * 8; i += 128) {             // 32 bodies = 8 x 16 bytes per row
      const int k = i / 8, q = i % 8;
      cp_async16_zfill(&pfs[buf][k][q * 4], a.pfT + (size_t)row_of(r0 + k) * a.Bpad + b0 + q * 4, 16);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  load_chunk(0, 0);
  for (int ch = 0; ch < n_chunks; ++ch) {
    const int buf = ch & 1;
    if (ch + 1 < n_chunks) {
      load_chunk(ch + 1, buf ^ 1);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    const int r0 = chunk_begin(ch), nr = min(n_rows, ch == 0 ? m.NB : r0 + KC) - r0;
#pragma unroll 4
    for (int k = 0; k < nr; ++k) {
      const float px = Ps[buf][k][3 * lane], py = Ps[buf][k][3 * lane + 1], pz = Ps[buf][k][3 * lane + 2];
      const float4 f0 = *reinterpret_cast<const float4 *>(&pfs[buf][k][warp * 8]);
      const float4 f1 = *reinterpret_cast<const float4 *>(&pfs[buf][k][warp * 8 + 4]);
      const float f[8] = {f0.x, f0.y, f0.z, f0.w, f1.x, f1.y, f1.z, f1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        acc[i][0] += f[i] * px; acc[i][1] += f[i] * py; acc[i][2] += f[i] * pz;
      }
    }
    if (ch == 0 && a.v_shaped && vok) {
      // v_shaped = v_template + shapedirs[:, :, :NB] . betas  (body_models.py:763-765)
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int b = b0 + warp * 8 + i;
        if (b < a.B) {
          float *o = a.v_shaped + ((size_t)b * m.V + v) * 3;
          o[0] = acc[i][0]; o[1] = acc[i][1]; o[2] = acc[i][2];
        }
      }
    }
    __syncthreads();
  }
  if (!posed || !vok) return;
  // ---- sparse linear blend skinning: out = sum_j w_vj (A_j . [v_posed; 1])
  float out[8][3];
#pragma unroll
  for (int i = 0; i < 8; ++i) out[i][0] = out[i][1] = out[i][2] = 0.f;
  for (int s = 0; s < m.ell_w_n; ++s) {
    float w = m.ell_w[(size_t)s * m.V + v];
    if (w == 0.f) continue;
    int j = m.ell_idx[(size_t)s * m.V + v];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int b = b0 + warp * 8 + i;
      if (b >= a.B) break;
      const float4 *Ab = reinterpret_cast<const float4 *>(a.A + ((size_t)b * m.J + j) * 12);
      float4 r0 = __ldg(Ab), r1 = __ldg(Ab + 1), r2 = __ldg(Ab + 2);
      float x = acc[i][0], y = acc[i][1], z = acc[i][2];
      out[i][0] += w * (r0.x * x + r0.y * y + r0.z * z + r0.w);
      out[i][1] += w * (r1.x * x + r1.y * y + r1.z * z + r1.w);
      out[i][2] += w * (r2.x * x + r2.y * y + r2.z * z + r2.w);
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    int b = b0 + warp * 8 + i;
    if (b < a.B) {
      float *o = a.vertices + ((size_t)b * m.V + v) * 3;
      o[0] = out[i][0]; o[1] = out[i][1]; o[2] = out[i][2];
    }
  }
}

// ----------------------------------------------------------------------------------------------
struct JointsArgs {
  SmplxDev m;
  const float *vertices, *camera;
  const int *lut;
  int B;
  float *joints, *proj;
};

__global__ void __launch_bounds__(512) smplx_joints_kernel(JointsArgs a) {
  // launched as a programmatic dependent of the kernel that writes the vertices: its launch latency overlaps that
  // kernel's tail; everything below reads the predecessor's output, so wait for its completion first
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const SmplxDev &m = a.m;
  const int b = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  extern __shared__ float sm[];
  float *jt = sm;               // [K][3]
  float *reg = sm + m.K * 3;    // [n_extra][3]
  const float *vb = a.vertices + (size_t)b * m.V * 3;
  float *jout = a.joints + (size_t)b * m.K * 3;
  for (int i = t; i < m.J * 3; i += blockDim.x) jt[i] = jout[i];  // posed joints from the pose kernel
  for (int i = t; i < m.L + m.D; i += blockDim.x) {
    const int *vi;
    const float *bc;
    if (i < m.L) { vi = m.lmk_vidx + 3 * i; bc = m.lmk_bc + 3 * i; }
    else {
      size_t o = ((size_t)a.lut[b] * m.D + (i - m.L)) * 3;
      vi = m.dyn_vidx + o; bc = m.dyn_bc + o;
    }
    for (int c = 0; c < 3; ++c)
      jt[(m.J + i) * 3 + c] = vb[3 * vi[0] + c] * bc[0] + vb[3 * vi[1] + c] * bc[1] + vb[3 * vi[2] + c] * bc[2];
  }
  for (int r = warp; r < m.n_extra; r += blockDim.x / 32) {
    float sx = 0.f, sy = 0.f, sz = 0.f;
    for (int e = m.ex_ptr[r] + lane; e < m.ex_ptr[r + 1]; e += 32) {
      int c = m.ex_col[e];
      float w = m.ex_val[e];
      sx += w * vb[3 * c]; sy += w * vb[3 * c + 1]; sz += w * vb[3 * c + 2];
    }
    for (int o = 16; o; o >>= 1) {
      sx += __shfl_xor_sync(0xffffffffu, sx, o);
      sy += __shfl_xor_sync(0xffffffffu, sy, o);
      sz += __shfl_xor_sync(0xffffffffu, sz, o);
    }
    if (lane == 0) { reg[3 * r] = sx; reg[3 * r + 1] = sy; reg[3 * r + 2] = sz; }
  }
  __syncthreads();
  for (int i = t; i < m.n_over * 3; i += blockDim.x) {
    int q = i / 3, c = i % 3;
    jt[m.over_src[q] * 3 + c] = reg[m.over_tgt[q] * 3 + c];
  }
  __syncthreads();
  for (int i = t; i < m.K * 3; i += blockDim.x) jout[i] = jt[i];
  if (a.proj && a.camera) {
    float c0 = a.camera[3 * b];
    float s = c0 > 20.f ? c0 : log1pf(expf(c0));  // F.softplus (beta=1, threshold=20)
    float tx = a.camera[3 * b + 1], ty = a.camera[3 * b + 2];
    for (int i = t; i < m.K; i += blockDim.x) {
      a.proj[((size_t)b * m.K + i) * 2 + 0] = s * (jt[3 * i] + tx);
      a.proj[((size_t)b * m.K + i) * 2 + 1] = s * (jt[3 * i + 1] + ty);
    }
  }
}

// ----------------------------------------------------------------------------------------------
// T-pose path: v_shaped[b][c] = T[c] + sum_l beta[b][l] S[l][c].  One thread per coordinate, the NB
// shape coefficients of that coordinate live in registers and are reused for SB bodies, so the only
// HBM traffic is the (B, 3V) output stream (S and T are 1.4 MB and stay in L2).
constexpr int SB = 64;
constexpr int SBP = 12;   // padded beta row (float4 x 3) so a body's coefficients are 3 broadcast LDS.128
template <int NB>
__global__ void __launch_bounds__(256) smplx_shape_kernel(const float *__restrict__ T, const float *__restrict__ S,
                                                          const float *__restrict__ betas, int V3, int B,
                                                          float *__restrict__ out) {
  static_assert(NB <= SBP, "beta row padding");
  __shared__ __align__(16) float bs[SB][SBP];
  // two coordinates per thread (c and c + 256): the same 3 LDS.128 of betas feed 20 FMAs
  const int c0 = blockIdx.x * 512 + threadIdx.x, c1 = c0 + 256;
  const int b0 = blockIdx.y * SB;
  for (int i = threadIdx.x; i < SB * SBP; i += blockDim.x) {
    int b = b0 + i / SBP, l = i % SBP;
    bs[i / SBP][l] = (b < B && l < NB) ? betas[(size_t)b * NB + l] : 0.f;
  }
  float s0[SBP], s1[SBP], t0 = 0.f, t1 = 0.f;
#pragma unroll
  for (int l = 0; l < SBP; ++l) { s0[l] = 0.f; s1[l] = 0.f; }
  if (c0 < V3) {
    t0 = T[c0];
#pragma unroll
    for (int l = 0; l < NB; ++l) s0[l] = S[(size_t)l * V3 + c0];
  }
  if (c1 < V3) {
    t1 = T[c1];
#pragma unroll
    for (int l = 0; l < NB; ++l) s1[l] = S[(size_t)l * V3 + c1];
  }
  __syncthreads();
  const int nb = min(SB, B - b0);
  float *o = out + (size_t)b0 * V3;
#pragma unroll 2
  for (int i = 0; i < nb; ++i) {
    const float4 q0 = *reinterpret_cast<const float4 *>(&bs[i][0]);
    const float4 q1 = *reinterpret_cast<const float4 *>(&bs[i][4]);
    const float4 q2 = *reinterpret_cast<const float4 *>(&bs[i][8]);
    const float bb[SBP] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w};
    float v0 = t0, v1 = t1;
#pragma unroll
    for (int l = 0; l < NB; ++l) { v0 += bb[l] * s0[l]; v1 += bb[l] * s1[l]; }
    if (c0 < V3) __stcs(o + (size_t)i * V3 + c0, v0);
    if (c1 < V3) __stcs(o + (size_t)i * V3 + c1, v1);
  }
}

__global__ void smplx_shape_kernel_generic(const float *__restrict__ T, const float *__restrict__ S,
                                           const float *__restrict__ betas, int NB, int V3, int B,
                                           float *__restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (c >= V3) return;
  float v = T[c];
  for (int l = 0; l < NB; ++l) v += betas[(size_t)b * NB + l] * S[(size_t)l * V3 + c];
  out[(size_t)b * V3 + c] = v;
}

// Backward of the T-pose path: grad_betas[b][l] = sum_c S[l][c] grad_v[b][c] for the NB shape rows of the [NC][3V]
// basis.  A CTA takes SBW bodies x SLW betas: each thread walks the coordinates c = tid, tid + 256, ... (one read of
// each gradient row, streaming; the basis rows come from L2), then a fixed shuffle tree and a fixed sum over the
// warps.  A body's result is the same arithmetic wherever it sits in the batch.
constexpr int SBW = 8, SLW = 10;
__global__ void __launch_bounds__(256) smplx_shape_backward_kernel(const float *__restrict__ S,
                                                                   const float *__restrict__ g, int NB, int V3, int B,
                                                                   float *__restrict__ out) {
  __shared__ float red[8][SBW * SLW];
  const int b0 = blockIdx.x * SBW, l0 = blockIdx.y * SLW;
  const int nb = min(SBW, B - b0), nl = min(SLW, NB - l0);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float acc[SBW][SLW];
#pragma unroll
  for (int i = 0; i < SBW; ++i)
#pragma unroll
    for (int l = 0; l < SLW; ++l) acc[i][l] = 0.f;
  for (int c = threadIdx.x; c < V3; c += 256) {
    float s[SLW];
#pragma unroll
    for (int l = 0; l < SLW; ++l) s[l] = l < nl ? __ldg(S + (size_t)(l0 + l) * V3 + c) : 0.f;
#pragma unroll
    for (int i = 0; i < SBW; ++i) {
      if (i < nb) {
        const float gv = __ldcs(g + (size_t)(b0 + i) * V3 + c);
#pragma unroll
        for (int l = 0; l < SLW; ++l) acc[i][l] += gv * s[l];
      }
    }
  }
#pragma unroll
  for (int i = 0; i < SBW; ++i)
#pragma unroll
    for (int l = 0; l < SLW; ++l) {
      float v = acc[i][l];
      for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) red[warp][i * SLW + l] = v;
    }
  __syncthreads();
  for (int j = threadIdx.x; j < SBW * SLW; j += 256) {
    const int i = j / SLW, l = j % SLW;
    if (i >= nb || l >= nl) continue;
    float v = 0.f;
    for (int w = 0; w < 8; ++w) v += red[w][j];
    out[(size_t)(b0 + i) * NB + l0 + l] = v;
  }
}

template <typename T>
static T *upload(shapy_smplx *m, const std::vector<T> &h, cudaError_t &err) {
  T *p = nullptr;
  if (err != cudaSuccess) return nullptr;
  err = cudaMalloc((void **)&p, std::max<size_t>(h.size(), 1) * sizeof(T));
  if (err != cudaSuccess) return nullptr;
  m->allocs.push_back(p);
  if (!h.empty()) err = cudaMemcpy(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice);
  return p;
}

}  // namespace shapy

using namespace shapy;

extern "C" int shapy_smplx_create(shapy_smplx_t **out, const shapy_smplx_desc_t *d) {
  SHAPY_REQUIRE(out && d, "shapy_smplx_create: null argument");
  SHAPY_REQUIRE(d->num_joints >= 1 && d->num_joints <= kMaxJoints, "num_joints %d unsupported", d->num_joints);
  SHAPY_REQUIRE(d->num_betas >= 1 && d->num_betas + d->num_expr <= kMaxCoef, "too many shape coefficients");
  SHAPY_REQUIRE(d->v_template && d->shapedirs && d->posedirs && d->J_regressor && d->lbs_weights && d->parents &&
                    d->faces, "shapy_smplx_create: missing model tensor");
  const int V = d->num_verts, J = d->num_joints, NB = d->num_betas, NE = d->expr_dirs ? d->num_expr : 0;
  const int NC = NB + NE, F = d->num_faces;
  auto *m = new shapy_smplx();
  SmplxDev &s = m->d;
  memset(&s, 0, sizeof(s));
  s.V = V; s.J = J; s.NB = NB; s.NE = NE; s.NC = NC; s.F = F;
  cudaError_t err = cudaSuccess;
  s.v_template = upload(m, std::vector<float>(d->v_template, d->v_template + (size_t)V * 3), err);
  // shapedirs -> [NC][3V]
  std::vector<float> S((size_t)NC * V * 3);
  for (int c = 0; c < V * 3; ++c) {
    for (int l = 0; l < NB; ++l) S[(size_t)l * V * 3 + c] = d->shapedirs[(size_t)c * NB + l];
    for (int l = 0; l < NE; ++l) S[(size_t)(NB + l) * V * 3 + c] = d->expr_dirs[(size_t)c * NE + l];
  }
  s.shapedirs = upload(m, S, err);
  s.posedirs = upload(m, std::vector<float>(d->posedirs, d->posedirs + (size_t)(J - 1) * 9 * V * 3), err);
  {
    // unified blend-shape basis with rows padded to a multiple of 4 floats (16-byte cp.async)
    const int V3 = V * 3, V3p = (V3 + 3) / 4 * 4, KP = (J - 1) * 9;
    std::vector<float> basis((size_t)(NC + KP) * V3p, 0.f);
    for (int l = 0; l < NC; ++l) memcpy(&basis[(size_t)l * V3p], &S[(size_t)l * V3], (size_t)V3 * sizeof(float));
    for (int k = 0; k < KP; ++k) memcpy(&basis[(size_t)(NC + k) * V3p], d->posedirs + (size_t)k * V3, (size_t)V3 * sizeof(float));
    s.V3p = V3p;
    s.basis = upload(m, basis, err);
  }
  // joint regression contracted with the template and the shape basis (fp64 accumulate)
  std::vector<float> Jt((size_t)J * 3), Jd((size_t)J * 3 * NC);
  for (int j = 0; j < J; ++j) {
    std::vector<double> at(3, 0.0), ad((size_t)3 * NC, 0.0);
    for (int v = 0; v < V; ++v) {
      double w = d->J_regressor[(size_t)j * V + v];
      if (w == 0.0) continue;
      for (int c = 0; c < 3; ++c) {
        at[c] += w * d->v_template[(size_t)v * 3 + c];
        for (int l = 0; l < NC; ++l) ad[(size_t)c * NC + l] += w * S[(size_t)l * V * 3 + v * 3 + c];
      }
    }
    for (int c = 0; c < 3; ++c) {
      Jt[j * 3 + c] = (float)at[c];
      for (int l = 0; l < NC; ++l) Jd[((size_t)j * 3 + c) * NC + l] = (float)ad[(size_t)c * NC + l];
    }
  }
  s.J_template = upload(m, Jt, err);
  s.J_dirs = upload(m, Jd, err);
  // ELL skinning weights
  int W = 1;
  for (int v = 0; v < V; ++v) {
    int n = 0;
    for (int j = 0; j < J; ++j) n += d->lbs_weights[(size_t)v * J + j] != 0.f;
    W = std::max(W, n);
  }
  std::vector<int> eidx((size_t)W * V, 0);
  std::vector<float> ew((size_t)W * V, 0.f);
  for (int v = 0; v < V; ++v) {
    int n = 0;
    for (int j = 0; j < J; ++j) {
      float w = d->lbs_weights[(size_t)v * J + j];
      if (w != 0.f) { eidx[(size_t)n * V + v] = j; ew[(size_t)n * V + v] = w; ++n; }
    }
  }
  s.ell_w_n = W;
  s.ell_idx = upload(m, eidx, err);
  s.ell_w = upload(m, ew, err);
  // kinematic levels
  std::vector<int> par(J), depth(J, 0);
  for (int j = 0; j < J; ++j) par[j] = j == 0 ? -1 : (int)d->parents[j];
  int maxd = 0;
  for (int j = 1; j < J; ++j) {
    if (par[j] < 0 || par[j] >= j) { delete m; set_error("parents[%d] = %d is not a topologically ordered tree", j, par[j]); return SHAPY_ERR_ARG; }
    depth[j] = depth[par[j]] + 1;
    maxd = std::max(maxd, depth[j]);
  }
  std::vector<int> lj, lo;
  for (int lv = 0; lv <= maxd; ++lv) {
    lo.push_back((int)lj.size());
    for (int j = 0; j < J; ++j) if (depth[j] == lv) lj.push_back(j);
  }
  lo.push_back((int)lj.size());
  s.n_levels = maxd + 1;
  s.parents = upload(m, par, err);
  s.level_joints = upload(m, lj, err);
  s.level_off = upload(m, lo, err);
  std::vector<int> faces((size_t)F * 3);
  for (size_t i = 0; i < faces.size(); ++i) faces[i] = (int)d->faces[i];
  s.faces = upload(m, faces, err);
  // landmarks resolved to vertex triples
  s.L = d->lmk_faces_idx ? d->num_static_lmk : 0;
  std::vector<int> lv((size_t)s.L * 3);
  for (int i = 0; i < s.L; ++i)
    for (int c = 0; c < 3; ++c) lv[i * 3 + c] = faces[(size_t)d->lmk_faces_idx[i] * 3 + c];
  s.lmk_vidx = upload(m, lv, err);
  s.lmk_bc = upload(m, std::vector<float>(d->lmk_bary_coords, d->lmk_bary_coords + (size_t)s.L * 3), err);
  s.D = d->dynamic_lmk_faces_idx ? d->num_dyn_lmk : 0;
  s.rows = s.D ? d->num_dyn_rows : 0;
  std::vector<int> dv((size_t)s.rows * s.D * 3);
  for (size_t i = 0; i < (size_t)s.rows * s.D; ++i)
    for (int c = 0; c < 3; ++c) dv[i * 3 + c] = faces[(size_t)d->dynamic_lmk_faces_idx[i] * 3 + c];
  s.dyn_vidx = upload(m, dv, err);
  s.dyn_bc = upload(m, std::vector<float>(d->dynamic_lmk_bary_coords,
                                          d->dynamic_lmk_bary_coords + (s.D ? (size_t)s.rows * s.D * 3 : 0)), err);
  s.n_chain = s.D ? d->neck_chain_len : 0;
  std::vector<int> neck(s.n_chain);
  for (int i = 0; i < s.n_chain; ++i) neck[i] = (int)d->neck_kin_chain[i];
  s.neck = upload(m, neck, err);
  s.K = J + s.L + s.D;
  // J14 regressor -> CSR
  s.n_extra = d->extra_joint_regressor ? d->num_extra : 0;
  std::vector<int> ep(1, 0), ec;
  std::vector<float> ev;
  for (int r = 0; r < s.n_extra; ++r) {
    for (int v = 0; v < V; ++v) {
      float w = d->extra_joint_regressor[(size_t)r * V + v];
      if (w != 0.f) { ec.push_back(v); ev.push_back(w); }
    }
    ep.push_back((int)ec.size());
  }
  s.ex_ptr = upload(m, ep, err);
  s.ex_col = upload(m, ec, err);
  s.ex_val = upload(m, ev, err);
  s.n_over = s.n_extra ? d->num_overwrite : 0;
  std::vector<int> os(s.n_over), ot(s.n_over);
  for (int i = 0; i < s.n_over; ++i) { os[i] = (int)d->source_idxs[i]; ot[i] = (int)d->target_idxs[i]; }
  s.over_src = upload(m, os, err);
  s.over_tgt = upload(m, ot, err);
  {
    // ---- operands of the fused tcgen05 LBS kernel (smplx_lbs.cu)
    const int Vpad = (V + 127) / 128 * 128, KP = (J - 1) * 9, KPpad = (KP + 63) / 64 * 64;
    s.Vpad = Vpad; s.KPpad = KPpad;
    const int nKB = KPpad / 32;
    std::vector<__half> pb((size_t)nKB * 3 * Vpad * 64, __float2half_rn(0.f));
    for (int k = 0; k < KP; ++k) {
      const float *row = d->posedirs + (size_t)k * V * 3;
      const int kb = k / 32, kk = k % 32;
      for (int v = 0; v < V; ++v)
        for (int c = 0; c < 3; ++c) {
          const float x = row[(size_t)v * 3 + c] * kPoseScale;
          const __half h = __float2half_rn(x);
          const size_t o = (((size_t)kb * 3 + c) * Vpad + v) * 64 + kk;
          pb[o] = h;
          pb[o + 32] = __float2half_rn((x - __half2float(h)) * 2048.0f);
        }
    }
    s.pbasis = upload(m, pb, err);
    std::vector<float> sp((size_t)(NB + 1) * 3 * Vpad, 0.f);
    for (int v = 0; v < V; ++v)
      for (int c = 0; c < 3; ++c) {
        for (int l = 0; l < NB; ++l) sp[(size_t)(l * 3 + c) * Vpad + v] = d->shapedirs[((size_t)v * 3 + c) * NB + l];
        sp[(size_t)(NB * 3 + c) * Vpad + v] = d->v_template[(size_t)v * 3 + c];
      }
    s.shape_planes = upload(m, sp, err);
    m->h_lbs_weights.assign(d->lbs_weights, d->lbs_weights + (size_t)V * J);
    m->h_parents = par;
    m->fused_ok = false;
    if (err == cudaSuccess && get_encode()) {
      cuuint64_t dims[4] = {64, (cuuint64_t)Vpad, 3, (cuuint64_t)nKB};
      cuuint64_t strides[3] = {128, (cuuint64_t)Vpad * 128, (cuuint64_t)3 * Vpad * 128};
      cuuint32_t box[4] = {64, 128, 3, 1};
      m->fused_ok = encode(&m->basis_map, s.pbasis, 4, dims, strides, box, 64);
    }
  }
  if (err != cudaSuccess) {
    set_error("shapy_smplx_create: %s", cudaGetErrorString(err));
    shapy_smplx_destroy(m);
    return (int)err;
  }
  *out = m;
  return SHAPY_OK;
}

extern "C" void shapy_smplx_destroy(shapy_smplx_t *m) {
  if (!m) return;
  for (void *p : m->allocs) cudaFree(p);
  for (auto &kv : m->wtiles) if (kv.second.dev) cudaFree(kv.second.dev);
  delete m;
}

extern "C" int shapy_smplx_num_keypoints(const shapy_smplx_t *m) { return m ? m->d.K : 0; }
extern "C" const int32_t *shapy_smplx_faces_i32(const shapy_smplx_t *m) { return m ? m->d.faces : nullptr; }

static inline int bpad(int B) { return (B + 31) / 32 * 32; }

extern "C" size_t shapy_smplx_workspace_bytes(const shapy_smplx_t *m, int B) {
  if (!m || B <= 0) return 0;
  size_t a = align_up((size_t)B * m->d.J * 12 * sizeof(float), 256);
  size_t p = align_up((size_t)((m->d.J - 1) * 9 + m->d.NC) * bpad(B) * sizeof(float), 256);
  size_t l = align_up((size_t)B * sizeof(int), 256);
  size_t j = align_up((size_t)B * m->d.K * 3 * sizeof(float), 256);
  return a + p + l + j;
}

extern "C" int shapy_decode_rot6d(const float *raw, int n, float *rot, void *stream) {
  SHAPY_REQUIRE(raw && rot && n >= 0, "shapy_decode_rot6d: bad argument");
  if (n == 0) return SHAPY_OK;
  decode_rot6d_kernel<<<ceil_div(n, 128), 128, 0, (cudaStream_t)stream>>>(raw, n, rot);
  SHAPY_LAUNCH_CHECK();
  return SHAPY_OK;
}

extern "C" int shapy_smplx_forward(const shapy_smplx_t *m, const float *betas, const float *rot, int n_rot,
                                   const float *expr, const float *camera, int B, float *vertices, float *v_shaped,
                                   float *joints, float *proj_joints, void *workspace, size_t workspace_bytes,
                                   void *stream) {
  SHAPY_REQUIRE(m && betas && rot, "shapy_smplx_forward: null argument");
  SHAPY_REQUIRE(B > 0, "shapy_smplx_forward: batch %d", B);
  SHAPY_REQUIRE(n_rot >= 1 && n_rot <= m->d.J, "shapy_smplx_forward: n_rot %d out of range", n_rot);
  SHAPY_REQUIRE(workspace && workspace_bytes >= shapy_smplx_workspace_bytes(m, B), "shapy_smplx_forward: workspace too small");
  SHAPY_REQUIRE(!(proj_joints && !joints) , "proj_joints requires joints");
  SHAPY_REQUIRE(!(joints && !vertices && (m->d.L + m->d.D + m->d.n_extra) > 0), "joints require vertices");
  cudaStream_t st = (cudaStream_t)stream;
  const SmplxDev &d = m->d;
  char *w = (char *)workspace;
  float *A = (float *)w; w += align_up((size_t)B * d.J * 12 * sizeof(float), 256);
  float *pfT = (float *)w; w += align_up((size_t)((d.J - 1) * 9 + d.NC) * bpad(B) * sizeof(float), 256);
  int *lut = (int *)w; w += align_up((size_t)B * sizeof(int), 256);
  float *jscratch = (float *)w;
  const int Kp = (n_rot - 1) * 9;
  // fused tcgen05 kernel (pose chain + shape + pose blend + skinning in one launch) when the configuration allows:
  // no expression coefficients, posed vertices requested, 10 betas, n_rot <= 29
  bool fused = false;
  if (vertices && !(d.NE && expr)) {
    const int rc = launch_lbs_fused(m, betas, rot, n_rot, B, vertices, v_shaped, joints ? joints : jscratch, lut, st);
    if (rc == SHAPY_OK) fused = true;
    else if (rc != SHAPY_ERR_UNSUPPORTED) return rc;
  }
  if (!fused) {
    PoseArgs pa{d, betas, d.NE ? expr : nullptr, rot, n_rot, B, bpad(B), Kp, A, pfT, joints ? joints : jscratch, lut};
    smplx_pose_kernel<<<B, 128, 0, st>>>(pa);
    SHAPY_LAUNCH_CHECK();
    if (vertices || v_shaped) {
      VertexArgs va{d, betas, d.NE ? expr : nullptr, A, pfT, B, bpad(B), Kp, vertices, v_shaped};
      dim3 grid(ceil_div(d.V, TV), ceil_div(B, TB));
      smplx_vertex_kernel<<<grid, 128, 0, st>>>(va);
      SHAPY_LAUNCH_CHECK();
    }
  }
  if (joints && (d.L + d.D + d.n_extra > 0 || proj_joints)) {
    JointsArgs ja{d, vertices, camera, lut, B, joints, proj_joints};
    size_t smem = ((size_t)d.K * 3 + (size_t)std::max(d.n_extra, 1) * 3) * sizeof(float);
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(B);
    cfg.blockDim = dim3(512);     // 16 warps: the 14 sparse J14 rows and the 68 landmarks are each one pass of dependent loads
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    SHAPY_CUDA_TRY(cudaLaunchKernelEx(&cfg, smplx_joints_kernel, ja));
    count_launch();
  }
  return SHAPY_OK;
}

extern "C" int shapy_smplx_forward_shape(const shapy_smplx_t *m, const float *betas, int B, float *v_shaped,
                                         void *stream) {
  SHAPY_REQUIRE(m && betas && v_shaped && B > 0, "shapy_smplx_forward_shape: bad argument");
  const SmplxDev &d = m->d;
  cudaStream_t st = (cudaStream_t)stream;
  const int V3 = d.V * 3;
  if (d.NB == 10) {
    dim3 grid(ceil_div(V3, 512), ceil_div(B, SB));
    smplx_shape_kernel<10><<<grid, 256, 0, st>>>(d.v_template, d.shapedirs, betas, V3, B, v_shaped);
  } else {
    dim3 grid(ceil_div(V3, 256), B);
    smplx_shape_kernel_generic<<<grid, 256, 0, st>>>(d.v_template, d.shapedirs, betas, d.NB, V3, B, v_shaped);
  }
  SHAPY_LAUNCH_CHECK();
  return SHAPY_OK;
}

extern "C" int shapy_smplx_shape_backward(const shapy_smplx_t *m, const float *grad_v_shaped, int B,
                                          float *grad_betas, void *stream) {
  SHAPY_REQUIRE(m && grad_v_shaped && grad_betas && B > 0, "shapy_smplx_shape_backward: bad argument");
  const SmplxDev &d = m->d;
  dim3 grid(ceil_div(B, SBW), ceil_div(d.NB, SLW));
  smplx_shape_backward_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d.shapedirs, grad_v_shaped, d.NB, d.V * 3, B,
                                                                      grad_betas);
  SHAPY_LAUNCH_CHECK();
  return SHAPY_OK;
}
