// flame.cu -- FLAME blendshapes + linear blend skinning, forward (2 launches) and backward (2 launches).
// Replaces FlameHead.forward(..., zero_centered_at_root_node=False, return_landmarks=False, return_verts_cano=True)
// and its autograd (flame_model/flame.py:485-558, flame_model/lbs.py:25-57,101-304) for one mesh per call:
//   betas    = [shape | expr]
//   v_shaped = v_template + shapedirs . betas + static_offset            (the offset moves the joints)
//   J        = J_template + J_shapedirs . betas + J_regressor . static_offset
//   R_j      = I + sin(a) K + (1 - cos(a)) K^2,  a = |r_j + 1e-8| (1e-8 added per component), K = skew(r_j / a)
//   v_posed  = v_shaped + posedirs^T . pose_feature,  pose_feature = (R_j - I), j = 1..4, row-major
//   G_0 = [R_0 | J_0], G_j = G_parent(j) [R_j | J_j - J_parent(j)],  A_j = G_j - [0 | G_j J_j]
//   verts    = (sum_j W_vj A_j) [v_posed; 1] + translation
// Per-timestep parameters arrive as (T, k) tables plus a device row index, so a CUDA graph replays any timestep, and
// the backward ADDS into row `row` of the (T, k) gradient tables.
//
// Launches: forward = joints (1 CTA: betas gather, joint regression, Rodrigues + chain in double) -> skin (a warp per
// vertex: the 3 rows of the shapedirs GEMV with lanes over the betas, pose blendshapes, skinning).  Backward = per
// chunk of vertices partial sums of dL/dA, dL/dtranslation, dL/dpose_feature and dL/dbetas -> chain (1 CTA: reduces
// the partials in a fixed order, then the chain and Rodrigues backward and J_shapedirs^T dL/dJ).  No atomics, no host
// synchronisation: capturable and deterministic.
#include "common.cuh"
#include "kernels.cuh"

namespace gab {

namespace {

constexpr int FL_J = 5;
constexpr int FL_STATE_A = 0;        // [5][3][4]
constexpr int FL_STATE_PF = 60;      // [36]
constexpr int FL_STATE_TRANS = 96;   // [3]
constexpr int FL_STATE_VALID = 99;   // 1: row index in range and parents well formed
constexpr int FL_STATE_J = 100;      // [5][3]
constexpr int FL_STATE_BETAS = 128;  // [NB]
constexpr int FL_CHUNK = 64;         // vertices per CTA of the backward partial sums
constexpr int FL_PART_HEAD = 100;    // per-CTA partial: gA (60) | gtrans (3) | pad | gpf (36) at 64 | gbetas (NB) at 100

struct FlameLayout {
  float* state;
  float* v_posed;
  float* partials;
  int n_chunks;
  size_t bytes;
};

__host__ __device__ inline FlameLayout flame_layout(void* ws, int V, int NB) {
  Carver c(ws);
  FlameLayout L;
  L.state = c.take<float>(FL_STATE_BETAS + NB);
  L.v_posed = c.take<float>(3 * (size_t)V);
  L.n_chunks = (V + FL_CHUNK - 1) / FL_CHUNK;
  L.partials = c.take<float>((size_t)L.n_chunks * (FL_PART_HEAD + NB));
  L.bytes = c.bytes();
  return L;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ int flame_row(const gab200_flame_args& a) { return a.row ? *a.row : 0; }

__device__ __forceinline__ const float* joint_pose(const gab200_flame_args& a, int t, int j) {
  switch (j) {
    case 0: return a.rotation + 3 * (size_t)t;
    case 1: return a.neck + 3 * (size_t)t;
    case 2: return a.jaw + 3 * (size_t)t;
    case 3: return a.eyes + 6 * (size_t)t;
    default: return a.eyes + 6 * (size_t)t + 3;
  }
}

// R = I + s K + (1 - c) K^2 with the reference's epsilon placement; keeps what the backward needs
struct Rodrigues {
  double r[3], a, d[3], s, c, K[9], K2[9], R[9];
};

__device__ void rodrigues(const float* rf, Rodrigues& o) {
  for (int i = 0; i < 3; ++i) o.r[i] = rf[i];
  const double e0 = o.r[0] + 1e-8, e1 = o.r[1] + 1e-8, e2 = o.r[2] + 1e-8;
  o.a = sqrt(e0 * e0 + e1 * e1 + e2 * e2);
  for (int i = 0; i < 3; ++i) o.d[i] = o.r[i] / o.a;
  o.s = sin(o.a);
  o.c = cos(o.a);
  const double x = o.d[0], y = o.d[1], z = o.d[2];
  const double K[9] = {0, -z, y, z, 0, -x, -y, x, 0};
  for (int i = 0; i < 9; ++i) o.K[i] = K[i];
  for (int i = 0; i < 3; ++i)
    for (int k = 0; k < 3; ++k) {
      double acc = 0;
      for (int m = 0; m < 3; ++m) acc += K[3 * i + m] * K[3 * m + k];
      o.K2[3 * i + k] = acc;
    }
  for (int i = 0; i < 9; ++i) o.R[i] = (i % 4 == 0 ? 1.0 : 0.0) + o.s * o.K[i] + (1.0 - o.c) * o.K2[i];
}

// gR (3x3) -> gr (3)
__device__ void rodrigues_bwd(const Rodrigues& o, const double* gR, double* gr) {
  // R = I + s K + (1-c) K^2
  double gs = 0, gomc = 0, gK[9];
  for (int i = 0; i < 9; ++i) {
    gs += gR[i] * o.K[i];
    gomc += gR[i] * o.K2[i];
  }
  const double w = 1.0 - o.c;
  for (int i = 0; i < 3; ++i)
    for (int k = 0; k < 3; ++k) {
      // d(K K)/dK: gK += w (gR K^T + K^T gR)
      double acc = 0;
      for (int m = 0; m < 3; ++m) acc += gR[3 * i + m] * o.K[3 * k + m] + o.K[3 * m + i] * gR[3 * m + k];
      gK[3 * i + k] = o.s * gR[3 * i + k] + w * acc;
    }
  double ga = o.c * gs + o.s * gomc;
  const double gd[3] = {gK[7] - gK[5], gK[2] - gK[6], gK[3] - gK[1]};
  // d = r / a
  double gd_r = 0;
  for (int i = 0; i < 3; ++i) gd_r += gd[i] * o.r[i];
  ga -= gd_r / (o.a * o.a);
  for (int i = 0; i < 3; ++i) gr[i] = gd[i] / o.a + ga * (o.r[i] + 1e-8) / o.a;
}

__device__ inline void mat3_mul(const double* A, const double* B, double* C) {
  for (int i = 0; i < 3; ++i)
    for (int k = 0; k < 3; ++k) C[3 * i + k] = A[3 * i] * B[k] + A[3 * i + 1] * B[3 + k] + A[3 * i + 2] * B[6 + k];
}
__device__ inline void mat3_vec(const double* A, const double* x, double* y) {
  for (int i = 0; i < 3; ++i) y[i] = A[3 * i] * x[0] + A[3 * i + 1] * x[1] + A[3 * i + 2] * x[2];
}
__device__ inline void mat3T_vec(const double* A, const double* x, double* y) {
  for (int i = 0; i < 3; ++i) y[i] = A[i] * x[0] + A[3 + i] * x[1] + A[6 + i] * x[2];
}

// The kinematic chain of one call (single thread, double).
struct Chain {
  Rodrigues rod[FL_J];
  double J[FL_J][3], rel[FL_J][3], Rg[FL_J][9], tg[FL_J][3];
  int parent[FL_J];
};

__device__ bool chain_forward(const gab200_flame_args& a, int t, const float* Jf, Chain& ch) {
  bool ok = true;
  for (int j = 0; j < FL_J; ++j) {
    rodrigues(joint_pose(a, t, j), ch.rod[j]);
    for (int k = 0; k < 3; ++k) ch.J[j][k] = Jf[3 * j + k];
    const int p = j == 0 ? -1 : a.parents[j];
    if (j > 0 && (p < 0 || p >= j)) ok = false;
    ch.parent[j] = (j > 0 && ok) ? p : 0;
  }
  for (int j = 0; j < FL_J; ++j) {
    if (j == 0) {
      for (int i = 0; i < 9; ++i) ch.Rg[0][i] = ch.rod[0].R[i];
      for (int k = 0; k < 3; ++k) ch.tg[0][k] = ch.rel[0][k] = ch.J[0][k];
      continue;
    }
    const int p = ch.parent[j];
    for (int k = 0; k < 3; ++k) ch.rel[j][k] = ch.J[j][k] - ch.J[p][k];
    mat3_mul(ch.Rg[p], ch.rod[j].R, ch.Rg[j]);
    double v[3];
    mat3_vec(ch.Rg[p], ch.rel[j], v);
    for (int k = 0; k < 3; ++k) ch.tg[j][k] = v[k] + ch.tg[p][k];
  }
  return ok;
}

// ---- forward ----------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) flame_joints_kernel(gab200_flame_args a, FlameLayout L) {
  const int NB = a.n_shape + a.n_expr;
  extern __shared__ float s_betas[];
  __shared__ float sJ[3 * FL_J];
  __shared__ int s_t;
  if (threadIdx.x == 0) {
    const int t = flame_row(a);
    s_t = (t >= 0 && t < a.T) ? t : -1;
  }
  __syncthreads();
  const int t = s_t;
  if (t < 0) {  // row out of range: every output of this call becomes NaN (visible, memory-safe)
    if (threadIdx.x == 0) {
      for (int i = 0; i < FL_STATE_BETAS; ++i) L.state[i] = __int_as_float(0x7fc00000);
      L.state[FL_STATE_VALID] = 0.f;
    }
    for (int l = threadIdx.x; l < NB; l += blockDim.x) L.state[FL_STATE_BETAS + l] = 0.f;
    return;
  }
  for (int l = threadIdx.x; l < NB; l += blockDim.x) {
    const float b = l < a.n_shape ? (a.shape ? a.shape[l] : 0.f) : a.expr[(size_t)t * a.n_expr + (l - a.n_shape)];
    s_betas[l] = b;
    L.state[FL_STATE_BETAS + l] = b;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  for (int jk = warp; jk < 3 * FL_J; jk += nwarps) {
    const float* row = a.J_shapedirs + (size_t)jk * NB;
    float acc = 0.f;
    for (int l = lane; l < NB; l += 32) acc = fmaf(row[l], s_betas[l], acc);
    if (a.static_offset) {
      const float* jr = a.J_regressor + (size_t)(jk / 3) * a.V;
      const int k = jk % 3;
      for (int v = lane; v < a.V; v += 32) acc = fmaf(jr[v], a.static_offset[3 * (size_t)v + k], acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) sJ[jk] = a.J_template[jk] + acc;
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  Chain ch;
  const bool ok = chain_forward(a, t, sJ, ch);
  float* S = L.state;
  for (int j = 0; j < FL_J; ++j) {
    double RJ[3];
    mat3_vec(ch.Rg[j], ch.J[j], RJ);
    for (int r = 0; r < 3; ++r) {
      for (int c = 0; c < 3; ++c) S[FL_STATE_A + 12 * j + 4 * r + c] = (float)ch.Rg[j][3 * r + c];
      S[FL_STATE_A + 12 * j + 4 * r + 3] = (float)(ch.tg[j][r] - RJ[r]);
    }
    for (int k = 0; k < 3; ++k) S[FL_STATE_J + 3 * j + k] = sJ[3 * j + k];
    if (j > 0)
      for (int i = 0; i < 9; ++i) S[FL_STATE_PF + 9 * (j - 1) + i] = (float)(ch.rod[j].R[i] - (i % 4 == 0 ? 1.0 : 0.0));
  }
  for (int k = 0; k < 3; ++k) S[FL_STATE_TRANS + k] = a.translation[3 * (size_t)t + k];
  S[FL_STATE_VALID] = ok ? 1.f : 0.f;
  if (!ok)
    for (int i = 0; i < FL_STATE_VALID; ++i) S[i] = __int_as_float(0x7fc00000);
}

// One warp per vertex.  Lanes stride over the betas of each of the vertex's three shapedirs rows (3 x NB contiguous
// floats), then over the 36 pose-feature rows of posedirs.
__global__ void __launch_bounds__(256) flame_skin_kernel(gab200_flame_args a, FlameLayout L) {
  const int NB = a.n_shape + a.n_expr;
  extern __shared__ float s_betas[];
  __shared__ float sS[FL_STATE_J];
  for (int i = threadIdx.x; i < FL_STATE_J; i += blockDim.x) sS[i] = L.state[i];
  for (int l = threadIdx.x; l < NB; l += blockDim.x) s_betas[l] = L.state[FL_STATE_BETAS + l];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int v = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (v >= a.V) return;
  float acc[3];
  const float* sd = a.shapedirs + 3 * (size_t)v * NB;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    float s = 0.f;
    for (int l = lane; l < NB; l += 32) s = fmaf(sd[(size_t)k * NB + l], s_betas[l], s);
    acc[k] = s;
  }
  float pacc[3] = {0.f, 0.f, 0.f};
  const size_t V3 = 3 * (size_t)a.V;
  for (int p = lane; p < 36; p += 32) {
    const float f = sS[FL_STATE_PF + p];
    const float* pd = a.posedirs + (size_t)p * V3 + 3 * (size_t)v;
#pragma unroll
    for (int k = 0; k < 3; ++k) pacc[k] = fmaf(f, pd[k], pacc[k]);
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    acc[k] = warp_sum(acc[k]);
    pacc[k] = warp_sum(pacc[k]);
  }
  if (lane != 0) return;
  float vs[3], vp[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    vs[k] = a.v_template[3 * (size_t)v + k] + acc[k];
    if (a.static_offset) vs[k] += a.static_offset[3 * (size_t)v + k];
    vp[k] = vs[k] + pacc[k];
  }
  float T[12];
#pragma unroll
  for (int i = 0; i < 12; ++i) T[i] = 0.f;
  for (int j = 0; j < FL_J; ++j) {
    const float w = a.lbs_weights[(size_t)v * FL_J + j];
#pragma unroll
    for (int i = 0; i < 12; ++i) T[i] = fmaf(w, sS[FL_STATE_A + 12 * j + i], T[i]);
  }
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const float o = T[4 * r] * vp[0] + T[4 * r + 1] * vp[1] + T[4 * r + 2] * vp[2] + T[4 * r + 3];
    a.verts[3 * (size_t)v + r] = o + sS[FL_STATE_TRANS + r];
    L.v_posed[3 * (size_t)v + r] = vp[r];
    if (a.verts_cano) a.verts_cano[3 * (size_t)v + r] = vs[r];
  }
}

// ---- backward -----------------------------------------------------------------------------------------------------
// CTA c covers vertices [64c, 64c + 64): writes its partial sums (no atomics) and adds dL/dv_shaped into
// grad_static_offset for its own rows.  Columns [0, n_shape) of shapedirs are read only when grad_shape is wanted.
__global__ void __launch_bounds__(256) flame_skin_bwd_kernel(gab200_flame_args a, const float* __restrict__ g_verts,
                                                             FlameLayout L) {
  const int NB = a.n_shape + a.n_expr;
  __shared__ float sA[60];
  __shared__ float s_gvs[3 * FL_CHUNK];
  __shared__ float s_contrib[FL_CHUNK][64];
  const int v0 = blockIdx.x * FL_CHUNK;
  const int nv = min(FL_CHUNK, a.V - v0);
  const bool valid = L.state[FL_STATE_VALID] != 0.f;
  float* part = L.partials + (size_t)blockIdx.x * (FL_PART_HEAD + NB);
  for (int i = threadIdx.x; i < 60; i += blockDim.x) sA[i] = L.state[FL_STATE_A + i];
  __syncthreads();
  if (threadIdx.x < FL_CHUNK) {
    const int i = threadIdx.x;
    float* cb = s_contrib[i];
    if (i < nv && valid) {
      const size_t v = v0 + i;
      float g[3], vp[4], w[FL_J], T[12];
      for (int k = 0; k < 3; ++k) {
        g[k] = g_verts[3 * v + k];
        vp[k] = L.v_posed[3 * v + k];
      }
      vp[3] = 1.f;
      for (int q = 0; q < 12; ++q) T[q] = 0.f;
      for (int j = 0; j < FL_J; ++j) {
        w[j] = a.lbs_weights[v * FL_J + j];
        for (int q = 0; q < 12; ++q) T[q] = fmaf(w[j], sA[12 * j + q], T[q]);
      }
      for (int j = 0; j < FL_J; ++j)
        for (int r = 0; r < 3; ++r)
          for (int c = 0; c < 4; ++c) cb[12 * j + 4 * r + c] = w[j] * g[r] * vp[c];
      cb[63] = 0.f;
      for (int k = 0; k < 3; ++k) {
        cb[60 + k] = g[k];
        s_gvs[3 * i + k] = T[k] * g[0] + T[4 + k] * g[1] + T[8 + k] * g[2];
      }
    } else {
      for (int q = 0; q < 64; ++q) cb[q] = 0.f;
      for (int k = 0; k < 3; ++k) s_gvs[3 * i + k] = 0.f;
    }
  }
  __syncthreads();
  // dL/dA, dL/dtranslation: fixed-order sums over the chunk
  if (threadIdx.x < 64) {
    float s = 0.f;
    for (int i = 0; i < FL_CHUNK; ++i) s += s_contrib[i][threadIdx.x];
    part[threadIdx.x] = s;
  }
  // dL/dpose_feature: row p of posedirs over the chunk's 3 * nv contiguous columns, a warp per row
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const size_t V3 = 3 * (size_t)a.V;
  for (int p = warp; p < 36; p += nwarps) {
    const float* pd = a.posedirs + (size_t)p * V3 + 3 * (size_t)v0;
    float s = 0.f;
    for (int m = lane; m < 3 * nv; m += 32) s = fmaf(pd[m], s_gvs[m], s);
    s = warp_sum(s);
    if (lane == 0) part[64 + p] = s;
  }
  // dL/dbetas: a thread per beta over the chunk's 3 * nv shapedirs rows
  const int l0 = a.grad_shape ? 0 : a.n_shape;
  const float* sd = a.shapedirs + 3 * (size_t)v0 * NB;
  for (int l = l0 + threadIdx.x; l < NB; l += blockDim.x) {
    float s = 0.f;
    for (int m = 0; m < 3 * nv; ++m) s = fmaf(sd[(size_t)m * NB + l], s_gvs[m], s);
    part[FL_PART_HEAD + l] = s;
  }
  if (a.grad_static_offset)
    for (int m = threadIdx.x; m < 3 * nv; m += blockDim.x) a.grad_static_offset[3 * (size_t)v0 + m] += s_gvs[m];
}

__global__ void __launch_bounds__(256) flame_chain_bwd_kernel(gab200_flame_args a, FlameLayout L) {
  const int NB = a.n_shape + a.n_expr;
  extern __shared__ double s_red[];  // [FL_PART_HEAD + NB]: summed partials, then dL/dbetas
  __shared__ double s_gJ[3 * FL_J];
  if (L.state[FL_STATE_VALID] == 0.f) return;
  const int t = flame_row(a);
  const int l0 = a.grad_shape ? 0 : a.n_shape;
  for (int i = threadIdx.x; i < FL_PART_HEAD + NB; i += blockDim.x) {
    double s = 0.0;
    if (i < FL_PART_HEAD || i - FL_PART_HEAD >= l0)
      for (int c = 0; c < L.n_chunks; ++c) s += L.partials[(size_t)c * (FL_PART_HEAD + NB) + i];
    s_red[i] = s;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    Chain ch;
    chain_forward(a, t, L.state + FL_STATE_J, ch);
    double gRg[FL_J][9], gtg[FL_J][3], gJ[FL_J][3], gR[FL_J][9];
    for (int j = 0; j < FL_J; ++j) {
      // A_j = [Rg_j | tg_j - Rg_j J_j]
      double gAt[3];
      for (int r = 0; r < 3; ++r) gAt[r] = s_red[12 * j + 4 * r + 3];
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) gRg[j][3 * r + c] = s_red[12 * j + 4 * r + c] - gAt[r] * ch.J[j][c];
      double RtgAt[3];
      mat3T_vec(ch.Rg[j], gAt, RtgAt);
      for (int k = 0; k < 3; ++k) {
        gtg[j][k] = gAt[k];
        gJ[j][k] = -RtgAt[k];
      }
      for (int i = 0; i < 9; ++i) gR[j][i] = j > 0 ? s_red[64 + 9 * (j - 1) + i] : 0.0;
    }
    for (int j = FL_J - 1; j >= 1; --j) {  // children before parents (parents[j] < j)
      const int p = ch.parent[j];
      // tg_j = Rg_p rel_j + tg_p
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) gRg[p][3 * r + c] += gtg[j][r] * ch.rel[j][c];
      double grel[3];
      mat3T_vec(ch.Rg[p], gtg[j], grel);
      for (int k = 0; k < 3; ++k) {
        gtg[p][k] += gtg[j][k];
        gJ[j][k] += grel[k];
        gJ[p][k] -= grel[k];
      }
      // Rg_j = Rg_p R_j
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) {
          double x = 0, y = 0;
          for (int m = 0; m < 3; ++m) {
            x += gRg[j][3 * r + m] * ch.rod[j].R[3 * c + m];  // (gRg_j R_j^T)[r][c]
            y += ch.Rg[p][3 * m + r] * gRg[j][3 * m + c];      // (Rg_p^T gRg_j)[r][c]
          }
          gRg[p][3 * r + c] += x;
          gR[j][3 * r + c] += y;
        }
    }
    for (int i = 0; i < 9; ++i) gR[0][i] += gRg[0][i];
    for (int k = 0; k < 3; ++k) gJ[0][k] += gtg[0][k];
    for (int j = 0; j < FL_J; ++j) {
      double gr[3];
      rodrigues_bwd(ch.rod[j], gR[j], gr);
      float* dst = j == 0 ? a.grad_rotation : j == 1 ? a.grad_neck : j == 2 ? a.grad_jaw : a.grad_eyes;
      if (dst) {
        const size_t base = j < 3 ? 3 * (size_t)t : 6 * (size_t)t + 3 * (j - 3);
        for (int k = 0; k < 3; ++k) dst[base + k] += (float)gr[k];
      }
      for (int k = 0; k < 3; ++k) s_gJ[3 * j + k] = gJ[j][k];
    }
    if (a.grad_translation)
      for (int k = 0; k < 3; ++k) a.grad_translation[3 * (size_t)t + k] += (float)s_red[60 + k];
  }
  __syncthreads();
  // betas: vertex part + J_shapedirs^T dL/dJ
  for (int l = l0 + threadIdx.x; l < NB; l += blockDim.x) {
    double s = s_red[FL_PART_HEAD + l];
    for (int jk = 0; jk < 3 * FL_J; ++jk) s += (double)a.J_shapedirs[(size_t)jk * NB + l] * s_gJ[jk];
    if (l < a.n_shape)
      a.grad_shape[l] += (float)s;
    else if (a.grad_expr)
      a.grad_expr[(size_t)t * a.n_expr + (l - a.n_shape)] += (float)s;
  }
  if (a.grad_static_offset)
    for (int m = threadIdx.x; m < 3 * a.V; m += blockDim.x) {
      const int v = m / 3, k = m - 3 * v;
      double s = 0.0;
      for (int j = 0; j < FL_J; ++j) s += (double)a.J_regressor[(size_t)j * a.V + v] * s_gJ[3 * j + k];
      a.grad_static_offset[m] += (float)s;
    }
}

}  // namespace

size_t flame_workspace_bytes(int V, int NB) { return flame_layout(nullptr, V, NB).bytes; }

void launch_flame_forward(const gab200_flame_args& a, cudaStream_t stream) {
  const int NB = a.n_shape + a.n_expr;
  const FlameLayout L = flame_layout(a.workspace, a.V, NB);
  flame_joints_kernel<<<1, 256, sizeof(float) * NB, stream>>>(a, L);
  count_launch();
  flame_skin_kernel<<<(a.V + 7) / 8, 256, sizeof(float) * NB, stream>>>(a, L);
  count_launch();
}

void launch_flame_backward(const gab200_flame_args& a, const float* g_verts, cudaStream_t stream) {
  const int NB = a.n_shape + a.n_expr;
  const FlameLayout L = flame_layout(a.workspace, a.V, NB);
  flame_skin_bwd_kernel<<<L.n_chunks, 256, 0, stream>>>(a, g_verts, L);
  count_launch();
  flame_chain_bwd_kernel<<<1, 256, sizeof(double) * (FL_PART_HEAD + NB), stream>>>(a, L);
  count_launch();
}

}  // namespace gab
