// MANO hand layer (linear blend skinning): 10 shape + 3 global-orientation + PCA pose parameters -> 778 vertices.
// Replaces the third-party call at network/gen_net.py:116-118
//     self.rh_mano(betas=recon[:, :10], global_orient=0, hand_pose=recon[:, 10:55], transl=0).vertices
// (package `mano`, created at gen_diverse_grasp_obman.py:355-360 with use_pca=True, num_pca_comps=45,
// flat_hand_mean=True; the arithmetic is smplx/lbs.py's, restated in oracle/mano_oracle.py) so that the decoder's 55
// parameters reach the 778-point PointNet without leaving the device or the stream.
//
// One CTA per hand, everything but the model tables in shared memory:
//   1  full pose = [global_orient | coeffs @ components] + pose_mean; Rodrigues per joint (angle = |r + 1e-8|)
//   2  v_shaped = v_template + shapedirs . betas   (thread = vertex coordinate, coalesced table rows)
//   3  J = J_regressor @ v_shaped                  (warp per joint, shuffle reduction)
//   4  kinematic chain: the five fingers are independent three-joint chains off the root (a lane per finger)
//   5  v_posed = v_shaped + posedirs . vec(R_1..15 - I)   (135 coalesced table rows per coordinate: the bulk of the work,
//      1.26 MB of L2-resident table per hand)
//   6  skinning: thread = vertex, T = sum_j w_vj A_j, out = T [v_posed; 1] + transl
// FP32 with fmaf throughout; agreement with the float64 oracle ~1e-7 of the hand size.
//
// The backward (vector-Jacobian product for betas, global_orient, hand_pose and transl) is a second kernel, also one CTA
// per hand.  It saves nothing from the forward: stages 1-5 are recomputed by the same device code, then the stages are
// walked in reverse (see mano_lbs_backward_kernel).
#include "dvq_common.cuh"

namespace dvq {
namespace {

constexpr int NV = 778, NJ = 16, NB = 10, NP = 45, NPF = 9 * (NJ - 1), NC = NV * 3;
constexpr int MT = 256;

// One hand's forward intermediates (G = [R | t], A = [G.R | G.t - G.R J], 3 x 4 row-major).
struct LbsShared {
  float pose[3 * NJ], R[NJ][9], pf[NPF], beta[NB], J[NJ][3], G[NJ][12], A[NJ][12];
  float vs[NC];   // v_shaped, then v_posed
};

// Stages 1-5 for hand b; leaves R, J, G, A and v_posed in shared memory and ends at a barrier.
__device__ __forceinline__ void lbs_recompute(const DvqManoModel& m, const float* __restrict__ betas, const float* __restrict__ global_orient,
                                              const float* __restrict__ hand_pose, int b, LbsShared& s) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // ---- 1: pose ----
  if (tid < 3) s.pose[tid] = (global_orient ? global_orient[(size_t)b * 3 + tid] : 0.f) + m.pose_mean[tid];
  if (tid >= 32 && tid < 32 + NP) {
    const int k = tid - 32;
    float v;
    if (m.ncomps > 0) {   // PCA coefficients -> axis-angle: sum over the first ncomps components, in order
      v = 0.f;
      for (int i = 0; i < m.ncomps; ++i) v = fmaf(hand_pose[(size_t)b * m.ncomps + i], m.hands_components[i * NP + k], v);
    } else {
      v = hand_pose[(size_t)b * NP + k];
    }
    s.pose[3 + k] = v + m.pose_mean[3 + k];
  }
  if (tid >= 96 && tid < 96 + NB) s.beta[tid - 96] = betas[(size_t)b * NB + tid - 96];
  __syncthreads();
  if (tid < NJ) {
    const float rx = s.pose[3 * tid], ry = s.pose[3 * tid + 1], rz = s.pose[3 * tid + 2];
    const float ex = rx + 1e-8f, ey = ry + 1e-8f, ez = rz + 1e-8f;
    const float angle = sqrtf(fmaf(ez, ez, fmaf(ey, ey, ex * ex)));
    const float dx = rx / angle, dy = ry / angle, dz = rz / angle;
    float sn, c;
    sincosf(angle, &sn, &c);
    const float t = 1.f - c;
    // R = I + s K + t K^2,  K = [[0,-dz,dy],[dz,0,-dx],[-dy,dx,0]],  K^2 = d d^T - |d|^2 I
    const float n2 = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
    float* r = s.R[tid];
    r[0] = 1.f + t * (dx * dx - n2); r[1] = fmaf(t, dx * dy, -sn * dz);  r[2] = fmaf(t, dx * dz, sn * dy);
    r[3] = fmaf(t, dx * dy, sn * dz);  r[4] = 1.f + t * (dy * dy - n2); r[5] = fmaf(t, dy * dz, -sn * dx);
    r[6] = fmaf(t, dx * dz, -sn * dy); r[7] = fmaf(t, dy * dz, sn * dx);  r[8] = 1.f + t * (dz * dz - n2);
  }
  __syncthreads();
  if (tid < NPF) { const int j = tid / 9 + 1, e = tid % 9; s.pf[tid] = s.R[j][e] - ((e == 0 || e == 4 || e == 8) ? 1.f : 0.f); }
  // ---- 2: shape blend ----
  for (int o = tid; o < NC; o += MT) {
    float v = __ldg(m.v_template + o);
#pragma unroll
    for (int l = 0; l < NB; ++l) v = fmaf(s.beta[l], __ldg(m.shapedirs + l * NC + o), v);
    s.vs[o] = v;
  }
  __syncthreads();
  // ---- 3: joints ----
  for (int j = warp; j < NJ; j += MT / 32) {
    float ax = 0.f, ay = 0.f, az = 0.f;
    for (int v = lane; v < NV; v += 32) {
      const float w = __ldg(m.j_regressor + j * NV + v);
      ax = fmaf(w, s.vs[3 * v], ax); ay = fmaf(w, s.vs[3 * v + 1], ay); az = fmaf(w, s.vs[3 * v + 2], az);
    }
    ax = warp_sum(ax); ay = warp_sum(ay); az = warp_sum(az);
    if (lane == 0) { s.J[j][0] = ax; s.J[j][1] = ay; s.J[j][2] = az; }
  }
  __syncthreads();
  // ---- 4: kinematic chain ----
  if (tid == 0) {
#pragma unroll
    for (int e = 0; e < 9; ++e) s.G[0][(e / 3) * 4 + e % 3] = s.R[0][e];
    s.G[0][3] = s.J[0][0]; s.G[0][7] = s.J[0][1]; s.G[0][11] = s.J[0][2];
  }
  __syncthreads();
  if (tid < 5) {   // finger tid: joints 3 tid + 1 .. 3 tid + 3 (MANO's tree: parents 0,1,2 / 0,4,5 / ...; checked on the host)
    for (int j = 3 * tid + 1; j <= 3 * tid + 3; ++j) {
      const int pj = m.parents[j];
      const float tx = s.J[j][0] - s.J[pj][0], ty = s.J[j][1] - s.J[pj][1], tz = s.J[j][2] - s.J[pj][2];
      const float* gp = s.G[pj];
      const float* r = s.R[j];
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const float g0 = gp[4 * i], g1 = gp[4 * i + 1], g2 = gp[4 * i + 2];
        s.G[j][4 * i + 0] = fmaf(g2, r[6], fmaf(g1, r[3], g0 * r[0]));
        s.G[j][4 * i + 1] = fmaf(g2, r[7], fmaf(g1, r[4], g0 * r[1]));
        s.G[j][4 * i + 2] = fmaf(g2, r[8], fmaf(g1, r[5], g0 * r[2]));
        s.G[j][4 * i + 3] = fmaf(g2, tz, fmaf(g1, ty, g0 * tx)) + gp[4 * i + 3];
      }
    }
  }
  __syncthreads();
  if (tid < NJ) {
    const float* g = s.G[tid];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      s.A[tid][4 * i] = g[4 * i]; s.A[tid][4 * i + 1] = g[4 * i + 1]; s.A[tid][4 * i + 2] = g[4 * i + 2];
      s.A[tid][4 * i + 3] = g[4 * i + 3] - fmaf(g[4 * i + 2], s.J[tid][2], fmaf(g[4 * i + 1], s.J[tid][1], g[4 * i] * s.J[tid][0]));
    }
  }
  // ---- 5: pose blend (in place: vs becomes v_posed) ----
  for (int o = tid; o < NC; o += MT) {
    float v = 0.f;
#pragma unroll 9
    for (int k = 0; k < NPF; ++k) v = fmaf(s.pf[k], __ldg(m.posedirs + k * NC + o), v);
    s.vs[o] += v;
  }
  __syncthreads();
}

// T = sum_j w_vj A_j for vertex v (3 x 4 row-major).
__device__ __forceinline__ void skin_transform(const DvqManoModel& m, const LbsShared& s, int v, float T[12]) {
#pragma unroll
  for (int e = 0; e < 12; ++e) T[e] = 0.f;
  const float4* wv = reinterpret_cast<const float4*>(m.weights + (size_t)v * NJ);
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float4 w4 = __ldg(wv + q);
    const float w[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      const float* a = s.A[4 * q + jj];
#pragma unroll
      for (int e = 0; e < 12; ++e) T[e] = fmaf(w[jj], a[e], T[e]);
    }
  }
}

__global__ void __launch_bounds__(MT) mano_lbs_kernel(const DvqManoModel m, const float* __restrict__ betas, const float* __restrict__ global_orient,
                                                      const float* __restrict__ hand_pose, const float* __restrict__ transl, int B,
                                                      float* __restrict__ vertices, float* __restrict__ joints) {
  __shared__ LbsShared s;
  const int b = blockIdx.x, tid = threadIdx.x;
  if (b >= B) return;
  lbs_recompute(m, betas, global_orient, hand_pose, b, s);
  const float tx = transl ? transl[(size_t)b * 3] : 0.f, ty = transl ? transl[(size_t)b * 3 + 1] : 0.f, tz = transl ? transl[(size_t)b * 3 + 2] : 0.f;
  if (joints && tid < NJ) {
    const float* g = s.G[tid];
    float* jo = joints + ((size_t)b * NJ + tid) * 3;
    jo[0] = g[3] + tx; jo[1] = g[7] + ty; jo[2] = g[11] + tz;
  }
  // ---- 6: skinning ----
  for (int v = tid; v < NV; v += MT) {
    float T[12];
    skin_transform(m, s, v, T);
    const float x = s.vs[3 * v], y = s.vs[3 * v + 1], z = s.vs[3 * v + 2];
    float* o = vertices + ((size_t)b * NV + v) * 3;
    o[0] = fmaf(T[2], z, fmaf(T[1], y, T[0] * x)) + T[3] + tx;
    o[1] = fmaf(T[6], z, fmaf(T[5], y, T[4] * x)) + T[7] + ty;
    o[2] = fmaf(T[10], z, fmaf(T[9], y, T[8] * x)) + T[11] + tz;
  }
}

// Vector-Jacobian product of mano_lbs_kernel for one hand per CTA.  gV [B,778,3] / gJo [B,16,3] may be NULL (zero).
// Every output element is written once by its hand's CTA, and every sum runs in a fixed order: deterministic.
//   B1  dA_j = sum_v w_vj gV_v (x) [v_posed_v; 1]   (warp per joint, shuffle reduction; a 17th task sums gV for transl)
//   B2  dv_posed_v = T_v.R^T gV_v                    (thread = vertex)
//   B3  A_j = [G_j.R | G_j.t - G_j.R J_j]  ->  dG_j, dJ_j   (gJo enters dG_j.t)
//   B4  kinematic chain in reverse, a lane per finger; the five fingers' shares of the root are summed in finger order
//   B5  dpf = posedirs . dv_posed                    (warp per table row, coalesced: the bulk of the work) -> dR_1..15
//   B6  Rodrigues backward per joint -> d(full pose); PCA / identity to the hand_pose gradient
//   B7  dv_shaped = dv_posed + J_regressor^T dJ; dbetas = shapedirs . dv_shaped (thread = coordinate, block reduction)
__global__ void __launch_bounds__(MT) mano_lbs_backward_kernel(const DvqManoModel m, const float* __restrict__ betas,
                                                               const float* __restrict__ global_orient, const float* __restrict__ hand_pose, int B,
                                                               const float* __restrict__ gV, const float* __restrict__ gJo,
                                                               float* __restrict__ g_betas, float* __restrict__ g_global_orient,
                                                               float* __restrict__ g_hand_pose, float* __restrict__ g_transl) {
  __shared__ LbsShared s;
  __shared__ float gv[NC];                       // this hand's grad_vertices
  __shared__ float dA[NJ + 1][12];               // row NJ: sum_v gV_v in columns 3, 7, 11
  __shared__ float dG[NJ][12], dJ[NJ][3], dR[NJ][9], dpf[NPF], gjo[NJ][3], gpose[3 * NJ];
  __shared__ float droot[5][15];                 // finger f's share of the root: dG_0 (12), dJ_0 (3)
  __shared__ float part[MT / 32][NB];
  const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (b >= B) return;
  for (int o = tid; o < NC; o += MT) gv[o] = gV ? gV[(size_t)b * NC + o] : 0.f;
  if (tid < 3 * NJ) gjo[tid / 3][tid % 3] = gJo ? gJo[(size_t)b * NJ * 3 + tid] : 0.f;
  lbs_recompute(m, betas, global_orient, hand_pose, b, s);
  // ---- B1 ----
  for (int j = warp; j <= NJ; j += MT / 32) {
    float a[12];
#pragma unroll
    for (int e = 0; e < 12; ++e) a[e] = 0.f;
    for (int v = lane; v < NV; v += 32) {
      const float w = j < NJ ? __ldg(m.weights + v * NJ + j) : 1.f;
      const float x = s.vs[3 * v], y = s.vs[3 * v + 1], z = s.vs[3 * v + 2];
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const float g = w * gv[3 * v + i];
        a[4 * i] = fmaf(g, x, a[4 * i]); a[4 * i + 1] = fmaf(g, y, a[4 * i + 1]); a[4 * i + 2] = fmaf(g, z, a[4 * i + 2]);
        a[4 * i + 3] += g;
      }
    }
#pragma unroll
    for (int e = 0; e < 12; ++e) a[e] = warp_sum(a[e]);
    if (lane == 0) {
#pragma unroll
      for (int e = 0; e < 12; ++e) dA[j][e] = a[e];
    }
  }
  __syncthreads();
  // ---- B2 (in place: vs becomes dv_posed) ----
  for (int v = tid; v < NV; v += MT) {
    float T[12];
    skin_transform(m, s, v, T);
    const float g0 = gv[3 * v], g1 = gv[3 * v + 1], g2 = gv[3 * v + 2];
#pragma unroll
    for (int c = 0; c < 3; ++c) s.vs[3 * v + c] = fmaf(T[8 + c], g2, fmaf(T[4 + c], g1, T[c] * g0));
  }
  // ---- B3 ----
  if (tid < NJ) {
    const float* a = dA[tid];
    const float* g = s.G[tid];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
      for (int k = 0; k < 3; ++k) dG[tid][4 * i + k] = fmaf(-a[4 * i + 3], s.J[tid][k], a[4 * i + k]);
      dG[tid][4 * i + 3] = a[4 * i + 3] + gjo[tid][i];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) dJ[tid][k] = -fmaf(g[8 + k], a[11], fmaf(g[4 + k], a[7], g[k] * a[3]));
  }
  __syncthreads();
  // ---- B4: G_j = G_p [R_j | t_j], t_j = J_j - J_p; joints in reverse order along each finger ----
  if (tid < 5) {
    for (int j = 3 * tid + 3; j >= 3 * tid + 1; --j) {
      const int pj = m.parents[j];
      const float t[3] = {s.J[j][0] - s.J[pj][0], s.J[j][1] - s.J[pj][1], s.J[j][2] - s.J[pj][2]};
      const float* gp = s.G[pj];
      const float* r = s.R[j];
      const float* dg = dG[j];
      float dt[3], pg[12];
#pragma unroll
      for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int c = 0; c < 3; ++c) dR[j][3 * a + c] = fmaf(gp[8 + a], dg[8 + c], fmaf(gp[4 + a], dg[4 + c], gp[a] * dg[c]));   // G_p.R^T dG_j.R
        dt[a] = fmaf(gp[8 + a], dg[11], fmaf(gp[4 + a], dg[7], gp[a] * dg[3]));                                                // G_p.R^T dG_j.t
      }
#pragma unroll
      for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int c = 0; c < 3; ++c)   // dG_p.R += dG_j.R R_j^T + dG_j.t t_j^T
          pg[4 * i + c] = fmaf(dg[4 * i + 3], t[c], fmaf(dg[4 * i + 2], r[3 * c + 2], fmaf(dg[4 * i + 1], r[3 * c + 1], dg[4 * i] * r[3 * c])));
        pg[4 * i + 3] = dg[4 * i + 3];
      }
#pragma unroll
      for (int k = 0; k < 3; ++k) dJ[j][k] += dt[k];
      if (pj == 0) {
#pragma unroll
        for (int e = 0; e < 12; ++e) droot[tid][e] = pg[e];
#pragma unroll
        for (int k = 0; k < 3; ++k) droot[tid][12 + k] = -dt[k];
      } else {
#pragma unroll
        for (int e = 0; e < 12; ++e) dG[pj][e] += pg[e];
#pragma unroll
        for (int k = 0; k < 3; ++k) dJ[pj][k] -= dt[k];
      }
    }
  }
  // ---- B5 ----
  for (int k = warp; k < NPF; k += MT / 32) {
    const float* row = m.posedirs + (size_t)k * NC;
    float a = 0.f;
#pragma unroll 8
    for (int o = lane; o < NC; o += 32) a = fmaf(__ldg(row + o), s.vs[o], a);
    a = warp_sum(a);
    if (lane == 0) dpf[k] = a;
  }
  __syncthreads();
  if (tid == 0) {   // root: G_0 = [R_0 | J_0]
    float g[15];
#pragma unroll
    for (int e = 0; e < 12; ++e) g[e] = dG[0][e];
#pragma unroll
    for (int k = 0; k < 3; ++k) g[12 + k] = dJ[0][k];
    for (int f = 0; f < 5; ++f) {
#pragma unroll
      for (int e = 0; e < 15; ++e) g[e] += droot[f][e];
    }
#pragma unroll
    for (int e = 0; e < 9; ++e) dR[0][e] = g[(e / 3) * 4 + e % 3];
#pragma unroll
    for (int k = 0; k < 3; ++k) dJ[0][k] = g[12 + k] + g[4 * k + 3];
  } else if (tid < NJ) {
#pragma unroll
    for (int e = 0; e < 9; ++e) dR[tid][e] += dpf[9 * (tid - 1) + e];
  }
  __syncthreads();
  // ---- B6: R = I + s K + t (d d^T - |d|^2 I), d = r / angle, angle = |r + 1e-8|, s = sin, t = 1 - cos ----
  if (tid < NJ) {
    const float rx = s.pose[3 * tid], ry = s.pose[3 * tid + 1], rz = s.pose[3 * tid + 2];
    const float ex = rx + 1e-8f, ey = ry + 1e-8f, ez = rz + 1e-8f;
    const float angle = sqrtf(fmaf(ez, ez, fmaf(ey, ey, ex * ex)));
    const float dx = rx / angle, dy = ry / angle, dz = rz / angle;
    float sn, c;
    sincosf(angle, &sn, &c);
    const float t = 1.f - c;
    const float n2 = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
    const float* g = dR[tid];
    const float kx = g[7] - g[5], ky = g[2] - g[6], kz = g[3] - g[1];     // d<g, K>/dd
    const float tr = g[0] + g[4] + g[8];
    const float gdx = fmaf(g[2], dz, fmaf(g[1], dy, g[0] * dx)), gdy = fmaf(g[5], dz, fmaf(g[4], dy, g[3] * dx)),
                gdz = fmaf(g[8], dz, fmaf(g[7], dy, g[6] * dx));         // g d
    const float hdx = fmaf(g[6], dz, fmaf(g[3], dy, g[0] * dx)), hdy = fmaf(g[7], dz, fmaf(g[4], dy, g[1] * dx)),
                hdz = fmaf(g[8], dz, fmaf(g[5], dy, g[2] * dx));         // g^T d
    const float gs = fmaf(dz, kz, fmaf(dy, ky, dx * kx));                                  // dL/ds
    const float gt = fmaf(dz, gdz, fmaf(dy, gdy, dx * gdx)) - n2 * tr;                     // dL/dt
    const float t2 = 2.f * t * tr;
    const float ddx = fmaf(sn, kx, t * (gdx + hdx)) - t2 * dx;                             // dL/dd
    const float ddy = fmaf(sn, ky, t * (gdy + hdy)) - t2 * dy;
    const float ddz = fmaf(sn, kz, t * (gdz + hdz)) - t2 * dz;
    const float inv = 1.f / angle;
    const float ga = fmaf(gs, c, gt * sn) - fmaf(ddz, rz, fmaf(ddy, ry, ddx * rx)) * inv * inv;   // dL/dangle
    const float ge = ga * inv;
    gpose[3 * tid] = fmaf(ge, ex, ddx * inv);
    gpose[3 * tid + 1] = fmaf(ge, ey, ddy * inv);
    gpose[3 * tid + 2] = fmaf(ge, ez, ddz * inv);
  }
  // ---- B7 ----
  float acc[NB];
#pragma unroll
  for (int l = 0; l < NB; ++l) acc[l] = 0.f;
  for (int o = tid; o < NC; o += MT) {
    const int v = o / 3, c = o - 3 * v;
    float d = s.vs[o];
#pragma unroll
    for (int j = 0; j < NJ; ++j) d = fmaf(__ldg(m.j_regressor + j * NV + v), dJ[j][c], d);
#pragma unroll
    for (int l = 0; l < NB; ++l) acc[l] = fmaf(__ldg(m.shapedirs + l * NC + o), d, acc[l]);
  }
#pragma unroll
  for (int l = 0; l < NB; ++l) acc[l] = warp_sum(acc[l]);
  if (lane == 0) {
#pragma unroll
    for (int l = 0; l < NB; ++l) part[warp][l] = acc[l];
  }
  __syncthreads();
  // ---- outputs ----
  if (g_global_orient && tid < 3) g_global_orient[(size_t)b * 3 + tid] = gpose[tid];
  if (g_hand_pose && tid >= 32 && tid < 32 + NP) {
    const int k = tid - 32;
    if (m.ncomps > 0) {   // hand_pose = coeffs @ components[:ncomps]  ->  g_coeffs = components[:ncomps] . g_pose
      if (k < m.ncomps) {
        float v = 0.f;
        for (int i = 0; i < NP; ++i) v = fmaf(m.hands_components[k * NP + i], gpose[3 + i], v);
        g_hand_pose[(size_t)b * m.ncomps + k] = v;
      }
    } else {
      g_hand_pose[(size_t)b * NP + k] = gpose[3 + k];
    }
  }
  if (g_betas && tid >= 96 && tid < 96 + NB) {
    const int l = tid - 96;
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < MT / 32; ++w) v += part[w][l];
    g_betas[(size_t)b * NB + l] = v;
  }
  if (g_transl && tid >= 128 && tid < 131) {
    const int i = tid - 128;
    float v = dA[NJ][4 * i + 3];
    for (int j = 0; j < NJ; ++j) v += gjo[j][i];
    g_transl[(size_t)b * 3 + i] = v;
  }
}

}  // namespace

int launch_mano(const DvqManoModel* m, const float* betas, const float* global_orient, const float* hand_pose, const float* transl, int B,
                float* vertices, float* joints, cudaStream_t s) {
  if (B == 0) return DVQ_OK;
  mano_lbs_kernel<<<B, MT, 0, s>>>(*m, betas, global_orient, hand_pose, transl, B, vertices, joints);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

int launch_mano_backward(const DvqManoModel* m, const float* betas, const float* global_orient, const float* hand_pose, int B,
                         const float* grad_vertices, const float* grad_joints, float* grad_betas, float* grad_global_orient,
                         float* grad_hand_pose, float* grad_transl, cudaStream_t s) {
  if (B == 0) return DVQ_OK;
  mano_lbs_backward_kernel<<<B, MT, 0, s>>>(*m, betas, global_orient, hand_pose, B, grad_vertices, grad_joints, grad_betas,
                                            grad_global_orient, grad_hand_pose, grad_transl);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

}  // namespace dvq
