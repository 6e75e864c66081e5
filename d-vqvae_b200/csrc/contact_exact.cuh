// The exact FP32 contract of the hand-object nearest-point kernels (contact_sm100.cu).  oracle/contact_oracle.py restates
// it in numpy, and the tests compare the kernels' bits with that restatement.
//
// Points are fp32 [B, n, 3], contiguous; batch item b's src points are searched against batch item b's trg points only.
//
//   distance   d(s, t) = fma(dz, dz, fma(dy, dy, fl(dx * dx))), dx = fl(s.x - t.x) (likewise y, z): the squared Euclidean
//              distance, as pytorch3d's knn_points returns it.  Every operation is an explicit _rn intrinsic or a packed
//              f32x2 instruction, so nvcc's contraction cannot change the bits (nn_dist / nn_dist2).
//   argmin     idx[b,i] = the lowest j among the exact fp32 minima of d(s_i, t_j), dist[b,i] = that d.  A NaN distance
//              counts as +inf; when no j gives a distance below +inf, idx = 0 and dist = d(s_i, t_0).
//   backward   g = dL/d dist[b,i], j = idx[b,i], dv = fl(s_i - t_j) per component, term_i = fl(fl(2 g) * dv):
//              g_src[b,i] = term_i;  g_trg[b,j] = -(sum of term_i over the i with idx[b,i] = j), summed in ascending i from
//              +0, one fp32 add at a time (no float atomics: deterministic run to run).  idx gets no gradient.
//   normals    n_f = cross(fl(v2 - v1), fl(v0 - v1)), components like fl(fl(a.y * b.z) - fl(a.z * b.y)), no FMA;
//              acc_v = sum of n_f over the faces listing v, ascending f, once per occurrence, from +0;
//              normal_v = acc_v / max(sqrt(fl(fl(fl(x^2) + fl(y^2)) + fl(z^2))), 1e-6) with IEEE sqrt and division
//              (pytorch3d's area-weighted vertex normal followed by F.normalize(eps=1e-6)).
//   interior   (src = object points, trg = hand vertices) interior[b,i] = dot(fl(t_j - s_i), normal_j) > 0, j = idx[b,i],
//              dot = fl(fl(fl(ax * nx) + fl(ay * ny)) + fl(az * nz)), no FMA.  fl(t - s) = -fl(s - t) exactly, so the
//              kernel reuses dv.
#pragma once

#include "f32x2.cuh"

namespace dvq {

__device__ __forceinline__ float nn_dist(float dx, float dy, float dz) {
  return __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
}
// the same for two points at once: packed (s.x - t.x) etc. of two pairs
__device__ __forceinline__ uint64_t nn_dist2(uint64_t dx, uint64_t dy, uint64_t dz) {
  return ffma2(dz, dz, ffma2(dy, dy, fmul2(dx, dx)));
}

// interior test from dv = fl(s - t_j) and the unit normal of t_j: dot(-dv, n) > 0
__device__ __forceinline__ bool nn_interior(float dx, float dy, float dz, float nx, float ny, float nz) {
  const float dot = __fadd_rn(__fadd_rn(__fmul_rn(-dx, nx), __fmul_rn(-dy, ny)), __fmul_rn(-dz, nz));
  return dot > 0.f;
}

// n_f = cross(a, b), a = fl(v2 - v1), b = fl(v0 - v1), no FMA
__device__ __forceinline__ float3 face_normal(float3 v0, float3 v1, float3 v2) {
  const float ax = __fsub_rn(v2.x, v1.x), ay = __fsub_rn(v2.y, v1.y), az = __fsub_rn(v2.z, v1.z);
  const float bx = __fsub_rn(v0.x, v1.x), by = __fsub_rn(v0.y, v1.y), bz = __fsub_rn(v0.z, v1.z);
  return make_float3(__fsub_rn(__fmul_rn(ay, bz), __fmul_rn(az, by)), __fsub_rn(__fmul_rn(az, bx), __fmul_rn(ax, bz)),
                     __fsub_rn(__fmul_rn(ax, by), __fmul_rn(ay, bx)));
}

// F.normalize(acc, eps=1e-6); the max propagates a NaN norm, as clamp_min does
__device__ __forceinline__ float3 normalize_eps(float3 a) {
  const float n2 = __fadd_rn(__fadd_rn(__fmul_rn(a.x, a.x), __fmul_rn(a.y, a.y)), __fmul_rn(a.z, a.z));
  const float norm = __fsqrt_rn(n2);
  const float den = norm < 1e-6f ? 1e-6f : norm;
  return make_float3(__fdiv_rn(a.x, den), __fdiv_rn(a.y, den), __fdiv_rn(a.z, den));
}

}  // namespace dvq
