// The FP32 contract of the mesh kernels (mesh_sm100.cu): generalised winding number, point-to-mesh distance and the grasp
// metrics built on them.  oracle/mesh_oracle.py restates it in float64 numpy; the tests compare the kernels with that
// restatement within bars that cover the fp32 rounding of the arithmetic below.
//
// A mesh is fp32 vertices [V, 3] plus int32 faces [F, 3].  A face with a vertex id outside [0, V) contributes nothing.
//
//   winding    a = fl(v0 - q), b = fl(v1 - q), c = fl(v2 - q) (componentwise),
//              Omega_f = 2 atan2(a . (b x c), |a||b||c| + (a . b)|c| + (b . c)|a| + (c . a)|b|) (Van Oosterom-Strackee),
//              w(q) = fl(S / fl(4 pi)), S = the sum of Omega_f over ascending f from +0, one fp32 add per face, in the query's
//              owner thread (deterministic).  atan2f / sqrtf are CUDA's accurate functions, not fast-math intrinsics.
//              For an outward-oriented closed mesh w = 1 inside and 0 outside (-1 inside a flipped one).
//   inside     w >= 0.5, the robust rule for open meshes such as MANO's hand (open at the wrist).  NaN is outside.
//   box rule   a query outside the axis-aligned box of its mesh item's V vertices gets w = 0 without being evaluated: exact
//              for a closed mesh, and what makes the kernel's culling legal.  The box is the per-axis min / max over the
//              item's vertices with NaN coordinates ignored (fminf / fmaxf); a query is inside it when lo <= q <= hi holds on
//              every axis, so a NaN query is outside.
//   distance   dist2(q) = min over f of the squared distance from q to the closest point of triangle f (Ericson, Real-Time
//              Collision Detection 5.1.5, written as closest = a + v ab + w ac, dist2 = |ap - v ab - w ac|^2).  A triangle
//              whose fp32 area^2 = |ab x ac|^2 is 0 is degenerate (no 0/0 in the interior region): it is its three edge
//              segments ab, ac, bc, in that order (face_segments), and its dist2 is the minimum of their segment_dist2.
//   face       the lowest f among exact fp32 minima of dist2; NaN counts as +inf (so a triangle with a non-finite corner
//              never wins).  When no face gives a finite distance, face = 0 and dist2 = +inf.
//   penetration  per query: depth2 = dist2 and face = the closest face when w >= 0.5, else depth2 = +0 and face = -1, with w,
//              dist2 and face exactly the winding and distance values above (so sqrt(depth2) maxed over a hand's vertices
//              is GraspQuality's depth, bit for bit).
//
// Gradient of dist2 (envelope theorem: the closest point's barycentrics are held fixed), for a query with its face f:
//   offset     triangle (fp32 area^2 != 0): from the forward's staged a = v0, ab = fl(v1 - v0), ac = fl(v2 - v0), aa, cc,
//              bc and ap = fl(q - a): (v, w) = closest_vw, d = ap - v ab - w ac in tri_offset2's FMA order, so
//              fma(dz, dz, fma(dy, dy, dx dx)) is the forward's dist2 bit for bit; lambda = (fl(fl(1 - v) - w), v, w).
//              Degenerate face: the first of its segments whose segment_dist2 equals that minimum, its t and offset from
//              segment_offset, its two endpoints weighted (fl(1 - t), t), the third 0.
//   g_pts      = fl(2 g) d per component, g the upstream gradient of dist2.
//   g_verts    corner k of face f gets the term -fl(lambda_k g_pts); g_verts[b, vertex] is the sum of its terms in
//              ascending (query, corner) order from +0 (no atomics).
//   nothing    a query contributes nothing (g_pts = 0, no term) when face = -1, face is outside [0, F), its face has a
//              vertex id outside [0, V), or its recomputed offset is not finite.
//
// Grasp metrics of hand b against one object (dvq.GraspQuality; the last reductions are device-side torch on the kernels'
// outputs):
//   voxels     lo = the object's vertex min, n = max(1, ceil((hi - lo) / pitch)) cells per axis (sized on the host once),
//              centre c = fl(lo + fl((i + 0.5) pitch)), kept when inside the object: an fp32 list [M, 3] in (i, j, k) order,
//              k fastest, so consecutive query tiles are spatially compact (and mostly culled by the box rule).
//   volume[b]  = count[b] pitch^3, count[b] = the number of voxel centres inside hand b (one integer atomicAdd per CTA).
//   depth[b]   = max of sqrt(dist2) over the hand vertices inside the object, 0 if there are none.
//   contact[b] = some hand vertex is inside the object or has dist2 <= contact_tol^2.
#pragma once

#include <math.h>

#include "f32x2.cuh"

namespace dvq {

constexpr float MESH_4PI = 12.566370614359172f;     // fl(4 pi)

__device__ __forceinline__ uint64_t dot2(uint64_t ax, uint64_t ay, uint64_t az, uint64_t bx, uint64_t by, uint64_t bz) {
  return ffma2(az, bz, ffma2(ay, by, fmul2(ax, bx)));
}

// Omega_f of one face for two queries at once: packed corner offsets a = fl(v0 - q), b, c of the two queries
__device__ __forceinline__ void solid_angle2(uint64_t ax, uint64_t ay, uint64_t az, uint64_t bx, uint64_t by, uint64_t bz,
                                             uint64_t cx, uint64_t cy, uint64_t cz, float& o0, float& o1) {
  const uint64_t rx = fsub2(fmul2(by, cz), fmul2(bz, cy));
  const uint64_t ry = fsub2(fmul2(bz, cx), fmul2(bx, cz));
  const uint64_t rz = fsub2(fmul2(bx, cy), fmul2(by, cx));
  const uint64_t det = dot2(ax, ay, az, rx, ry, rz);
  float a0, a1, b0, b1, c0, c1;
  unpack_f32x2(dot2(ax, ay, az, ax, ay, az), a0, a1);
  unpack_f32x2(dot2(bx, by, bz, bx, by, bz), b0, b1);
  unpack_f32x2(dot2(cx, cy, cz, cx, cy, cz), c0, c1);
  const uint64_t la = pack_f32x2(sqrtf(a0), sqrtf(a1)), lb = pack_f32x2(sqrtf(b0), sqrtf(b1)), lc = pack_f32x2(sqrtf(c0), sqrtf(c1));
  const uint64_t den = ffma2(dot2(cx, cy, cz, ax, ay, az), lb,
                             ffma2(dot2(bx, by, bz, cx, cy, cz), la, ffma2(dot2(ax, ay, az, bx, by, bz), lc, fmul2(fmul2(la, lb), lc))));
  float d0, d1, n0, n1;
  unpack_f32x2(det, n0, n1);
  unpack_f32x2(den, d0, d1);
  o0 = 2.f * atan2f(n0, d0);
  o1 = 2.f * atan2f(n1, d1);
}

// Ericson's region cascade for one query: (v, w) of the closest point a + v ab + w ac, from d1 = ab . ap, d2 = ac . ap and
// the face's aa = ab . ab, cc = ac . ac, bc = ab . ac (so d3 = ab . bp = d1 - aa, d4 = ac . bp = d2 - bc, d5 = ab . cp =
// d1 - bc, d6 = ac . cp = d2 - cc).  A NaN anywhere falls through to the interior case and gives NaN.
__device__ __forceinline__ void closest_vw(float d1, float d2, float aa, float cc, float bc, float& v, float& w) {
  const float d3 = d1 - aa, d4 = d2 - bc, d5 = d1 - bc, d6 = d2 - cc;
  const float vc = d1 * d4 - d3 * d2, vb = d5 * d2 - d1 * d6, va = d3 * d6 - d5 * d4;
  float nv, nw, den = 1.f;
  if (d1 <= 0.f && d2 <= 0.f) {                              // vertex a
    nv = 0.f, nw = 0.f;
  } else if (d3 >= 0.f && d4 <= d3) {                        // vertex b
    nv = 1.f, nw = 0.f;
  } else if (vc <= 0.f && d1 >= 0.f && d3 <= 0.f) {          // edge ab
    nv = d1, nw = 0.f, den = d1 - d3;
  } else if (d6 >= 0.f && d5 <= d6) {                        // vertex c
    nv = 0.f, nw = 1.f;
  } else if (vb <= 0.f && d2 >= 0.f && d6 <= 0.f) {          // edge ac
    nv = 0.f, nw = d2, den = d2 - d6;
  } else if (va <= 0.f && d4 - d3 >= 0.f && d5 - d6 >= 0.f) {  // edge bc: b + t (c - b) = a + (1 - t) ab + t ac
    nv = d5 - d6, nw = d4 - d3, den = (d4 - d3) + (d5 - d6);
  } else {                                                   // interior
    nv = vb, nw = vc, den = va + vb + vc;
  }
  const float r = 1.f / den;
  v = nv * r;
  w = nw * r;
}

// |ab x ac|^2 of the edges ab = fl(v1 - v0), ac = fl(v2 - v0), every operation rounded (no FMA), so the degenerate-face
// decision is reproducible bit for bit
__device__ __forceinline__ float area2(const float* e1, const float* e2) {
  const float nx = __fsub_rn(__fmul_rn(e1[1], e2[2]), __fmul_rn(e1[2], e2[1]));
  const float ny = __fsub_rn(__fmul_rn(e1[2], e2[0]), __fmul_rn(e1[0], e2[2]));
  const float nz = __fsub_rn(__fmul_rn(e1[0], e2[1]), __fmul_rn(e1[1], e2[0]));
  return __fadd_rn(__fadd_rn(__fmul_rn(nx, nx), __fmul_rn(ny, ny)), __fmul_rn(nz, nz));
}

// The face data both the distance and its gradient stage: a = v0, ab = fl(v1 - v0), ac = fl(v2 - v0) from the corners
// p0, p1, p2, and aa = ab . ab, cc = ac . ac, bc = ab . ac.
__device__ __forceinline__ void face_frame(const float* p0, const float* p1, const float* p2, float (&a)[3], float (&e1)[3],
                                           float (&e2)[3], float& aa, float& cc, float& bc) {
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    a[d] = p0[d];
    e1[d] = p1[d] - a[d];
    e2[d] = p2[d] - a[d];
  }
  aa = e1[0] * e1[0] + e1[1] * e1[1] + e1[2] * e1[2];
  cc = e2[0] * e2[0] + e2[1] * e2[1] + e2[2] * e2[2];
  bc = e1[0] * e2[0] + e1[1] * e2[1] + e1[2] * e2[2];
}

// Triangle offset d = ap - v ab - w ac of two queries (packed ap; packed ab = e[0..2], ac = e[3..5]); (v, w) per query
// from closest_vw.  dist2 = dot2(d, d).
__device__ __forceinline__ void tri_offset2(uint64_t px, uint64_t py, uint64_t pz, const uint64_t* e, float aa, float cc, float bc,
                                            float (&vv)[2], float (&ww)[2], uint64_t& dx, uint64_t& dy, uint64_t& dz) {
  float d1[2], d2[2];
  unpack_f32x2(dot2(e[0], e[1], e[2], px, py, pz), d1[0], d1[1]);
  unpack_f32x2(dot2(e[3], e[4], e[5], px, py, pz), d2[0], d2[1]);
#pragma unroll
  for (int h = 0; h < 2; ++h) closest_vw(d1[h], d2[h], aa, cc, bc, vv[h], ww[h]);
  const uint64_t nv = pack_f32x2(-vv[0], -vv[1]), nw = pack_f32x2(-ww[0], -ww[1]);
  dx = ffma2(nw, e[3], ffma2(nv, e[0], px));
  dy = ffma2(nw, e[4], ffma2(nv, e[1], py));
  dz = ffma2(nw, e[5], ffma2(nv, e[2], pz));
}

// Offset d = p - t e from p = a + ap to the closest point of the segment a + t e, t in [0, 1] (a zero-length segment is
// its point); returns t.
__device__ __forceinline__ float segment_offset(float px, float py, float pz, float ex, float ey, float ez, float& dx, float& dy,
                                                float& dz) {
  const float ee = ex * ex + ey * ey + ez * ez, pe = px * ex + py * ey + pz * ez;
  const float t = ee > 0.f ? fminf(fmaxf(pe / ee, 0.f), 1.f) : 0.f;
  dx = px - t * ex, dy = py - t * ey, dz = pz - t * ez;
  return t;
}

// squared distance from p = a + ap to the segment a + t e
__device__ __forceinline__ float segment_dist2(float px, float py, float pz, float ex, float ey, float ez) {
  float dx, dy, dz;
  segment_offset(px, py, pz, ex, ey, ez, dx, dy, dz);
  return dx * dx + dy * dy + dz * dz;
}

// The segments of a degenerate face, k = 0 ab, 1 ac, 2 bc, from the query's offset ap = fl(q - a) and the face's ab = e1,
// ac = e2: segment k is a' + t e[k] with p[k] = fl(q - a') -- (ap, ab), (ap, ac), (fl(ap - ab), fl(ac - ab)) -- and s[k] =
// its segment_dist2.
__device__ __forceinline__ void face_segments(const float (&ap)[3], const float (&e1)[3], const float (&e2)[3], float (&p)[3][3],
                                              float (&e)[3][3], float (&s)[3]) {
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    p[0][d] = ap[d], e[0][d] = e1[d];
    p[1][d] = ap[d], e[1][d] = e2[d];
    p[2][d] = ap[d] - e1[d], e[2][d] = e2[d] - e1[d];
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) s[k] = segment_dist2(p[k][0], p[k][1], p[k][2], e[k][0], e[k][1], e[k][2]);
}

}  // namespace dvq
