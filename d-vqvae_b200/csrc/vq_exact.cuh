// The exact FP32 contract of the VQ kernels.  The all-FP32 kernel (vq_simt_fp32.cu) and the three refine kernels of the
// tcgen05 path (vq_refine.cu, vq_refine_binned.cu, vq_refine_stationary.cu) give every row the same idx, the same z_q
// bits and the same histogram entry, because each evaluates exactly this, with the helpers below:
//
//   dot(z, e_k) = sequential fmaf over d = 0 .. D-1, from +0
//   zz = ||z||^2: lane l of a 32-lane warp accumulates elements l, l + 32, ... with fmaf (sq_partial), then an xor-shuffle
//        tree over offsets 16, 8, 4, 2, 1; ee_k = ||e_k||^2 the same way (code_norms_kernel)
//   distance = fma(-2, dot, fl(zz + ee_k))   (exact_dist; == fl(fl(zz + ee_k) - 2 dot), 2 dot is exact)
//   winner = lexicographic minimum of (distance, code): exact ties keep the lowest code.  A NaN distance counts as +inf
//            and a row without a finite distance on its candidate codes gets code 0.  A distance is never -0 (zz + ee_k
//            >= +0, and an exact cancellation rounds to +0), so the order of dist_key and the float order agree.
//   outputs: z_q = fl(z + fl(e - z)) (the straight-through value), sse += (double)fl(e - z)^2 per element in train mode
//            (st_step4 / st_step1); z_q = e in inference.
#pragma once

#include "dvq_common.cuh"

namespace dvq {

__device__ __forceinline__ float exact_dist(float dot, float zz, float eek) { return __fmaf_rn(-2.0f, dot, __fadd_rn(zz, eek)); }

// order-preserving unsigned image of a distance; NaN counts as +inf (never a winner)
constexpr uint32_t KEY_INF = 0xff800000u;   // dist_key(+inf)
__device__ __forceinline__ uint32_t dist_key(float d) {
  if (!(d == d)) d = INFINITY;
  const uint32_t b = __float_as_uint(d);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// lexicographic (key, code) minimum over a warp whose lane l holds code code0 + l: one REDUX.MIN, then the lowest lane
// holding it (the lowest code among ties).  Packed as key << 32 | code, so that an unsigned 64-bit minimum of such
// values is again the lexicographic minimum (~0 = nothing evaluated yet).
__device__ __forceinline__ unsigned long long warp_argmin(uint32_t key, int code0) {
  const uint32_t kmin = __reduce_min_sync(0xffffffffu, key);
  const int src = __ffs(__ballot_sync(0xffffffffu, key == kmin)) - 1;
  return ((unsigned long long)kmin << 32) | (unsigned)(code0 + src);
}
// the code a packed minimum stands for: no finite distance -> code 0
__device__ __forceinline__ int packed_winner(unsigned long long best) { return (uint32_t)(best >> 32) >= KEY_INF ? 0 : (int)(uint32_t)best; }

// z_q and the SSE contribution of four elements (train mode)
__device__ __forceinline__ float4 st_step4(float4 e4, float4 z4, double& sse) {
  const float dx = __fsub_rn(e4.x, z4.x), dy = __fsub_rn(e4.y, z4.y);
  const float dz = __fsub_rn(e4.z, z4.z), dw = __fsub_rn(e4.w, z4.w);
  sse += (double)dx * dx + (double)dy * dy + (double)dz * dz + (double)dw * dw;
  return make_float4(__fadd_rn(z4.x, dx), __fadd_rn(z4.y, dy), __fadd_rn(z4.z, dz), __fadd_rn(z4.w, dw));
}
__device__ __forceinline__ float st_step1(float e, float z, double& sse) {
  const float d = __fsub_rn(e, z);
  sse += (double)d * d;
  return __fadd_rn(z, d);
}

// this lane's partial of ||row||^2 (the caller adds the lanes with its xor-shuffle tree).  DT elements known at compile
// time (rows staged in shared memory), or D elements read through the read-only path.
template <int DT, typename T>
__device__ __forceinline__ float sq_partial(const T* row, int lane) {
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < DT; c += 32) {
    if (c + lane < DT) { const float v = zf(row[c + lane]); s = fmaf(v, v, s); }
  }
  return s;
}
template <typename T>
__device__ __forceinline__ float sq_partial_ldg(const T* __restrict__ row, int D, int lane) {
  float s = 0.f;
  for (int c = lane; c < D; c += 32) { const float v = zf(__ldg(row + c)); s = fmaf(v, v, s); }
  return s;
}

}  // namespace dvq
