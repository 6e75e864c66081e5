// Hand-object nearest-point search (dvq_nn_forward / dvq_nn_backward / dvq_vertex_normals): batched 1-NN with a
// penetration mask and a deterministic backward, the pytorch3d knn_points(K=1) / Meshes.verts_normals_packed /
// interior test that GraspTTA-style grasp refinement runs every step.  The arithmetic is contact_exact.cuh's contract.
//
// nn_forward_kernel: one CTA per (batch item, tile of NN_TILE src points).  A thread keeps NN_SRC src points in registers
// as packed x / y / z pairs, so one broadcast shared-memory read of a trg point serves NN_SRC distances at three packed
// instructions per two distances.  The item's trg points are staged in shared memory NN_STAGE at a time, each coordinate
// duplicated into both halves of a 64-bit word (the packed operand), the stage padded with NaN points to a multiple of
// NN_BLK.  Argmin bookkeeping: per block of NN_BLK trg points, a 3-input fminf tree (FMNMX3, NaN = missing) gives the
// block minimum, compared once with the running best.  Only when a block improves does the thread recompute the block's
// distances and take the first j holding that value.  Blocks run in ascending j and the comparison is strict, so exact
// ties keep the lowest index.  The epilogue recomputes d and dv for the winner from global memory (the same bits), which
// also gives d(s, t_0) for a row with no distance below +inf, and the interior test when normals are given.
#include "contact_exact.cuh"
#include "dvq_common.cuh"

namespace dvq {
namespace {

constexpr int NN_THREADS = 128;
constexpr int NN_PAIRS = 4;                     // packed src pairs per thread
constexpr int NN_SRC = 2 * NN_PAIRS;            // src points per thread
constexpr int NN_TILE = NN_THREADS * NN_SRC;    // src points per CTA
constexpr int NN_STAGE = 1024;                  // trg points per shared-memory stage (24 KB)
constexpr int NN_BLK = 8;                       // trg points per block minimum

__global__ void __launch_bounds__(NN_THREADS) nn_forward_kernel(const float* __restrict__ src, const float* __restrict__ trg,
                                                                 const float* __restrict__ trg_normals, int N1, int N2, int tiles,
                                                                 float* __restrict__ dist, int64_t* __restrict__ idx,
                                                                 uint8_t* __restrict__ interior) {
  __shared__ __align__(16) uint64_t tx2[NN_STAGE], ty2[NN_STAGE], tz2[NN_STAGE];
  const int b = blockIdx.x / tiles, tile = blockIdx.x - b * tiles, tid = threadIdx.x;
  const float* S = src + (size_t)b * N1 * 3;
  const float* T = trg + (size_t)b * N2 * 3;
  const int i0 = tile * NN_TILE + tid;          // src point p of this thread: i0 + p * NN_THREADS

  uint64_t sx[NN_PAIRS], sy[NN_PAIRS], sz[NN_PAIRS];
#pragma unroll
  for (int q = 0; q < NN_PAIRS; ++q) {
    float c[2][3];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int i = i0 + (2 * q + h) * NN_THREADS;
#pragma unroll
      for (int k = 0; k < 3; ++k) c[h][k] = i < N1 ? __ldg(S + i * 3 + k) : 0.f;
    }
    sx[q] = pack_f32x2(c[0][0], c[1][0]);
    sy[q] = pack_f32x2(c[0][1], c[1][1]);
    sz[q] = pack_f32x2(c[0][2], c[1][2]);
  }
  float best[NN_SRC];
  int bj[NN_SRC];
#pragma unroll
  for (int p = 0; p < NN_SRC; ++p) {
    best[p] = INFINITY;
    bj[p] = 0;
  }

  for (int j0 = 0; j0 < N2; j0 += NN_STAGE) {
    const int n = min(NN_STAGE, N2 - j0), nr = (n + NN_BLK - 1) / NN_BLK * NN_BLK;
    __syncthreads();
    for (int k = tid; k < nr; k += NN_THREADS) {
      float x = __int_as_float(0x7fffffff), y = x, z = x;
      if (k < n) {
        x = __ldg(T + (j0 + k) * 3);
        y = __ldg(T + (j0 + k) * 3 + 1);
        z = __ldg(T + (j0 + k) * 3 + 2);
      }
      tx2[k] = pack_f32x2(x, x);
      ty2[k] = pack_f32x2(y, y);
      tz2[k] = pack_f32x2(z, z);
    }
    __syncthreads();
    for (int k0 = 0; k0 < nr; k0 += NN_BLK) {
      float m[NN_SRC];
#pragma unroll
      for (int kk = 0; kk < NN_BLK; kk += 2) {
        const ulonglong2 X = *reinterpret_cast<const ulonglong2*>(tx2 + k0 + kk);
        const ulonglong2 Y = *reinterpret_cast<const ulonglong2*>(ty2 + k0 + kk);
        const ulonglong2 Z = *reinterpret_cast<const ulonglong2*>(tz2 + k0 + kk);
#pragma unroll
        for (int q = 0; q < NN_PAIRS; ++q) {
          float a0, a1, c0, c1;
          unpack_f32x2(nn_dist2(fsub2(sx[q], X.x), fsub2(sy[q], Y.x), fsub2(sz[q], Z.x)), a0, a1);
          unpack_f32x2(nn_dist2(fsub2(sx[q], X.y), fsub2(sy[q], Y.y), fsub2(sz[q], Z.y)), c0, c1);
          m[2 * q] = kk == 0 ? fminf(a0, c0) : fminf(m[2 * q], fminf(a0, c0));
          m[2 * q + 1] = kk == 0 ? fminf(a1, c1) : fminf(m[2 * q + 1], fminf(a1, c1));
        }
      }
#pragma unroll
      for (int p = 0; p < NN_SRC; ++p) {
        if (m[p] < best[p]) {           // rare after the first blocks: find the first j of the block holding m[p]
          best[p] = m[p];
          float x, y, z, unused;
          if (p & 1) {
            unpack_f32x2(sx[p / 2], unused, x);
            unpack_f32x2(sy[p / 2], unused, y);
            unpack_f32x2(sz[p / 2], unused, z);
          } else {
            unpack_f32x2(sx[p / 2], x, unused);
            unpack_f32x2(sy[p / 2], y, unused);
            unpack_f32x2(sz[p / 2], z, unused);
          }
          for (int kk = 0; kk < NN_BLK; ++kk) {
            float tx, ty, tz;
            unpack_f32x2(tx2[k0 + kk], tx, unused);
            unpack_f32x2(ty2[k0 + kk], ty, unused);
            unpack_f32x2(tz2[k0 + kk], tz, unused);
            if (nn_dist(__fsub_rn(x, tx), __fsub_rn(y, ty), __fsub_rn(z, tz)) == m[p]) {
              bj[p] = j0 + k0 + kk;
              break;
            }
          }
        }
      }
    }
  }

#pragma unroll
  for (int p = 0; p < NN_SRC; ++p) {
    const int i = i0 + p * NN_THREADS;
    if (i >= N1) continue;
    const int j = bj[p];
    const float dx = __fsub_rn(S[i * 3], T[j * 3]), dy = __fsub_rn(S[i * 3 + 1], T[j * 3 + 1]), dz = __fsub_rn(S[i * 3 + 2], T[j * 3 + 2]);
    const size_t o = (size_t)b * N1 + i;
    dist[o] = nn_dist(dx, dy, dz);
    idx[o] = j;
    if (interior) {
      const float* nj = trg_normals + ((size_t)b * N2 + j) * 3;
      interior[o] = nn_interior(dx, dy, dz, nj[0], nj[1], nj[2]);
    }
  }
}

// One warp per batch item.  g_src is elementwise; g_trg is the ascending-i segmented sum: the warp walks its item's src
// points 32 at a time and adds each chunk's terms into the item's g_trg rows with one warp_add_rows pass; the rows are
// negated last.  An idx outside [0, N2) contributes nothing.
constexpr int BW_WARPS = 4;

__global__ void __launch_bounds__(BW_WARPS * 32) nn_backward_kernel(const float* __restrict__ src, const float* __restrict__ trg,
                                                                    const int64_t* __restrict__ idx, const float* __restrict__ g_dist,
                                                                    int B, int N1, int N2, float* __restrict__ g_src,
                                                                    float* __restrict__ g_trg) {
  __shared__ float term[BW_WARPS][3][32];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, b = blockIdx.x * BW_WARPS + w;
  if (b >= B) return;
  const float* S = src + (size_t)b * N1 * 3;
  const float* T = trg + (size_t)b * N2 * 3;
  const int64_t* I = idx + (size_t)b * N1;
  const float* G = g_dist + (size_t)b * N1;
  float* GS = g_src ? g_src + (size_t)b * N1 * 3 : nullptr;
  float* GT = g_trg ? g_trg + (size_t)b * N2 * 3 : nullptr;
  if (GT) warp_zero_rows(GT, N2);
  for (int c0 = 0; c0 < N1; c0 += 32) {
    const int i = c0 + lane;
    const int64_t j64 = i < N1 ? I[i] : -1;
    const bool valid = j64 >= 0 && j64 < N2;
    const int j = (int)j64;
    float t[3] = {0.f, 0.f, 0.f};
    if (valid) {
      const float g2 = __fmul_rn(2.f, G[i]);
#pragma unroll
      for (int k = 0; k < 3; ++k) t[k] = __fmul_rn(g2, __fsub_rn(S[i * 3 + k], T[j * 3 + k]));
    }
    if (GS && i < N1) {
#pragma unroll
      for (int k = 0; k < 3; ++k) GS[i * 3 + k] = t[k];
    }
    if (GT) {
#pragma unroll
      for (int k = 0; k < 3; ++k) term[w][k][lane] = t[k];
      __syncwarp();
      warp_add_rows(GT, valid ? j : -1, term[w], 0);
    }
  }
  if (GT) {
    for (int k = lane; k < N2 * 3; k += 32) GT[k] = -GT[k];
  }
}

// One thread per (b, v): the incident faces through the CSR (vf_offsets [V+1], vf_faces ascending f per vertex, one
// entry per occurrence), n_f recomputed from the face's corners.  A face with a vertex id outside [0, V) is skipped.
__global__ void __launch_bounds__(128) vertex_normals_kernel(const float* __restrict__ verts, int B, int V, const int* __restrict__ faces,
                                                             const int* __restrict__ vf_offsets, const int* __restrict__ vf_faces,
                                                             float* __restrict__ normals) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)B * V) return;
  const int b = (int)(t / V), v = (int)(t - (long long)b * V);
  const float* P = verts + (size_t)b * V * 3;
  float3 acc = make_float3(0.f, 0.f, 0.f);
  for (int e = vf_offsets[v], e1 = vf_offsets[v + 1]; e < e1; ++e) {
    int id[3];
    if (!face_ids(faces, vf_faces[e], V, id)) continue;
    const float3 n = face_normal(make_float3(P[id[0] * 3], P[id[0] * 3 + 1], P[id[0] * 3 + 2]),
                                 make_float3(P[id[1] * 3], P[id[1] * 3 + 1], P[id[1] * 3 + 2]),
                                 make_float3(P[id[2] * 3], P[id[2] * 3 + 1], P[id[2] * 3 + 2]));
    acc = make_float3(__fadd_rn(acc.x, n.x), __fadd_rn(acc.y, n.y), __fadd_rn(acc.z, n.z));
  }
  const float3 r = normalize_eps(acc);
  float* o = normals + (size_t)t * 3;
  o[0] = r.x;
  o[1] = r.y;
  o[2] = r.z;
}

}  // namespace

int launch_nn_forward(const float* src, const float* trg, int B, int N1, int N2, const float* trg_normals, float* dist, int64_t* idx,
                      uint8_t* interior, cudaStream_t s) {
  if (B == 0 || N1 == 0) return DVQ_OK;
  const int tiles = (N1 + NN_TILE - 1) / NN_TILE;
  nn_forward_kernel<<<(unsigned)((long long)B * tiles), NN_THREADS, 0, s>>>(src, trg, trg_normals, N1, N2, tiles, dist, idx,
                                                                           interior);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

int launch_nn_backward(const float* src, const float* trg, const int64_t* idx, const float* g_dist, int B, int N1, int N2,
                       float* g_src, float* g_trg, cudaStream_t s) {
  if (B == 0 || (!g_src && !g_trg)) return DVQ_OK;
  nn_backward_kernel<<<(B + BW_WARPS - 1) / BW_WARPS, BW_WARPS * 32, 0, s>>>(src, trg, idx, g_dist, B, N1, N2, g_src, g_trg);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

int launch_vertex_normals(const float* verts, int B, int V, const int* faces, const int* vf_offsets, const int* vf_faces,
                          float* normals, cudaStream_t s) {
  const long long n = (long long)B * V;
  if (n == 0) return DVQ_OK;
  vertex_normals_kernel<<<(unsigned)((n + 127) / 128), 128, 0, s>>>(verts, B, V, faces, vf_offsets, vf_faces, normals);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

}  // namespace dvq
