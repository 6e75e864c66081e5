// Batched mesh queries for grasp scoring (dvq_mesh_winding / dvq_mesh_distance): generalised winding numbers (inside
// tests, voxel volumes) and point-to-mesh distances, on the FP32 SIMT pipe.  The arithmetic is mesh_exact.cuh's contract.
//
// Both kernels share one layout: one CTA per (batch item, tile of MESH_TILE queries).  A thread keeps MESH_Q queries in
// registers as packed x / y / z pairs, so one broadcast shared-memory read of a face's data serves MESH_Q queries and the
// polynomial part of the arithmetic runs as f32x2 instructions (two queries per instruction); sqrtf, atan2f and the
// region selection of the distance run per query.  The item's faces are staged in shared memory MESH_STAGE at a time as
// structure-of-arrays, each value duplicated into both halves of a 64-bit word (the packed operand), with one flag per
// face (skip: a vertex id outside [0, V); triangle; or degenerate: area^2 = 0, taken as three segments).  The flag is the
// same for every thread, so its branch never diverges.
//
// Mesh batch Bm and query batch Bp are each 1 or B: the item's mesh is verts[Bm == 1 ? 0 : b], its queries
// pts[Bp == 1 ? 0 : b] (an object's voxel list shared by every hand, or every hand's vertices against one object).
//
// mesh_winding_kernel first reduces the item's vertex box over the CTA; a query outside it gets w = 0 (the box rule), and
// a CTA none of whose queries lies inside exits before staging a face: that keeps the voxel-volume pass proportional to
// the hand/object overlap rather than to (voxels x hands).  The per-CTA inside count is one integer atomicAdd.
#include "dvq_common.cuh"
#include "mesh_exact.cuh"

namespace dvq {
namespace {

constexpr int MESH_THREADS = 128;
constexpr int MESH_PAIRS = 2;                          // packed query pairs per thread
constexpr int MESH_Q = 2 * MESH_PAIRS;                 // queries per thread
constexpr int MESH_TILE = MESH_THREADS * MESH_Q;       // queries per CTA
constexpr int MESH_STAGE = 256;                        // faces per shared-memory stage
constexpr int MESH_WARPS = MESH_THREADS / 32;

enum : uint8_t { FACE_SKIP = 0, FACE_TRI = 1, FACE_SEGS = 2 };

__device__ __forceinline__ bool face_ids(const int* __restrict__ faces, int f, int V, int& i0, int& i1, int& i2) {
  i0 = __ldg(faces + (size_t)f * 3);
  i1 = __ldg(faces + (size_t)f * 3 + 1);
  i2 = __ldg(faces + (size_t)f * 3 + 2);
  return (unsigned)i0 < (unsigned)V && (unsigned)i1 < (unsigned)V && (unsigned)i2 < (unsigned)V;
}

// The CTA's queries: thread tid holds i0 + p * MESH_THREADS, p < MESH_Q, as packed pairs (2q, 2q + 1); past Q -> 0.
__device__ __forceinline__ void load_queries(const float* __restrict__ S, int Q, int i0, float (&c)[MESH_Q][3], uint64_t (&qx)[MESH_PAIRS],
                                             uint64_t (&qy)[MESH_PAIRS], uint64_t (&qz)[MESH_PAIRS]) {
#pragma unroll
  for (int p = 0; p < MESH_Q; ++p) {
    const int i = i0 + p * MESH_THREADS;
#pragma unroll
    for (int k = 0; k < 3; ++k) c[p][k] = i < Q ? __ldg(S + (size_t)i * 3 + k) : 0.f;
  }
#pragma unroll
  for (int q = 0; q < MESH_PAIRS; ++q) {
    qx[q] = pack_f32x2(c[2 * q][0], c[2 * q + 1][0]);
    qy[q] = pack_f32x2(c[2 * q][1], c[2 * q + 1][1]);
    qz[q] = pack_f32x2(c[2 * q][2], c[2 * q + 1][2]);
  }
}

// Per-axis min / max of P [V, 3] over the CTA, NaN coordinates ignored; box[0..2] = lo, box[3..5] = hi.
__device__ void mesh_box(const float* __restrict__ P, int V, float* box, float (*red)[6]) {
  float b[6] = {INFINITY, INFINITY, INFINITY, -INFINITY, -INFINITY, -INFINITY};
  for (int v = threadIdx.x; v < V; v += MESH_THREADS) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float x = __ldg(P + (size_t)v * 3 + k);
      b[k] = fminf(b[k], x);
      b[k + 3] = fmaxf(b[k + 3], x);
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      b[k] = fminf(b[k], __shfl_xor_sync(0xffffffffu, b[k], o));
      b[k + 3] = fmaxf(b[k + 3], __shfl_xor_sync(0xffffffffu, b[k + 3], o));
    }
  }
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int k = 0; k < 6; ++k) red[w][k] = b[k];
  }
  __syncthreads();
  if (threadIdx.x < 6) {
    const int k = threadIdx.x;
    float r = red[0][k];
    for (int j = 1; j < MESH_WARPS; ++j) r = k < 3 ? fminf(r, red[j][k]) : fmaxf(r, red[j][k]);
    box[k] = r;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(MESH_THREADS) mesh_winding_kernel(const float* __restrict__ verts, int Bm, int V,
                                                                     const int* __restrict__ faces, int F, const float* __restrict__ pts,
                                                                     int Bp, int Q, int tiles, float* __restrict__ w,
                                                                     int* __restrict__ inside_count) {
  __shared__ __align__(16) uint64_t sv[9][MESH_STAGE];     // corners v0 x y z, v1 x y z, v2 x y z (18 KB)
  __shared__ uint8_t sflag[MESH_STAGE];
  __shared__ float red[MESH_WARPS][6];
  __shared__ float box[6];
  const int b = blockIdx.x / tiles, tile = blockIdx.x - b * tiles, tid = threadIdx.x;
  const float* P = verts + (size_t)(Bm == 1 ? 0 : b) * V * 3;
  const float* S = pts + (size_t)(Bp == 1 ? 0 : b) * Q * 3;
  const int i0 = tile * MESH_TILE + tid;

  mesh_box(P, V, box, red);
  float c[MESH_Q][3];
  uint64_t qx[MESH_PAIRS], qy[MESH_PAIRS], qz[MESH_PAIRS];
  load_queries(S, Q, i0, c, qx, qy, qz);
  bool inbox[MESH_Q], any = false;
#pragma unroll
  for (int p = 0; p < MESH_Q; ++p) {
    inbox[p] = i0 + p * MESH_THREADS < Q && box[0] <= c[p][0] && c[p][0] <= box[3] && box[1] <= c[p][1] && c[p][1] <= box[4] &&
               box[2] <= c[p][2] && c[p][2] <= box[5];
    any |= inbox[p];
  }
  if (!__syncthreads_or(any)) {                 // the whole tile is outside the box: w = 0, nothing inside
    if (w) {
#pragma unroll
      for (int p = 0; p < MESH_Q; ++p) {
        const int i = i0 + p * MESH_THREADS;
        if (i < Q) w[(size_t)b * Q + i] = 0.f;
      }
    }
    return;
  }

  float acc[MESH_Q];
#pragma unroll
  for (int p = 0; p < MESH_Q; ++p) acc[p] = 0.f;
  for (int f0 = 0; f0 < F; f0 += MESH_STAGE) {
    const int n = min(MESH_STAGE, F - f0);
    __syncthreads();
    for (int k = tid; k < n; k += MESH_THREADS) {
      int id[3];
      const bool ok = face_ids(faces, f0 + k, V, id[0], id[1], id[2]);
      sflag[k] = ok ? FACE_TRI : FACE_SKIP;
#pragma unroll
      for (int j = 0; j < 3; ++j) {
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          const float x = ok ? __ldg(P + (size_t)id[j] * 3 + d) : 0.f;
          sv[j * 3 + d][k] = pack_f32x2(x, x);
        }
      }
    }
    __syncthreads();
    for (int k = 0; k < n; ++k) {
      if (sflag[k] == FACE_SKIP) continue;
      uint64_t v[9];
#pragma unroll
      for (int j = 0; j < 9; ++j) v[j] = sv[j][k];
#pragma unroll
      for (int q = 0; q < MESH_PAIRS; ++q) {
        float o0, o1;
        solid_angle2(fsub2(v[0], qx[q]), fsub2(v[1], qy[q]), fsub2(v[2], qz[q]), fsub2(v[3], qx[q]), fsub2(v[4], qy[q]),
                     fsub2(v[5], qz[q]), fsub2(v[6], qx[q]), fsub2(v[7], qy[q]), fsub2(v[8], qz[q]), o0, o1);
        acc[2 * q] = __fadd_rn(acc[2 * q], o0);
        acc[2 * q + 1] = __fadd_rn(acc[2 * q + 1], o1);
      }
    }
  }

  int mine[MESH_Q];
#pragma unroll
  for (int p = 0; p < MESH_Q; ++p) {
    const int i = i0 + p * MESH_THREADS;
    const float wv = inbox[p] ? __fdiv_rn(acc[p], MESH_4PI) : 0.f;
    mine[p] = i < Q && wv >= 0.5f;
    if (w && i < Q) w[(size_t)b * Q + i] = wv;
  }
  if (inside_count) {
    int total = 0;
#pragma unroll
    for (int p = 0; p < MESH_Q; ++p) total += __syncthreads_count(mine[p]);
    if (tid == 0 && total) atomicAdd(inside_count + b, total);
  }
}

__global__ void __launch_bounds__(MESH_THREADS) mesh_distance_kernel(const float* __restrict__ verts, int Bm, int V,
                                                                      const int* __restrict__ faces, int F, const float* __restrict__ pts,
                                                                      int Bp, int Q, int tiles, float* __restrict__ dist2,
                                                                      int64_t* __restrict__ face) {
  __shared__ __align__(16) uint64_t sv[9][MESH_STAGE];     // a x y z, ab x y z, ac x y z (18 KB)
  __shared__ float sd[3][MESH_STAGE];                      // ab . ab, ac . ac, ab . ac
  __shared__ uint8_t sflag[MESH_STAGE];
  const int b = blockIdx.x / tiles, tile = blockIdx.x - b * tiles, tid = threadIdx.x;
  const float* P = verts + (size_t)(Bm == 1 ? 0 : b) * V * 3;
  const float* S = pts + (size_t)(Bp == 1 ? 0 : b) * Q * 3;
  const int i0 = tile * MESH_TILE + tid;

  float c[MESH_Q][3];
  uint64_t qx[MESH_PAIRS], qy[MESH_PAIRS], qz[MESH_PAIRS];
  load_queries(S, Q, i0, c, qx, qy, qz);
  float best[MESH_Q];
  int bf[MESH_Q];
#pragma unroll
  for (int p = 0; p < MESH_Q; ++p) {
    best[p] = INFINITY;
    bf[p] = 0;
  }

  for (int f0 = 0; f0 < F; f0 += MESH_STAGE) {
    const int n = min(MESH_STAGE, F - f0);
    __syncthreads();
    for (int k = tid; k < n; k += MESH_THREADS) {
      int id[3];
      const bool ok = face_ids(faces, f0 + k, V, id[0], id[1], id[2]);
      float a[3] = {0.f, 0.f, 0.f}, e1[3] = {0.f, 0.f, 0.f}, e2[3] = {0.f, 0.f, 0.f};
      if (ok) {
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          a[d] = __ldg(P + (size_t)id[0] * 3 + d);
          e1[d] = __ldg(P + (size_t)id[1] * 3 + d) - a[d];
          e2[d] = __ldg(P + (size_t)id[2] * 3 + d) - a[d];
        }
      }
      sflag[k] = !ok ? FACE_SKIP : (area2(e1, e2) == 0.f ? FACE_SEGS : FACE_TRI);
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        sv[d][k] = pack_f32x2(a[d], a[d]);
        sv[3 + d][k] = pack_f32x2(e1[d], e1[d]);
        sv[6 + d][k] = pack_f32x2(e2[d], e2[d]);
      }
      sd[0][k] = e1[0] * e1[0] + e1[1] * e1[1] + e1[2] * e1[2];
      sd[1][k] = e2[0] * e2[0] + e2[1] * e2[1] + e2[2] * e2[2];
      sd[2][k] = e1[0] * e2[0] + e1[1] * e2[1] + e1[2] * e2[2];
    }
    __syncthreads();
    for (int k = 0; k < n; ++k) {
      const uint8_t flag = sflag[k];
      if (flag == FACE_SKIP) continue;
      uint64_t v[9];
#pragma unroll
      for (int j = 0; j < 9; ++j) v[j] = sv[j][k];
      const float aa = sd[0][k], cc = sd[1][k], bc = sd[2][k];
#pragma unroll
      for (int q = 0; q < MESH_PAIRS; ++q) {
        const uint64_t px = fsub2(qx[q], v[0]), py = fsub2(qy[q], v[1]), pz = fsub2(qz[q], v[2]);
        float d[2];
        if (flag == FACE_TRI) {
          float d1[2], d2[2], vv[2], ww[2];
          unpack_f32x2(dot2(v[3], v[4], v[5], px, py, pz), d1[0], d1[1]);
          unpack_f32x2(dot2(v[6], v[7], v[8], px, py, pz), d2[0], d2[1]);
#pragma unroll
          for (int h = 0; h < 2; ++h) closest_vw(d1[h], d2[h], aa, cc, bc, vv[h], ww[h]);
          const uint64_t nv = pack_f32x2(-vv[0], -vv[1]), nw = pack_f32x2(-ww[0], -ww[1]);
          const uint64_t dx = ffma2(nw, v[6], ffma2(nv, v[3], px)), dy = ffma2(nw, v[7], ffma2(nv, v[4], py)),
                         dz = ffma2(nw, v[8], ffma2(nv, v[5], pz));
          unpack_f32x2(dot2(dx, dy, dz, dx, dy, dz), d[0], d[1]);
        } else {                                           // degenerate: the three edges ab, ac, bc
          float ap[2][3], e1[3], e2[3], unused;
          unpack_f32x2(px, ap[0][0], ap[1][0]);
          unpack_f32x2(py, ap[0][1], ap[1][1]);
          unpack_f32x2(pz, ap[0][2], ap[1][2]);
#pragma unroll
          for (int j = 0; j < 3; ++j) {
            unpack_f32x2(v[3 + j], e1[j], unused);
            unpack_f32x2(v[6 + j], e2[j], unused);
          }
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const float sab = segment_dist2(ap[h][0], ap[h][1], ap[h][2], e1[0], e1[1], e1[2]);
            const float sac = segment_dist2(ap[h][0], ap[h][1], ap[h][2], e2[0], e2[1], e2[2]);
            const float sbc = segment_dist2(ap[h][0] - e1[0], ap[h][1] - e1[1], ap[h][2] - e1[2], e2[0] - e1[0], e2[1] - e1[1],
                                            e2[2] - e1[2]);
            d[h] = fminf(fminf(sab, sac), sbc);
          }
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          if (d[h] < best[2 * q + h]) {                  // strict, ascending f: the lowest f among exact minima; NaN never wins
            best[2 * q + h] = d[h];
            bf[2 * q + h] = f0 + k;
          }
        }
      }
    }
  }

#pragma unroll
  for (int p = 0; p < MESH_Q; ++p) {
    const int i = i0 + p * MESH_THREADS;
    if (i >= Q) continue;
    dist2[(size_t)b * Q + i] = best[p];
    face[(size_t)b * Q + i] = bf[p];
  }
}

}  // namespace

int launch_mesh_winding(const float* verts, int Bm, int V, const int* faces, int F, const float* pts, int Bp, int Q, int B, float* w,
                        int* inside_count, cudaStream_t s) {
  if (B == 0 || Q == 0) return DVQ_OK;
  const int tiles = (Q + MESH_TILE - 1) / MESH_TILE;
  mesh_winding_kernel<<<(unsigned)((long long)B * tiles), MESH_THREADS, 0, s>>>(verts, Bm, V, faces, F, pts, Bp, Q, tiles, w,
                                                                                inside_count);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

int launch_mesh_distance(const float* verts, int Bm, int V, const int* faces, int F, const float* pts, int Bp, int Q, int B,
                         float* dist2, int64_t* face, cudaStream_t s) {
  if (B == 0 || Q == 0) return DVQ_OK;
  const int tiles = (Q + MESH_TILE - 1) / MESH_TILE;
  mesh_distance_kernel<<<(unsigned)((long long)B * tiles), MESH_THREADS, 0, s>>>(verts, Bm, V, faces, F, pts, Bp, Q, tiles, dist2,
                                                                                 face);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

}  // namespace dvq
