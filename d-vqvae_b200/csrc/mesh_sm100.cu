// Batched mesh queries for grasp scoring and refinement (dvq_mesh_winding / dvq_mesh_distance / dvq_mesh_penetration /
// dvq_mesh_distance_backward): generalised winding numbers (inside tests, voxel volumes), point-to-mesh distances, the
// fused penetration query and the gradient of the distance, on the FP32 SIMT pipe.  The arithmetic is mesh_exact.cuh's
// contract.
//
// The forward kernels share one layout: one CTA per (batch item, tile of MESH_TILE queries).  A thread keeps MESH_Q
// queries in registers as packed x / y / z pairs, so one broadcast shared-memory read of a face's data serves MESH_Q
// queries and the polynomial part of the arithmetic runs as f32x2 instructions (two queries per instruction); sqrtf, atan2f
// and the region selection of the distance run per query.  The item's faces are staged in shared memory MESH_STAGE at a
// time as structure-of-arrays, each value duplicated into both halves of a 64-bit word (the packed operand), with one flag
// per face (skip: a vertex id outside [0, V); triangle; or degenerate: area^2 = 0, taken as three segments).  The flag is
// the same for every thread, so its branch never diverges.
//
// The winding phase (winding_phase) first reduces the item's vertex box over the CTA; a query outside it gets w = 0 (the
// box rule), and a CTA none of whose queries lies inside stages no face: that keeps the voxel-volume pass proportional to
// the hand/object overlap rather than to (voxels x hands).  mesh_winding_kernel's per-CTA inside count is one integer
// atomicAdd.
//
// mesh_penetration_kernel runs the winding phase, compacts the CTA's inside queries into a shared-memory list and runs the
// distance sweep over that list only; a CTA with no inside query never stages a face for distances.
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

struct WindingStage {
  uint64_t sv[9][MESH_STAGE];                          // corners v0 x y z, v1 x y z, v2 x y z (18 KB)
  uint8_t sflag[MESH_STAGE];
};

struct DistanceStage {
  uint64_t sv[9][MESH_STAGE];                          // a x y z, ab x y z, ac x y z (18 KB)
  float sd[3][MESH_STAGE];                             // ab . ab, ac . ac, ab . ac
  uint8_t sflag[MESH_STAGE];
};

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

// The box rule for the thread's queries (inbox[p]); returns whether any query of the CTA is inside the box.
__device__ __forceinline__ bool box_rule(const float* __restrict__ P, int V, int Q, int i0, const float (&c)[MESH_Q][3],
                                         bool (&inbox)[MESH_Q], float* box, float (*red)[6]) {
  mesh_box(P, V, box, red);
  bool any = false;
#pragma unroll
  for (int p = 0; p < MESH_Q; ++p) {
    inbox[p] = i0 + p * MESH_THREADS < Q && box[0] <= c[p][0] && c[p][0] <= box[3] && box[1] <= c[p][1] && c[p][1] <= box[4] &&
               box[2] <= c[p][2] && c[p][2] <= box[5];
    any |= inbox[p];
  }
  return __syncthreads_or(any);
}

// S = the sum of Omega_f over ascending f for the thread's MESH_Q queries; every face is staged through st.
__device__ __forceinline__ void winding_sum(const float* __restrict__ P, int V, const int* __restrict__ faces, int F,
                                            const uint64_t (&qx)[MESH_PAIRS], const uint64_t (&qy)[MESH_PAIRS],
                                            const uint64_t (&qz)[MESH_PAIRS], float (&acc)[MESH_Q], WindingStage& st) {
  const int tid = threadIdx.x;
#pragma unroll
  for (int p = 0; p < MESH_Q; ++p) acc[p] = 0.f;
  for (int f0 = 0; f0 < F; f0 += MESH_STAGE) {
    const int n = min(MESH_STAGE, F - f0);
    __syncthreads();
    for (int k = tid; k < n; k += MESH_THREADS) {
      int id[3];
      const bool ok = face_ids(faces, f0 + k, V, id);
      st.sflag[k] = ok ? FACE_TRI : FACE_SKIP;
#pragma unroll
      for (int j = 0; j < 3; ++j) {
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          const float x = ok ? __ldg(P + (size_t)id[j] * 3 + d) : 0.f;
          st.sv[j * 3 + d][k] = pack_f32x2(x, x);
        }
      }
    }
    __syncthreads();
    for (int k = 0; k < n; ++k) {
      if (st.sflag[k] == FACE_SKIP) continue;
      uint64_t v[9];
#pragma unroll
      for (int j = 0; j < 9; ++j) v[j] = st.sv[j][k];
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
}

// The winding phase of the CTA's queries (P, S: the item's mesh and queries): per query of the thread, w = 0 outside the
// item's vertex box, fl(S / fl(4 pi)) inside it; returns box_rule's vote (false: the CTA staged no face).
__device__ __forceinline__ bool winding_phase(const MeshQuery& m, const float* P, const float* S, int i0, float (&w)[MESH_Q],
                                              float* box, float (*red)[6], WindingStage& st) {
  float c[MESH_Q][3];
  uint64_t qx[MESH_PAIRS], qy[MESH_PAIRS], qz[MESH_PAIRS];
  load_queries(S, m.Q, i0, c, qx, qy, qz);
  bool inbox[MESH_Q];
  if (!box_rule(P, m.V, m.Q, i0, c, inbox, box, red)) {
#pragma unroll
    for (int p = 0; p < MESH_Q; ++p) w[p] = 0.f;
    return false;
  }
  float acc[MESH_Q];
  winding_sum(P, m.V, m.faces, m.F, qx, qy, qz, acc, st);
#pragma unroll
  for (int p = 0; p < MESH_Q; ++p) w[p] = inbox[p] ? __fdiv_rn(acc[p], MESH_4PI) : 0.f;
  return true;
}

// Stages faces f0 .. f0 + n - 1 of P for the distance: a, ab, ac packed, the three dot products and the flag.
__device__ __forceinline__ void distance_stage(const float* __restrict__ P, int V, const int* __restrict__ faces, int f0, int n,
                                               DistanceStage& st) {
  for (int k = threadIdx.x; k < n; k += MESH_THREADS) {
    int id[3];
    const bool ok = face_ids(faces, f0 + k, V, id);
    float p[3][3] = {{0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
    if (ok) {
#pragma unroll
      for (int j = 0; j < 3; ++j) {
#pragma unroll
        for (int d = 0; d < 3; ++d) p[j][d] = __ldg(P + (size_t)id[j] * 3 + d);
      }
    }
    float a[3], e1[3], e2[3];
    face_frame(p[0], p[1], p[2], a, e1, e2, st.sd[0][k], st.sd[1][k], st.sd[2][k]);
    st.sflag[k] = !ok ? FACE_SKIP : (area2(e1, e2) == 0.f ? FACE_SEGS : FACE_TRI);
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      st.sv[d][k] = pack_f32x2(a[d], a[d]);
      st.sv[3 + d][k] = pack_f32x2(e1[d], e1[d]);
      st.sv[6 + d][k] = pack_f32x2(e2[d], e2[d]);
    }
  }
}

// dist2 of one staged face (flag != FACE_SKIP) for a packed query pair with offsets (px, py, pz) = fl(q - a)
__device__ __forceinline__ void face_dist2(uint8_t flag, const uint64_t (&v)[9], float aa, float cc, float bc, uint64_t px,
                                           uint64_t py, uint64_t pz, float (&d)[2]) {
  if (flag == FACE_TRI) {
    float vv[2], ww[2];
    uint64_t dx, dy, dz;
    tri_offset2(px, py, pz, v + 3, aa, cc, bc, vv, ww, dx, dy, dz);
    unpack_f32x2(dot2(dx, dy, dz, dx, dy, dz), d[0], d[1]);
  } else {                                           // degenerate: its three segments
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
      float p[3][3], e[3][3], s[3];
      face_segments(ap[h], e1, e2, p, e, s);
      d[h] = fminf(fminf(s[0], s[1]), s[2]);
    }
  }
}

// The distance sweep: best / bf = the smallest dist2 over ascending f and its lowest face for the thread's packed pairs
// q < pairs (pairs is the same for the whole CTA).  Every thread joins the staging barriers; an inactive one skips the
// arithmetic.
__device__ __forceinline__ void distance_sweep(const float* __restrict__ P, int V, const int* __restrict__ faces, int F,
                                               const uint64_t (&qx)[MESH_PAIRS], const uint64_t (&qy)[MESH_PAIRS],
                                               const uint64_t (&qz)[MESH_PAIRS], int pairs, bool active, float (&best)[MESH_Q],
                                               int (&bf)[MESH_Q], DistanceStage& st) {
#pragma unroll
  for (int p = 0; p < MESH_Q; ++p) {
    best[p] = INFINITY;
    bf[p] = 0;
  }
  for (int f0 = 0; f0 < F; f0 += MESH_STAGE) {
    const int n = min(MESH_STAGE, F - f0);
    __syncthreads();
    distance_stage(P, V, faces, f0, n, st);
    __syncthreads();
    if (!active) continue;
    for (int k = 0; k < n; ++k) {
      const uint8_t flag = st.sflag[k];
      if (flag == FACE_SKIP) continue;
      uint64_t v[9];
#pragma unroll
      for (int j = 0; j < 9; ++j) v[j] = st.sv[j][k];
      const float aa = st.sd[0][k], cc = st.sd[1][k], bc = st.sd[2][k];
#pragma unroll
      for (int q = 0; q < MESH_PAIRS; ++q) {
        if (q >= pairs) break;
        float d[2];
        face_dist2(flag, v, aa, cc, bc, fsub2(qx[q], v[0]), fsub2(qy[q], v[1]), fsub2(qz[q], v[2]), d);
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
}

__global__ void __launch_bounds__(MESH_THREADS) mesh_winding_kernel(__grid_constant__ const MeshQuery m, int tiles,
                                                                     float* __restrict__ w, int* __restrict__ inside_count) {
  __shared__ __align__(16) WindingStage st;
  __shared__ float red[MESH_WARPS][6];
  __shared__ float box[6];
  const int b = blockIdx.x / tiles, tile = blockIdx.x - b * tiles, tid = threadIdx.x, Q = m.Q;
  const int i0 = tile * MESH_TILE + tid;

  float wv[MESH_Q];
  if (!winding_phase(m, m.mesh(b), m.queries(b), i0, wv, box, red, st)) {   // the whole tile is outside the box: w = 0
    if (w) {
#pragma unroll
      for (int p = 0; p < MESH_Q; ++p) {
        const int i = i0 + p * MESH_THREADS;
        if (i < Q) w[(size_t)b * Q + i] = 0.f;
      }
    }
    return;
  }
  int mine[MESH_Q];
#pragma unroll
  for (int p = 0; p < MESH_Q; ++p) {
    const int i = i0 + p * MESH_THREADS;
    mine[p] = i < Q && wv[p] >= 0.5f;
    if (w && i < Q) w[(size_t)b * Q + i] = wv[p];
  }
  if (inside_count) {
    int total = 0;
#pragma unroll
    for (int p = 0; p < MESH_Q; ++p) total += __syncthreads_count(mine[p]);
    if (tid == 0 && total) atomicAdd(inside_count + b, total);
  }
}

__global__ void __launch_bounds__(MESH_THREADS) mesh_distance_kernel(__grid_constant__ const MeshQuery m, int tiles,
                                                                      float* __restrict__ dist2, int64_t* __restrict__ face) {
  __shared__ __align__(16) DistanceStage st;
  const int b = blockIdx.x / tiles, tile = blockIdx.x - b * tiles, tid = threadIdx.x, Q = m.Q;
  const int i0 = tile * MESH_TILE + tid;

  float c[MESH_Q][3];
  uint64_t qx[MESH_PAIRS], qy[MESH_PAIRS], qz[MESH_PAIRS];
  load_queries(m.queries(b), Q, i0, c, qx, qy, qz);
  float best[MESH_Q];
  int bf[MESH_Q];
  distance_sweep(m.mesh(b), m.V, m.faces, m.F, qx, qy, qz, MESH_PAIRS, true, best, bf, st);

#pragma unroll
  for (int p = 0; p < MESH_Q; ++p) {
    const int i = i0 + p * MESH_THREADS;
    if (i >= Q) continue;
    dist2[(size_t)b * Q + i] = best[p];
    face[(size_t)b * Q + i] = bf[p];
  }
}

// Phase 1 is the winding phase.  Phase 2 compacts the inside queries, in ascending query order, into slist; list entry j
// is held by thread (j mod 256) / 2 in half j mod 2 of pair j / 256, so n inside queries occupy the first ceil(n / 64)
// warps and one pair per thread while n <= 256.  The distance faces are staged into the same shared memory as the winding
// faces.  The bound of 6 CTAs per SM caps ptxas at 80 registers; without it, ptxas takes 94 (5 CTAs per SM).
__global__ void __launch_bounds__(MESH_THREADS, 6) mesh_penetration_kernel(__grid_constant__ const MeshQuery m, int tiles,
                                                                            float* __restrict__ depth2, int64_t* __restrict__ face) {
  __shared__ __align__(16) union {
    WindingStage w;
    DistanceStage d;
  } st;
  __shared__ float red[MESH_WARPS][6];
  __shared__ float box[6];
  __shared__ float slist[3][MESH_TILE];
  __shared__ int sidx[MESH_TILE];
  __shared__ int wcount[MESH_Q][MESH_WARPS];
  const int b = blockIdx.x / tiles, tile = blockIdx.x - b * tiles, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, Q = m.Q;
  const float* P = m.mesh(b);
  const float* S = m.queries(b);
  const int i0 = tile * MESH_TILE + tid;
  float* D = depth2 + (size_t)b * Q;
  int64_t* FC = face + (size_t)b * Q;

  bool inside[MESH_Q];
  {
    float wv[MESH_Q];
    const bool any = winding_phase(m, P, S, i0, wv, box, red, st.w);
#pragma unroll
    for (int p = 0; p < MESH_Q; ++p) {
      const int i = i0 + p * MESH_THREADS;
      inside[p] = wv[p] >= 0.5f;
      if (i < Q && !inside[p]) {
        D[i] = 0.f;
        FC[i] = -1;
      }
    }
    if (!any) return;                                  // CTA-uniform: box_rule's vote
  }

  unsigned mask[MESH_Q];
#pragma unroll
  for (int p = 0; p < MESH_Q; ++p) {
    mask[p] = __ballot_sync(0xffffffffu, inside[p]);
    if (lane == 0) wcount[p][warp] = __popc(mask[p]);
  }
  __syncthreads();
  int n_in = 0, off[MESH_Q];
#pragma unroll
  for (int p = 0; p < MESH_Q; ++p) {
#pragma unroll
    for (int j = 0; j < MESH_WARPS; ++j) {
      if (j == warp) off[p] = n_in;
      n_in += wcount[p][j];
    }
  }
  if (n_in == 0) return;                               // CTA-uniform
#pragma unroll
  for (int p = 0; p < MESH_Q; ++p) {
    if (inside[p]) {
      const int j = off[p] + __popc(mask[p] & ((1u << lane) - 1u)), i = i0 + p * MESH_THREADS;
#pragma unroll
      for (int k = 0; k < 3; ++k) slist[k][j] = __ldg(S + (size_t)i * 3 + k);
      sidx[j] = i;
    }
  }
  __syncthreads();

  uint64_t qx[MESH_PAIRS], qy[MESH_PAIRS], qz[MESH_PAIRS];
#pragma unroll
  for (int q = 0; q < MESH_PAIRS; ++q) {
    float c[2][3];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int j = q * 2 * MESH_THREADS + 2 * tid + h;
#pragma unroll
      for (int k = 0; k < 3; ++k) c[h][k] = j < n_in ? slist[k][j] : 0.f;
    }
    qx[q] = pack_f32x2(c[0][0], c[1][0]);
    qy[q] = pack_f32x2(c[0][1], c[1][1]);
    qz[q] = pack_f32x2(c[0][2], c[1][2]);
  }
  const int pairs = (n_in + 2 * MESH_THREADS - 1) / (2 * MESH_THREADS);
  const bool active = warp * 64 < n_in;
  float best[MESH_Q];
  int bf[MESH_Q];
  distance_sweep(P, m.V, m.faces, m.F, qx, qy, qz, pairs, active, best, bf, st.d);
#pragma unroll
  for (int p = 0; p < MESH_Q; ++p) {
    const int j = (p >> 1) * 2 * MESH_THREADS + 2 * tid + (p & 1);
    if (j < n_in) {
      const int i = sidx[j];
      D[i] = best[p];
      FC[i] = bf[p];
    }
  }
}

// One warp per broadcast item b, which owns (zero-fills, then accumulates) the item's g_verts rows: no races, no atomics.
// The warp walks the item's queries 32 at a time; each lane recomputes its query's offset at its face (mesh_exact.cuh)
// and writes g_pts.  The chunk's 96 (query, corner) terms go to shared memory in ascending (query, corner) order and are
// added into g_verts by three warp_add_rows passes, so every vertex's terms are summed in ascending (query, corner) order.
constexpr int BW_WARPS = 4;

__global__ void __launch_bounds__(BW_WARPS * 32) mesh_distance_backward_kernel(__grid_constant__ const MeshQuery m,
                                                                               const int64_t* __restrict__ face,
                                                                               const float* __restrict__ g_dist2,
                                                                               float* __restrict__ g_pts, float* __restrict__ g_verts) {
  __shared__ float term[BW_WARPS][3][96];
  __shared__ int tvert[BW_WARPS][96];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, b = blockIdx.x * BW_WARPS + w;
  if (b >= m.B) return;
  const int V = m.V, Q = m.Q;
  const float* P = m.mesh(b);
  const float* S = m.queries(b);
  const int64_t* I = face + (size_t)b * Q;
  const float* G = g_dist2 + (size_t)b * Q;
  float* GP = g_pts ? g_pts + (size_t)b * Q * 3 : nullptr;
  float* GV = g_verts ? g_verts + (size_t)b * V * 3 : nullptr;
  if (GV) warp_zero_rows(GV, V);
  for (int c0 = 0; c0 < Q; c0 += 32) {
    const int i = c0 + lane;
    int id[3] = {-1, -1, -1};
    float lam[3] = {0.f, 0.f, 0.f}, t[3] = {0.f, 0.f, 0.f};
    bool valid = false;
    const int64_t f64 = i < Q ? I[i] : -1;
    if (f64 >= 0 && f64 < m.F && face_ids(m.faces, (int)f64, V, id)) {
      float p[3][3], q[3];
#pragma unroll
      for (int j = 0; j < 3; ++j) {
#pragma unroll
        for (int k = 0; k < 3; ++k) p[j][k] = __ldg(P + (size_t)id[j] * 3 + k);
      }
#pragma unroll
      for (int k = 0; k < 3; ++k) q[k] = __ldg(S + (size_t)i * 3 + k);
      float a[3], e1[3], e2[3], aa, cc, bc, d[3];
      face_frame(p[0], p[1], p[2], a, e1, e2, aa, cc, bc);
      if (area2(e1, e2) != 0.f) {                       // the forward's packed arithmetic, both halves the same query
        uint64_t e[6];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          e[k] = pack_f32x2(e1[k], e1[k]);
          e[3 + k] = pack_f32x2(e2[k], e2[k]);
        }
        float vv[2], ww[2], unused;
        uint64_t dx, dy, dz;
        tri_offset2(fsub2(pack_f32x2(q[0], q[0]), pack_f32x2(a[0], a[0])), fsub2(pack_f32x2(q[1], q[1]), pack_f32x2(a[1], a[1])),
                    fsub2(pack_f32x2(q[2], q[2]), pack_f32x2(a[2], a[2])), e, aa, cc, bc, vv, ww, dx, dy, dz);
        unpack_f32x2(dx, d[0], unused);
        unpack_f32x2(dy, d[1], unused);
        unpack_f32x2(dz, d[2], unused);
        lam[0] = __fsub_rn(__fsub_rn(1.f, vv[0]), ww[0]);
        lam[1] = vv[0];
        lam[2] = ww[0];
      } else {                                          // degenerate: the first segment attaining the forward's minimum
        float ap[3], sp[3][3], se[3][3], s[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) ap[k] = q[k] - a[k];
        face_segments(ap, e1, e2, sp, se, s);
        const float mn = fminf(fminf(s[0], s[1]), s[2]);
        auto take = [&](int k, int c0, int c1) {        // segment k, from corner c0 to corner c1
          const float t = segment_offset(sp[k][0], sp[k][1], sp[k][2], se[k][0], se[k][1], se[k][2], d[0], d[1], d[2]);
          lam[c0] = __fsub_rn(1.f, t);
          lam[c1] = t;
        };
        if (s[0] == mn) {
          take(0, 0, 1);
        } else if (s[1] == mn) {
          take(1, 0, 2);
        } else {
          take(2, 1, 2);
        }
      }
      valid = isfinite(d[0]) && isfinite(d[1]) && isfinite(d[2]);
      if (valid) {
        const float g2 = __fmul_rn(2.f, G[i]);
#pragma unroll
        for (int k = 0; k < 3; ++k) t[k] = __fmul_rn(g2, d[k]);
      }
    }
    if (GP && i < Q) {
#pragma unroll
      for (int k = 0; k < 3; ++k) GP[(size_t)i * 3 + k] = t[k];
    }
    if (GV && __ballot_sync(0xffffffffu, valid)) {     // warp-uniform
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        tvert[w][3 * lane + j] = valid ? id[j] : -1;
#pragma unroll
        for (int k = 0; k < 3; ++k) term[w][k][3 * lane + j] = -__fmul_rn(lam[j], t[k]);
      }
      __syncwarp();
#pragma unroll
      for (int r = 0; r < 3; ++r) warp_add_rows(GV, tvert[w][32 * r + lane], term[w], 32 * r);
    }
  }
}

// One CTA per (batch item, tile of MESH_TILE queries).
template <typename... Out>
int launch_mesh_tiles(void (*kernel)(MeshQuery, int, Out...), const MeshQuery& m, cudaStream_t s, Out... out) {
  if (m.B == 0 || m.Q == 0) return DVQ_OK;
  const int tiles = (m.Q + MESH_TILE - 1) / MESH_TILE;
  kernel<<<(unsigned)((long long)m.B * tiles), MESH_THREADS, 0, s>>>(m, tiles, out...);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

}  // namespace

int launch_mesh_winding(const MeshQuery& m, float* w, int* inside_count, cudaStream_t s) {
  return launch_mesh_tiles(mesh_winding_kernel, m, s, w, inside_count);
}

int launch_mesh_distance(const MeshQuery& m, float* dist2, int64_t* face, cudaStream_t s) {
  return launch_mesh_tiles(mesh_distance_kernel, m, s, dist2, face);
}

int launch_mesh_penetration(const MeshQuery& m, float* depth2, int64_t* face, cudaStream_t s) {
  return launch_mesh_tiles(mesh_penetration_kernel, m, s, depth2, face);
}

int launch_mesh_distance_backward(const MeshQuery& m, const int64_t* face, const float* g_dist2, float* g_pts, float* g_verts,
                                  cudaStream_t s) {
  if (m.B == 0 || (m.Q == 0 && !g_verts)) return DVQ_OK;
  mesh_distance_backward_kernel<<<(m.B + BW_WARPS - 1) / BW_WARPS, BW_WARPS * 32, 0, s>>>(m, face, g_dist2, g_pts, g_verts);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

}  // namespace dvq
