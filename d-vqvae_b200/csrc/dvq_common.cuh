// Shared internals of libdvq_sm100.so (not part of the public ABI).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "dvq.h"

namespace dvq {

// thread-local last-error text behind dvq_last_error()
void set_error(const char* fmt, ...);
int fail(int code, const char* fmt, ...);

#define DVQ_CUDA_CHECK(expr)                                                              \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess)                                                                \
      return ::dvq::fail(DVQ_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                         __FILE__, __LINE__);                                             \
  } while (0)

struct DeviceProps {
  int ordinal;  // the current device, 0 <= ordinal < 64
  int sm_count;
  int cc_major;
  int cc_minor;
  int max_smem_optin;
};
int device_props(DeviceProps* out);  // cached per device

// instrumentation (dvq_api.cu)
void count_launch(int n = 1);
void profile_mark(int stage, bool begin, cudaStream_t s);  // no-op unless dvq_profile_enable(1)

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---- workspace layout of dvq_vq_forward (all offsets 256-byte aligned) -------------------
// The areas after the counters exist only when the tcgen05 path may run for the call.
struct VqWorkspace {
  size_t off_ee;        // float [K]            ||e_k||^2
  size_t off_counters;  // int   [CNT_WORDS]    see CounterSlot
  size_t off_rowlist;   // int   [N]            rows the tensor-core filter could not decide (RefineList)
  size_t off_candlist;  // int   [N]            their candidate records
  size_t off_bop;       // operand image of the codebook for the tcgen05 path
  size_t off_binned;    // bin tables + (row, sub-chunk) pair list of the binned refine (vq_refine_binned.cu)
  size_t total;
};
VqWorkspace vq_workspace_layout(int64_t N, int K, int D, int flags);

// ---- the refine list: how the tcgen05 filter (vq_tc_sm100.cu) hands its undecided rows to the exact kernels ----------
// Slots of the int counters in the workspace, reset on every call.
enum CounterSlot {
  CNT_LISTED = 0,         // rows in the refine list: row_list[0 .. n)
  CNT_ERROR = 1,          // pipeline protocol error of the filter kernel (0 = none)
  CNT_OVF = 2,            // list mode: rows in the overflow list, stored downwards from row_list[N - 1]
  CNT_PAIRS = 4,          // binned refine: (row, sub-chunk) pairs
  CNT_HANDBACK = 5,       // binned refine: listed rows handed to the per-row kernel (the pairs did not fit)
  CNT_HANDBACK_OVF = 6,   //   and overflow rows
  CNT_STATS = 8,          // DVQ_TC_STATS builds: 64-bit wait-time accounting from here on
  CNT_WORDS = 64
};

// Candidate record of a listed row (cand_list[i]).  In the filter's hand-off word, CAND_UNDECIDED marks an undecided row
// and the low 31 bits hold the record.  Mask mode (K <= 992): bit g <-> 32-code sub-chunk g held a key inside the row's
// error band.  List mode (larger codebooks, where 31 bits would be too coarse): up to three CAND_ENTRY_BITS-bit entries
// (sub-chunk index + 1, 0 = empty, packed from the low bits, in no particular order); CAND_LIST_OVERFLOW = more than three,
// such a row goes to the overflow list.  Every code: 0 in either mode, CAND_MASK_ALL (a degenerate row) in mask mode,
// CAND_LIST_OVERFLOW in list mode.
constexpr uint32_t CAND_UNDECIDED = 0x80000000u;
constexpr uint32_t CAND_MASK_ALL = 0x7fffffffu;
constexpr uint32_t CAND_LIST_OVERFLOW = 0x3fffffffu;
constexpr int CAND_ENTRY_BITS = 10;
__host__ __device__ inline bool cand_list_mode(int K) { return K > 31 * 32; }

// sub-chunk of list entry k (0..2) of a record, -1 when empty
__device__ __forceinline__ int cand_entry(uint32_t cand, int k) {
  return (int)((cand >> (CAND_ENTRY_BITS * k)) & ((1u << CAND_ENTRY_BITS) - 1u)) - 1;
}
__device__ __forceinline__ bool cand_is_all(uint32_t cand, bool list_mode) {
  return cand == 0u || cand == (list_mode ? CAND_LIST_OVERFLOW : CAND_MASK_ALL);
}
// the candidate sub-chunks of a record (every one of the nsc sub-chunks when `all`), spread over a group of `gs` lanes
// (gl = lane in the group)
template <typename F>
__device__ __forceinline__ void for_each_candidate(uint32_t cand, bool all, bool list_mode, int nsc, int gl, int gs, F&& f) {
  if (all) {
    for (int b = gl; b < nsc; b += gs) f(b);
  } else if (list_mode) {
    for (int k = gl; k < 3; k += gs) {
      const int e = cand_entry(cand, k);
      if (e >= 0 && e < nsc) f(e);
    }
  } else {
    for (int b = gl; b < 31 && b < nsc; b += gs)
      if ((cand >> b) & 1u) f(b);
  }
}

// The refine list as the exact kernels read it, counts on the device: rows[0 .. *n) with their records cand[0 .. *n), and in
// list mode the overflow rows ovf_last[0], ovf_last[-1], ... ovf_last[-(*n_ovf - 1)] (ovf_last = row_list + N - 1).
struct RefineList {
  const int* rows;
  const int* cand;
  const int* n;
  const int* ovf_last;   // nullptr in mask mode
  const int* n_ovf;      // nullptr in mask mode
  bool list_mode;
};

// ---- one dvq_vq_forward call, as its launchers see it ------------------------------------
// Filled once by dvq_vq_forward after validation; the workspace views are the VqWorkspace areas.
struct VqCall {
  const void* z;                // [N, D] fp32, or bf16 when zbf (DVQ_Z_BF16): every VQ kernel computes in fp32 on the upcast rows
  const float* E;               // [K, D]
  void* z_q;                    // [N, D], the type of z
  int64_t* idx;                 // [N]
  unsigned long long* hist;     // [K]   train only
  double* sse;                  //       train only
  int64_t N;
  int K, D, train;
  bool zbf;
  cudaStream_t s;
  int sm_count;                 // of the current device
  float* ee;
  int* counters;
  int* row_list;
  int* cand_list;
  void* bop;
  void* binned;
};

// f(z, z_q) with z / z_q typed as the call's element type: const float* / float*, or the __nv_bfloat16 pair
template <typename F>
int with_z_type(const VqCall& c, F&& f) {
  if (c.zbf) return f(static_cast<const __nv_bfloat16*>(c.z), static_cast<__nv_bfloat16*>(c.z_q));
  return f(static_cast<const float*>(c.z), static_cast<float*>(c.z_q));
}

// ---- kernels launched by the API layer ---------------------------------------------------
// ee[k] = sum_d E[k,d]^2
int launch_code_norms(const float* E, int K, int D, float* ee, cudaStream_t s);

// Exact FP32 CUDA-core path over rows [0, N): every shape, the path when the tcgen05 kernel does not run.
int launch_vq_simt(const VqCall& c);

// tcgen05 filter kernel (vq_tc_sm100.cu, whose plan_vq_tc makes every decision below); supported(N,K,D) says whether the shape is handled.
bool vq_tc_supported(int64_t N, int K, int D);
size_t vq_tc_operand_bytes(int K, int D);
// dvq_debug_tc_layout (kernel 0), _pair_layout (1), _layout_ex (-1); zbytes: size of a z element
void vq_tc_plan_info(int64_t N, int K, int D, int zbytes, int kernel, int* out8);
long long vq_tc_image_offset(int k, int d, int K, int D, int pair, long long* image_bytes);   // dvq_debug_tc_image_offset
// z, E and z_q 16-byte aligned
int launch_vq_tc(const VqCall& c, bool codebook_cached);
// DVQ_TC_STATS_PRINT: prints the filter's wait-time sums and pipeline timeline, which DVQ_TC_STATS builds record
int vq_tc_print_stats(const int* counters, const int* row_list, int64_t N);

// The exact refine stage of the tcgen05 path (vq_refine.cu): re-evaluates the rows of the filter's refine list with the
// refine kernels its plan picks for the shape.  mode and pair_cap as in dvq_vq_set_refine (0 = automatic / default).
int launch_vq_refine_stage(const VqCall& c, int mode, long long pair_cap);

// code-stationary exact refine (vq_refine_stationary.cu): mask-mode codebooks whose K/32 warps hold e_dim code floats
// per lane in registers
bool vq_refine_stationary_supported(int K, int D);
int launch_vq_refine_stationary(const VqCall& c, const RefineList& list);

// binned exact refine (vq_refine_binned.cu): (row, sub-chunk) pairs bucketed by sub-chunk; hands the list to the per-row
// kernel through counters[CNT_HANDBACK] / [CNT_HANDBACK_OVF] when the pairs do not fit min(pair_cap, 2 N) (pair_cap 0:
// 2 N, the workspace's capacity)
size_t vq_refine_binned_bytes(int64_t N);
size_t vq_refine_binned_zero_bytes();
int launch_vq_refine_binned(const VqCall& c, const RefineList& list, long long pair_cap);

int launch_onehot(const int64_t* idx, int64_t N, int K, float* onehot, cudaStream_t s);
int launch_finalize(const unsigned long long* hist, const double* sse, int64_t N, int K, int D, float al,
                    float beta, float* loss, float* ppl, cudaStream_t s);
int launch_vq_backward(const void* z, const float* E, const int64_t* idx, const void* g_zq, const float* g_loss,
                       const float* rows, int64_t N, int D, float al, float beta, void* dz, float* dE, bool zbf, cudaStream_t s);
int launch_gather_multi(const float* const* E, int G, const int64_t* codes, int64_t N, int K, int D, float* out, int64_t out_stride,
                        int* oob, cudaStream_t s);
int launch_vq_code_sums(const void* z, const int64_t* idx, int64_t N, int D, float* sums, bool zbf, cudaStream_t s);
int launch_gather(const float* E, const int64_t* idx, int64_t N, int K, int D, float* out, int* oob,
                  cudaStream_t s);

int launch_umma_probe(const void* a_img, uint32_t a_bytes, const void* b_img, uint32_t b_bytes, int ksteps,
                      const uint32_t* strides, uint32_t idesc, int n_cols, float* out, int* err, cudaStream_t s);

// GatedPixelCNN sampler (pcnn_sm100.cu)
int launch_pcnn_gemm(const DvqPcnnGemm* g, cudaStream_t s);
int launch_pcnn_embed(const int64_t* x, int x_stride, int W, int B, int Bp, const float* emb, int n_emb, int d, void* img16,
                      float* img32, cudaStream_t s);
int launch_pcnn_rows_to_image(const int64_t* label, int B, int Bp, const float* table, int n_rows, int kd, void* img16, cudaStream_t s);

// MANO hand layer (mano_sm100.cu)
int launch_mano(const DvqManoModel* m, const float* betas, const float* global_orient, const float* hand_pose, const float* transl, int B,
                float* vertices, float* joints, cudaStream_t s);
int launch_mano_backward(const DvqManoModel* m, const float* betas, const float* global_orient, const float* hand_pose, int B,
                         const float* grad_vertices, const float* grad_joints, float* grad_betas, float* grad_global_orient,
                         float* grad_hand_pose, float* grad_transl, cudaStream_t s);

// hand-object nearest-point search (contact_sm100.cu)
int launch_nn_forward(const float* src, const float* trg, int B, int N1, int N2, const float* trg_normals, float* dist, int64_t* idx,
                      uint8_t* interior, cudaStream_t s);
int launch_nn_backward(const float* src, const float* trg, const int64_t* idx, const float* g_dist, int B, int N1, int N2,
                       float* g_src, float* g_trg, cudaStream_t s);
int launch_vertex_normals(const float* verts, int B, int V, const int* faces, const int* vf_offsets, const int* vf_faces,
                          float* normals, cudaStream_t s);

// ---- one mesh query call (mesh_sm100.cu), as its launchers and kernels see it -------------
// Filled by check_mesh_shape.  Mesh batch Bm and query batch Bp are each 1 or B: item b's mesh is verts[Bm == 1 ? 0 : b],
// its queries pts[Bp == 1 ? 0 : b] (an object's voxel list shared by every hand, or every hand's vertices against one
// object).
struct MeshQuery {
  const float* verts;   // [Bm, V, 3]
  int Bm, V;
  const int* faces;     // [F, 3]
  int F;
  const float* pts;     // [Bp, Q, 3]
  int Bp, Q;
  int B;                // the broadcast batch
  __host__ __device__ const float* mesh(int b) const { return verts + (size_t)(Bm == 1 ? 0 : b) * V * 3; }
  __host__ __device__ const float* queries(int b) const { return pts + (size_t)(Bp == 1 ? 0 : b) * Q * 3; }
};

// mesh winding numbers, point-to-mesh distances, penetration and the distance gradient (mesh_sm100.cu)
int launch_mesh_winding(const MeshQuery& m, float* w, int* inside_count, cudaStream_t s);
int launch_mesh_distance(const MeshQuery& m, float* dist2, int64_t* face, cudaStream_t s);
int launch_mesh_penetration(const MeshQuery& m, float* depth2, int64_t* face, cudaStream_t s);
int launch_mesh_distance_backward(const MeshQuery& m, const int64_t* face, const float* g_dist2, float* g_pts, float* g_verts,
                                  cudaStream_t s);

// PointNet
size_t pointnet_workspace_bytes(int B, int C, int P, int flags);
int launch_pointnet(const float* x, const DvqPointNetWeights* w, int B, int C, int P, int flags, float* feat,
                    float* trans, void* ws, size_t ws_bytes, cudaStream_t s);
size_t pointnet_tc_image_bytes();
int launch_pointnet_tc_trunk(const float* x, const float* trans, const float* w1, const float* b1, const float* w2,
                             const float* b2, const float* w3, int B, int C, int P, float* maxbuf, void* images,
                             bool main_trunk, cudaStream_t s);

// ---- small device helpers ----------------------------------------------------------------
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// z rows as fp32 or bf16 (DVQ_Z_BF16).  A bf16 value upcasts exactly (a 16-bit shift), so every kernel runs the fp32
// arithmetic of the fp32 call on the upcast values; stores round to nearest even once.  The 4-element forms need
// 16-byte (fp32) / 8-byte (bf16) alignment.
__device__ __forceinline__ float zf(float v) { return v; }
__device__ __forceinline__ float zf(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float4 bf4_to_f4(uint2 u) {
  return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u), __uint_as_float(u.y << 16),
                     __uint_as_float(u.y & 0xffff0000u));
}
__device__ __forceinline__ uint32_t f2_to_bf2(float lo, float hi) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ uint2 f4_to_bf4(float4 v) { return make_uint2(f2_to_bf2(v.x, v.y), f2_to_bf2(v.z, v.w)); }
__device__ __forceinline__ float4 zld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 zld4(const __nv_bfloat16* p) { return bf4_to_f4(*reinterpret_cast<const uint2*>(p)); }
__device__ __forceinline__ float4 zldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 zldg4(const __nv_bfloat16* p) { return bf4_to_f4(__ldg(reinterpret_cast<const uint2*>(p))); }
__device__ __forceinline__ float4 zldcs4(const float* p) { return __ldcs(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 zldcs4(const __nv_bfloat16* p) { return bf4_to_f4(__ldcs(reinterpret_cast<const uint2*>(p))); }
__device__ __forceinline__ void zst4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void zst4(__nv_bfloat16* p, float4 v) { *reinterpret_cast<uint2*>(p) = f4_to_bf4(v); }
__device__ __forceinline__ void zstcs4(float* p, float4 v) { __stcs(reinterpret_cast<float4*>(p), v); }
__device__ __forceinline__ void zstcs4(__nv_bfloat16* p, float4 v) { __stcs(reinterpret_cast<uint2*>(p), f4_to_bf4(v)); }
__device__ __forceinline__ void zst1(float* p, float v) { *p = v; }
__device__ __forceinline__ void zst1(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

// cp.async global -> shared copies (dst: shared-window address, (uint32_t)__cvta_generic_to_shared(p)): .ca caches in L1,
// .cg only in L2; with src_bytes (16 or 0) the copy reads that many bytes and zero-fills the rest of the 16.  Completion:
// cp_async_commit() closes a group, cp_async_wait<N>() waits until at most N of this thread's groups are pending.
__device__ __forceinline__ void cp_async_ca4(uint32_t dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_ca16(uint32_t dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_cg16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_cg16(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// the vertex ids of face f of faces [F, 3]; false when one of them lies outside [0, V), which skips the face
__device__ __forceinline__ bool face_ids(const int* __restrict__ faces, int f, int V, int (&id)[3]) {
#pragma unroll
  for (int j = 0; j < 3; ++j) id[j] = __ldg(faces + (size_t)f * 3 + j);
  return (unsigned)id[0] < (unsigned)V && (unsigned)id[1] < (unsigned)V && (unsigned)id[2] < (unsigned)V;
}

// Ordered, atomic-free row sums of a warp (the backward kernels' scatter of per-slot terms into [n_rows, 3] rows).  The
// warp owns its item's rows, so there are no races and no atomics: warp_zero_rows zero-fills them, then each
// warp_add_rows pass takes 32 slots, slot l (lane l) adding terms term[0..2][base + l] into row `row` (-1: nothing).
// __match_any_sync groups the slots that share a row and the group's lowest lane adds them in ascending slot order, so
// over passes in ascending base every row's terms are summed in ascending slot order from +0.
__device__ __forceinline__ void warp_zero_rows(float* rows, int n_rows) {
  for (int k = threadIdx.x & 31; k < n_rows * 3; k += 32) rows[k] = 0.f;
  __syncwarp();
}
template <int N>
__device__ __forceinline__ void warp_add_rows(float* rows, int row, const float (&term)[3][N], int base) {
  const unsigned vmask = __ballot_sync(0xffffffffu, row >= 0);
  if (row >= 0) {
    const unsigned peers = __match_any_sync(vmask, row);
    if ((threadIdx.x & 31) == __ffs(peers) - 1) {
      float acc[3] = {rows[(size_t)row * 3], rows[(size_t)row * 3 + 1], rows[(size_t)row * 3 + 2]};
      for (unsigned rest = peers; rest; rest &= rest - 1) {
        const int l = base + __ffs(rest) - 1;
#pragma unroll
        for (int k = 0; k < 3; ++k) acc[k] = __fadd_rn(acc[k], term[k][l]);
      }
#pragma unroll
      for (int k = 0; k < 3; ++k) rows[(size_t)row * 3 + k] = acc[k];
    }
  }
  __syncwarp();
}

}  // namespace dvq
