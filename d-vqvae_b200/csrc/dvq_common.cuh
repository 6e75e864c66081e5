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
struct VqWorkspace {
  size_t off_ee;        // float [K]            ||e_k||^2
  size_t off_counters;  // int   [CNT_WORDS]    see CounterSlot
  size_t off_rowlist;   // int   [2][N]         rows the tensor-core filter could not decide + their candidate records
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

// ---- kernels launched by the API layer ---------------------------------------------------
// ee[k] = sum_d E[k,d]^2
int launch_code_norms(const float* E, int K, int D, float* ee, cudaStream_t s);

// Exact FP32 CUDA-core path.  row_list == nullptr: rows [0,N).  Otherwise rows
// row_list[0 .. *n_list) (device-side count), used as the refine stage of the tcgen05 path.
// zbf: z / z_q are bf16 rows (DVQ_Z_BF16), else fp32 — every VQ kernel below computes in fp32 on the upcast rows
int launch_vq_simt(const void* z, const float* E, const float* ee, int64_t N, int K, int D, int train,
                   void* z_q, int64_t* idx, unsigned long long* hist, double* sse,
                   const int* row_list, const int* n_list, int list_stride, bool zbf, cudaStream_t s);

// tcgen05 filter kernel (vq_tc_sm100.cu); supported(K,D) says whether the shape is handled.
bool vq_tc_supported(int64_t N, int K, int D);
void vq_tc_layout_info(int K, int D, int* out8, int zbytes = 4);   // dvq_debug_tc_layout (zbytes: size of a z element)
bool vq_tc_pair_selected(int64_t N, int K, int D);   // CTA-pair (cta_group::2) kernel for this shape?
void vq_tc_pair_layout_info(int64_t N, int K, int D, int* out8, int zbytes = 4);   // dvq_debug_tc_pair_layout
long long vq_tc_image_offset(int k, int d, int K, int D, int pair, long long* image_bytes);   // dvq_debug_tc_image_offset
size_t vq_tc_operand_bytes(int K, int D);
int launch_vq_tc(const void* z, const float* E, const float* ee, int64_t N, int K, int D, int train,
                 void* z_q, int64_t* idx, unsigned long long* hist, double* sse,
                 void* bop, int* counters, int* row_list, int* cand_list, int* zero_ints, int zero_n,
                 bool codebook_cached, bool zbf, cudaStream_t s);

// candidate-restricted exact refine (vq_refine.cu): one warp per listed row
bool vq_refine_supported(int K, int D);
bool vq_refine_codebook_in_smem(int K, int D);
int launch_vq_refine(const void* z, const float* E, const float* ee, int K, int D, int train, void* z_q, int64_t* idx,
                     unsigned long long* hist, double* sse, const RefineList& list, bool zbf, cudaStream_t s);

// code-stationary exact refine (vq_refine_stationary.cu): mask-mode codebooks whose K/32 warps hold e_dim code floats
// per lane in registers
bool vq_refine_stationary_supported(int K, int D);
bool vq_refine_stationary_default(int K, int D);   // the subset the automatic refine choice gives it (measured faster)
int launch_vq_refine_stationary(const void* z, const float* E, const float* ee, int K, int D, int train, void* z_q, int64_t* idx,
                                unsigned long long* hist, double* sse, const RefineList& list, bool zbf, cudaStream_t s);

// binned exact refine (vq_refine_binned.cu): (row, sub-chunk) pairs bucketed by sub-chunk; hands the list to
// launch_vq_refine through counters[CNT_HANDBACK] / [CNT_HANDBACK_OVF] when the pairs do not fit its workspace
long long refine_pair_cap_override();   // dvq_vq_set_refine (dvq_api.cu); 0 = default
size_t vq_refine_binned_bytes(int64_t N);
size_t vq_refine_binned_zero_bytes();
int launch_vq_refine_binned(const void* z, const float* E, const float* ee, int64_t N, int K, int D, int train, void* z_q,
                            int64_t* idx, unsigned long long* hist, double* sse, const RefineList& list, int* counters,
                            void* ws, bool zbf, cudaStream_t s);

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

}  // namespace dvq
