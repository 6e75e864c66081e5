/* dvq.h — C ABI of the B200-native D-VQVAE hot path (libdvq_sm100.so).
 *
 * The reference (florasion/D-VQVAE) is pure Python and has no FFI of its own;
 * its boundary for this path is the Python class surface.  Each entry point
 * below names the reference code it replaces (paths relative to the reference
 * root).  The Python mirror of that surface lives in d-vqvae_b200/dvq/ and
 * binds these symbols with ctypes — see INTEGRATION.md.
 *
 * Conventions
 *  - All data pointers are DEVICE pointers on the current CUDA device unless the
 *    name ends in _host; tensors are row-major and contiguous; fp32 unless said.
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *  - Device entry points only enqueue work on `stream`: no host synchronisation,
 *    no allocation; the caller owns every buffer including the workspace.
 *  - Return value: 0 (DVQ_OK) or a negative DvqStatus; a human-readable message
 *    for the last failure on the calling thread is at dvq_last_error().
 *  - There is no CPU fallback: on a machine without an sm_100 device the compute
 *    entry points return DVQ_ERR_UNSUPPORTED_ARCH / DVQ_ERR_CUDA.
 */
#ifndef DVQ_H_
#define DVQ_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DVQ_ABI_VERSION 1

#if defined(__GNUC__)
#define DVQ_API __attribute__((visibility("default")))
#else
#define DVQ_API
#endif

typedef enum DvqStatus {
  DVQ_OK = 0,
  DVQ_ERR_BAD_SHAPE = -1,
  DVQ_ERR_BAD_ALIGN = -2,
  DVQ_ERR_UNSUPPORTED_ARCH = -3,
  DVQ_ERR_WORKSPACE = -4,
  DVQ_ERR_CUDA = -5,
  DVQ_ERR_NCCL = -6,
  DVQ_ERR_BAD_ARG = -7
} DvqStatus;

/* flags for dvq_vq_forward / dvq_vq_workspace_bytes */
#define DVQ_TRAIN 0x1         /* istrain=True: z_q = fl(z + fl(e - z)), accumulate hist + sse   */
#define DVQ_WRITE_ONEHOT 0x2  /* also materialise min_encodings [N,K] fp32                      */
#define DVQ_PATH_AUTO 0x00    /* tensor-core filter + exact refine when the shape allows        */
#define DVQ_PATH_SIMT 0x10    /* force the all-FP32 CUDA-core kernel                            */
#define DVQ_PATH_TC 0x20      /* force the tcgen05 kernel (error if the shape is unsupported)   */
#define DVQ_PATH_MASK 0x30
#define DVQ_CODEBOOK_CACHED 0x200 /* dvq_vq_forward: the caller vouches that `workspace` still holds the codebook
                                   * preparation (code norms, FP16 operand image, scale / residual bounds) of a previous
                                   * call with the SAME E contents, N, K, D, flags & DVQ_PATH_MASK and workspace — it is
                                   * reused instead of rebuilt (three small launches fewer per call) */
#define DVQ_HOST_COPY_ONLY 0x100 /* dvq_vq_forward_host only: run the chunk pipeline's H2D / D2H copies without the
                                    kernels (outputs are undefined) - the copy-only ceiling of the host-buffer path */
#define DVQ_Z_BF16 0x400      /* dvq_vq_forward / _workspace_bytes / _read_counters, dvq_vq_backward_ex, dvq_vq_code_sums_ex,
                               * dvq_debug_tc_layout_ex: the `z` / `z_q` (and `g_zq` / `dz`) pointers are reinterpreted as
                               * bf16 rows (2-byte alignment; the tcgen05 path needs 16 bytes as in fp32).  The call is the fp32
                               * call on the upcast rows: same indices, histogram and SSE; z_q is its result rounded to
                               * nearest-even bf16.  The codebook stays fp32.  Not accepted by dvq_vq_forward_host. */

DVQ_API int dvq_abi_version(void);
DVQ_API const char* dvq_last_error(void);

/* Instrumentation for bench.py: number of kernels this library has launched in the process, and
 * (when enabled) CUDA-event times of the stages of the calling thread's dvq_vq_forward calls,
 * averaged over the calls since dvq_profile_enable(1) (at most 128 are kept):
 * ms[0] code norms, ms[1] main kernel (tcgen05 filter or FP32 kernel), ms[2] FP32 refine,
 * ms[3] one-hot; count[i] = calls averaged.  Events are recorded on the launching stream;
 * dvq_profile_mean synchronises on them. */
DVQ_API long long dvq_launch_count(void);
DVQ_API int dvq_profile_enable(int on);
DVQ_API int dvq_profile_mean(float* ms, int* count, int n);

/* Test / measurement hook for the exact refine stage of the tcgen05 path (all variants give identical
 * results): mode 0 = automatic (the code-stationary kernel on the mask-mode codebooks that fit in registers
 * where it is the faster one, else the per-row kernel while the FP32 codebook fits its shared memory, binned
 * kernels otherwise), 1 = per-row kernel only, 2 = binned kernels, 3 = code-stationary kernel
 * (dvq_vq_forward fails with DVQ_ERR_BAD_SHAPE on a shape it does not cover); pair_cap > 0 overrides the capacity
 * of the binned (row, sub-chunk) pair list (default 2 N) so that tests can exercise the device-side
 * hand-back to the per-row kernel, <= 0 restores the default.  Process-wide. */
DVQ_API int dvq_vq_set_refine(int mode, long long pair_cap);

/* Diagnostic (host-only, no GPU needed): the shared-memory plan the tcgen05 VQ kernel would use for a codebook
 * shape.  out8 = { handled by the tensor-core path (0/1), e_dim slice width, slices per row, A images (1-2),
 * operand ring slots (2-4), z staging slots (1-2), dynamic shared memory in bytes, histogram kept in shared
 * memory (0/1) }.  Used by tests/test_cabi_symbols.py to pin the per-shape choices. */
DVQ_API int dvq_debug_tc_layout(int K, int D, int* out8);

/* Diagnostic (host-only): streamed codebooks (the operand image does not fit shared memory) with e_dim 512, or e_dim
 * 128 / 256 from K = 2048 on, run on CTA pairs (clusters of two CTAs, tcgen05 cta_group::2: one M = 256 MMA over both
 * SMs' row tiles, each CTA streaming half of every operand block).  out8 = { pair kernel selected for (N, K, D) (0/1;
 * honours DVQ_TC_PAIR=0/1), e_dim slice width, slices per row, A images, ring slots (2-8), z staging slots, dynamic
 * shared memory in bytes, codes per ring slot (128) } of the pair kernel's plan. */
DVQ_API int dvq_debug_tc_pair_layout(long long N, int K, int D, int* out8);

/* Diagnostic (host-only): the plan of the tcgen05 kernel variant dvq_vq_forward would launch for (N, K, D, flags) (flags:
 * DVQ_Z_BF16 or 0; other bits are ignored).  When the CTA-pair kernel is selected, out8 is filled as by
 * dvq_debug_tc_pair_layout, otherwise as by dvq_debug_tc_layout — with flags = 0 exactly their output — with the plan
 * of the z element type: the dynamic shared memory out8[6] includes the z staging slots of 128 rows x (slice width)
 * x (4 bytes fp32 / 2 bytes bf16) each. */
DVQ_API int dvq_debug_tc_layout_ex(long long N, int K, int D, int flags, int* out8);

/* Diagnostic (host-only): byte offset of element (code k, column d) of the FP16 operand image the tcgen05 VQ kernel keeps in
 * its workspace — d in [0, D) the scaled code, d in [D, D + 16) the fold columns — for the single-CTA layout (pair = 0: blocks
 * of 256 codes) or the CTA-pair layout (pair = 1: half blocks of 128-code capacity, lower / upper half of a chunk's codes),
 * and the image size in *image_bytes (may be NULL).  -1 for an unsupported shape or an index out of range. */
DVQ_API long long dvq_debug_tc_image_offset(int k, int d, int K, int D, int pair, long long* image_bytes);

/* Diagnostic used by tests/test_tc_probe_gpu.py: run `ksteps` tcgen05.mma (M=128, N=n_cols,
 * kind::f16) on caller-built shared-memory operand images and dump the [128,n_cols] fp32
 * accumulator.  strides = {a_lbo, a_sbo, a_kstep, b_lbo, b_sbo, b_kstep} in bytes; *err (device
 * int) is set non-zero if the MMA never signalled completion (bounded wait, no hang). */
DVQ_API int dvq_debug_umma(const void* a_img, uint32_t a_bytes, const void* b_img, uint32_t b_bytes, int ksteps,
                           const uint32_t* strides, uint32_t idesc, int n_cols, float* out, int* err, void* stream);

/* Device probe: SM count and compute capability of the current device. */
DVQ_API int dvq_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- VectorQuantizer.forward — network/vqvae/quantizer.py:30-67 -------------------------
 * d = fl(fl(sum z^2 + sum e^2) - 2 z.e) (:36-38), idx = first argmin (:39), z_q = E[idx]
 * (:43/:53) or z + (z_q - z) (:60); the N x K distance matrix is never materialised.
 *   z [N,D], E [K,D]  ->  z_q [N,D], idx [N] int64 (== the reference's [N,1]),
 *   onehot [N,K] or NULL (:40-42), hist [K] += code usage, sse [1] += sum (e-z)^2.
 * hist/sse must be zeroed by the caller before the first shard and are only touched
 * under DVQ_TRAIN (they may be NULL otherwise).  Splitting forward from finalize lets a
 * multi-GPU caller all-reduce (hist, sse) in between (dvq_allreduce_stats). */
DVQ_API int dvq_vq_workspace_bytes(int64_t N, int K, int D, int flags, size_t* bytes);
DVQ_API int dvq_vq_forward(const float* z, const float* E, int64_t N, int K, int D, int flags,
                   float* z_q, int64_t* idx, float* onehot,
                   unsigned long long* hist, double* sse,
                   void* workspace, size_t workspace_bytes, void* stream);

/* Diagnostics of the last dvq_vq_forward that used `workspace` (synchronous device->host read):
 * out[0] = rows the tensor-core filter sent to the exact FP32 kernel, out[1] = pipeline protocol
 * error code of the tcgen05 kernel (0 = none), out[2..3] reserved.  Zeros on the FP32-only path. */
DVQ_API int dvq_vq_read_counters(const void* workspace, int64_t N, int K, int D, int flags, int* out4);

/* loss = al*mean((z_q-z)^2) + beta*mean((z_q-z)^2) (quantizer.py:56-57),
 * perplexity = exp(-sum p log(p+1e-10)), p = hist/N_total (:63-64).  N_total == 0 means "use the
 * histogram total" (every row is counted once), which spares a row-sharded caller a second collective. */
DVQ_API int dvq_vq_finalize(const unsigned long long* hist, const double* sse, int64_t N_total, int K, int D,
                    float al, float beta, float* loss, float* perplexity, void* stream);

/* Backward of the forward above — the autograd graph of quantizer.py:56-60 (loss = al*mean((sg[z_q]-z)^2) +
 * beta*mean((z_q-sg[z])^2), z_q_out = z + sg[z_q - z]):
 *   dz[n,:]       = g_zq[n,:] + g_loss * al   * 2/(rows*D) * (z[n,:] - E[idx[n],:])     (dz may be NULL)
 *   dE[idx[n],:] +=             g_loss * beta * 2/(rows*D) * (E[idx[n],:] - z[n,:])     (dE may be NULL; zero it first)
 * g_loss [1] and rows [1] are DEVICE floats (rows = number of rows the loss was averaged over: N, or the
 * all-reduced histogram total on a row-sharded run); g_zq may be NULL (no gradient reaches z_q).  D % 4 == 0. */
DVQ_API int dvq_vq_backward(const float* z, const float* E, const int64_t* idx, const float* g_zq, const float* g_loss,
                    const float* rows, int64_t N, int K, int D, float al, float beta, float* dz, float* dE, void* stream);
/* The same with flags: DVQ_Z_BF16 = z, g_zq and dz are bf16 rows (8-byte aligned; E and dE stay fp32, 16-byte aligned).
 * The formulas are evaluated in fp32 on the upcast values and dz is rounded to bf16 once.  flags = 0 is dvq_vq_backward. */
DVQ_API int dvq_vq_backward_ex(const float* z, const float* E, const int64_t* idx, const float* g_zq, const float* g_loss,
                               const float* rows, int64_t N, int K, int D, float al, float beta, int flags, float* dz, float* dE,
                               void* stream);

/* sums[k,:] += sum of the rows z[n,:] with idx[n] == k — the per-code input sums of an EMA codebook update
 * (together with the usage histogram of dvq_vq_forward).  sums [K,D] must be zeroed by the caller.  D % 4 == 0. */
DVQ_API int dvq_vq_code_sums(const float* z, const int64_t* idx, int64_t N, int K, int D, float* sums, void* stream);
/* The same with flags: DVQ_Z_BF16 = z is bf16 rows (8-byte aligned), summed in fp32.  flags = 0 is dvq_vq_code_sums. */
DVQ_API int dvq_vq_code_sums_ex(const float* z, const int64_t* idx, int64_t N, int K, int D, int flags, float* sums, void* stream);

/* VectorQuantizer.get_emb — quantizer.py:68-75 (batched meaning: out[n,:] = E[idx[n],:]).
 * Out-of-range indices set *oob (device int, may be NULL) and write zeros. */
DVQ_API int dvq_gather(const float* E, const int64_t* idx, int64_t N, int K, int D, float* out, int* oob, void* stream);

/* Grouped get_emb for the six part codebooks of GenNet.gen (gen_net.py:101-106) in ONE launch:
 * out[n, g*D .. g*D+D) = E[g][codes[n*G + g], :], row pitch out_stride floats (the concatenated decoder input, :109).
 * E: host array of G <= 8 device pointers to [K,D] codebooks.  Out-of-range codes set *oob and write zeros. */
DVQ_API int dvq_gather_multi(const float* const* E, int G, const int64_t* codes, int64_t N, int K, int D, float* out,
                     int64_t out_stride, int* oob, void* stream);

/* min_encodings — quantizer.py:40-42: out[n,k] = (k == idx[n]) as fp32, every element written
 * once (no memset + scatter).  Separate entry so the [N,K] matrix can be produced on demand. */
DVQ_API int dvq_onehot(const int64_t* idx, int64_t N, int K, float* out, void* stream);

/* ---- GatedPixelCNN prior: tcgen05 GEMM with fused epilogues (network/pixelcnn/models.py:65-88,176-197) ----------
 * C[m,n] = sum_s A_s[m + 128*tile_shift_s, :] . W_s[:, n], FP16 operands, FP32 accumulation.  Activations are FP16
 * operand images: rows in tiles of 128, a tile stored [K/8][128][8 halfs]; weights are images [n/256][K/8][256][8].
 * A grid row's rows are ordered column-major (m = column * B + b), so a convolution tap is a K-segment with a
 * whole-tile shift; a segment is skipped for tiles whose grid column + col_shift falls outside [0, ncols_src).
 * mode 0 GATE: 128 'a' + 128 'b' columns per tile, out = tanh(a + bias + cond_a) * sigmoid(b + bias + cond_b) -> FP16 image
 *   (out_kd = d wide) and, if pre_img, the raw a|b pre-activations (+ bias) -> FP16 image (2 d wide); cond_img: FP16 image
 *   [B, 2 d] of the class-conditional rows (may be NULL); d_gate = d.
 * mode 1 RES: acc + bias (+ res_img if res_in) -> res_img (FP32 image [K/4][128][4]) and out_img (FP16 image).
 * mode 2 RELU: relu(acc + bias) -> out_img.   mode 3 LOGITS: acc + bias -> logits, row-major [m_tiles*128, n_tiles*256].
 * bias holds n_tiles * 256 floats in tile column order.  *err (device int, may be NULL) is set on a pipeline time-out. */
typedef struct DvqPcnnSeg {
  const void* a_img;
  const void* w_img;
  int a_kd, ks, tile_shift, col_shift;
} DvqPcnnSeg;
typedef struct DvqPcnnGemm {
  DvqPcnnSeg seg[12];
  int nseg, m_tiles, n_tiles, tiles_per_col, ncols_src, mode;
  const float* bias;
  const void* cond_img;
  void* out_img;
  void* pre_img;
  float* res_img;
  float* logits;
  int out_kd, res_in, d_gate;
  int* err;
} DvqPcnnGemm;
DVQ_API int dvq_pcnn_gemm(const DvqPcnnGemm* g, void* stream);
/* x[b * x_stride + c] (int64 indices of one grid row, c < W) -> emb rows as FP16 image (and FP32 image if img32),
 * rows m = c * Bp + b, Bp a multiple of 128 (rows b >= B are zero). */
DVQ_API int dvq_pcnn_embed(const int64_t* x, int x_stride, int W, int B, int Bp, const float* emb, int n_emb, int d,
                           void* img16, float* img32, void* stream);
/* table[label[b], :] (FP32 [n_rows, kd]) -> FP16 image [Bp, kd]. */
DVQ_API int dvq_pcnn_rows_to_image(const int64_t* label, int B, int Bp, const float* table, int n_rows, int kd,
                                   void* img16, void* stream);

/* ---- MANO hand layer — the third-party call at network/gen_net.py:116-118
 *      self.rh_mano(betas=recon[:, :10], global_orient=0, hand_pose=recon[:, 10:55], transl=0).vertices
 * (package `mano`, created at gen_diverse_grasp_obman.py:355-360: use_pca=True, num_pca_comps=45, flat_hand_mean=True).
 * Linear blend skinning of MANO_{LEFT,RIGHT}.pkl (778 vertices, 16 joints, 10 shape and 45 pose dimensions); every
 * table is a device pointer to fp32 data in the layout given here, 16-byte aligned. */
typedef struct DvqManoModel {
  const float* v_template;       /* [778*3]        vertex-major xyz                                              */
  const float* shapedirs;        /* [10][778*3]    shape blend directions, one contiguous row per shape parameter */
  const float* posedirs;         /* [135][778*3]   pose blend directions, one row per element of vec(R_1..15 - I) */
  const float* j_regressor;      /* [16][778]                                                                     */
  const float* weights;          /* [778][16]      skinning weights                                               */
  const float* hands_components; /* [ncomps][45]   PCA basis rows (unused when ncomps == 0)                       */
  const float* pose_mean;        /* [48]           added to [global_orient | hand pose]; zeros for flat_hand_mean */
  const int* parents;            /* [16]           kinematic tree; joint 3f+1..3f+3 must form finger f's chain off joint 0 */
  int ncomps;                    /* PCA components in hand_pose (0: hand_pose holds 45 axis-angle values)          */
} DvqManoModel;
/* betas [B,10], global_orient [B,3] or NULL (zeros), hand_pose [B, ncomps ? ncomps : 45], transl [B,3] or NULL
 * -> vertices [B,778,3], joints [B,16,3] (posed joints; NULL to skip). */
DVQ_API int dvq_mano_forward(const DvqManoModel* model, const float* betas, const float* global_orient, const float* hand_pose,
                             const float* transl, int B, float* vertices, float* joints, void* stream);
/* Vector-Jacobian product of dvq_mano_forward with respect to betas, global_orient, hand_pose and transl (the forward is
 * recomputed from the same inputs; transl does not enter it).  grad_vertices [B,778,3] and grad_joints [B,16,3] are the
 * upstream gradients, NULL meaning zero.  Each of grad_betas [B,10], grad_global_orient [B,3],
 * grad_hand_pose [B, ncomps ? ncomps : 45] and grad_transl [B,3] is written when non-NULL.  An ordinary stream launch
 * (no host synchronisation, no allocation; CUDA-graph capturable), deterministic run to run. */
DVQ_API int dvq_mano_backward(const DvqManoModel* model, const float* betas, const float* global_orient, const float* hand_pose,
                              int B, const float* grad_vertices, const float* grad_joints, float* grad_betas,
                              float* grad_global_orient, float* grad_hand_pose, float* grad_transl, void* stream);

/* ---- hand-object nearest-point search (grasp refinement: pytorch3d knn_points(K=1), Meshes.verts_normals_packed and
 * GraspTTA's interior test) — the exact FP32 contract is stated in csrc/contact_exact.cuh.
 * Points are fp32 [B, n, 3], contiguous; item b's src points are searched against item b's trg points only.  Each entry is
 * an ordinary stream launch (no host synchronisation, no allocation; CUDA-graph capturable).  Shapes: B, N1 >= 0, N2 > 0
 * (DVQ_ERR_BAD_SHAPE otherwise), and B * max(N1, N2) * 3 < 2^31, which keeps the kernels' index arithmetic in 32 bits.
 * B = 0 or N1 = 0 launches nothing. */
/* src [B,N1,3], trg [B,N2,3] -> dist [B,N1] (squared distance to the nearest trg point), idx [B,N1] (its index, lowest
 * among exact ties); with trg_normals [B,N2,3] (unit vertex normals) also interior [B,N1] (1 when the offset from the src
 * point to its nearest trg point points along that point's normal), else interior may be NULL. */
DVQ_API int dvq_nn_forward(const float* src, const float* trg, int B, int N1, int N2, const float* trg_normals, float* dist,
                           int64_t* idx, uint8_t* interior, void* stream);
/* Gradient of dist with respect to src and trg, given the forward's idx and the upstream g_dist [B,N1].  g_src [B,N1,3]
 * and g_trg [B,N2,3] are each written when non-NULL.  Deterministic: g_trg sums in ascending src index, no atomics. */
DVQ_API int dvq_nn_backward(const float* src, const float* trg, const int64_t* idx, const float* g_dist, int B, int N1, int N2,
                            float* g_src, float* g_trg, void* stream);
/* Area-weighted unit vertex normals of a triangle mesh: verts [B,V,3], faces [F,3] (int32 ids in [0, V)), vf_offsets [V+1]
 * and vf_faces [vf_offsets[V]] list the faces of each vertex in ascending order, once per occurrence -> normals [B,V,3].
 * Needs V > 0, F >= 0, B * V * 3 < 2^31 and F * 3 < 2^31. */
DVQ_API int dvq_vertex_normals(const float* verts, int B, int V, const int* faces, int F, const int* vf_offsets,
                               const int* vf_faces, float* normals, void* stream);

/* Host-buffer (end-to-end) form of the same forward: z_host/E_host/zq_host/idx_host are
 * HOST pointers (pinned for full overlap).  Rows are streamed through the GPU in chunks on
 * three internal streams (H2D, compute, D2H).  loss/perplexity are host floats (train only). */
typedef struct DvqHostCtx DvqHostCtx;
DVQ_API int dvq_host_ctx_create(int64_t chunk_rows, int K_max, int D_max, DvqHostCtx** ctx);
DVQ_API int dvq_host_ctx_destroy(DvqHostCtx* ctx);
DVQ_API int dvq_vq_forward_host(DvqHostCtx* ctx, const float* z_host, const float* E_host, int64_t N, int K, int D,
                        int flags, float al, float beta, float* zq_host, int64_t* idx_host,
                        float* loss_host, float* perplexity_host);

/* ---- PointNetEncoder.forward — network/pointnet_encoder.py:140-169 (+STN3d :27-45) ------
 * Eval mode, global_feat=True, feature_transform=False.  BatchNorm is folded into the
 * preceding conv/linear by the caller: W' = W*g/sqrt(var+eps), b' = (b-mean)*g/sqrt(var+eps)+beta.
 *   x [B,C,P] (C = 3 or 4)  ->  feat [B,1024], trans [B,3,3]. */
typedef struct DvqPointNetWeights {
  const float *stn_w1, *stn_b1;       /* [64,C],   [64]   conv1+bn1 (ReLU)   :29 */
  const float *stn_w2, *stn_b2;       /* [128,64], [128]  conv2+bn2 (ReLU)   :30 */
  const float *stn_w3, *stn_b3;       /* [1024,128],[1024] conv3+bn3 (ReLU)  :31 */
  const float *stn_fc1_w, *stn_fc1_b; /* [512,1024],[512] fc1+bn4 (ReLU)     :35 */
  const float *stn_fc2_w, *stn_fc2_b; /* [256,512],[256]  fc2+bn5 (ReLU)     :36 */
  const float *stn_fc3_w, *stn_fc3_b; /* [9,256], [9]     fc3; +I by kernel  :37-43 */
  const float *w1, *b1;               /* [64,C]    conv1+bn1 (ReLU)          :150 */
  const float *w2, *b2;               /* [128,64]  conv2+bn2 (ReLU)          :161 */
  const float *w3, *b3;               /* [1024,128] conv3+bn3 (no ReLU)      :162 */
} DvqPointNetWeights;
DVQ_API int dvq_pointnet_workspace_bytes(int B, int C, int P, size_t* bytes);
/* Same forward with a precision choice.  flags = 0: all-FP32 CUDA-core kernel (parity reference, 5e-5);
 * DVQ_PN_FP16_TC: the 64->128 and 128->1024 layers on tcgen05 tensor cores with FP16 operands and FP32
 * accumulation (10-bit mantissa, as the TF32 cuDNN convolutions the reference runs on a GPU; 3e-3). */
#define DVQ_PN_FP16_TC 0x1
DVQ_API int dvq_pointnet_workspace_bytes_ex(int B, int C, int P, int flags, size_t* bytes);
DVQ_API int dvq_pointnet_forward_ex(const float* x, const DvqPointNetWeights* w, int B, int C, int P, int flags,
                                    float* feat, float* trans, void* workspace, size_t workspace_bytes, void* stream);
DVQ_API int dvq_pointnet_forward(const float* x, const DvqPointNetWeights* w, int B, int C, int P,
                         float* feat, float* trans, void* workspace, size_t workspace_bytes, void* stream);

/* ---- the one collective of the sharded path (SURVEY §8e) ---------------------------------
 * In-place sum over ranks of hist [K] (uint64) and sse [1] (double) on `nccl_comm`
 * (an ncclComm_t passed as void*), enqueued on `stream`.  libnccl is resolved at run time
 * (dlopen of the already-loaded library); DVQ_ERR_NCCL if it cannot be found. */
DVQ_API int dvq_allreduce_stats(void* nccl_comm, unsigned long long* hist, double* sse, int K, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DVQ_H_ */
