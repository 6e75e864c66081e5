// C-ABI entry points of libdvq_sm100.so (declared in include/dvq.h): argument validation,
// workspace carving, path selection, the host-buffer streaming pipeline and the NCCL hook.
#include <dlfcn.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include "dvq_common.cuh"

namespace dvq {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int device_props(DeviceProps* out) {
  static DeviceProps cache[64];
  static bool have[64] = {};
  int dev = 0;
  DVQ_CUDA_CHECK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return fail(DVQ_ERR_CUDA, "device ordinal %d out of range", dev);
  if (!have[dev]) {
    DeviceProps p;
    DVQ_CUDA_CHECK(cudaDeviceGetAttribute(&p.sm_count, cudaDevAttrMultiProcessorCount, dev));
    DVQ_CUDA_CHECK(cudaDeviceGetAttribute(&p.cc_major, cudaDevAttrComputeCapabilityMajor, dev));
    DVQ_CUDA_CHECK(cudaDeviceGetAttribute(&p.cc_minor, cudaDevAttrComputeCapabilityMinor, dev));
    DVQ_CUDA_CHECK(cudaDeviceGetAttribute(&p.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    cache[dev] = p;
    have[dev] = true;
  }
  *out = cache[dev];
  return DVQ_OK;
}

static long long g_launches = 0;
void count_launch(int n) { __atomic_fetch_add(&g_launches, (long long)n, __ATOMIC_RELAXED); }

static int g_refine_mode = 0;            // dvq_vq_set_refine
static long long g_refine_pair_cap = 0;
long long refine_pair_cap_override() { return __atomic_load_n(&g_refine_pair_cap, __ATOMIC_RELAXED); }

static const int kStages = 4;
static const int kProfSlots = 128;  // event pairs per stage between enable and read-out
static thread_local bool g_prof_on = false;
static thread_local cudaEvent_t g_prof_ev[kStages][kProfSlots][2] = {};
static thread_local int g_prof_n[kStages] = {};

void profile_mark(int stage, bool begin, cudaStream_t s) {
  if (!g_prof_on || stage < 0 || stage >= kStages) return;
  const int slot = g_prof_n[stage];
  if (slot >= kProfSlots) return;
  cudaEvent_t& e = g_prof_ev[stage][slot][begin ? 0 : 1];
  if (!e && cudaEventCreate(&e) != cudaSuccess) return;
  cudaEventRecord(e, s);
  if (!begin) g_prof_n[stage] = slot + 1;
}

static int require_sm100() {
  DeviceProps dp;
  int rc = device_props(&dp);
  if (rc) return rc;
  if (dp.cc_major != 10)
    return fail(DVQ_ERR_UNSUPPORTED_ARCH, "libdvq_sm100 is built for sm_100a only; device is sm_%d%d",
                dp.cc_major, dp.cc_minor);
  return DVQ_OK;
}

VqWorkspace vq_workspace_layout(int64_t N, int K, int D, int flags) {
  VqWorkspace w;
  size_t off = 0;
  w.off_ee = off;
  off = align_up(off + sizeof(float) * (size_t)K, 256);
  w.off_counters = off;
  off = align_up(off + sizeof(int) * CNT_WORDS, 256);
  const bool may_tc = (flags & DVQ_PATH_MASK) != DVQ_PATH_SIMT && vq_tc_supported(N, K, D);
  w.off_rowlist = off;
  if (may_tc) off = align_up(off + 2 * align_up(sizeof(int) * (size_t)N, 256), 256);
  w.off_bop = off;
  if (may_tc) off = align_up(off + vq_tc_operand_bytes(K, D), 1024);
  w.off_binned = off;
  if (may_tc) off = align_up(off + vq_refine_binned_bytes(N), 256);
  w.total = off;
  return w;
}

}  // namespace dvq

using namespace dvq;

extern "C" {

int dvq_abi_version(void) { return DVQ_ABI_VERSION; }

const char* dvq_last_error(void) { return g_err; }

long long dvq_launch_count(void) { return __atomic_load_n(&g_launches, __ATOMIC_RELAXED); }

int dvq_vq_set_refine(int mode, long long pair_cap) {
  if (mode < 0 || mode > 3) return fail(DVQ_ERR_BAD_ARG, "refine mode must be 0 (auto), 1 (per-row), 2 (binned) or 3 (code-stationary)");
  __atomic_store_n(&g_refine_mode, mode, __ATOMIC_RELAXED);
  __atomic_store_n(&g_refine_pair_cap, pair_cap > 0 ? pair_cap : 0, __ATOMIC_RELAXED);
  return DVQ_OK;
}

int dvq_debug_tc_layout(int K, int D, int* out8) {
  if (!out8) return fail(DVQ_ERR_BAD_ARG, "out8 is NULL");
  if (K <= 0 || D <= 0) return fail(DVQ_ERR_BAD_SHAPE, "need K > 0, D > 0");
  vq_tc_layout_info(K, D, out8);
  return DVQ_OK;
}

int dvq_debug_tc_pair_layout(long long N, int K, int D, int* out8) {
  if (!out8) return fail(DVQ_ERR_BAD_ARG, "out8 is NULL");
  if (K <= 0 || D <= 0) return fail(DVQ_ERR_BAD_SHAPE, "need K > 0, D > 0");
  vq_tc_pair_layout_info((int64_t)N, K, D, out8);
  return DVQ_OK;
}

int dvq_debug_tc_layout_ex(long long N, int K, int D, int flags, int* out8) {
  if (!out8) return fail(DVQ_ERR_BAD_ARG, "out8 is NULL");
  if (K <= 0 || D <= 0) return fail(DVQ_ERR_BAD_SHAPE, "need K > 0, D > 0");
  const int zbytes = (flags & DVQ_Z_BF16) ? 2 : 4;
  if (vq_tc_pair_selected((int64_t)N, K, D)) vq_tc_pair_layout_info((int64_t)N, K, D, out8, zbytes);
  else vq_tc_layout_info(K, D, out8, zbytes);
  return DVQ_OK;
}

long long dvq_debug_tc_image_offset(int k, int d, int K, int D, int pair, long long* image_bytes) {
  if (K <= 0 || D <= 0 || k < 0 || k >= K || d < 0 || d >= D + 16 || !vq_tc_supported(1, K, D)) return -1;
  return vq_tc_image_offset(k, d, K, D, pair, image_bytes);
}

int dvq_profile_enable(int on) {
  g_prof_on = on != 0;
  for (int i = 0; i < kStages; ++i) g_prof_n[i] = 0;
  return DVQ_OK;
}

int dvq_profile_mean(float* ms, int* count, int n) {
  if (!ms || n <= 0) return fail(DVQ_ERR_BAD_ARG, "ms is NULL or n <= 0");
  for (int i = 0; i < n; ++i) {
    ms[i] = 0.f;
    if (count) count[i] = 0;
    if (i >= kStages) continue;
    double sum = 0.0;
    for (int j = 0; j < g_prof_n[i]; ++j) {
      float t = 0.f;
      DVQ_CUDA_CHECK(cudaEventSynchronize(g_prof_ev[i][j][1]));
      DVQ_CUDA_CHECK(cudaEventElapsedTime(&t, g_prof_ev[i][j][0], g_prof_ev[i][j][1]));
      sum += t;
    }
    if (g_prof_n[i] > 0) ms[i] = (float)(sum / g_prof_n[i]);
    if (count) count[i] = g_prof_n[i];
  }
  return DVQ_OK;
}

int dvq_device_info(int* sm_count, int* cc_major, int* cc_minor) {
  DeviceProps dp;
  int rc = device_props(&dp);
  if (rc) return rc;
  if (sm_count) *sm_count = dp.sm_count;
  if (cc_major) *cc_major = dp.cc_major;
  if (cc_minor) *cc_minor = dp.cc_minor;
  return DVQ_OK;
}

static int check_vq_shape(int64_t N, int K, int D) {
  if (N < 0 || K <= 0 || D <= 0) return fail(DVQ_ERR_BAD_SHAPE, "need N >= 0, K > 0, D > 0 (got N=%lld K=%d D=%d)", (long long)N, K, D);
  if (N > 2147483647LL - 256) return fail(DVQ_ERR_BAD_SHAPE, "N=%lld exceeds the per-call limit of 2^31-257 rows; shard the call", (long long)N);
  return DVQ_OK;
}

int dvq_vq_workspace_bytes(int64_t N, int K, int D, int flags, size_t* bytes) {
  if (!bytes) return fail(DVQ_ERR_BAD_ARG, "bytes is NULL");
  int rc = check_vq_shape(N, K, D);
  if (rc) return rc;
  *bytes = vq_workspace_layout(N, K, D, flags).total;
  return DVQ_OK;
}

int dvq_vq_forward(const float* z, const float* E, int64_t N, int K, int D, int flags, float* z_q, int64_t* idx,
                   float* onehot, unsigned long long* hist, double* sse, void* workspace, size_t workspace_bytes,
                   void* stream) {
  int rc = check_vq_shape(N, K, D);
  if (rc) return rc;
  const int train = (flags & DVQ_TRAIN) ? 1 : 0;
  if (!E || !workspace) return fail(DVQ_ERR_BAD_ARG, "E / workspace must not be NULL");
  if (N > 0 && (!z || !z_q || !idx)) return fail(DVQ_ERR_BAD_ARG, "z, z_q and idx must not be NULL");
  if (train && (!hist || !sse)) return fail(DVQ_ERR_BAD_ARG, "DVQ_TRAIN needs hist and sse");
  if ((flags & DVQ_WRITE_ONEHOT) && !onehot) return fail(DVQ_ERR_BAD_ARG, "DVQ_WRITE_ONEHOT needs onehot");
  const bool zbf = (flags & DVQ_Z_BF16) != 0;   // z / z_q are bf16 rows
  if ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(z_q)) % (zbf ? 2 : 4) != 0 || reinterpret_cast<uintptr_t>(E) % 4 != 0 ||
      reinterpret_cast<uintptr_t>(idx) % 8 != 0 || reinterpret_cast<uintptr_t>(workspace) % 256 != 0)
    return fail(DVQ_ERR_BAD_ALIGN, "z/z_q need %d-byte, E 4-byte, idx 8-byte, workspace 256-byte alignment", zbf ? 2 : 4);
  const VqWorkspace w = vq_workspace_layout(N, K, D, flags);
  if (workspace_bytes < w.total)
    return fail(DVQ_ERR_WORKSPACE, "workspace too small: %zu < %zu bytes", workspace_bytes, w.total);
  rc = require_sm100();
  if (rc) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  float* ee = reinterpret_cast<float*>(ws + w.off_ee);

  const int path = flags & DVQ_PATH_MASK;
  const bool tc_ok = vq_tc_supported(N, K, D);
  if (path == DVQ_PATH_TC && !tc_ok)
    return fail(DVQ_ERR_BAD_SHAPE, "DVQ_PATH_TC: shape N=%lld K=%d D=%d is not handled by the tcgen05 kernel", (long long)N, K, D);
  // the tcgen05 kernel moves rows with bulk copies / 128-bit accesses: AUTO falls back to the FP32 kernel for a
  // (valid) 4-byte-aligned view such as a contiguous tensor with an odd storage offset; an explicit DVQ_PATH_TC
  // request errors in launch_vq_tc
  const bool aligned16 = (reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(E) | reinterpret_cast<uintptr_t>(z_q)) % 16 == 0;
  const bool use_tc = tc_ok && path != DVQ_PATH_SIMT && (aligned16 || path == DVQ_PATH_TC);

  const bool cached = (flags & DVQ_CODEBOOK_CACHED) != 0;   // the caller vouches for ee / CbMeta / operand image in the workspace
  profile_mark(0, true, s);
  if (!cached) rc = launch_code_norms(E, K, D, ee, s);
  profile_mark(0, false, s);
  if (rc) return rc;
  if (N > 0) {
    if (use_tc) {
      int* counters = reinterpret_cast<int*>(ws + w.off_counters);
      int* row_list = reinterpret_cast<int*>(ws + w.off_rowlist);
      int* cand_list = reinterpret_cast<int*>(ws + w.off_rowlist + align_up(sizeof(int) * (size_t)N, 256));
      profile_mark(1, true, s);
      rc = launch_vq_tc(z, E, ee, N, K, D, train, z_q, idx, hist, sse, ws + w.off_bop, counters, row_list, cand_list,
                        reinterpret_cast<int*>(ws + w.off_binned), (int)(vq_refine_binned_zero_bytes() / sizeof(int)), cached, zbf, s);
      profile_mark(1, false, s);
      if (rc) return rc;
      // exact FP32 refine of the rows the filter flagged (device-side count, no host sync): restricted to
      // the recorded candidate groups when that kernel covers the shape, else the full FP32 kernel on the list
      profile_mark(2, true, s);
      // (large codebooks: rows with too many candidates for the list record, and degenerate rows, sit in a second
      //  list stored downwards from the end of the same buffer; both kernels re-evaluate them against every code)
      const bool list_mode = cand_list_mode(K);
      const RefineList list{row_list, cand_list, counters + CNT_LISTED, list_mode ? row_list + (N - 1) : nullptr,
                            list_mode ? counters + CNT_OVF : nullptr, list_mode};
      if (vq_refine_supported(K, D)) {
        // Three exact refine paths with identical results.  The code-stationary kernel (code rows register-resident, one
        // warp per 32-code sub-chunk, z rows streamed past them) covers mask-mode codebooks whose K/32 warps hold e_dim
        // floats per lane; the automatic choice takes it where it measured faster than the per-row kernel
        // (vq_refine_stationary_default: K >= 128 up to e_dim 64, K = 256 at e_dim 128; config 2: 0.077 vs 0.101 ms).
        // Otherwise the per-row kernel (one warp per undecided row) while the FP32 codebook fits its shared memory
        // (measured at K = 512, e_dim = 64: 0.105 vs 0.128 ms for 108 k rows against the binned kernels); beyond that the
        // binned kernels win by 2-5x (code rows register-resident per bucket instead of re-read from L2 per row).  The
        // binned path hands its list back to the per-row kernel through the hand-back counters when the pairs do not
        // fit its workspace (normally both stay zero and the per-row kernel exits at once).  dvq_vq_set_refine /
        // DVQ_REFINE_PER_ROW / DVQ_REFINE_BINNED force one path.
        static const bool env_per_row = getenv("DVQ_REFINE_PER_ROW") != nullptr;
        static const bool env_binned = getenv("DVQ_REFINE_BINNED") != nullptr;
        const int mode = __atomic_load_n(&g_refine_mode, __ATOMIC_RELAXED);
        const bool force_per_row = env_per_row || mode == 1, force_binned = env_binned || mode == 2;
        const bool stationary = mode == 3 || (!force_per_row && !force_binned && vq_refine_stationary_default(K, D));
        const bool per_row_only = force_per_row || (!force_binned && vq_refine_codebook_in_smem(K, D));
        RefineList handback = list;
        handback.n = counters + CNT_HANDBACK;
        if (list_mode) handback.n_ovf = counters + CNT_HANDBACK_OVF;
        if (stationary)
          rc = launch_vq_refine_stationary(z, E, ee, K, D, train, z_q, idx, hist, sse, list, zbf, s);
        else if (!per_row_only)
          rc = launch_vq_refine_binned(z, E, ee, N, K, D, train, z_q, idx, hist, sse, list, counters, ws + w.off_binned, zbf, s);
        if (!rc && !stationary)
          rc = launch_vq_refine(z, E, ee, K, D, train, z_q, idx, hist, sse, per_row_only ? list : handback, zbf, s);
      } else {
        rc = launch_vq_simt(z, E, ee, N, K, D, train, z_q, idx, hist, sse, list.rows, list.n, 1, zbf, s);
        if (!rc && list_mode)
          rc = launch_vq_simt(z, E, ee, N, K, D, train, z_q, idx, hist, sse, list.ovf_last, list.n_ovf, -1, zbf, s);
      }
      profile_mark(2, false, s);
      if (rc) return rc;
    } else {
      profile_mark(1, true, s);
      rc = launch_vq_simt(z, E, ee, N, K, D, train, z_q, idx, hist, sse, nullptr, nullptr, 1, zbf, s);
      profile_mark(1, false, s);
      if (rc) return rc;
    }
    if (flags & DVQ_WRITE_ONEHOT) {
      profile_mark(3, true, s);
      rc = launch_onehot(idx, N, K, onehot, s);
      profile_mark(3, false, s);
      if (rc) return rc;
    }
  }
  return DVQ_OK;
}

int dvq_vq_read_counters(const void* workspace, int64_t N, int K, int D, int flags, int* out4) {
  if (!workspace || !out4) return fail(DVQ_ERR_BAD_ARG, "NULL argument");
  int rc = check_vq_shape(N, K, D);
  if (rc) return rc;
  out4[0] = out4[1] = out4[2] = out4[3] = 0;
  const bool use_tc = vq_tc_supported(N, K, D) && (flags & DVQ_PATH_MASK) != DVQ_PATH_SIMT;
  if (!use_tc) return DVQ_OK;
  const VqWorkspace w = vq_workspace_layout(N, K, D, flags);
  DVQ_CUDA_CHECK(cudaMemcpy(out4, static_cast<const char*>(workspace) + w.off_counters, 4 * sizeof(int), cudaMemcpyDeviceToHost));
  if (getenv("DVQ_TC_STATS_PRINT")) {
    unsigned long long st[17];
    DVQ_CUDA_CHECK(cudaMemcpy(st, static_cast<const char*>(workspace) + w.off_counters + CNT_STATS * sizeof(int), sizeof(st),
                              cudaMemcpyDeviceToHost));
    static const char* names[17] = {"producer.wait_stage_empty", "mma.wait_a_full", "mma.wait_acc_empty", "mma.total",
                                    "conv.wait_stage_full", "conv.wait_a_empty", "conv.total", "epi0.wait_acc_full",
                                    "epi4.wait_fin_empty", "epi0.wait_fin_full", "epi0.wait_sidx_empty", "epi0.total",
                                    "gather.wait_sidx_full", "gather.total", "mma.wait_b_full", "(unused)", "mma.wait_peer_acc_empty"};
    for (int i = 0; i < 17; ++i) fprintf(stderr, "[dvq tc stats] %-28s %14llu cycles (sum over CTAs)\n", names[i], st[i]);
    if (N >= 65536) {   // pipeline timeline of CTA 3, tiles 8..11 (see TRACE in vq_tc_sm100.cu)
      static long long tr[5 * 8 * 8];
      DVQ_CUDA_CHECK(cudaMemcpy(tr, static_cast<const char*>(workspace) + w.off_rowlist + (size_t)(N - 8192) * sizeof(int), sizeof(tr),
                                cudaMemcpyDeviceToHost));
      static const char* ev[5][4] = {{"mma.a_full", "mma.acc_empty", "mma.issued", "mma.complete"},
                                     {"own.acc_full", "own.chunk_done", "own.fin_full", "own.sidx_out"},
                                     {"hlp.acc_full", "hlp.chunk_done", "hlp.fin_out", "hlp.stage_freed"},
                                     {"cnv.stage_full", "cnv.pass1_done", "cnv.a_empty", "cnv.a_full_out"},
                                     {"gth.sidx_full", "gth.done", "", ""}};
      long long base = tr[(0 * 8 + 0) * 8 + 0];
      for (int role = 0; role < 5; ++role)
        for (int e = 0; e < 4; ++e) {
          if (!ev[role][e][0]) continue;
          fprintf(stderr, "[dvq tc trace] %-16s", ev[role][e]);
          for (int k = 0; k < 8; ++k) {
            const long long v = tr[(role * 8 + e) * 8 + k];
            fprintf(stderr, " %7lld", v ? v - base : -1);
          }
          fprintf(stderr, "\n");
        }
    }
  }
  return DVQ_OK;
}

int dvq_vq_finalize(const unsigned long long* hist, const double* sse, int64_t N_total, int K, int D, float al,
                    float beta, float* loss, float* perplexity, void* stream) {
  if (!hist || !sse || !loss || !perplexity) return fail(DVQ_ERR_BAD_ARG, "NULL argument");
  if (N_total < 0 || K <= 0 || D <= 0) return fail(DVQ_ERR_BAD_SHAPE, "need N_total >= 0 (0 = take the histogram total), K, D > 0");
  int rc = require_sm100();
  if (rc) return rc;
  return launch_finalize(hist, sse, N_total, K, D, al, beta, loss, perplexity, static_cast<cudaStream_t>(stream));
}

int dvq_gather(const float* E, const int64_t* idx, int64_t N, int K, int D, float* out, int* oob, void* stream) {
  if (N < 0 || K <= 0 || D <= 0) return fail(DVQ_ERR_BAD_SHAPE, "need N >= 0, K > 0, D > 0");
  if (N > 0 && (!E || !idx || !out)) return fail(DVQ_ERR_BAD_ARG, "NULL argument");
  int rc = require_sm100();
  if (rc) return rc;
  return launch_gather(E, idx, N, K, D, out, oob, static_cast<cudaStream_t>(stream));
}

int dvq_vq_backward_ex(const float* z, const float* E, const int64_t* idx, const float* g_zq, const float* g_loss,
                       const float* rows, int64_t N, int K, int D, float al, float beta, int flags, float* dz, float* dE,
                       void* stream) {
  if (N < 0 || K <= 0 || D <= 0 || (D & 3)) return fail(DVQ_ERR_BAD_SHAPE, "need N >= 0, K > 0, D a positive multiple of 4");
  if (flags & ~DVQ_Z_BF16) return fail(DVQ_ERR_BAD_ARG, "dvq_vq_backward_ex accepts DVQ_Z_BF16 only");
  if (!g_loss || !rows || (N > 0 && (!z || !E || !idx))) return fail(DVQ_ERR_BAD_ARG, "NULL argument");
  const bool zbf = (flags & DVQ_Z_BF16) != 0;   // z, g_zq and dz move 4 elements at a time: 16 bytes fp32, 8 bytes bf16
  if ((reinterpret_cast<uintptr_t>(E) | reinterpret_cast<uintptr_t>(dE)) % 16 != 0 ||
      (reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(g_zq) | reinterpret_cast<uintptr_t>(dz)) % (zbf ? 8 : 16) != 0)
    return fail(DVQ_ERR_BAD_ALIGN, "dvq_vq_backward needs 16-byte aligned E / dE and %d-byte aligned z / g_zq / dz", zbf ? 8 : 16);
  int rc = require_sm100();
  if (rc) return rc;
  return launch_vq_backward(z, E, idx, g_zq, g_loss, rows, N, D, al, beta, dz, dE, zbf, static_cast<cudaStream_t>(stream));
}

int dvq_vq_backward(const float* z, const float* E, const int64_t* idx, const float* g_zq, const float* g_loss,
                    const float* rows, int64_t N, int K, int D, float al, float beta, float* dz, float* dE, void* stream) {
  return dvq_vq_backward_ex(z, E, idx, g_zq, g_loss, rows, N, K, D, al, beta, 0, dz, dE, stream);
}

int dvq_vq_code_sums_ex(const float* z, const int64_t* idx, int64_t N, int K, int D, int flags, float* sums, void* stream) {
  if (N < 0 || K <= 0 || D <= 0 || (D & 3)) return fail(DVQ_ERR_BAD_SHAPE, "need N >= 0, K > 0, D a positive multiple of 4");
  if (flags & ~DVQ_Z_BF16) return fail(DVQ_ERR_BAD_ARG, "dvq_vq_code_sums_ex accepts DVQ_Z_BF16 only");
  if (N > 0 && (!z || !idx || !sums)) return fail(DVQ_ERR_BAD_ARG, "NULL argument");
  const bool zbf = (flags & DVQ_Z_BF16) != 0;
  if (reinterpret_cast<uintptr_t>(sums) % 16 != 0 || reinterpret_cast<uintptr_t>(z) % (zbf ? 8 : 16) != 0)
    return fail(DVQ_ERR_BAD_ALIGN, "dvq_vq_code_sums needs 16-byte aligned sums and a %d-byte aligned z", zbf ? 8 : 16);
  int rc = require_sm100();
  if (rc) return rc;
  return launch_vq_code_sums(z, idx, N, D, sums, zbf, static_cast<cudaStream_t>(stream));
}

int dvq_vq_code_sums(const float* z, const int64_t* idx, int64_t N, int K, int D, float* sums, void* stream) {
  return dvq_vq_code_sums_ex(z, idx, N, K, D, 0, sums, stream);
}

int dvq_gather_multi(const float* const* E, int G, const int64_t* codes, int64_t N, int K, int D, float* out, int64_t out_stride,
                     int* oob, void* stream) {
  if (G <= 0 || G > 8 || N < 0 || K <= 0 || D <= 0 || (D & 3) || out_stride < (int64_t)G * D || (out_stride & 3))
    return fail(DVQ_ERR_BAD_SHAPE, "need 1 <= G <= 8, D %% 4 == 0, out_stride >= G * D and a multiple of 4");
  if (!E || (N > 0 && (!codes || !out))) return fail(DVQ_ERR_BAD_ARG, "NULL argument");
  for (int g = 0; g < G; ++g)
    if (!E[g] || reinterpret_cast<uintptr_t>(E[g]) % 16) return fail(DVQ_ERR_BAD_ALIGN, "codebook %d is NULL or not 16-byte aligned", g);
  if (reinterpret_cast<uintptr_t>(out) % 16) return fail(DVQ_ERR_BAD_ALIGN, "out needs 16-byte alignment");
  int rc = require_sm100();
  if (rc) return rc;
  return launch_gather_multi(E, G, codes, N, K, D, out, out_stride, oob, static_cast<cudaStream_t>(stream));
}

static int check_mano_model(const DvqManoModel* model) {
  if (!model->v_template || !model->shapedirs || !model->posedirs || !model->j_regressor || !model->weights || !model->pose_mean ||
      !model->parents || (model->ncomps > 0 && !model->hands_components))
    return fail(DVQ_ERR_BAD_ARG, "DvqManoModel has a NULL table");
  if (model->ncomps < 0 || model->ncomps > 45) return fail(DVQ_ERR_BAD_SHAPE, "ncomps must be in [0, 45]");
  if (reinterpret_cast<uintptr_t>(model->weights) % 16) return fail(DVQ_ERR_BAD_ALIGN, "the skinning weights need 16-byte alignment");
  return require_sm100();
}

int dvq_mano_forward(const DvqManoModel* model, const float* betas, const float* global_orient, const float* hand_pose,
                     const float* transl, int B, float* vertices, float* joints, void* stream) {
  if (B < 0) return fail(DVQ_ERR_BAD_SHAPE, "B must be >= 0");
  if (!model || (B > 0 && (!betas || !hand_pose || !vertices))) return fail(DVQ_ERR_BAD_ARG, "NULL argument");
  int rc = check_mano_model(model);
  if (rc) return rc;
  return launch_mano(model, betas, global_orient, hand_pose, transl, B, vertices, joints, static_cast<cudaStream_t>(stream));
}

int dvq_mano_backward(const DvqManoModel* model, const float* betas, const float* global_orient, const float* hand_pose, int B,
                      const float* grad_vertices, const float* grad_joints, float* grad_betas, float* grad_global_orient,
                      float* grad_hand_pose, float* grad_transl, void* stream) {
  if (B < 0) return fail(DVQ_ERR_BAD_SHAPE, "B must be >= 0");
  if (!model || (B > 0 && (!betas || !hand_pose))) return fail(DVQ_ERR_BAD_ARG, "NULL argument");
  int rc = check_mano_model(model);
  if (rc) return rc;
  return launch_mano_backward(model, betas, global_orient, hand_pose, B, grad_vertices, grad_joints, grad_betas, grad_global_orient,
                              grad_hand_pose, grad_transl, static_cast<cudaStream_t>(stream));
}

// the contact kernels index within a call in 32 bits: every [B, n, 3] tensor they touch must have fewer than 2^31 elements
static int check_nn_shape(int B, int N1, int N2) {
  if (B < 0 || N1 < 0 || N2 <= 0) return fail(DVQ_ERR_BAD_SHAPE, "need B >= 0, N1 >= 0, N2 > 0 (got B=%d N1=%d N2=%d)", B, N1, N2);
  if ((long long)B * (N1 > N2 ? N1 : N2) * 3 >= (1LL << 31))
    return fail(DVQ_ERR_BAD_SHAPE, "B * max(N1, N2) * 3 = %lld must be below 2^31; split the batch", (long long)B * (N1 > N2 ? N1 : N2) * 3);
  return DVQ_OK;
}

int dvq_nn_forward(const float* src, const float* trg, int B, int N1, int N2, const float* trg_normals, float* dist, int64_t* idx,
                   uint8_t* interior, void* stream) {
  int rc = check_nn_shape(B, N1, N2);
  if (rc) return rc;
  const bool work = (long long)B * N1 > 0;    // empty tensors may have NULL data pointers
  if (work && (!src || !trg || !dist || !idx)) return fail(DVQ_ERR_BAD_ARG, "src, trg, dist and idx must not be NULL");
  if (work && !trg_normals != !interior) return fail(DVQ_ERR_BAD_ARG, "trg_normals and interior go together (both NULL or both set)");
  rc = require_sm100();
  if (rc) return rc;
  return launch_nn_forward(src, trg, B, N1, N2, trg_normals, dist, idx, interior, static_cast<cudaStream_t>(stream));
}

int dvq_nn_backward(const float* src, const float* trg, const int64_t* idx, const float* g_dist, int B, int N1, int N2, float* g_src,
                    float* g_trg, void* stream) {
  int rc = check_nn_shape(B, N1, N2);
  if (rc) return rc;
  if ((long long)B * N1 > 0 && (!src || !trg || !idx || !g_dist)) return fail(DVQ_ERR_BAD_ARG, "src, trg, idx and g_dist must not be NULL");
  rc = require_sm100();
  if (rc) return rc;
  return launch_nn_backward(src, trg, idx, g_dist, B, N1, N2, g_src, g_trg, static_cast<cudaStream_t>(stream));
}

int dvq_vertex_normals(const float* verts, int B, int V, const int* faces, int F, const int* vf_offsets, const int* vf_faces,
                       float* normals, void* stream) {
  if (B < 0 || V <= 0 || F < 0) return fail(DVQ_ERR_BAD_SHAPE, "need B >= 0, V > 0, F >= 0 (got B=%d V=%d F=%d)", B, V, F);
  if ((long long)B * V * 3 >= (1LL << 31) || (long long)F * 3 >= (1LL << 31))
    return fail(DVQ_ERR_BAD_SHAPE, "B * V * 3 and F * 3 must be below 2^31; split the batch");
  if (!vf_offsets || (B > 0 && (!verts || !normals)) || (F > 0 && (!faces || !vf_faces))) return fail(DVQ_ERR_BAD_ARG, "NULL argument");
  int rc = require_sm100();
  if (rc) return rc;
  return launch_vertex_normals(verts, B, V, faces, vf_offsets, vf_faces, normals, static_cast<cudaStream_t>(stream));
}

int dvq_pcnn_gemm(const DvqPcnnGemm* g, void* stream) {
  int rc = require_sm100();
  if (rc) return rc;
  return launch_pcnn_gemm(g, static_cast<cudaStream_t>(stream));
}

int dvq_pcnn_embed(const int64_t* x, int x_stride, int W, int B, int Bp, const float* emb, int n_emb, int d, void* img16,
                   float* img32, void* stream) {
  if (!x || !emb || !img16) return fail(DVQ_ERR_BAD_ARG, "NULL argument");
  if (W <= 0 || B <= 0 || Bp < B || Bp % 128 || d <= 0 || d % 8 || n_emb <= 0) return fail(DVQ_ERR_BAD_SHAPE, "need Bp %% 128 == 0, Bp >= B > 0, d %% 8 == 0");
  int rc = require_sm100();
  if (rc) return rc;
  return launch_pcnn_embed(x, x_stride, W, B, Bp, emb, n_emb, d, img16, img32, static_cast<cudaStream_t>(stream));
}

int dvq_pcnn_rows_to_image(const int64_t* label, int B, int Bp, const float* table, int n_rows, int kd, void* img16, void* stream) {
  if (!label || !table || !img16) return fail(DVQ_ERR_BAD_ARG, "NULL argument");
  if (B <= 0 || Bp < B || Bp % 128 || kd <= 0 || kd % 8 || n_rows <= 0) return fail(DVQ_ERR_BAD_SHAPE, "need Bp %% 128 == 0, Bp >= B > 0, kd %% 8 == 0");
  int rc = require_sm100();
  if (rc) return rc;
  return launch_pcnn_rows_to_image(label, B, Bp, table, n_rows, kd, img16, static_cast<cudaStream_t>(stream));
}

int dvq_debug_umma(const void* a_img, uint32_t a_bytes, const void* b_img, uint32_t b_bytes, int ksteps,
                   const uint32_t* strides, uint32_t idesc, int n_cols, float* out, int* err, void* stream) {
  if (!a_img || !b_img || !strides || !out || !err) return fail(DVQ_ERR_BAD_ARG, "NULL argument");
  if (a_bytes % 16 || b_bytes % 16 || n_cols % 32 || n_cols <= 0 || n_cols > 256 || ksteps <= 0)
    return fail(DVQ_ERR_BAD_SHAPE, "images must be multiples of 16 bytes, n_cols a multiple of 32 in (0,256]");
  if ((size_t)a_bytes + b_bytes > 200 * 1024) return fail(DVQ_ERR_BAD_SHAPE, "operand images exceed 200 KB");
  int rc = require_sm100();
  if (rc) return rc;
  return launch_umma_probe(a_img, a_bytes, b_img, b_bytes, ksteps, strides, idesc, n_cols, out, err, static_cast<cudaStream_t>(stream));
}

int dvq_onehot(const int64_t* idx, int64_t N, int K, float* out, void* stream) {
  if (N < 0 || K <= 0) return fail(DVQ_ERR_BAD_SHAPE, "need N >= 0, K > 0");
  if (N > 0 && (!idx || !out)) return fail(DVQ_ERR_BAD_ARG, "NULL argument");
  int rc = require_sm100();
  if (rc) return rc;
  return launch_onehot(idx, N, K, out, static_cast<cudaStream_t>(stream));
}

static int check_pn_shape(int B, int C, int P) {
  if (B < 0 || P <= 0 || (C != 3 && C != 4)) return fail(DVQ_ERR_BAD_SHAPE, "need B >= 0, P > 0, C in {3,4} (got B=%d C=%d P=%d)", B, C, P);
  return DVQ_OK;
}

int dvq_pointnet_workspace_bytes_ex(int B, int C, int P, int flags, size_t* bytes) {
  if (!bytes) return fail(DVQ_ERR_BAD_ARG, "bytes is NULL");
  int rc = check_pn_shape(B, C, P);
  if (rc) return rc;
  *bytes = pointnet_workspace_bytes(B, C, P, flags);
  return DVQ_OK;
}

int dvq_pointnet_workspace_bytes(int B, int C, int P, size_t* bytes) { return dvq_pointnet_workspace_bytes_ex(B, C, P, 0, bytes); }

int dvq_pointnet_forward_ex(const float* x, const DvqPointNetWeights* w, int B, int C, int P, int flags, float* feat,
                            float* trans, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_pn_shape(B, C, P);
  if (rc) return rc;
  if (!w) return fail(DVQ_ERR_BAD_ARG, "weights struct is NULL");
  if (B > 0 && (!x || !feat || !trans || !workspace)) return fail(DVQ_ERR_BAD_ARG, "NULL argument");
  if (workspace_bytes < pointnet_workspace_bytes(B, C, P, flags))
    return fail(DVQ_ERR_WORKSPACE, "workspace too small: %zu < %zu bytes", workspace_bytes, pointnet_workspace_bytes(B, C, P, flags));
  rc = require_sm100();
  if (rc) return rc;
  if (B == 0) return DVQ_OK;
  return launch_pointnet(x, w, B, C, P, flags, feat, trans, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

int dvq_pointnet_forward(const float* x, const DvqPointNetWeights* w, int B, int C, int P, float* feat, float* trans,
                         void* workspace, size_t workspace_bytes, void* stream) {
  return dvq_pointnet_forward_ex(x, w, B, C, P, 0, feat, trans, workspace, workspace_bytes, stream);
}

// ---------------------------------------------------------------------------------------------
// Host-buffer pipeline: rows streamed through three device slots on three streams so that the
// PCIe uplink, the kernels and the PCIe downlink of consecutive chunks overlap.
// ---------------------------------------------------------------------------------------------
struct DvqHostCtx {
  static const int kSlots = 3;
  int64_t chunk_rows;
  int K_max, D_max;
  cudaStream_t s_in, s_run, s_out;
  float* z_dev[kSlots];
  float* zq_dev[kSlots];
  int64_t* idx_dev[kSlots];
  cudaEvent_t ev_in[kSlots], ev_run[kSlots], ev_out[kSlots];
  float* E_dev;
  unsigned long long* hist_dev;  // [K_max] followed by sse (double) and loss/ppl (2 floats)
  double* sse_dev;
  float* scal_dev;
  void* ws;
  size_t ws_bytes;
};

int dvq_host_ctx_destroy(DvqHostCtx* c) {
  if (!c) return DVQ_OK;
  for (int i = 0; i < DvqHostCtx::kSlots; ++i) {
    if (c->z_dev[i]) cudaFree(c->z_dev[i]);
    if (c->zq_dev[i]) cudaFree(c->zq_dev[i]);
    if (c->idx_dev[i]) cudaFree(c->idx_dev[i]);
    if (c->ev_in[i]) cudaEventDestroy(c->ev_in[i]);
    if (c->ev_run[i]) cudaEventDestroy(c->ev_run[i]);
    if (c->ev_out[i]) cudaEventDestroy(c->ev_out[i]);
  }
  if (c->E_dev) cudaFree(c->E_dev);
  if (c->hist_dev) cudaFree(c->hist_dev);
  if (c->ws) cudaFree(c->ws);
  if (c->s_in) cudaStreamDestroy(c->s_in);
  if (c->s_run) cudaStreamDestroy(c->s_run);
  if (c->s_out) cudaStreamDestroy(c->s_out);
  free(c);
  return DVQ_OK;
}

int dvq_host_ctx_create(int64_t chunk_rows, int K_max, int D_max, DvqHostCtx** out) {
  if (!out) return fail(DVQ_ERR_BAD_ARG, "ctx out pointer is NULL");
  int rc = check_vq_shape(chunk_rows, K_max, D_max);
  if (rc) return rc;
  if (chunk_rows <= 0) return fail(DVQ_ERR_BAD_SHAPE, "chunk_rows must be positive");
  rc = require_sm100();
  if (rc) return rc;
  DvqHostCtx* c = static_cast<DvqHostCtx*>(calloc(1, sizeof(DvqHostCtx)));
  if (!c) return fail(DVQ_ERR_CUDA, "out of host memory");
  c->chunk_rows = chunk_rows;
  c->K_max = K_max;
  c->D_max = D_max;
#define CTX_CHECK(expr)                                                                     \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess) {                                                                \
      dvq_host_ctx_destroy(c);                                                              \
      return fail(DVQ_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(_e));           \
    }                                                                                       \
  } while (0)
  CTX_CHECK(cudaStreamCreateWithFlags(&c->s_in, cudaStreamNonBlocking));
  CTX_CHECK(cudaStreamCreateWithFlags(&c->s_run, cudaStreamNonBlocking));
  CTX_CHECK(cudaStreamCreateWithFlags(&c->s_out, cudaStreamNonBlocking));
  const size_t row_bytes = sizeof(float) * (size_t)D_max;
  for (int i = 0; i < DvqHostCtx::kSlots; ++i) {
    CTX_CHECK(cudaMalloc(&c->z_dev[i], row_bytes * chunk_rows));
    CTX_CHECK(cudaMalloc(&c->zq_dev[i], row_bytes * chunk_rows));
    CTX_CHECK(cudaMalloc(&c->idx_dev[i], sizeof(int64_t) * chunk_rows));
    CTX_CHECK(cudaEventCreateWithFlags(&c->ev_in[i], cudaEventDisableTiming));
    CTX_CHECK(cudaEventCreateWithFlags(&c->ev_run[i], cudaEventDisableTiming));
    CTX_CHECK(cudaEventCreateWithFlags(&c->ev_out[i], cudaEventDisableTiming));
  }
  CTX_CHECK(cudaMalloc(&c->E_dev, row_bytes * K_max));
  const size_t stat_bytes = align_up(sizeof(unsigned long long) * (size_t)K_max, 16) + 32;
  CTX_CHECK(cudaMalloc(&c->hist_dev, stat_bytes));
  c->sse_dev = reinterpret_cast<double*>(reinterpret_cast<char*>(c->hist_dev) + align_up(sizeof(unsigned long long) * (size_t)K_max, 16));
  c->scal_dev = reinterpret_cast<float*>(c->sse_dev + 1);
  // the workspace must serve every shape up to (K_max, D_max): the layout is not monotone in K and D (the tcgen05
  // path and its buffers exist only for some shapes), so take the maximum over the shape classes
  size_t ws_need = 0;
  for (int k = 32; ; k *= 2) {
    const int kk = k < K_max ? k : K_max;
    for (int d = 16; ; d *= 2) {
      const int dd = d < D_max ? d : D_max;
      const size_t t = vq_workspace_layout(chunk_rows, kk, dd, 0).total;
      ws_need = t > ws_need ? t : ws_need;
      if (dd == D_max) break;
    }
    if (kk == K_max) break;
  }
  c->ws_bytes = ws_need + 4096;
  CTX_CHECK(cudaMalloc(&c->ws, c->ws_bytes));
#undef CTX_CHECK
  *out = c;
  return DVQ_OK;
}

int dvq_vq_forward_host(DvqHostCtx* c, const float* z_host, const float* E_host, int64_t N, int K, int D, int flags,
                        float al, float beta, float* zq_host, int64_t* idx_host, float* loss_host,
                        float* perplexity_host) {
  if (!c) return fail(DVQ_ERR_BAD_ARG, "ctx is NULL");
  int rc = check_vq_shape(N, K, D);
  if (rc) return rc;
  if (K > c->K_max || D > c->D_max)
    return fail(DVQ_ERR_BAD_SHAPE, "K=%d D=%d exceed the context limits K_max=%d D_max=%d", K, D, c->K_max, c->D_max);
  if (flags & DVQ_WRITE_ONEHOT) return fail(DVQ_ERR_BAD_ARG, "the host-buffer entry does not materialise the one-hot matrix");
  if (flags & DVQ_Z_BF16) return fail(DVQ_ERR_BAD_ARG, "the host-buffer entry takes fp32 rows only (DVQ_Z_BF16 is not accepted)");
  if (!E_host || (N > 0 && (!z_host || !zq_host || !idx_host))) return fail(DVQ_ERR_BAD_ARG, "NULL host pointer");
  const int train = (flags & DVQ_TRAIN) ? 1 : 0;
  if (train && (!loss_host || !perplexity_host)) return fail(DVQ_ERR_BAD_ARG, "DVQ_TRAIN needs loss_host and perplexity_host");
  const int64_t chunk = c->chunk_rows;  // D <= D_max, so chunk_rows rows always fit a slot
  const size_t row_bytes = sizeof(float) * (size_t)D;

  DVQ_CUDA_CHECK(cudaMemcpyAsync(c->E_dev, E_host, row_bytes * K, cudaMemcpyHostToDevice, c->s_in));
  cudaEvent_t ev_E = c->ev_in[0];
  DVQ_CUDA_CHECK(cudaEventRecord(ev_E, c->s_in));
  DVQ_CUDA_CHECK(cudaStreamWaitEvent(c->s_run, ev_E, 0));
  if (train)
    DVQ_CUDA_CHECK(cudaMemsetAsync(c->hist_dev, 0, align_up(sizeof(unsigned long long) * (size_t)c->K_max, 16) + 32, c->s_run));

  int64_t n_chunks = (N + chunk - 1) / chunk;
  for (int64_t ci = 0; ci < n_chunks; ++ci) {
    const int b = (int)(ci % DvqHostCtx::kSlots);
    const int64_t r0 = ci * chunk;
    const int64_t rows = (N - r0 < chunk) ? (N - r0) : chunk;
    if (ci >= DvqHostCtx::kSlots) {
      DVQ_CUDA_CHECK(cudaStreamWaitEvent(c->s_in, c->ev_run[b], 0));   // z slot consumed
      DVQ_CUDA_CHECK(cudaStreamWaitEvent(c->s_run, c->ev_out[b], 0));  // z_q / idx slot drained
    }
    DVQ_CUDA_CHECK(cudaMemcpyAsync(c->z_dev[b], z_host + r0 * D, row_bytes * rows, cudaMemcpyHostToDevice, c->s_in));
    DVQ_CUDA_CHECK(cudaEventRecord(c->ev_in[b], c->s_in));
    DVQ_CUDA_CHECK(cudaStreamWaitEvent(c->s_run, c->ev_in[b], 0));
    if (!(flags & DVQ_HOST_COPY_ONLY)) {
      // every full chunk after the first finds the codebook preparation of this call in the workspace (same E, rows, K, D)
      const int cflags = flags | ((ci > 0 && rows == chunk) ? DVQ_CODEBOOK_CACHED : 0);
      rc = dvq_vq_forward(c->z_dev[b], c->E_dev, rows, K, D, cflags, c->zq_dev[b], c->idx_dev[b], nullptr, c->hist_dev,
                          c->sse_dev, c->ws, c->ws_bytes, c->s_run);
      if (rc) return rc;
    }
    DVQ_CUDA_CHECK(cudaEventRecord(c->ev_run[b], c->s_run));
    DVQ_CUDA_CHECK(cudaStreamWaitEvent(c->s_out, c->ev_run[b], 0));
    DVQ_CUDA_CHECK(cudaMemcpyAsync(zq_host + r0 * D, c->zq_dev[b], row_bytes * rows, cudaMemcpyDeviceToHost, c->s_out));
    DVQ_CUDA_CHECK(cudaMemcpyAsync(idx_host + r0, c->idx_dev[b], sizeof(int64_t) * rows, cudaMemcpyDeviceToHost, c->s_out));
    DVQ_CUDA_CHECK(cudaEventRecord(c->ev_out[b], c->s_out));
  }
  float scal[2] = {0.f, 0.f};
  if (train && N > 0 && !(flags & DVQ_HOST_COPY_ONLY)) {
    rc = launch_finalize(c->hist_dev, c->sse_dev, N, K, D, al, beta, c->scal_dev, c->scal_dev + 1, c->s_run);
    if (rc) return rc;
    DVQ_CUDA_CHECK(cudaMemcpyAsync(scal, c->scal_dev, sizeof(scal), cudaMemcpyDeviceToHost, c->s_run));
  }
  DVQ_CUDA_CHECK(cudaStreamSynchronize(c->s_in));
  DVQ_CUDA_CHECK(cudaStreamSynchronize(c->s_run));
  DVQ_CUDA_CHECK(cudaStreamSynchronize(c->s_out));
  if (train) {
    *loss_host = scal[0];
    *perplexity_host = scal[1];
  }
  return DVQ_OK;
}

// ---------------------------------------------------------------------------------------------
// NCCL hook: resolved lazily from the libnccl already mapped into the process (torch's), so the
// library itself has no link-time NCCL dependency.
// ---------------------------------------------------------------------------------------------
typedef int (*nccl_allreduce_fn)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef int (*nccl_group_fn)(void);
typedef const char* (*nccl_errstr_fn)(int);

int dvq_allreduce_stats(void* nccl_comm, unsigned long long* hist, double* sse, int K, void* stream) {
  static nccl_allreduce_fn p_allreduce = nullptr;
  static nccl_group_fn p_start = nullptr, p_end = nullptr;
  static nccl_errstr_fn p_err = nullptr;
  if (!nccl_comm || !hist || !sse || K <= 0) return fail(DVQ_ERR_BAD_ARG, "NULL communicator / buffer or K <= 0");
  if (!p_allreduce) {
    const char* override_path = getenv("DVQ_NCCL_LIB");
    void* h = nullptr;
    if (override_path) h = dlopen(override_path, RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return fail(DVQ_ERR_NCCL, "libnccl not found (set DVQ_NCCL_LIB): %s", dlerror());
    p_allreduce = reinterpret_cast<nccl_allreduce_fn>(dlsym(h, "ncclAllReduce"));
    p_start = reinterpret_cast<nccl_group_fn>(dlsym(h, "ncclGroupStart"));
    p_end = reinterpret_cast<nccl_group_fn>(dlsym(h, "ncclGroupEnd"));
    p_err = reinterpret_cast<nccl_errstr_fn>(dlsym(h, "ncclGetErrorString"));
    if (!p_allreduce || !p_start || !p_end) {
      p_allreduce = nullptr;
      return fail(DVQ_ERR_NCCL, "libnccl is missing ncclAllReduce/ncclGroupStart/ncclGroupEnd");
    }
  }
  const int kUint64 = 5, kFloat64 = 8, kSum = 0;  // ncclDataType_t / ncclRedOp_t (nccl.h 2.2x)
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int r = p_start();
  if (!r) r = p_allreduce(hist, hist, (size_t)K, kUint64, kSum, nccl_comm, s);
  if (!r) r = p_allreduce(sse, sse, 1, kFloat64, kSum, nccl_comm, s);
  int r2 = p_end();
  if (!r) r = r2;
  if (r) return fail(DVQ_ERR_NCCL, "NCCL all-reduce failed: %s", p_err ? p_err(r) : "unknown");
  return DVQ_OK;
}

}  // extern "C"
