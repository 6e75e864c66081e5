// Exact FP32 re-evaluation of the undecided rows, code-stationary: for mask-mode codebooks (K <= 992) small enough that
// every lane of a CTA can hold one code row in registers.  One warp per 32-code sub-chunk (K / 32 warps), lane = code;
// the code rows are loaded once per CTA and the z rows stream past them.
//
// Each CTA takes a contiguous share of the filter's row list (sized on the device from its count) and stages it in
// batches of SB rows: row ids and candidate masks by 4-byte cp.async two batches ahead, the z rows by 16-byte cp.async
// one batch ahead (double-buffered, fp32 or bf16 as stored).  Per batch: ||z||^2 once per row (one warp per row), then
// every warp evaluates the rows whose mask names its sub-chunk (mask 0 = degenerate row: every warp), four rows at a
// time so that four independent FMA chains share the code registers and a z value is a broadcast LDS.128 (one read per
// 4 FMAs per row, where the per-row kernel of vq_refine.cu reads a 512-byte code row per 4 FMAs).  Each warp's
// (order-preserving distance image << 32 | code) minimum of a row goes into a per-(warp, row) table, one thread per row
// takes the table's minimum and writes idx, and all threads write z_q / SSE as independent (row, 4-column) items; the
// histogram is kept in shared memory and flushed once per CTA.
//
// Arithmetic: the contract of vq_exact.cuh.
#include "vq_exact.cuh"

namespace dvq {
namespace {

constexpr int SB = 128;           // rows per staged batch
constexpr int SMAX_WARPS = 31;    // mask mode: at most 31 sub-chunks

// warps (sub-chunks) a CTA can hold with DT code floats per lane in registers: 1024 threads leave 64 registers a
// thread, 512 leave 128, 256 leave 255
template <int DT>
constexpr int stationary_max_warps() { return DT <= 16 ? 31 : DT <= 64 ? 16 : DT == 128 ? 8 : 0; }

// distances of R staged rows (slots rs[0..R)) to this lane's code; the warp's (distance image, code) minimum of each row
// goes to cand[row] (this warp's column of the per-row candidate table)
template <int R, int DT, typename ZT>
__device__ __forceinline__ void eval_rows(const float (&e)[DT], float eek, int sc_base, const ZT* __restrict__ zb,
                                          const unsigned char* rs, const float* s_zz, unsigned long long* cand, int lane) {
  int r[R];
  float acc[R];
#pragma unroll
  for (int i = 0; i < R; ++i) { r[i] = rs[i]; acc[i] = 0.f; }
#pragma unroll
  for (int d = 0; d < DT; d += 4) {
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const float4 z4 = zld4(zb + r[i] * DT + d);   // broadcast read
      acc[i] = fmaf(z4.x, e[d], acc[i]);
      acc[i] = fmaf(z4.y, e[d + 1], acc[i]);
      acc[i] = fmaf(z4.z, e[d + 2], acc[i]);
      acc[i] = fmaf(z4.w, e[d + 3], acc[i]);
    }
  }
#pragma unroll
  for (int i = 0; i < R; ++i) {
    const unsigned long long best = warp_argmin(dist_key(exact_dist(acc[i], s_zz[r[i]], eek)), sc_base);
    if (lane == 0) cand[r[i]] = best;
  }
}

// ZT: element type of z / z_q (float, or __nv_bfloat16 under DVQ_Z_BF16: staged as bf16, upcast on read)
template <int DT, typename ZT>
__global__ void __launch_bounds__(stationary_max_warps<DT>() * 32, 1)
vq_refine_stationary_kernel(const ZT* __restrict__ z, const float* __restrict__ E, const float* __restrict__ ee, int K, int train,
                            ZT* __restrict__ zq, int64_t* __restrict__ idx_out, unsigned long long* __restrict__ hist,
                            double* __restrict__ sse, RefineList L) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ZT* zbuf = reinterpret_cast<ZT*>(smem_raw);   // [2][SB][DT]
  // [warps][SB]: each warp's (distance image << 32 | code) minimum per row, ~0 where the warp did not evaluate the row
  unsigned long long* s_cand = reinterpret_cast<unsigned long long*>(smem_raw + 2 * SB * DT * sizeof(ZT));
  __shared__ int s_row[3][SB];
  __shared__ unsigned s_mask[3][SB];
  __shared__ float s_zz[SB];
  __shared__ int s_bidx[SB];
  __shared__ unsigned char s_list[SMAX_WARPS][SB];
  __shared__ unsigned s_hist[SMAX_WARPS * 32];
  __shared__ double s_sse[SMAX_WARPS];   // per warp: keeps the fp64 sum out of the registers the evaluation needs
  constexpr int ZE = 16 / (int)sizeof(ZT);     // z elements per 16-byte piece
  constexpr int PPR = DT / ZE;                 // 16-byte pieces per z row
  constexpr int C4 = DT / 4;                   // 4-element columns per row
  const int nt = blockDim.x, nw = nt >> 5;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint32_t lanemask_lt;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(lanemask_lt));
  const int n = *L.n;
  const int start = (int)((int64_t)n * blockIdx.x / gridDim.x);
  const int end = (int)((int64_t)n * (blockIdx.x + 1) / gridDim.x);
  if (start >= end) return;
  const int nb = (end - start + SB - 1) / SB;

  auto stage_ids = [&](int b) {   // row ids and candidate masks of batch b (no commit of its own)
    const int i0 = start + b * SB, cnt = min(SB, end - i0);
    for (int t = tid; t < cnt; t += nt) {
      const uint32_t dr = (uint32_t)__cvta_generic_to_shared(&s_row[b % 3][t]);
      const uint32_t dm = (uint32_t)__cvta_generic_to_shared(&s_mask[b % 3][t]);
      cp_async_ca4(dr, L.rows + i0 + t);
      cp_async_ca4(dm, L.cand + i0 + t);
    }
  };
  auto stage_z = [&](int b) {     // z rows of batch b (ids landed and visible; no commit of its own)
    const int cnt = min(SB, end - (start + b * SB));
    const int* rows = s_row[b % 3];
    ZT* dst0 = zbuf + (b & 1) * SB * DT;
    for (int p = tid; p < cnt * PPR; p += nt) {
      const int r = p / PPR, c = p - r * PPR;
      const uint32_t dst = (uint32_t)__cvta_generic_to_shared(dst0 + r * DT + c * ZE);
      cp_async_cg16(dst, z + (int64_t)rows[r] * DT + c * ZE);
    }
  };

  stage_ids(0);
  cp_async_commit();
  // the code rows (loaded once) and the histogram reset overlap the first ids' round trip
  const int code = warp * 32 + lane;            // K is a multiple of 32: every lane holds a code
  float e[DT];
#pragma unroll
  for (int d = 0; d < DT; d += 4) {
    const float4 v = ldg4(E + (int64_t)code * DT + d);
    e[d] = v.x; e[d + 1] = v.y; e[d + 2] = v.z; e[d + 3] = v.w;
  }
  const float eek = __ldg(ee + code);
  if (train) {
    for (int k = tid; k < K; k += nt) s_hist[k] = 0u;
    if (lane == 0) s_sse[warp] = 0.0;
  }
  cp_async_wait<0>();
  __syncthreads();
  stage_z(0);
  if (nb > 1) stage_ids(1);
  cp_async_commit();

  for (int b = 0; b < nb; ++b) {
    const int cnt = min(SB, end - (start + b * SB));
    cp_async_wait<0>();
    __syncthreads();   // batch b's z rows and batch b+1's ids have landed; batch b-1 is written out (its buffers are free)
    if (b + 1 < nb) {
      stage_z(b + 1);
      if (b + 2 < nb) stage_ids(b + 2);
    }
    cp_async_commit();
    const ZT* zb = zbuf + (b & 1) * SB * DT;
    const int* rows = s_row[b % 3];
    const unsigned* masks = s_mask[b % 3];
    // ||z||^2, four rows of a warp at a time (independent shuffle trees)
    for (int r0 = warp; r0 < cnt; r0 += 4 * nw) {
      float s2[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) s2[u] = sq_partial<DT>(zb + min(r0 + u * nw, cnt - 1) * DT, lane);
#pragma unroll
      for (int u = 0; u < 4; ++u) s2[u] = warp_sum(s2[u]);
      if (lane == 0) {
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (r0 + u * nw < cnt) s_zz[r0 + u * nw] = s2[u];
      }
    }
    for (int i = tid; i < nw * SB; i += nt) s_cand[i] = ~0ull;
    __syncthreads();
    // the rows that name this warp's sub-chunk, in slot order
    unsigned char* list = s_list[warp];
    int m = 0;
    for (int g = 0; g < cnt; g += 32) {
      const int r = g + lane;
      const unsigned mk = r < cnt ? masks[r] : 1u;
      const bool sel = r < cnt && (cand_is_all(mk, false) || ((mk >> warp) & 1u));
      const unsigned bal = __ballot_sync(0xffffffffu, sel);
      if (sel) list[m + __popc(bal & lanemask_lt)] = (unsigned char)r;
      m += __popc(bal);
    }
    __syncwarp();
    unsigned long long* cand = s_cand + warp * SB;
    int j = 0;
    for (; j + 4 <= m; j += 4) eval_rows<4, DT>(e, eek, warp * 32, zb, list + j, s_zz, cand, lane);
    if (j + 2 <= m) { eval_rows<2, DT>(e, eek, warp * 32, zb, list + j, s_zz, cand, lane); j += 2; }
    if (j < m) eval_rows<1, DT>(e, eek, warp * 32, zb, list + j, s_zz, cand, lane);
    __syncthreads();
    // winner per row: lexicographic minimum over the warps' candidates
    for (int r = tid; r < cnt; r += nt) {
      unsigned long long best = ~0ull;
      for (int w = 0; w < nw; ++w) best = min(best, s_cand[w * SB + r]);
      const int bidx = packed_winner(best);
      s_bidx[r] = bidx;
      idx_out[rows[r]] = (int64_t)bidx;
      if (train) atomicAdd(s_hist + bidx, 1u);
    }
    __syncthreads();
    // z_q (and SSE) of the batch's rows: every thread a few (row, 4-column) items, their loads independent
    double lsse = 0.0;
#pragma unroll 4
    for (int p = tid; p < cnt * C4; p += nt) {
      const int r = p / C4, c = (p - r * C4) * 4;
      float4 o4 = ldg4(E + (int64_t)s_bidx[r] * DT + c);
      if (train) o4 = st_step4(o4, zld4(zb + r * DT + c), lsse);
      zst4(zq + (int64_t)rows[r] * DT + c, o4);
    }
    if (train) {
      lsse = warp_sum(lsse);
      if (lane == 0) s_sse[warp] += lsse;
    }
  }
  if (train) {
    __syncthreads();
    for (int k = tid; k < K; k += nt)
      if (s_hist[k]) atomicAdd(hist + k, (unsigned long long)s_hist[k]);
    if (lane == 0 && s_sse[warp] != 0.0) atomicAdd(sse, s_sse[warp]);
  }
}

template <int DT, typename ZT>
int launch_stationary_dt(const ZT* z, ZT* z_q, const VqCall& c, const RefineList& list) {
  auto kern = vq_refine_stationary_kernel<DT, ZT>;
  const int threads = c.K;   // one warp per 32-code sub-chunk
  const size_t bytes = (size_t)2 * SB * DT * sizeof(ZT) + (size_t)(c.K / 32) * SB * sizeof(unsigned long long);
  DVQ_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  int per_sm = 0;   // small codebooks (few warps) fit several CTAs per SM
  DVQ_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, bytes));
  kern<<<c.sm_count * (per_sm > 0 ? per_sm : 1), threads, bytes, c.s>>>(z, c.E, c.ee, c.K, c.train, z_q, c.idx, c.hist, c.sse, list);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

}  // namespace

bool vq_refine_stationary_supported(int K, int D) {
  int max_warps = 0;
  switch (D) {
    case 16: max_warps = stationary_max_warps<16>(); break;
    case 32: max_warps = stationary_max_warps<32>(); break;
    case 64: max_warps = stationary_max_warps<64>(); break;
    case 128: max_warps = stationary_max_warps<128>(); break;
    default: return false;
  }
  return !cand_list_mode(K) && K % 32 == 0 && K >= 32 && K / 32 <= max_warps;
}

int launch_vq_refine_stationary(const VqCall& c, const RefineList& list) {
  if (!vq_refine_stationary_supported(c.K, c.D))
    return fail(DVQ_ERR_BAD_SHAPE, "code-stationary refine: K=%d, e_dim %d does not fit (mask-mode K with K/32 warps x e_dim registers)", c.K, c.D);
  return with_z_type(c, [&](auto z, auto z_q) {
    switch (c.D) {
      case 16: return launch_stationary_dt<16>(z, z_q, c, list);
      case 32: return launch_stationary_dt<32>(z, z_q, c, list);
      case 64: return launch_stationary_dt<64>(z, z_q, c, list);
      case 128: return launch_stationary_dt<128>(z, z_q, c, list);
      default: return fail(DVQ_ERR_BAD_SHAPE, "code-stationary refine kernel is instantiated for e_dim 16..128 only");
    }
  });
}

}  // namespace dvq
