// Exact FP32 re-evaluation of the rows the tcgen05 filter could not decide, restricted to the
// candidate sub-chunks the filter recorded (the 32-code sub-chunks that held a key inside the row's
// error band).  One warp per undecided row; lane = code inside a sub-chunk.
//
// Arithmetic: the contract of vq_exact.cuh, so a row refined here gets exactly the index the all-FP32
// kernel would give it (the true minimiser is always inside the candidate sub-chunks: every key outside
// the band is provably farther, DESIGN.md §4.1).
//
// The codebook is staged once per CTA in shared memory with a (D+4)-float row pitch: 16-byte aligned
// rows whose 128-bit reads are conflict-free for lane = code (a quarter-warp covers all 32 banks).  The
// z row stays in shared memory too (broadcast 128-bit reads), so a thread needs ~40 registers and 32
// warps per SM hide the latency of the sequential FMA chain; each undecided row then costs ~2 groups
// x (32 LDS.128 + 64 FMAs) per lane instead of the K x D of the full kernel.
#include "vq_exact.cuh"

namespace dvq {
namespace {

constexpr int RTHREADS = 1024;

// ZT: element type of z / z_q (float, or __nv_bfloat16 under DVQ_Z_BF16: the z rows are staged as bf16 and upcast on read)
template <int DT, bool TRAIN, bool SMEM_E, typename ZT>
__global__ void __launch_bounds__(RTHREADS, 1)
vq_refine_kernel(const ZT* __restrict__ z, const float* __restrict__ E, const float* __restrict__ ee, int K,
                 ZT* __restrict__ zq, int64_t* __restrict__ idx_out, unsigned long long* __restrict__ hist,
                 double* __restrict__ sse, RefineList L) {
  extern __shared__ __align__(16) float smem_f[];   // zbuf[warps][2][DT] (ZT) | es[K][DT+4] when SMEM_E
  constexpr int PITCH = DT + 4;
  constexpr int NW = RTHREADS / 32;
  constexpr int ZE = 16 / (int)sizeof(ZT);          // z elements per 16-byte piece
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  ZT* zbuf = reinterpret_cast<ZT*>(smem_f) + warp * 2 * DT;   // double-buffered z row of this warp
  float* es = reinterpret_cast<float*>(reinterpret_cast<ZT*>(smem_f) + NW * 2 * DT);
  // nothing listed (the usual case when the binned kernels ran first): leave before staging the codebook
  if (*L.n == 0 && (L.n_ovf == nullptr || *L.n_ovf == 0)) return;
  if (SMEM_E) {
    for (int i = tid; i < K * (DT / 4); i += RTHREADS) {
      const int k = i / (DT / 4), d = (i - k * (DT / 4)) * 4;
      *reinterpret_cast<float4*>(es + k * PITCH + d) = ldg4(E + (size_t)k * DT + d);
    }
    __syncthreads();
  }
  const int n = *L.n;
  const int wglobal = blockIdx.x * NW + warp;
  const int wtotal = gridDim.x * NW;
  const int nsc = (K + 31) / 32;
  double lsse = 0.0;
  // cp.async prefetch of the next undecided row of this warp hides its (random-access) global latency
  auto prefetch = [&](int i, int buf) {
    if (i < n) {
      const ZT* src = z + (int64_t)L.rows[i] * DT;
#pragma unroll
      for (int v = lane; v < DT / ZE; v += 32) {
        const uint32_t dst = (uint32_t)__cvta_generic_to_shared(zbuf + buf * DT + v * ZE);
        cp_async_ca16(dst, src + v * ZE);
      }
    }
    cp_async_commit();
  };
  // outputs of one row, executed by one warp
  auto emit_row = [&](int64_t row, int bidx, const ZT* zsrc) {
    ZT* orow = zq + row * DT;
    const float* erow = E + (int64_t)bidx * DT;
    for (int c = lane * 4; c < DT; c += 128) {
      float4 o4 = ldg4(erow + c);
      if (TRAIN) o4 = st_step4(o4, zld4(zsrc + c), lsse);
      zst4(orow + c, o4);
    }
    if (lane == 0) {
      idx_out[row] = (int64_t)bidx;
      if (TRAIN) atomicAdd(hist + bidx, 1ull);
    }
  };
  prefetch(wglobal, 0);
  int buf = 0;
  for (int i = wglobal; i < n; i += wtotal, buf ^= 1) {
    prefetch(i + wtotal, buf ^ 1);
    cp_async_wait<1>();
    __syncwarp();
    const int64_t row = L.rows[i];
    const uint32_t cand = (uint32_t)L.cand[i];
    const ZT* zb = zbuf + buf * DT;
    const float zz = warp_sum(sq_partial<DT>(zb, lane));
    unsigned long long best = ~0ull;   // (distance key, code) minimum so far
    // candidate sub-chunks (32 codes each) in ascending code order (the tie-break relies on it), two at a time: one
    // broadcast read of z feeds both dot products, and the two sequential FMA chains interleave
    unsigned todo = 0u;                          // mask mode: the candidate bits
    int g_sc = 0, g_end = 0;                     // every code: sub-chunks g_sc .. g_end - 1
    int l0 = -1, l1 = -1, l2 = -1;               // list mode: the entries
    if (cand_is_all(cand, L.list_mode)) {
      g_end = nsc;
    } else if (L.list_mode) {
      // ascending order, empty entries (-1) last
      const int big = 1 << 30;
      const int e0 = cand_entry(cand, 0), e1 = cand_entry(cand, 1), e2 = cand_entry(cand, 2);
      int a0 = e0 < 0 ? big : e0, a1 = e1 < 0 ? big : e1, a2 = e2 < 0 ? big : e2;
      int t;
      if (a0 > a1) { t = a0; a0 = a1; a1 = t; }
      if (a1 > a2) { t = a1; a1 = a2; a2 = t; }
      if (a0 > a1) { t = a0; a0 = a1; a1 = t; }
      l0 = a0 == big ? -1 : a0; l1 = a1 == big ? -1 : a1; l2 = a2 == big ? -1 : a2;
    } else {
      todo = cand;
    }
    auto next_sc = [&]() -> int {   // warp-uniform; -1 when exhausted
      if (g_sc < g_end) return g_sc++;
      if (L.list_mode) {
        const int r = l0;
        l0 = l1; l1 = l2; l2 = -1;
        return r < nsc ? r : -1;
      }
      if (!todo) return -1;
      const int g = __ffs(todo) - 1;
      todo &= todo - 1u;
      return g;
    };
    for (;;) {
      const int sa = next_sc();
      if (sa < 0) break;
      const int sb = next_sc();
      const int code_a = sa * 32 + lane, code_b = (sb < 0 ? sa : sb) * 32 + lane;
      const bool va = code_a < K, vb = sb >= 0 && code_b < K;
      float acc_a = 0.f, acc_b = 0.f;
      if (SMEM_E && sb < 0) {
        // a single sub-chunk left (about half of the rows have an odd number of candidate sub-chunks): one FMA chain, half the
        // shared-memory reads of the paired pass
        const float* ea = es + (va ? code_a : 0) * PITCH;
#pragma unroll
        for (int d = 0; d < DT; d += 4) {
          const float4 z4 = zld4(zb + d);   // broadcast read
          const float4 a4 = *reinterpret_cast<const float4*>(ea + d);
          acc_a = fmaf(z4.x, a4.x, acc_a); acc_a = fmaf(z4.y, a4.y, acc_a);
          acc_a = fmaf(z4.z, a4.z, acc_a); acc_a = fmaf(z4.w, a4.w, acc_a);
        }
      } else if (SMEM_E) {
        const float* ea = es + (va ? code_a : 0) * PITCH;
        const float* eb = es + (vb ? code_b : 0) * PITCH;
#pragma unroll
        for (int d = 0; d < DT; d += 4) {
          const float4 z4 = zld4(zb + d);   // broadcast read
          const float4 a4 = *reinterpret_cast<const float4*>(ea + d);
          const float4 b4 = *reinterpret_cast<const float4*>(eb + d);
          acc_a = fmaf(z4.x, a4.x, acc_a); acc_b = fmaf(z4.x, b4.x, acc_b);
          acc_a = fmaf(z4.y, a4.y, acc_a); acc_b = fmaf(z4.y, b4.y, acc_b);
          acc_a = fmaf(z4.z, a4.z, acc_a); acc_b = fmaf(z4.z, b4.z, acc_b);
          acc_a = fmaf(z4.w, a4.w, acc_a); acc_b = fmaf(z4.w, b4.w, acc_b);
        }
      } else {
        const float* ea = E + (int64_t)(va ? code_a : 0) * DT;
        const float* eb = E + (int64_t)(vb ? code_b : 0) * DT;
#pragma unroll
        for (int d = 0; d < DT; d += 4) {
          const float4 z4 = zld4(zb + d);
          const float4 a4 = ldg4(ea + d);
          const float4 b4 = ldg4(eb + d);
          acc_a = fmaf(z4.x, a4.x, acc_a); acc_b = fmaf(z4.x, b4.x, acc_b);
          acc_a = fmaf(z4.y, a4.y, acc_a); acc_b = fmaf(z4.y, b4.y, acc_b);
          acc_a = fmaf(z4.z, a4.z, acc_a); acc_b = fmaf(z4.z, b4.z, acc_b);
          acc_a = fmaf(z4.w, a4.w, acc_a); acc_b = fmaf(z4.w, b4.w, acc_b);
        }
      }
      best = min(best, warp_argmin(dist_key(va ? exact_dist(acc_a, zz, __ldg(ee + code_a)) : INFINITY), sa * 32));
      if (sb >= 0) best = min(best, warp_argmin(dist_key(vb ? exact_dist(acc_b, zz, __ldg(ee + code_b)) : INFINITY), sb * 32));
    }
    emit_row(row, packed_winner(best), zbuf + buf * DT);
    __syncwarp();   // everyone is done with zbuf[buf] before the next-but-one prefetch overwrites it
  }
  cp_async_wait<0>();
  // ---- overflow rows (list mode: more than three candidate sub-chunks, degenerate rows): one CTA per row, the
  //      warps split the sub-chunks of the whole codebook, lexicographic (distance, code) minimum across warps ----
  if (L.n_ovf != nullptr) {
    __shared__ unsigned long long red[NW];
    const int n2 = *L.n_ovf;
    ZT* zrow = reinterpret_cast<ZT*>(smem_f);   // every warp is done with its z buffers after the barrier below
    for (int j = blockIdx.x; j < n2; j += gridDim.x) {
      __syncthreads();
      const int64_t row = L.ovf_last[-(int64_t)j];
      for (int v = tid; v < DT / ZE; v += RTHREADS) reinterpret_cast<uint4*>(zrow)[v] = __ldg(reinterpret_cast<const uint4*>(z + row * DT) + v);
      __syncthreads();
      const float zz = warp_sum(sq_partial<DT>(zrow, lane));
      unsigned long long best = ~0ull;
      for (int sc = warp; sc < nsc; sc += NW) {
        const int code = sc * 32 + lane;
        float dist = INFINITY;
        if (code < K) {
          const float* er = SMEM_E ? es + code * PITCH : E + (int64_t)code * DT;
          float acc = 0.f;
#pragma unroll 8
          for (int d = 0; d < DT; d += 4) {
            const float4 z4 = zld4(zrow + d);
            const float4 e4 = SMEM_E ? *reinterpret_cast<const float4*>(er + d) : ldg4(er + d);
            acc = fmaf(z4.x, e4.x, acc); acc = fmaf(z4.y, e4.y, acc);
            acc = fmaf(z4.z, e4.z, acc); acc = fmaf(z4.w, e4.w, acc);
          }
          dist = exact_dist(acc, zz, __ldg(ee + code));
        }
        best = min(best, warp_argmin(dist_key(dist), sc * 32));
      }
      if (lane == 0) red[warp] = best;
      __syncthreads();
      if (warp == 0) {
        unsigned long long b = red[lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) b = min(b, __shfl_xor_sync(0xffffffffu, b, o));
        emit_row(row, packed_winner(b), zrow);
      }
    }
  }
  if (TRAIN) {
    lsse = warp_sum(lsse);
    if (lane == 0 && lsse != 0.0) atomicAdd(sse, lsse);
  }
}

}  // namespace

// true when the per-row kernel can keep the whole FP32 codebook in shared memory (its fast regime)
static bool codebook_in_smem(int K, int D) {
  return (size_t)K * (D + 4) * sizeof(float) + (size_t)(RTHREADS / 32) * 2 * D * sizeof(float) <= 200 * 1024;
}

template <int DT, typename ZT>
static int launch_refine_dt(const ZT* z, ZT* z_q, const VqCall& c, const RefineList& list) {
  const size_t zbuf_bytes = (size_t)(RTHREADS / 32) * 2 * DT * sizeof(ZT);
  const size_t smem_e = (size_t)c.K * (DT + 4) * sizeof(float);
  const bool in_smem = codebook_in_smem(c.K, DT);
#define DVQ_LAUNCH_REFINE(TR_, SM_)                                                                                      \
  do {                                                                                                                   \
    const size_t bytes = zbuf_bytes + (SM_ ? smem_e : 0);                                                                \
    DVQ_CUDA_CHECK(cudaFuncSetAttribute(vq_refine_kernel<DT, TR_, SM_, ZT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes)); \
    vq_refine_kernel<DT, TR_, SM_, ZT><<<c.sm_count, RTHREADS, bytes, c.s>>>(z, c.E, c.ee, c.K, z_q, c.idx, c.hist, c.sse, list); \
  } while (0)
  if (c.train) { if (in_smem) DVQ_LAUNCH_REFINE(true, true); else DVQ_LAUNCH_REFINE(true, false); }
  else         { if (in_smem) DVQ_LAUNCH_REFINE(false, true); else DVQ_LAUNCH_REFINE(false, false); }
#undef DVQ_LAUNCH_REFINE
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

// the per-row kernel on `list`: the filter's refine list, or the binned kernels' hand-back list
static int launch_vq_refine(const VqCall& c, const RefineList& list) {
  return with_z_type(c, [&](auto z, auto z_q) {
    switch (c.D) {
      case 16: return launch_refine_dt<16>(z, z_q, c, list);
      case 32: return launch_refine_dt<32>(z, z_q, c, list);
      case 64: return launch_refine_dt<64>(z, z_q, c, list);
      case 128: return launch_refine_dt<128>(z, z_q, c, list);
      case 256: return launch_refine_dt<256>(z, z_q, c, list);
      case 512: return launch_refine_dt<512>(z, z_q, c, list);
      default: return fail(DVQ_ERR_BAD_SHAPE, "candidate refine kernel is instantiated for e_dim 16..512 (powers of two) only");
    }
  });
}

// The refine plan.  The three refine kernels give identical results; the automatic choice (mode 0) takes the one that
// measured fastest for the shape (NVIDIA B200, 1000 W power limit, refine stage):
//  - code-stationary (code rows register-resident, one warp per 32-code sub-chunk, z rows streamed past them) where it covers
//    the shape and K >= 128 up to e_dim 64, K >= 256 at e_dim 128: N = 4M, K = 512 / e_dim 64 (config 2) 0.077 vs 0.101 ms
//    for the per-row kernel, K = 128 / e_dim 64 0.062 vs 0.077, K = 256 / e_dim 128 0.149 vs 0.185.  With fewer sub-chunks a
//    CTA has too few warps to hide the FMA chains' latency (K = 64 / e_dim 64: 0.072 vs 0.065 ms; K = 128 / e_dim 128: 0.169
//    vs 0.162 ms);
//  - otherwise per-row (one warp per listed row) while the FP32 codebook fits its shared memory: K = 512 / e_dim 64, 108 k
//    rows, 0.105 vs 0.128 ms for the binned kernels;
//  - otherwise binned, 2-5x faster than per-row reading its code rows from L2 (code rows register-resident per bucket).  The
//    per-row kernel then runs on the hand-back list, which the binned kernels fill when their pairs do not fit the pair list
//    (normally both hand-back counts stay zero and it exits at once).
int launch_vq_refine_stage(const VqCall& c, int mode, long long pair_cap) {
  // the filter's list: rows [0, counters[CNT_LISTED]) with their candidate records; in list mode (large codebooks) also the
  // overflow list (too many candidates for a record, degenerate rows), stored downwards from the end of the row list
  const bool lm = cand_list_mode(c.K);
  const RefineList list{c.row_list, c.cand_list, c.counters + CNT_LISTED, lm ? c.row_list + (c.N - 1) : nullptr,
                        lm ? c.counters + CNT_OVF : nullptr, lm};
  if (mode == 0) {
    const bool stationary = vq_refine_stationary_supported(c.K, c.D) && c.K >= (c.D <= 64 ? 128 : 256);
    mode = stationary ? 3 : codebook_in_smem(c.K, c.D) ? 1 : 2;
  }
  if (mode == 3) return launch_vq_refine_stationary(c, list);
  if (mode == 1) return launch_vq_refine(c, list);
  const int rc = launch_vq_refine_binned(c, list, pair_cap);
  if (rc) return rc;
  RefineList handback = list;
  handback.n = c.counters + CNT_HANDBACK;
  if (lm) handback.n_ovf = c.counters + CNT_HANDBACK_OVF;
  return launch_vq_refine(c, handback);
}

}  // namespace dvq
