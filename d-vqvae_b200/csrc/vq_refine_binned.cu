// Binned exact refine of the rows the tcgen05 filter could not decide.
//
// vq_refine.cu gives every undecided row its own warp (lane = code of a candidate sub-chunk), so each
// (row, sub-chunk) pair re-reads 32 code rows from shared memory: 2 x 512-byte reads per 8 FMAs, bound by
// the shared-memory pipe (and by L2 when the codebook does not fit).  Here the (row, sub-chunk) pairs are
// bucketed by sub-chunk first; a warp then keeps the 32 code rows of ONE sub-chunk in registers and streams
// the z rows of that bucket past them (broadcast shared-memory reads, 1 read per 4 FMAs): the FP32 FMA pipe
// is the bound and a code row is fetched once per bucket slice instead of once per row.
//
//   refine_prep_kernel     one warp per listed row: ||z||^2 (stashed in the row's still unwritten z_q slot),
//                          idx[row] := ~0 (the 64-bit (distance, code) minimum is taken in place), pair counts
//                          per sub-chunk (shared-memory histogram per CTA, one global atomic per bin per CTA)
//   refine_scatter_kernel  exclusive scan of the counts (every CTA, in shared memory), CTA-local counting +
//                          one reservation per (CTA, bin), pairs[pos] = listed-row index; work-item table
//   refine_pairs_kernel    one work item = (sub-chunk, slice of its bucket): exact distances of 16 rows at a
//                          time against the warp's 32 codes, warp argmin, atomicMin on idx[row]
//   refine_emit_kernel     one warp per listed row: winner -> idx, z_q, SSE, histogram
//
// Arithmetic: the contract of vq_exact.cuh; the (distance, code) minimum is an unsigned 64-bit minimum of
// warp_argmin's packed values, so the order in which pairs are processed is irrelevant.
//
// Rows whose candidate record says "every code" (degenerate rows; list mode: more than three candidate
// sub-chunks) are paired with every sub-chunk.  If the pairs do not fit the workspace (2 N entries) the
// scatter kernel hands the whole list to vq_refine.cu instead (device-side switch, no host sync).
#include "vq_exact.cuh"

namespace dvq {
namespace {

constexpr int PREP_THREADS = 1024;
constexpr int PAIR_THREADS = 384;
constexpr int RB = 16;                 // rows per batch of the pairs kernel
constexpr int MAX_BINS = 1024;         // K <= 32 768

struct BinTables {        // int arrays in the workspace
  int* count;             // [MAX_BINS]   pairs per sub-chunk            (zeroed per call)
  int* cursor;            // [MAX_BINS]   scatter reservations           (zeroed per call)
  int* start;             // [MAX_BINS+1] exclusive scan of count
  int* item_start;        // [MAX_BINS+1] exclusive scan of ceil(count / ch); [MAX_BINS+1] = ch
};

// listed row i: the refine list, then the overflow list
__device__ __forceinline__ int64_t listed_row(int i, int n, const int* __restrict__ rows, const int* __restrict__ ovf_last) {
  return i < n ? rows[i] : ovf_last[-(int64_t)(i - n)];
}

// ||z||^2 of a listed row is stashed as a float in the first 4 bytes of its z_q row (rewritten by the emit kernel): 2 D >= 32
// bytes of a bf16 row (DVQ_Z_BF16), at a 32-byte aligned offset
template <typename ZT>
__device__ __forceinline__ float* zz_stash(ZT* zq, int64_t row, int D) { return reinterpret_cast<float*>(zq + row * D); }

template <typename ZT>
__global__ void __launch_bounds__(PREP_THREADS, 1)
refine_prep_kernel(const ZT* __restrict__ z, int D, int K, ZT* __restrict__ zq, unsigned long long* __restrict__ idx64,
                   RefineList L, int* __restrict__ counters, BinTables bt) {
  __shared__ int s_cnt[MAX_BINS];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n = counters[CNT_LISTED], n2 = L.list_mode ? counters[CNT_OVF] : 0;
  if (n + n2 == 0) return;
  const int nbins = (K + 31) / 32;
  for (int b = tid; b < nbins; b += PREP_THREADS) s_cnt[b] = 0;
  __syncthreads();
  // Four rows per warp (8 lanes each) so that four independent row fetches are in flight per warp.  ||z||^2 is the
  // 32-lane sum of vq_exact.cuh bit for bit: lane j of a group plays the virtual lanes j, j + 8, j + 16, j + 24; the
  // first two tree levels (xor 16, xor 8) are in-thread sums of the same operand pairs, the last three are shuffles.
  const int wtotal = gridDim.x * (PREP_THREADS / 32);
  const int g = lane >> 3, j = lane & 7;
  int my_pairs = 0;
  for (int base = (blockIdx.x * (PREP_THREADS / 32) + warp) * 4; base < n + n2; base += wtotal * 4) {
    const int i = base + g;
    const bool active = i < n + n2;
    const int64_t row = active ? (i < n ? L.rows[i] : L.ovf_last[-(int64_t)(i - n)]) : 0;
    const uint32_t cand = (active && i < n) ? (uint32_t)L.cand[i] : 0u;
    const ZT* zr = z + row * D;
    float pm[4] = {0.f, 0.f, 0.f, 0.f};
    for (int c = 0; c < D; c += 32) {
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        const int d = c + j + 8 * m;
        if (d < D) { const float v = zf(__ldg(zr + d)); pm[m] = fmaf(v, v, pm[m]); }
      }
    }
    float zz = (pm[0] + pm[2]) + (pm[1] + pm[3]);
    zz += __shfl_xor_sync(0xffffffffu, zz, 4);
    zz += __shfl_xor_sync(0xffffffffu, zz, 2);
    zz += __shfl_xor_sync(0xffffffffu, zz, 1);
    if (active) {
      if (j == 0) {
        *zz_stash(zq, row, D) = zz;    // the row's z_q is rewritten by the emit kernel
        idx64[row] = ~0ull;
      }
      const bool all = i >= n || cand_is_all(cand, L.list_mode);   // overflow rows: every code
      for_each_candidate(cand, all, L.list_mode, nbins, j, 8, [&](int b) { atomicAdd(&s_cnt[b], 1); ++my_pairs; });
    }
  }
  __syncthreads();
  for (int b = tid; b < nbins; b += PREP_THREADS) {
    const int c = s_cnt[b];
    if (c) atomicAdd(bt.count + b, c);
  }
  my_pairs = (int)warp_sum((float)my_pairs);   // < 2^24 per warp: exact in FP32
  if (lane == 0 && my_pairs) atomicAdd(counters + CNT_PAIRS, my_pairs);
}

// exclusive scan of v[0..n) (n <= MAX_BINS) by a 1024-thread block; out[n] = total
__device__ __forceinline__ void block_scan_1024(int v, int n, int* out, int* s_warp) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int w = s_warp[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += t;
    }
    s_warp[lane] = w;   // inclusive over warps
  }
  __syncthreads();
  const int base = warp ? s_warp[warp - 1] : 0;
  if (tid < n) out[tid] = base + inc - v;
  if (tid == n - 1) out[n] = base + inc;
  __syncthreads();
}

__global__ void __launch_bounds__(PREP_THREADS, 1)
refine_scatter_kernel(int K, RefineList L, int* __restrict__ counters, BinTables bt, int* __restrict__ pairs, long long pair_cap,
                      int pair_warps) {
  __shared__ int s_start[MAX_BINS + 1];
  __shared__ int s_items[MAX_BINS + 1];
  __shared__ int s_cnt[MAX_BINS];
  __shared__ int s_base[MAX_BINS];
  __shared__ int s_warp[32];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n = counters[CNT_LISTED], n2 = L.list_mode ? counters[CNT_OVF] : 0;
  if (n + n2 == 0) return;
  const long long total = counters[CNT_PAIRS];
  if (total > pair_cap || total >= (1ll << 30)) {   // does not fit: the per-row kernel takes the whole list
    if (blockIdx.x == 0 && tid == 0) { counters[CNT_HANDBACK] = n; counters[CNT_HANDBACK_OVF] = n2; }
    return;
  }
  const int nbins = (K + 31) / 32;
  const int cnt = tid < nbins ? bt.count[tid] : 0;
  block_scan_1024(cnt, nbins, s_start, s_warp);
  // bucket slice per work item: about two items per warp of the pairs kernel, a multiple of the batch size
  int ch = (int)((total + 2ll * pair_warps - 1) / (2ll * pair_warps));
  ch = (ch + RB - 1) / RB * RB;
  ch = ch < RB ? RB : (ch > 4096 ? 4096 : ch);
  block_scan_1024((cnt + ch - 1) / ch, nbins, s_items, s_warp);
  if (blockIdx.x == 0) {
    for (int b = tid; b <= nbins; b += PREP_THREADS) { bt.start[b] = s_start[b]; bt.item_start[b] = s_items[b]; }
    if (tid == 0) bt.item_start[MAX_BINS + 1] = ch;
  }
  for (int b = tid; b < nbins; b += PREP_THREADS) s_cnt[b] = 0;
  __syncthreads();
  // this CTA's contiguous share of the listed rows: count, reserve, place.  One thread per row (a row has two or
  // three candidates); rows paired with every sub-chunk are spread over the warp.
  const int per = (n + n2 + gridDim.x - 1) / gridDim.x;
  const int i0 = blockIdx.x * per, i1 = min(n + n2, i0 + per);
  auto sweep = [&](auto&& f) {
    for (int ib = i0 + warp * 32; ib < i1; ib += PREP_THREADS) {
      const int i = ib + lane;
      const bool active = i < i1;
      const uint32_t cand = (active && i < n) ? (uint32_t)L.cand[i] : 0u;
      const bool all = active && (i >= n || cand_is_all(cand, L.list_mode));
      if (active && !all) for_each_candidate(cand, false, L.list_mode, nbins, 0, 1, [&](int b) { f(b, i); });
      unsigned am = __ballot_sync(0xffffffffu, all);
      while (am) {
        const int ii = ib + __ffs(am) - 1;
        am &= am - 1u;
        for (int b = lane; b < nbins; b += 32) f(b, ii);
      }
    }
  };
  sweep([&](int b, int) { atomicAdd(&s_cnt[b], 1); });
  __syncthreads();
  for (int b = tid; b < nbins; b += PREP_THREADS) {
    const int c = s_cnt[b];
    s_base[b] = c ? s_start[b] + atomicAdd(bt.cursor + b, c) : 0;
    s_cnt[b] = 0;
  }
  __syncthreads();
  sweep([&](int b, int i) { pairs[s_base[b] + atomicAdd(&s_cnt[b], 1)] = i; });
}

template <int DS, typename ZT>
__global__ void __launch_bounds__(PAIR_THREADS, DS <= 32 ? 2 : 1)
refine_pairs_kernel(const ZT* __restrict__ z, const float* __restrict__ E, const float* __restrict__ ee, int K, int D,
                    ZT* __restrict__ zq, unsigned long long* __restrict__ idx64, RefineList L, const int* __restrict__ pairs,
                    const int* __restrict__ counters, BinTables bt, long long pair_cap) {
  extern __shared__ __align__(16) float smem_f[];   // zs[warps][2][RB][DS] (ZT: bf16 rows are staged as bf16) | es
  __shared__ int s_start[MAX_BINS + 1];
  __shared__ int s_items[MAX_BINS + 1];
  constexpr int NW = PAIR_THREADS / 32;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n = counters[CNT_LISTED], n2 = L.list_mode ? counters[CNT_OVF] : 0;
  const long long total = counters[CNT_PAIRS];
  if (n + n2 == 0 || total == 0 || total > pair_cap || total >= (1ll << 30)) return;
  const int nbins = (K + 31) / 32;
  for (int b = tid; b <= nbins; b += PAIR_THREADS) { s_start[b] = bt.start[b]; s_items[b] = bt.item_start[b]; }
  __syncthreads();
  const int ch = bt.item_start[MAX_BINS + 1];
  const int items = s_items[nbins];
  constexpr int ZE = 16 / (int)sizeof(ZT);    // z elements per 16-byte piece
  ZT* zs = reinterpret_cast<ZT*>(smem_f) + warp * 2 * RB * DS;   // two halves: one being read, one being filled
  const int ns = D / DS;
  // sliced e_dim: the 32 code rows' slices are staged too ([32][DS + 4] floats, single-buffered: filled by coalesced
  // cp.async for the next step as soon as every lane has copied its own row into registers — conflict-free 128-bit loads —,
  // i.e. under this step's FMAs).
  // Each lane fetching its own row straight from global memory — 32 different lines per load instruction — took two
  // thirds of the LSU data pipe, which the ncu capture showed to be the kernel's bound (74 % busy, FMA pipe 24 %).
  constexpr int EP = DS + 4;
  float* es = reinterpret_cast<float*>(reinterpret_cast<ZT*>(smem_f) + NW * 2 * RB * DS) + warp * 32 * EP;
  for (int item = blockIdx.x * NW + warp; item < items; item += gridDim.x * NW) {
    // bucket of this item: the last b with item_start[b] <= item
    int lo = 0, hi = nbins;   // invariant: s_items[lo] <= item < s_items[hi]
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (s_items[mid] <= item) lo = mid; else hi = mid;
    }
    const int b = lo;
    const int p0 = s_start[b] + (item - s_items[b]) * ch;
    const int p1 = min(p0 + ch, s_start[b + 1]);
    const int code = b * 32 + lane;
    const bool valid = code < K;
    const float* erow = E + (size_t)(valid ? code : 0) * D;
    const float eek = valid ? __ldg(ee + code) : 0.f;
    float e[DS];
    if (ns == 1) {
#pragma unroll
      for (int d = 0; d < DS; d += 4) {
        const float4 v = ldg4(erow + d);
        e[d] = v.x; e[d + 1] = v.y; e[d + 2] = v.z; e[d + 3] = v.w;
      }
    }
    // Software pipeline over the (batch, slice) steps of the item: the z rows of the next step are copied into the
    // other half of the warp's staging buffer with cp.async (zero-filled for missing rows), and the
    // (row, ||z||^2) records of the next batch are read, while the current step is computed.
    constexpr int ZL = RB * (DS / ZE) / 32;   // 16-byte pieces per lane of one staged slice
    auto fetch_rows = [&](int p, int64_t& row_, float& zz_) {
      row_ = -1; zz_ = 0.f;
      if (p < p1 && lane < min(RB, p1 - p)) {
        row_ = listed_row(pairs[p + lane], n, L.rows, L.ovf_last);
        zz_ = *zz_stash(zq, row_, D);
      }
    };
    auto stage_e = [&](int sl) {   // (no commit of its own)
#pragma unroll
      for (int k = 0; k < DS / 4; ++k) {
        const int f = k * 32 + lane;
        const int cl = f / (DS / 4), c4 = f - cl * (DS / 4);
        const bool cv = b * 32 + cl < K;
        const float* src = E + (size_t)(cv ? b * 32 + cl : 0) * D + sl * DS + c4 * 4;
        const uint32_t dst = (uint32_t)__cvta_generic_to_shared(es + cl * EP + c4 * 4);
        cp_async_cg16(dst, src, cv ? 16 : 0);
      }
    };
    auto stage_z = [&](int64_t row_, int sl, int buf) {
#pragma unroll
      for (int k = 0; k < ZL; ++k) {
        const int f = k * 32 + lane;
        const int r = f / (DS / ZE), c4 = f - r * (DS / ZE);
        const long long rr = __shfl_sync(0xffffffffu, (long long)row_, r);
        const ZT* src = rr >= 0 ? z + rr * D + sl * DS + c4 * ZE : z;
        const uint32_t dst = (uint32_t)__cvta_generic_to_shared(zs + buf * RB * DS + r * DS + c4 * ZE);
        cp_async_cg16(dst, src, rr >= 0 ? 16 : 0);
      }
      cp_async_commit();
    };
    int64_t row, row_n;
    float zz, zz_n;
    int buf = 0;
    fetch_rows(p0, row, zz);
    if (ns > 1) stage_e(0);   // same group as the first z rows
    stage_z(row, 0, 0);
    for (int p = p0; p < p1; p += RB) {
      const int nb = min(RB, p1 - p);
      fetch_rows(p + RB, row_n, zz_n);
      float acc[RB];
#pragma unroll
      for (int r = 0; r < RB; ++r) acc[r] = 0.f;
      for (int sl = 0; sl < ns; ++sl) {
        __syncwarp();   // the previous step's reads of the other half are done
        if (sl + 1 < ns) stage_z(row, sl + 1, buf ^ 1);
        else if (p + RB < p1) stage_z(row_n, 0, buf ^ 1);
        else cp_async_commit();   // keep one group per step
        cp_async_wait<1>();       // this step's rows (and code slices) have landed
        __syncwarp();
        if (ns > 1) {
          const float* eb = es + lane * EP;
#pragma unroll
          for (int d = 0; d < DS; d += 4) {
            const float4 v = *reinterpret_cast<const float4*>(eb + d);
            e[d] = v.x; e[d + 1] = v.y; e[d + 2] = v.z; e[d + 3] = v.w;
          }
          __syncwarp();   // every lane has its row: the buffer takes the next step's slices (a group of its own, older than
                          // the next step's z group, so that step's wait_group 1 covers it)
          if (sl + 1 < ns || p + RB < p1) {
            stage_e(sl + 1 < ns ? sl + 1 : 0);
            cp_async_commit();
          }
        }
        const ZT* zb = zs + buf * RB * DS;
        buf ^= 1;
#pragma unroll
        for (int d = 0; d < DS; d += 4) {
#pragma unroll
          for (int r = 0; r < RB; ++r) {
            const float4 z4 = zld4(zb + r * DS + d);   // broadcast read
            acc[r] = fmaf(z4.x, e[d], acc[r]);
            acc[r] = fmaf(z4.y, e[d + 1], acc[r]);
            acc[r] = fmaf(z4.z, e[d + 2], acc[r]);
            acc[r] = fmaf(z4.w, e[d + 3], acc[r]);
          }
        }
      }
#pragma unroll
      for (int r = 0; r < RB; ++r) {
        if (r < nb) {   // warp-uniform
          const float zzr = __shfl_sync(0xffffffffu, zz, r);
          const unsigned long long best = warp_argmin(dist_key(valid ? exact_dist(acc[r], zzr, eek) : INFINITY), b * 32);
          const long long rr = __shfl_sync(0xffffffffu, (long long)row, r);
          if (lane == 0) atomicMin(idx64 + rr, best);
        }
      }
      row = row_n; zz = zz_n;
    }
  }
}

template <bool TRAIN, typename ZT>
__global__ void __launch_bounds__(PREP_THREADS, 1)
refine_emit_kernel(const ZT* __restrict__ z, const float* __restrict__ E, int D, ZT* __restrict__ zq,
                   unsigned long long* __restrict__ idx64, unsigned long long* __restrict__ hist, double* __restrict__ sse,
                   RefineList L, const int* __restrict__ counters, long long pair_cap) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n = counters[CNT_LISTED], n2 = L.list_mode ? counters[CNT_OVF] : 0;
  const long long total = counters[CNT_PAIRS];
  if (n + n2 == 0 || total > pair_cap || total >= (1ll << 30)) return;
  const int wtotal = gridDim.x * (PREP_THREADS / 32);
  const int g = lane >> 3, j = lane & 7;   // four rows per warp, 8 lanes each: four independent fetch chains in flight
  double lsse = 0.0;
  for (int base = (blockIdx.x * (PREP_THREADS / 32) + warp) * 4; base < n + n2; base += wtotal * 4) {
    const int i = base + g;
    const bool active = i < n + n2;
    const int64_t row = active ? listed_row(i, n, L.rows, L.ovf_last) : 0;
    const int bidx = active ? packed_winner(idx64[row]) : 0;
    ZT* orow = zq + row * D;
    const float* erow = E + (int64_t)bidx * D;
    const ZT* zsrc = z + row * D;
    if (active) {
      for (int c = j * 4; c < D; c += 32) {
        float4 o4 = ldg4(erow + c);
        if (TRAIN) o4 = st_step4(o4, zldg4(zsrc + c), lsse);
        zst4(orow + c, o4);
      }
    }
    __syncwarp();   // every lane of the group has read idx64[row] before it is overwritten
    if (active && j == 0) {
      idx64[row] = (unsigned long long)bidx;
      if (TRAIN) atomicAdd(hist + bidx, 1ull);
    }
  }
  if (TRAIN) {
    lsse = warp_sum(lsse);
    if (lane == 0 && lsse != 0.0) atomicAdd(sse, lsse);
  }
}

}  // namespace

size_t vq_refine_binned_bytes(int64_t N) {
  return align_up(sizeof(int) * (size_t)(4 * MAX_BINS + 8), 256) + align_up(sizeof(int) * 2 * (size_t)N, 256);
}

// the bin tables are zeroed by the caller (count, cursor: the first 2 * MAX_BINS ints of `ws`)
size_t vq_refine_binned_zero_bytes() { return sizeof(int) * 2 * MAX_BINS; }

template <typename ZT>
static int launch_binned_t(const ZT* z, ZT* z_q, const VqCall& c, const RefineList& L, long long pair_cap) {
  const int K = c.K, D = c.D;
  if (K > 32 * MAX_BINS) return fail(DVQ_ERR_BAD_SHAPE, "binned refine handles K <= %d", 32 * MAX_BINS);
  int* wi = static_cast<int*>(c.binned);
  BinTables bt;
  bt.count = wi; bt.cursor = wi + MAX_BINS; bt.start = wi + 2 * MAX_BINS; bt.item_start = wi + 3 * MAX_BINS + 1;
  int* pairs = reinterpret_cast<int*>(static_cast<char*>(c.binned) + align_up(sizeof(int) * (size_t)(4 * MAX_BINS + 8), 256));
  if (pair_cap <= 0 || pair_cap > 2 * (long long)c.N) pair_cap = 2 * (long long)c.N;   // the pair list holds 2 N entries
  unsigned long long* idx64 = reinterpret_cast<unsigned long long*>(c.idx);
  // slice width of the pairs kernel: a lane keeps DS floats of its code row in registers.  DS = 64 (168 registers, one CTA
  // of 12 warps per SM) re-reads a code row half as often, DS = 32 (80 registers) fits two CTAs per SM: measured at
  // N = 2M-4M, refine stage: e_dim 128 / 256 / 512 at K = 16 384 / 16 384 / 4096: 0.60 -> 0.44, 1.85 -> 1.37, 2.32 -> 1.71 ms
  // with DS = 32; e_dim 64 (one slice at DS = 64: the code row stays in registers for the whole work item): 0.15 -> 0.19 ms at
  // K = 2048.  Hence 32 from e_dim 128 on.  DVQ_REFINE_DS=32|64 overrides (A/B runs).
  static const char* ds_env = getenv("DVQ_REFINE_DS");
  const int ds_want = ds_env ? atoi(ds_env) : (D >= 128 ? 32 : 64);
  const int DS = D < 64 ? D : (ds_want == 32 ? 32 : 64);
  const int pair_grid = c.sm_count * (DS <= 32 && D >= 64 ? 2 : 1);
  const int pair_warps = pair_grid * (PAIR_THREADS / 32);

  refine_prep_kernel<<<c.sm_count, PREP_THREADS, 0, c.s>>>(z, D, K, z_q, idx64, L, c.counters, bt);
  DVQ_CUDA_CHECK(cudaGetLastError());
  refine_scatter_kernel<<<c.sm_count, PREP_THREADS, 0, c.s>>>(K, L, c.counters, bt, pairs, pair_cap, pair_warps);
  DVQ_CUDA_CHECK(cudaGetLastError());
  const size_t smem = (size_t)(PAIR_THREADS / 32) * (2 * RB * DS * sizeof(ZT) + (D > DS ? 32 * (DS + 4) * sizeof(float) : 0));
#define DVQ_LAUNCH_PAIRS(DS_)                                                                                              \
  do {                                                                                                                     \
    DVQ_CUDA_CHECK(cudaFuncSetAttribute(refine_pairs_kernel<DS_, ZT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    refine_pairs_kernel<DS_, ZT><<<pair_grid, PAIR_THREADS, smem, c.s>>>(z, c.E, c.ee, K, D, z_q, idx64, L, pairs, c.counters, \
                                                                     bt, pair_cap);                                        \
  } while (0)
  if (DS == 64) DVQ_LAUNCH_PAIRS(64);
  else if (DS == 32) DVQ_LAUNCH_PAIRS(32);
  else if (DS == 16) DVQ_LAUNCH_PAIRS(16);
  else return fail(DVQ_ERR_BAD_SHAPE, "binned refine needs e_dim 16, 32 or a multiple of 64");
#undef DVQ_LAUNCH_PAIRS
  DVQ_CUDA_CHECK(cudaGetLastError());
  if (c.train)
    refine_emit_kernel<true, ZT><<<c.sm_count, PREP_THREADS, 0, c.s>>>(z, c.E, D, z_q, idx64, c.hist, c.sse, L, c.counters, pair_cap);
  else
    refine_emit_kernel<false, ZT><<<c.sm_count, PREP_THREADS, 0, c.s>>>(z, c.E, D, z_q, idx64, c.hist, c.sse, L, c.counters, pair_cap);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch(4);
  return DVQ_OK;
}

int launch_vq_refine_binned(const VqCall& c, const RefineList& list, long long pair_cap) {
  return with_z_type(c, [&](auto z, auto z_q) { return launch_binned_t(z, z_q, c, list, pair_cap); });
}

}  // namespace dvq
