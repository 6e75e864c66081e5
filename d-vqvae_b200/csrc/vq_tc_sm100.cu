// tcgen05 VQ kernel: tensor-core distance filter fused with the row argmin, the codebook gather,
// the straight-through / SSE reduction and the usage histogram.  The rows whose winner the filter
// cannot decide *rigorously* are appended to a device-side list and re-evaluated by the exact
// FP32 kernel (vq_simt_fp32.cu) — "filter and refine" (SURVEY §7.4).
//
// Contraction.  For a 128-row tile the accumulator is
//     acc[n,k] = g_n * (B_n + ee_k) - 2 z'_n . e'_k        (z' = s_n z, e' = s_E e, g_n = s_n s_E)
// with power-of-two scales s_n (per row) and s_E (per codebook) that put every operand inside the
// FP16 range, ee_k = ||e_k||^2 and the bias B_n >= 2 |z_n| max_k|e_k| which keeps acc >= 0.
// It is ONE chain of tcgen05.mma (kind::f16, FP32 accumulate in TMEM, M=128, N<=256, K=16):
//     A row  = [ zh (D) | fold (16) ]     zh = fp16(z')      (USE_ZL adds zl = fp16(z' - zh) as a second product)
//     B row  = [ eh (D) | fold (16) ]     eh = fp16(-2 e')
// issued as zh.eh + fold.fold; the fold columns carry g_n*B_n and g_n*ee_k as products of FP16 pairs
// (ee_k split in three FP16 terms).  Because acc >= 0 its bit pattern is monotone, so the epilogue
// reduces raw accumulators with 3-input FMNMX3 minima and recovers the winning column from the
// indicator bit masks of its ambiguity count (no per-element index packing).
//
// Rigor.  eps_n bounds |acc - exact| for every k of row n (operand rounding: |z'| * max_k||eh_k+2e'_k||
// measured exactly by the prep kernel; ||z' - zh|| * max_k||eh_k|| measured exactly by the converter;
// tensor-core FP32 accumulation; ee rounding).  A row is decided iff no other key lies within
// 2*eps_n of the minimum; the count of such keys is kept with a running (never too small) threshold,
// exact resets, and FFMA.SAT / FFMA2 arithmetic on the FMA pipe.  Undecided rows (a few %) go to the list.
//
// Pipeline (one persistent CTA per SM, 24 warps in six warpgroups; every SM sub-partition hosts 1 converter,
// 3 epilogue and 1 gather warp):
//   warp 0      producer : cp.async.bulk (TMA engine) z tile fp32 -> staging ring (2 x 128 x D x 4 B)
//   warp 1      MMA      : one elected lane issues tcgen05.mma from uniform-register descriptors; the warp
//                          then waits for the chunk's commit mbarrier and relays it on named barriers
//   warp 2      streamer : codebook chunks -> ring of 2-3 slots when the operand image is not resident
//   warp 3      relay    : waits for each chunk's tcgen05.commit mbarrier and releases the filter warps (named barriers)
//   warps 4-7   convert  : staging -> scales / norms / bounds -> FP16 A image (2 stages)
//   warps 8-19  epilogue : tcgen05.ld TMEM -> min tree + ambiguity masks per 32-code sub-chunk; three warps
//                          per TMEM lane quarter split the columns, the owner merges and writes idx / histogram
//   warps 20-23 gather   : E[idx] (128-bit loads, two batches in flight per lane, z rows requested before the
//                          codes arrive), z_q, SSE, refine-list append
// The control warpgroup (warps 0-3) releases registers with setmaxnreg and the gather warpgroup takes them.
// Warp-to-warp hand-offs are hardware named barriers (bar.arrive / bar.sync), mbarriers only where the
// async proxy signals.  TMEM: 512 columns = 2 accumulator stages of 256, so the MMA of one 256-code
// chunk overlaps the epilogue of the previous one.  The codebook operand image (K x (D+16) fp16) stays
// resident in shared memory for K <= 512 and is streamed per row tile above — by one CTA per SM, or (template
// parameter PAIR: e_dim 512, e_dim 128 / 256 from K = 2048 on) by CTA pairs that run one M = 256 tcgen05.mma.cta_group::2
// per k-step over both SMs' row tiles and stream half of every operand block each (see the comment above vq_tc_kernel).
#include <cuda.h>        // CUtensorMap (the encoder is fetched through cudaGetDriverEntryPoint: no libcuda link dependency)
#include <cuda_fp16.h>
#include <cstddef>
#include <cstdlib>
#include <cstring>

#include "dvq_common.cuh"
#include "f32x2.cuh"
#include "tc_prims.cuh"

namespace dvq {
namespace {

constexpr int TM = 128;                 // rows per tile
constexpr int A_CHUNK_BYTES = TM * 16 + 32;  // one 8-wide k-chunk of the A image (+32 B: bank spreading)
// Warp roles are laid out in aligned groups of four (warpgroups) so that a group can resize its register
// allocation with setmaxnreg: warps 0-3 producer / MMA issuer / codebook streamer / completion relay, 4-7 converters,
// 8-19 epilogue (three warpgroups: one warp per TMEM lane quarter each), 20-23 gather.
constexpr int BLOAD_WARP = 2;                // codebook streamer (active when the image is not resident)
constexpr int CONV_WARP0 = 4;
constexpr int EPI_WARP0 = 8;
#ifdef DVQ_EPQ4   // experiment: four epilogue warps per lane quarter (28 warps, 72 registers per thread at launch)
constexpr int EPQ = 4;
#else
constexpr int EPQ = 3;                       // epilogue warps per TMEM lane quarter (they split the columns)
#endif
constexpr int EPI_WARPS = 4 * EPQ;
constexpr int GATHER_WARP0 = EPI_WARP0 + EPI_WARPS;
constexpr int GATHER_WARPS = 4;
constexpr int NUM_WARPS = GATHER_WARP0 + GATHER_WARPS;
// The launch gives each of the 768 threads 80 registers (warp allocations come in units of 512).  The control
// group hands 32 per thread back and the gather group takes them: its two batches of 128-bit loads in flight
// (plus the z rows requested ahead of the codes) do not fit 80.  The trade must balance inside the CTA's own
// allocation — setmaxnreg.inc only draws from what the CTA released: 128 * (48 + 80 + 112) + 384 * 80 = 61 440.
#ifdef DVQ_EPQ4   // the launch hands out 896 * 72 = 64 512 registers: 128 * (40 + 72 + 104) + 512 * 72 = 64 512
constexpr int REGS_CTRL = 40, REGS_GATHER = 104;
#else
constexpr int REGS_CTRL = 48, REGS_GATHER = 112;
#endif
// streamed-codebook variant (ST): control 40, converter 64, gather 64, epilogue 104 (128 * (40 + 64 + 64) + 384 * 104 = 61 440)
constexpr int REGS_ST_CTRL = 40, REGS_ST_SIDE = 64, REGS_ST_EPI = 104;
constexpr int DSLICE = 64;                   // e_dim is contracted in slices of at most 64 columns
// slice width: the whole row up to 64 columns, 64-column slices up to e_dim 256, 32-column slices for e_dim 512
// (the resident A image of 128 x 528 halfs leaves room for only small staging / ring slots)
__host__ __device__ inline int slice_width(int D) { return D <= DSLICE ? D : (D <= 256 ? DSLICE : 32); }
constexpr int NTHREADS = NUM_WARPS * 32;
constexpr int META_SLOTS = 4;
// true: A row = [zh | zl | fold] (22-bit z, two products per code); false: A row = [zh | fold] and the exact norm
// of the dropped residual enters the error bound (about twice the band, hence twice the undecided rows, for
// 44 % fewer tensor-core k-steps and shared-memory operand reads)
constexpr bool USE_ZL = false;

enum ErrCode { ERR_STAGE_FULL = 1, ERR_STAGE_EMPTY, ERR_A_FULL, ERR_A_EMPTY, ERR_ACC_FULL, ERR_ACC_EMPTY, ERR_B_FULL, ERR_FIN, ERR_SIDX, ERR_NOT_PREPARED,
               ERR_PEER_A_FULL, ERR_PEER_ACC_EMPTY };

struct CbMeta {          // written by the prep kernels, read by the main kernel
  float s_E;             // power-of-two codebook scale
  float b0;              // fp16-representable upper bound of s_E * max_k ||e_k||
  float eh_norm_bound;   // >= max_k ||eh_k||
  float delta_max;       // >= max_k ||eh_k - (-2 s_E e_k)||   (exact FP16 rounding residual)
  int half_E;            // s_E = 2^(10 - half_E)
  int degenerate;        // 1: codebook all-zero / non-finite -> every row goes to the exact kernel
  int magic;             // cb_magic(K, D) once the preparation of this shape is complete (checked when DVQ_CODEBOOK_CACHED reuses it)
};
__host__ __device__ inline int cb_magic(int K, int D, bool pair = false) { return (0x44565100 ^ (K << 12) ^ D) + (pair ? 0x40000000 : 0); }

struct TcParams {
  CUtensorMap ztile;      // z as a [N, D] tensor, box = (slice columns, 128 rows): the staged slices of e_dim > 64 (one TMA load each)
  CUtensorMap bmap[2];    // CTA-pair kernel: the operand image as [bytes / 1024, 256] int32, box = one half block without ([0]) / with ([1]) the fold columns
  const void* z;          // [N, D] fp32 or bf16 (the kernel's ZT)
  const float* E;
  const uint8_t* bimg;
  const CbMeta* cb;
  int64_t N;
  int K, D, train;
  void* zq;               // [N, D] ZT
  int64_t* idx;
  unsigned long long* hist;
  double* sse;
  int* counters;        // CounterSlot (dvq_common.cuh)
  int* row_list;
  int* cand_list;       // candidate record of each listed row (dvq_common.cuh)
  int layout_ovr;       // smem_layout override (0 = automatic)
  unsigned long long* stats;   // optional wait-time accounting (DVQ_TC_STATS builds)
  int64_t ntiles;
};

constexpr int MAX_BSLOTS = 8;           // ring slots of the streamed codebook image (barrier arrays)
constexpr int MAX_BSLOTS_SOLO = 4;      // single-CTA kernel: largest ring the layout search considers (whole 256-code blocks)

struct SmemLayout {
  uint32_t bimg, a_img[2], stage[2], meta, fin, sidx, hist, total;
  uint32_t bimg_bytes, a_bytes, stage_bytes;   // bimg_bytes: the codebook ring (nslots slots) in shared memory
  uint32_t bchunk_bytes, hist_in_smem;           // one ring slot: (256 codes) x (one e_dim slice + the fold columns)
  uint32_t ns, ds, a_bufs, bslice_bytes;         // e_dim = ns slices of ds columns; a slice without the fold columns
  uint32_t nslots, nstage;                       // ring slots (2..MAX_BSLOTS), z staging slots (1..2)
  uint32_t bcodes;                               // codes per ring slot: 256, or 128 in the CTA-pair kernel (each CTA holds half a block)
};

constexpr uint32_t SMEM_LIMIT = 227u * 1024u - 640u;   // dynamic shared memory budget (alignment slack + static barriers)

__host__ __device__ inline uint32_t smem_place(SmemLayout& L, int K) {
  uint32_t off = 0;
  L.bimg_bytes = L.nslots * L.bchunk_bytes;
  L.bimg = off; off += (L.bimg_bytes + 127u) & ~127u;
  L.a_img[0] = off; off += (L.a_bytes + 127u) & ~127u;
  L.a_img[1] = L.a_bufs == 2 ? off : L.a_img[0];
  if (L.a_bufs == 2) off += (L.a_bytes + 127u) & ~127u;
  L.stage[0] = off; off += L.stage_bytes;
  L.stage[1] = L.nstage == 2 ? off : L.stage[0];
  if (L.nstage == 2) off += L.stage_bytes;
  L.meta = off; off += META_SLOTS * TM * 4;
  L.fin = off; off += EPQ * TM * 16;         // up to EPQ helper warps (EPQ + 1 warps per quarter when the converters join) x (key, col, cnt, cand); single slot
  L.sidx = off; off += 2 * TM * 4;      // 2 slots of the hand-off word (code offset | undecided flag + candidates)
  L.hist = off; off += L.hist_in_smem ? (uint32_t)K * 4 : 0u;
  L.total = off;
  return off;
}

// `ovr` != 0 forces (A images, z staging slots, ring slots) = (ovr / 100, ovr / 10 % 10, ovr % 10) for a streamed image
// (experiments: DVQ_TC_LAYOUT; the launch passes it to the kernel so that both sides agree)
// `pair`: layout of the CTA-pair kernel (cta_group::2) — always streamed, a ring slot holds this CTA's half (128 codes) of a block
// `zbytes`: size of a z element (4 fp32, 2 bf16): a staging slot holds 128 rows of one slice.  Which kernel and layout class a shape
// gets is decided on the fp32 plan (vq_tc_supported, vq_tc_pair_selected); the smaller bf16 slots only re-run the search below.
__host__ __device__ inline SmemLayout smem_layout(int K, int D, int ovr = 0, bool pair = false, int zbytes = 4) {
  SmemLayout L;
  L.ds = (uint32_t)slice_width(D);
  L.ns = (uint32_t)D / L.ds;
  L.bcodes = pair ? 128u : 256u;
  const uint32_t kc_s = L.ds / 8, kc_a = (uint32_t)((USE_ZL ? 2 : 1) * D + 16) / 8;
  L.bslice_bytes = kc_s * L.bcodes * 16u;
  L.bchunk_bytes = (kc_s + 2u) * L.bcodes * 16u;
  L.a_bytes = kc_a * A_CHUNK_BYTES;
  L.stage_bytes = (uint32_t)TM * L.ds * (uint32_t)zbytes;
  const uint32_t nchunks = (uint32_t)(K + 255) / 256;
  if (!pair && nchunks * L.ns <= 2) {
    // resident operand image (two slots hold it for the life of the CTA).  Preference order when shared memory is
    // short: drop the shared-memory histogram (global atomics), then the second A image (the converters then
    // wait for the previous tile's MMAs)
    L.nslots = 2; L.nstage = 2;
    for (int attempt = 0; attempt < 3; ++attempt) {
      L.hist_in_smem = (K <= 512 && attempt == 0) ? 1u : 0u;   // larger histograms go straight to global atomics
      L.a_bufs = attempt < 2 ? 2u : 1u;
      if (smem_place(L, K) <= SMEM_LIMIT) break;
    }
    return L;
  }
  // streamed image: blocks in flight hide the L2 latency.  Measured (N = 16.8 M): a third ring slot is worth +7 % at
  // e_dim 128, K = 16 384 even at the price of a single A image and a single staging slot, but with a single A
  // image K = 2048 / 4096 lose 10-17 % (the MMAs stall while each tile is converted).  Hence: from 32 chunks per
  // tile on the third slot comes first; from 8 chunks on it only replaces the second z staging slot (a tile lasts
  // long enough for one); below that the layout of the resident case is kept.
  L.hist_in_smem = 0u;
  if (ovr) {
    L.a_bufs = (uint32_t)(ovr / 100); L.nstage = (uint32_t)(ovr / 10 % 10); L.nslots = (uint32_t)(ovr % 10);
    smem_place(L, K);
    return L;
  }
  if (!pair && ((nchunks == 2 && (L.ns == 2 || L.ns == 4)) || (nchunks == 4 && L.ns == 2))) {
    // Few blocks per tile at e_dim 128 / 256: measured layouts (N = 16.8 M, filter kernel; profiles/README.md).  A tile is short,
    // so what counts is the per-tile chain load -> convert -> MMA -> filter, and a smaller footprint leaves the gather more L1:
    //   K <= 512, e_dim 128 (4 blocks):  (1, 1, 2) 5.17 ms, (2, 1, 2) 5.21, (1, 1, 3) 5.34, (1, 2, 2) 5.66, (2, 2, 2) 6.22
    //   K <= 512, e_dim 256 (8 blocks):  (1, 1, 2) 11.49 ms, (1, 2, 2) 13.43 / 13.48
    //   K = 1024, e_dim 128 (8 blocks):  (2, 1, 2) 6.23 ms, (2, 2, 2) 6.62, (1, 2, 2) 6.98, (1, 1, 2) 7.28, (1, 1, 3) 7.35
    const bool two_a = nchunks == 4;   // K = 1024 at e_dim 128: the second A image pays once a tile has four chunks
    L.a_bufs = two_a ? 2 : 1; L.nstage = 1; L.nslots = 2;
    if (smem_place(L, K) <= SMEM_LIMIT) return L;
  }
  if (pair) {
    // CTA-pair kernel, measured layouts (N = 4M, filter kernel; profiles/r02_ab_pair_layouts.jsonl); everything else
    // follows the general rule below, which was at or within 1 % of the best layout tried:
    //   e_dim 512, K >= 4096: one z staging slot and a ring of five (1, 1, 5) instead of (1, 2, 4):
    //                         K = 4096 19.5 vs 20.0 ms, K = 8192 35.3 vs 37.0, K = 16 384 64.2 vs 70.0 (K <= 2048: 6-13 % slower)
    //   e_dim 256, K = 4096: one A image, two staging slots, ring of four (1, 2, 4) instead of (2, 1, 2): 7.17 vs 7.93 ms
    //                         (N = 16.8M: 35.3 vs 38.7); K = 8192: 13.8 vs 14.2 at N = 4M but 62.8 vs 61.8 at N = 16.8M,
    //                         K = 2048 and K = 16 384 2 % slower: not applied there
    if (L.ns == 16 && nchunks >= 16) {
      L.a_bufs = 1; L.nstage = 1; L.nslots = 5;
      if (smem_place(L, K) <= SMEM_LIMIT) return L;
    }
    if (L.ns == 4 && nchunks >= 16 && nchunks < 32) {
      L.a_bufs = 1; L.nstage = 2; L.nslots = 4;
      if (smem_place(L, K) <= SMEM_LIMIT) return L;
    }
  }
  uint32_t best_score = 0, best_a = 1, best_st = 1, best_sl = 2;
  for (uint32_t a = 2; a >= 1; --a)
    for (uint32_t st = 2; st >= 1; --st)
      for (uint32_t sl = pair ? MAX_BSLOTS : MAX_BSLOTS_SOLO; sl >= 2; --sl) {
        L.a_bufs = a; L.nstage = st; L.nslots = sl;
        if (smem_place(L, K) > SMEM_LIMIT) continue;
        const uint32_t sl3 = sl < 3u ? sl : 3u;
        const uint32_t score = nchunks >= 32 ? sl3 * 100u + a * 10u + st + sl
                             : nchunks >= 8  ? a * 100u + sl3 * 10u + st
                                             : a * 100u + st * 10u + sl;
        if (score > best_score) { best_score = score; best_a = a; best_st = st; best_sl = sl; }
        break;   // the largest ring for this (a, st)
      }
  L.a_bufs = best_a; L.nstage = best_st; L.nslots = best_sl;
  smem_place(L, K);   // (total > SMEM_LIMIT if nothing fits: vq_tc_supported rejects the shape)
  return L;
}

// ------------------------------------------------------------------------------------------------
// codebook preparation (tiny): scale, FP16 operand image, exact rounding residual
// ------------------------------------------------------------------------------------------------
__global__ void tc_cb_stats_kernel(const float* __restrict__ ee, int K, int D, CbMeta* __restrict__ cb, int* __restrict__ counters,
                                   int* __restrict__ zero_ints, int zero_n, bool pair) {
  __shared__ float red[32];
  for (int i = threadIdx.x; i < zero_n; i += blockDim.x) zero_ints[i] = 0;   // bin tables of the binned refine
  float m = 0.f;
  bool bad = false;
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    const float v = ee[k];
    if (!(v >= 0.f) || v > 1e30f) bad = true;
    m = fmaxf(m, v);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  bad = __syncthreads_or(bad);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) m = fmaxf(m, red[w]);
    CbMeta c;
    c.degenerate = (bad || !(m > 1e-30f)) ? 1 : 0;
    const float emax = sqrtf(m) * (1.f + 1e-6f) ;
    int ex = 0;
    if (!c.degenerate) ex = (int)((__float_as_uint(emax) >> 23) & 255u) - 127;   // emax in [2^ex, 2^(ex+1))
    c.half_E = ex;
    c.s_E = c.degenerate ? 1.f : exp2f((float)(10 - ex));                        // s_E*emax in [2^10, 2^11)
    c.b0 = __half2float(__float2half_ru(c.s_E * emax * (1.f + 1e-6f)));
    c.eh_norm_bound = 2.f * c.s_E * emax * (1.f + 1.f / 512.f);
    c.delta_max = 0.f;
    c.magic = cb_magic(K, D, pair);
    *cb = c;
    for (int i = 0; i < CNT_WORDS; ++i) counters[i] = 0;
  }
}

// per-call reset when the codebook preparation is reused (DVQ_CODEBOOK_CACHED)
__global__ void tc_reset_kernel(int* __restrict__ counters, int* __restrict__ zero_ints, int zero_n) {
  for (int i = threadIdx.x; i < zero_n; i += blockDim.x) zero_ints[i] = 0;
  if (threadIdx.x < CNT_WORDS) counters[threadIdx.x] = 0;
}

// byte offset of element (code k, column d) in the global operand image: one block per (256-code chunk,
// e_dim slice), each block laid out [d' / 8][k % 256][d' % 8] halfs exactly as its shared-memory ring slot;
// the 16 fold columns (d >= D) follow the last slice of a chunk inside the same block
// CTA-pair image (`pair`): every block is stored as two half blocks [d' / 8][k' % nh][d' % 8] of 128-code capacity, the
// first holding the lower half of the chunk's codes (nh = codes in the chunk / 2; CTA 0's B operand), the second the upper
// half (CTA 1's) — the split cta_group::2 expects of an N-wide B operand.
__host__ __device__ inline size_t bimg_offset(int k, int d, int D, int K = 0, bool pair = false) {
  const int ds = slice_width(D), ns = D / ds;
  const size_t block_bytes = (size_t)(ds / 8 + 2) * 256 * 16;
  const int sl = d < D ? d / ds : ns - 1;
  const int dd = d < D ? d - sl * ds : ds + (d - D);
  if (pair) {
    const int c = k >> 8, kk = k & 255;
    const int nh = (K - c * 256 < 256 ? K - c * 256 : 256) / 2;
    const int half = kk >= nh ? 1 : 0;
    return (((size_t)c * ns + sl) * 2 + half) * (block_bytes / 2) + (size_t)(dd >> 3) * (128 * 16) + (size_t)(kk - half * nh) * 16 + (size_t)(dd & 7) * 2;
  }
  return ((size_t)(k >> 8) * ns + sl) * block_bytes + (size_t)(dd >> 3) * (256 * 16) + (size_t)(k & 255) * 16 + (size_t)(dd & 7) * 2;
}

// one warp per code: eh = fp16(-2 s_E e), fold columns, residual norm -> atomic max
__global__ void tc_cb_image_kernel(const float* __restrict__ E, const float* __restrict__ ee, int K, int D,
                                   CbMeta* __restrict__ cb, uint8_t* __restrict__ bimg, bool pair) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= K) return;
  const float sE = cb->s_E;
  const float* row = E + (int64_t)warp * D;
  float res = 0.f;
  for (int d = lane; d < D; d += 32) {
    const float v = -2.f * sE * __ldg(row + d);
    const __half h = __float2half_rn(v);
    const float r = v - __half2float(h);       // exact
    res = fmaf(r, r, res);
    *reinterpret_cast<__half*>(bimg + bimg_offset(warp, d, D, K, pair)) = h;
  }
  res = warp_sum(res);
  if (lane < 16) {   // fold k-chunks D/8 and D/8+1
    float v = 0.f;
    const float q = (sE * __ldg(ee + warp)) * sE * (1.f / 256.f);   // this order cannot overflow
    const float hi = __half2float(__float2half_rn(q));
    const float mid = __half2float(__float2half_rn(q - hi));
    const float lo = __half2float(__float2half_rn(q - hi - mid));
    if (lane == 0) v = cb->b0;
    if (lane == 1) v = hi;
    if (lane == 2) v = mid;
    if (lane == 3) v = lo;
    const int d = D + lane;
    *reinterpret_cast<__half*>(bimg + bimg_offset(warp, d, D, K, pair)) = __float2half_rn(v);
  }
  if (lane == 0) atomicMax(reinterpret_cast<int*>(&cb->delta_max), __float_as_int(sqrtf(res) * (1.f + 1e-5f)));
}

// ------------------------------------------------------------------------------------------------
// main kernel
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float min3f(float a, float b, float c) {
  float r;
  asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
__device__ __forceinline__ float fma_sat(float a, float b, float c) {
  float r;
  asm("fma.rn.sat.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
// tcgen05.wait::ld that also carries a register dependence on the loaded values, so the compiler
// cannot move their consumers above the wait
__device__ __forceinline__ void tmem_ld_wait_dep(uint32_t (&v)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                 "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]),
                 "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]),
                 "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
               :
               : "memory");
}
__device__ __forceinline__ void warp_arrive(uint32_t bar) {   // one arrival per warp, after all lanes are done
  __syncwarp();
  if ((threadIdx.x & 31) == 0) tc::mbar_arrive_a(bar);
}
// Hardware named barriers for the warp <-> warp hand-offs: a warp blocked in bar.sync issues nothing
// (an mbarrier poll loop was measured to burn ~19 % of the SM's issue slots).  bar.arrive / bar.sync
// order the participants' shared-memory accesses (PTX producer/consumer pattern).  `nthreads` counts
// arrivers + waiters.  mbarriers remain only where the async proxy signals (bulk copies, tcgen05.commit).
__device__ __forceinline__ void nb_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
__device__ __forceinline__ void nb_arrive(int id, int nthreads) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
// Bounded mbarrier wait; a protocol bug records its code and traps (a loud launch failure, never a hang).
__device__ __forceinline__ void wait_or_trap(uint32_t bar, uint32_t parity, int* err_out, int code) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b32 n;\n\t"
      "mov.b32 n, 0;\n\t"
      "DVQ_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "@p bra DVQ_DONE;\n\t"
      "add.u32 n, n, 1;\n\t"
      "setp.lt.u32 p, n, %4;\n\t"
      "@p bra DVQ_WAIT;\n\t"
      "DVQ_DONE:\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity), "r"(100000u), "r"(1u << 22)
      : "memory");
  if (!ok) {
    *err_out = code;
    __threadfence_system();
    __trap();
  }
}

// The same wait with acquire semantics at cluster scope: the phase was completed by the peer CTA's remote arrive
__device__ __forceinline__ void wait_or_trap_cluster(uint32_t bar, uint32_t parity, int* err_out, int code) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b32 n;\n\t"
      "mov.b32 n, 0;\n\t"
      "DVQ_CWAIT:\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "@p bra DVQ_CDONE;\n\t"
      "add.u32 n, n, 1;\n\t"
      "setp.lt.u32 p, n, %4;\n\t"
      "@p bra DVQ_CWAIT;\n\t"
      "DVQ_CDONE:\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity), "r"(100000u), "r"(1u << 22)
      : "memory");
  if (!ok) {
    *err_out = code;
    __threadfence_system();
    __trap();
  }
}

// Optional wait-time accounting (build with DVQ_TC_STATS=1): cycles spent in each wait site,
// summed over the lanes that wait, flushed to stats[site] at the end of the kernel.
#ifdef DVQ_TC_STATS
#define STAT_DECL(n) long long stat_acc[n] = {}
#define STAT_T0() const long long _t0 = clock64()
#define STAT_ADD(i) stat_acc[i] += clock64() - _t0
#define STAT_FLUSH(n, base)                                                              \
  do {                                                                                   \
    if ((threadIdx.x & 31) == 0)                                                         \
      for (int _i = 0; _i < (n); ++_i) atomicAdd(p.stats + (base) + _i, (unsigned long long)stat_acc[_i]); \
  } while (0)
#else
#define STAT_DECL(n)
#define STAT_T0()
#define STAT_ADD(i)
#define STAT_FLUSH(n, base)
#endif
// Pipeline timeline (DVQ_TC_STATS builds): clock64 stamps of one CTA for tiles 8..11, written to the unused
// tail of the refine row list (role, event, tile, chunk); printed by dvq_vq_read_counters.
#ifdef DVQ_TC_STATS
#define TRACE(role, ev, c_)                                                                                         \
  do {                                                                                                              \
    if (blockIdx.x == (PAIR ? 2 : 3) && (threadIdx.x & 31) == 0 && it >= 8 && it < 12 && p.N >= 65536)                            \
      reinterpret_cast<long long*>(p.row_list + p.N - 8192)[((role) * 8 + (ev)) * 8 + (int)(it - 8) * 2 + (c_)] = clock64(); \
  } while (0)
#else
#define TRACE(role, ev, c_)
#endif

// float(h) - a in one FHADD (PTX mixed-precision sub, sm_100+): h is one half of a packed pair
__device__ __forceinline__ float half_minus_float(uint32_t h16, float a) {
  float r;
  asm("sub.rn.f32.f16 %0, %1, %2;" : "=f"(r) : "h"((unsigned short)h16), "f"(a));
  return r;
}

// Reads of one staged z row: 4 elements at column 4 * c4 (one float4 / one 8-byte word of bf16, upcast exactly with a shift),
// and the 8-wide k-chunk c8 as two float4 (two 16-byte loads of fp32, one of bf16)
__device__ __forceinline__ void stage_ld8(const float4* row, int c8, float4& v0, float4& v1) {
  v0 = row[2 * c8];
  v1 = row[2 * c8 + 1];
}
__device__ __forceinline__ void stage_ld8(const uint2* row, int c8, float4& v0, float4& v1) {
  const uint4 u = reinterpret_cast<const uint4*>(row)[c8];
  v0 = bf4_to_f4(make_uint2(u.x, u.y));
  v1 = bf4_to_f4(make_uint2(u.z, u.w));
}
// four z elements of a gather lane as loaded (float4 / packed bf16: the bf16 form holds half the registers while in flight)
__device__ __forceinline__ float4 zraw_ldcs(const float* p) { return __ldcs(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ uint2 zraw_ldcs(const __nv_bfloat16* p) { return __ldcs(reinterpret_cast<const uint2*>(p)); }
__device__ __forceinline__ float4 zup(float4 v) { return v; }
__device__ __forceinline__ float4 zup(uint2 u) { return bf4_to_f4(u); }

// All barriers live in one shared struct so that a site addresses its barrier as base + immediate.
// (B_PEER_*: CTA-pair kernel, used in the leader CTA only — the peer CTA arrives on them remotely: its warp 1 once per tile
// on B_PEER_A_FULL, each of its filter warps once per chunk on B_PEER_ACC_EMPTY)
enum BarId { B_STAGE_FULL = 0, B_STAGE_EMPTY = 2, B_ACC_FULL = 4, B_A_EMPTY = 6, B_B_FULL = 8, B_B_EMPTY = 8 + MAX_BSLOTS,
             B_PEER_A_FULL = 8 + 2 * MAX_BSLOTS, B_PEER_ACC_EMPTY = 10 + 2 * MAX_BSLOTS, NBARS = 12 + 2 * MAX_BSLOTS };
// named barrier ids (0 is __syncthreads).  The accumulator-full relay has one barrier per (stage, warp group):
// the helper warps of a tile must not wait for the owner warps, which are still merging / writing the previous
// tile when the helpers are ready for the next one.
enum NamedBarId { NB_ACC_FULL_OWN = 1, NB_ACC_FULL_HLP = 3, NB_ACC_EMPTY = 5, NB_A_FULL = 7, NB_FIN_FULL = 9, NB_FIN_EMPTY = 10,
                  NB_SIDX_FULL = 11, NB_SIDX_EMPTY = 13 };
// (epq = warps per TMEM lane quarter that run the filter: EPQ, or EPQ + 1 when the converter warps join in)
__host__ __device__ constexpr int nb_acc_threads(int epq) { return 32 + 4 * epq * 32; }            // MMA warp + filter warps
constexpr int NB_ACC_OWN_THREADS = 32 + 4 * 32;                                                     // MMA warp + owner warps
__host__ __device__ constexpr int nb_acc_hlp_threads(int epq) { return 32 + 4 * (epq - 1) * 32; }  // MMA warp + helper warps
__host__ __device__ constexpr int nb_fin_threads(int epq) { return 4 * epq * 32; }                  // owners + helpers
constexpr int NB_A_THREADS = 32 + 128;                       // MMA warp + converter warps
constexpr int NB_SIDX_THREADS = 4 * 32 + GATHER_WARPS * 32;  // owner epilogue warps + gather warps
struct Ctl {
  uint64_t bars[NBARS];
  uint32_t tmem_slot;
};
#define BAR(id, i) (bar0 + 8u * (uint32_t)((id) + (i)))

struct RowState {   // per (row, column subset) running result of the filter
  float m1;         // smallest accumulator value so far
  int cnt;          // number of OTHER keys within `band` of m1 (a superset count)
  uint32_t bits;    // indicator mask of the last sub-chunk that held a key inside the band: even columns in the
                    // high half, odd columns in the low half, bit 15 - j/2 of a half <-> column j
  int col0;         // first code of that sub-chunk
  uint32_t cand;    // groups of sub-chunks holding a key within `band` of m1 (superset; always holds m1's own)
  int ncand;        // list mode: entries pushed into `cand` since the last reset (more than three = overflow)
};
// Record that sub-chunk `gbit` held a key inside the band.  Mask mode: set its bit.  List mode: push its 10-bit entry
// (newest in the low bits) and count; with more than three pushes the oldest entry has been shifted out and the
// record becomes CAND_LIST_OVERFLOW when the tile is finished (filter_tile) — two predicated instructions per sub-chunk
// instead of the branchy cand_union, which is kept for the once-per-tile merge of the warps' records.
template <bool LIST>
__device__ __forceinline__ void cand_push(RowState& st, uint32_t gbit) {
  if (LIST) { st.cand = (st.cand << CAND_ENTRY_BITS) | gbit; ++st.ncand; }
  else st.cand |= gbit;
}
// code index of a set bit of the mask (for a decided row the only set bit is the minimum itself)
__device__ __forceinline__ int row_state_col(const RowState& st) {
  const int zc = __clz(st.bits);                   // 0..15: even column 2*zc; 16..31: odd column 2*(zc-16)+1
  return st.col0 + (zc < 16 ? 2 * zc : 2 * zc - 31);
}

// Union of two candidate records (format: dvq_common.cuh); in list mode more than three entries become CAND_LIST_OVERFLOW.
template <bool LIST>
__device__ __forceinline__ uint32_t cand_union(uint32_t a, uint32_t b) {
  if (!LIST) return a | b;
  if (a == CAND_LIST_OVERFLOW || b == CAND_LIST_OVERFLOW) return CAND_LIST_OVERFLOW;
  constexpr uint32_t one = 1u << CAND_ENTRY_BITS, two = 1u << (2 * CAND_ENTRY_BITS);
  const int na = a == 0u ? 0 : (a < one ? 1 : (a < two ? 2 : 3));
  const int nb = b == 0u ? 0 : (b < one ? 1 : (b < two ? 2 : 3));
  return na + nb > 3 ? CAND_LIST_OVERFLOW : (a | (b << (CAND_ENTRY_BITS * na)));
}

// One 32-column sub-chunk of raw accumulators (all >= 0, so float order == bit order):
//   pass 1  FMNMX3 tree -> sub-chunk minimum -> running minimum with exact reset of the ambiguity state;
//   pass 2  indicator of "key < m1 + band" per element, fma.sat((T - key) * BIG) in {0, 1} exactly, shifted
//           into two 16-bit masks (even / odd columns) by a packed Horner step acc2 = 2 * acc2 + {s0, s1}
//           (one FFMA2 per two elements).  popc of the masks is the count; the position of the set bit is
//           the column of the minimum for a decided row (after the last reset the only key that was ever
//           inside the band is the minimum itself), so no per-element index packing is needed.
// ~3 issued instructions per element: 0.5 FMNMX3 (ALU) + 1 FFMA.SAT + 0.5 FFMA2 (FMA pipe).
__device__ __forceinline__ float subchunk_min(const float (&key)[32]) {
  float a0 = min3f(key[0], key[1], key[2]), a1 = min3f(key[3], key[4], key[5]);
  float a2 = min3f(key[6], key[7], key[8]), a3 = min3f(key[9], key[10], key[11]);
  float a4 = min3f(key[12], key[13], key[14]), a5 = min3f(key[15], key[16], key[17]);
  float a6 = min3f(key[18], key[19], key[20]), a7 = min3f(key[21], key[22], key[23]);
  float a8 = min3f(key[24], key[25], key[26]), a9 = min3f(key[27], key[28], key[29]);
  a0 = min3f(a0, a1, a2); a3 = min3f(a3, a4, a5); a6 = min3f(a6, a7, a8); a9 = min3f(a9, key[30], key[31]);
  return fminf(min3f(a0, a3, a6), a9);
}
// indicator masks of "key < T" for the 32 keys of a sub-chunk (TB = T * 2^20): even columns in the high half,
// odd columns in the low half, bit 15 - j/2 of a half <-> column j
__device__ __forceinline__ uint32_t subchunk_bits(const float (&key)[32], float TB) {
  const float BIG = 1048576.f;
  const uint64_t two = pack_f32x2(2.f, 2.f);
  // four independent Horner chains of 4 steps (columns 0-7, 8-15, 16-23, 24-31): short dependency chains
  uint64_t h0 = pack_f32x2(0.f, 0.f), h1 = h0, h2 = h0, h3 = h0;
#pragma unroll
  for (int j = 0; j < 8; j += 2) {
    h0 = ffma2(h0, two, pack_f32x2(fma_sat(key[j], -BIG, TB), fma_sat(key[j + 1], -BIG, TB)));
    h1 = ffma2(h1, two, pack_f32x2(fma_sat(key[8 + j], -BIG, TB), fma_sat(key[9 + j], -BIG, TB)));
    h2 = ffma2(h2, two, pack_f32x2(fma_sat(key[16 + j], -BIG, TB), fma_sat(key[17 + j], -BIG, TB)));
    h3 = ffma2(h3, two, pack_f32x2(fma_sat(key[24 + j], -BIG, TB), fma_sat(key[25 + j], -BIG, TB)));
  }
  // merge the four 4-bit masks per parity with exact FP32 arithmetic: m = ((h0 * 16 + h1) * 16 + h2) * 16 + h3
  const uint64_t sixteen = pack_f32x2(16.f, 16.f);
  const uint64_t acc2 = ffma2(ffma2(ffma2(h0, sixteen, h1), sixteen, h2), sixteen, h3);
  float fe, fo;
  unpack_f32x2(acc2, fe, fo);
  // both masks in one integer: fe * 65536 + fo would need 32 mantissa bits, so the halves are converted separately
  return ((uint32_t)__float2int_rn(fe) << 16) | (uint32_t)__float2int_rn(fo);
}

template <bool LIST>
__device__ __forceinline__ void filter_subchunk(uint32_t (&v)[32], int col0, uint32_t gbit, float band, float band_big, RowState& st) {
  const float BIG = 1048576.f;
  float key[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) key[j] = __uint_as_float(v[j]);
  const float m = subchunk_min(key);
  if (LIST) {
    // Large codebooks: after the first few dozen sub-chunks of a row most sub-chunks hold no key below the running
    // threshold (the chance is ~1/j for the j-th), and then nothing changes — no new minimum, no indicator bit.  The
    // test applies the indicator arithmetic itself to the sub-chunk minimum (monotone in the key, so a zero here means
    // 32 zeros below; any new minimum lies below the threshold and gives 1); when no row of the warp needs it the
    // indicator pass and the state update (two thirds of the instructions) are skipped.
    const bool need = fma_sat(m, -BIG, fmaf(st.m1, BIG, band_big)) != 0.f;
    if (!__any_sync(0xffffffffu, need)) return;
  }
  // running minimum: m1n = min(sub-chunk minimum, previous minimum)
  const float m1n = fminf(m, st.m1);
  // An improvement by more than the band voids every earlier key exactly (cnt := -1 cancels the new
  // minimum's own hit below); a smaller improvement (or none: 0) leaves the old minimum inside the band,
  // which the new minimum's own hit accounts for.
  if (st.m1 - m1n > band) { st.cnt = -1; st.cand = 0u; st.ncand = 0; }
  st.m1 = m1n;
  const float TB = fmaf(m1n, BIG, band_big);   // == (m1 + band) * 2^20: scaling by a power of two commutes with the rounding
#ifdef DVQ_KO_IND   // knock-out: no indicator pass — every row "decided" for the first code of its minimum's sub-chunk
  const uint32_t bits = (m <= m1n) ? 0x80000000u : 0u; (void)TB;
#else
  const uint32_t bits = subchunk_bits(key, TB);
  st.cnt += __popc(bits);
#endif
  if (bits) { cand_push<LIST>(st, gbit); st.bits = bits; st.col0 = col0; }   // the position is decoded once per row
}

// Two sub-chunks at once (A before B in code order): the same result as two calls of filter_subchunk, written so
// that the two min trees and the two indicator passes are independent instruction streams — a warp then fills the
// fixed-latency gaps of one with the other (the streamed-codebook variant gives the epilogue warps the registers).
template <bool LIST>
__device__ __forceinline__ void filter_subchunk2(uint32_t (&va)[32], uint32_t (&vb)[32], int col_a, int col_b, uint32_t gbit_a, uint32_t gbit_b,
                                                 float band, float band_big, RowState& st) {
  const float BIG = 1048576.f;
  float ka[32], kb[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) { ka[j] = __uint_as_float(va[j]); kb[j] = __uint_as_float(vb[j]); }
  const float ma = subchunk_min(ka), mb = subchunk_min(kb);   // two independent min trees
  if (LIST) {
    // the early-out of filter_subchunk for both sub-chunks at once (see there): nothing below the running threshold in
    // either, for every row of the warp -> no new minimum, no indicator bit, no state change
    const bool need = fma_sat(fminf(ma, mb), -BIG, fmaf(st.m1, BIG, band_big)) != 0.f;
    if (!__any_sync(0xffffffffu, need)) return;
  }
  const float m1a = fminf(ma, st.m1);
  const float m1b = fminf(mb, m1a);
  const bool reset_a = st.m1 - m1a > band, reset_b = m1a - m1b > band;
  const uint32_t bits_a = subchunk_bits(ka, fmaf(m1a, BIG, band_big));
  const uint32_t bits_b = subchunk_bits(kb, fmaf(m1b, BIG, band_big));
  if (reset_a) { st.cnt = -1; st.cand = 0u; st.ncand = 0; }
  st.cnt += __popc(bits_a);
  if (bits_a) { cand_push<LIST>(st, gbit_a); st.bits = bits_a; st.col0 = col_a; }
  if (reset_b) { st.cnt = -1; st.cand = 0u; st.ncand = 0; }
  st.cnt += __popc(bits_b);
  if (bits_b) { cand_push<LIST>(st, gbit_b); st.bits = bits_b; st.col0 = col_b; }
  st.m1 = m1b;
}

// DT > 0: e_dim known at compile time (strides, trip counts and index masks become immediates and the
// role loops unroll); DT == 0: generic.  TRAIN selects the straight-through / SSE / histogram epilogue.
// LIST selects the candidate record of the undecided rows (see cand_union): sub-chunk list for large codebooks.
// CE: the converter warps join the filter as a fourth warp per TMEM lane quarter (streamed codebooks with a
// double-buffered A image: a tile then has many accumulator chunks and the converters would idle for most of it;
// with four warps per quarter every warp takes exactly two of a chunk's eight sub-chunks instead of 3 / 3 / 2).
// ST: variant for streamed codebooks (many accumulator chunks per tile): the converter and gather warps work once per
// tile and can live with 64 registers, so the epilogue warps get 104 and filter two sub-chunks at a time.
// PAIR: CTA-pair kernel for streamed codebooks (cluster of two CTAs = the two SMs of a TPC, cta_group::2).  A streamed
// shape at M = 128 needs 64 bytes of operand image per tensor-pipe cycle and SM, 1.5x what the L2 delivers to 148 SMs
// (profiles/README.md), so the tensor pipe idles a third of the time.  The pair runs ONE M = 256 MMA per k-step: each CTA
// converts its own 128-row tile and streams only its HALF of every operand block (N / 2 codes), the accumulator of each
// CTA's rows lands in its own TMEM, and filter / gather work as in the single-CTA kernel.  The leader's (rank 0) warp 1
// issues; both CTAs' operand loads complete on the leader's ring barrier (cp.async.bulk.tensor with cta_group::2), the
// peer's warp 1 forwards "A image full" once per tile (remote arrive, release / acquire at cluster scope), the peer's filter
// warps announce a freed accumulator stage with one remote arrive each; completions are committed to both CTAs' barriers
// (multicast).
// ZT: element type of z / z_q — float, or __nv_bfloat16 (DVQ_Z_BF16: half the staging bytes, the converters and the gather
// warps upcast exactly and run the fp32 arithmetic unchanged, z_q is rounded to bf16 when stored).
template <int DT, bool TRAIN, bool LIST, bool CE, bool ST, bool PAIR = false, typename ZT = float>
__global__ void __launch_bounds__(NTHREADS, 1) vq_tc_kernel(const __grid_constant__ TcParams p) {
  static_assert(!(CE && ST), "the converter warps cannot hold the two-sub-chunk filter in 64 registers");
  static_assert(!PAIR || DT == 0, "the CTA-pair kernel is the generic streamed kernel");
  using ZRaw = decltype(zraw_ldcs(static_cast<const ZT*>(nullptr)));   // four z elements as loaded: float4 / uint2 (bf16)
  constexpr int EPQX = CE ? EPQ + 1 : EPQ;       // filter warps per TMEM lane quarter
  constexpr int NB_ACC_THREADS = nb_acc_threads(EPQX), NB_ACC_HLP_THREADS = nb_acc_hlp_threads(EPQX), NB_FIN_THREADS = nb_fin_threads(EPQX);
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ __align__(8) Ctl ctl;   // every mbarrier + the error word: addressed as base + constant
  // the opaque move keeps the window addresses in registers (the compiler otherwise rematerialises the
  // generic->shared conversion, S2R + LEA, at every use)
  uint32_t bar0, smem0;
  asm volatile("mov.u32 %0, %1;" : "=r"(bar0) : "r"(tc::smem_u32(ctl.bars)));
  asm volatile("mov.u32 %0, %1;" : "=r"(smem0) : "r"(tc::smem_u32(smem)));
  int* const err_out = p.counters + CNT_ERROR;

  const int D = DT > 0 ? DT : p.D;
  const int K = p.K;
  const SmemLayout L = smem_layout(K, D, p.layout_ovr, PAIR, (int)sizeof(ZT));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t crank = PAIR ? tc::cluster_ctarank() : 0u;   // 0 = leader (issues the MMAs), 1 = peer
  const int ns = DT > 0 ? (DT > DSLICE ? DT / DSLICE : 1) : (int)L.ns;   // e_dim slices
  const int ds = DT > 0 ? (DT > DSLICE ? DSLICE : DT) : (int)L.ds;        // columns per slice
  const int nk = ds / 16;                      // k-steps per slice
  const int nchunks = (K + 255) / 256;         // accumulator chunks per tile
  const bool resident = !PAIR && nchunks * ns <= 2;     // whole operand image fits the two ring slots
  // tile of iteration `it`: CTA b takes tiles b, b + grid, ...; a pair takes the tile pairs (2u, 2u + 1), u = cluster id,
  // cluster id + clusters, ... — both CTAs of a pair run the same number of iterations (the odd tile past the end has no rows)
  const int64_t pair_units = (p.ntiles + 1) / 2;
  const int64_t my_tiles = PAIR ? (pair_units > (int64_t)(blockIdx.x >> 1) ? (pair_units - 1 - (blockIdx.x >> 1)) / (gridDim.x >> 1) + 1 : 0)
                                : (p.ntiles > (int64_t)blockIdx.x ? (p.ntiles - 1 - blockIdx.x) / gridDim.x + 1 : 0);
  // (block and grid indices are read at the point of use: held in a register they are spill candidates)
  auto tile_of = [&](int64_t it) -> int64_t {
    return PAIR ? 2 * ((int64_t)(blockIdx.x >> 1) + it * (int64_t)(gridDim.x >> 1)) + (int64_t)crank : (int64_t)blockIdx.x + it * gridDim.x;
  };
  const int64_t total_chunks = my_tiles * nchunks;

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) {
      tc::mbar_init(&ctl.bars[B_STAGE_FULL + i], 1);
      tc::mbar_init(&ctl.bars[B_STAGE_EMPTY + i], 4);    // one arrival per converter warp
      tc::mbar_init(&ctl.bars[B_ACC_FULL + i], 1);       // tcgen05.commit
      tc::mbar_init(&ctl.bars[B_A_EMPTY + i], 1);        // tcgen05.commit
    }
    for (int i = 0; i < MAX_BSLOTS; ++i) {
      tc::mbar_init(&ctl.bars[B_B_FULL + i], 1);
      tc::mbar_init(&ctl.bars[B_B_EMPTY + i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      tc::mbar_init(&ctl.bars[B_PEER_A_FULL + i], 1);
      tc::mbar_init(&ctl.bars[B_PEER_ACC_EMPTY + i], 4 * EPQX);   // one remote arrival per filter warp of the peer CTA
    }
    tc::fence_barrier_init();
  }
  if (L.hist_in_smem) {
    int* shist = reinterpret_cast<int*>(smem + L.hist);
    for (int k = tid; k < K; k += NTHREADS) shist[k] = 0;
  }
  if (warp == 1) {
    if (PAIR) tc::tmem_alloc_pair(&ctl.tmem_slot, 512);
    else tc::tmem_alloc(&ctl.tmem_slot, 512);
  }
  tc::tc_fence_before();
  __syncthreads();
  if (PAIR) tc::cluster_sync_all();   // the peer's barriers exist before a commit or a remote arrive reaches them
  tc::tc_fence_after();
  const uint32_t tmem_base = ctl.tmem_slot;

  // ---- the filter over one row tile, shared by the epilogue warps and (CE) the converter warps -----------------
  // wq: 0 = owner of the warp's rows, 1..EPQX-1 = helpers (they split the columns); r = tile row = TMEM lane.
  // My sub-chunks of a 256-column chunk: every EPQX-th one; the owner takes the residue class with the fewest
  // members when they are uneven (it also merges, writes idx and the histogram).  The sub-chunk loop is kept
  // rolled so that the filter stays inside the instruction cache; the TMEM-load latency is covered by the other
  // warps of the sub-partition.  Mask mode: one candidate bit per 32-code sub-chunk (K <= 992, see
  // cand_list_mode); list mode: sub-chunk index + 1.
  auto filter_tile = [&](int64_t it, uint32_t& q, int wq, int r, RowState& st, float& band) {
    const uint32_t lane_addr = (uint32_t)(r & ~31) << 16;
    st.m1 = __uint_as_float(0x7f800000u); st.cnt = 0; st.bits = 0u; st.col0 = 0; st.cand = 0u; st.ncand = 0;
    float band_big = 0.f;
    const int sc0 = (wq + EPQX - 1) % EPQX;
    for (int c = 0; c < nchunks; ++c, ++q) {
      const uint32_t t = q & 1u;
#ifdef DVQ_ACC_MBAR   // experiment: every filter warp waits on the commit mbarrier itself (no lock-step with its sibling warps)
      if (resident) wait_or_trap(BAR(B_ACC_FULL, t), (q >> 1) & 1u, err_out, ERR_ACC_FULL);
      else
#endif
      if (wq == 0) nb_sync(NB_ACC_FULL_OWN + (int)t, NB_ACC_OWN_THREADS);
      else nb_sync(NB_ACC_FULL_HLP + (int)t, NB_ACC_HLP_THREADS);
      tc::tc_fence_after();
      if (wq == 0 && r < 32) TRACE(1, 0, c & 1);
      if (wq == 1 && r < 32) TRACE(2, 0, c & 1);
      if (c == 0) {
        band = reinterpret_cast<const float*>(smem + L.meta)[(it & (META_SLOTS - 1)) * TM + r];
        band_big = band * 1048576.f;
      }
      const int n = min(256, K - c * 256);
      int col = c * 256 + sc0 * 32;
      const int col_end = c * 256 + n;
      uint32_t taddr = tmem_base + lane_addr + t * 256u + (uint32_t)sc0 * 32u;
      uint32_t gbit = LIST ? (uint32_t)(c * 8 + sc0 + 1) : 1u << (c * 8 + sc0);
      if (ST) {
        // two of my sub-chunks per step (both loads issued before either is consumed)
#pragma unroll 1
        for (; col + 32 * EPQX < col_end; col += 64 * EPQX, taddr += 64u * EPQX, gbit = LIST ? gbit + 2 * EPQX : gbit << (2 * EPQX)) {
          uint32_t va[32], vb[32];
          tc::tmem_ld32(taddr, va);
          tc::tmem_ld32(taddr + 32u * EPQX, vb);
          tmem_ld_wait_dep(va);
          tmem_ld_wait_dep(vb);
          filter_subchunk2<LIST>(va, vb, col, col + 32 * EPQX, gbit, LIST ? gbit + EPQX : gbit << EPQX, band, band_big, st);
        }
      }
#pragma unroll 1
      for (; col < col_end; col += 32 * EPQX, taddr += 32u * EPQX, gbit = LIST ? gbit + EPQX : gbit << EPQX) {
        uint32_t v[32];
        tc::tmem_ld32(taddr, v);
        tmem_ld_wait_dep(v);
        filter_subchunk<LIST>(v, col, gbit, band, band_big, st);
      }
      tc::tc_fence_before();
      if (wq == 0 && r < 32) TRACE(1, 1, c & 1);
      if (wq == 1 && r < 32) TRACE(2, 1, c & 1);
      if ((int64_t)q + 2 < total_chunks) {
        if (PAIR && crank != 0) {
          // peer CTA of a pair: this warp's share of the stage is read (tcgen05.wait::ld above) — tell the leader's issuer
          // directly, one relaxed remote arrive per warp (a release at cluster scope would stall the warp for a fence)
          __syncwarp();
          if (lane == 0) tc::mbar_arrive_remote_relaxed(tc::map_to_cta(BAR(B_PEER_ACC_EMPTY, t), 0));
        } else {
          nb_arrive(NB_ACC_EMPTY + (int)t, NB_ACC_THREADS);
        }
      }
      if (wq == 1 && r < 32) TRACE(2, 3, c & 1);   // (stats builds) after the stage was handed back
    }
    if (LIST && st.ncand > 3) st.cand = CAND_LIST_OVERFLOW;   // an entry was shifted out: the refine scans every code of this row
  };
  // a helper hands its partial result of the tile to the owner warp of the same rows (single slot per helper)
  auto helper_handoff = [&](int64_t it, int wq, int r, const RowState& st) {
    float* fin_key = reinterpret_cast<float*>(smem + L.fin) + (wq - 1) * 4 * TM;
    if (it >= 1) nb_sync(NB_FIN_EMPTY, NB_FIN_THREADS);
    fin_key[r] = st.m1;
    reinterpret_cast<int*>(fin_key + TM)[r] = row_state_col(st);
    reinterpret_cast<int*>(fin_key + 2 * TM)[r] = st.cnt;
    reinterpret_cast<uint32_t*>(fin_key + 3 * TM)[r] = st.cand;
    nb_arrive(NB_FIN_FULL, NB_FIN_THREADS);
    if (wq == 1 && r < 32) TRACE(2, 2, 0);
  };

  if (warp < CONV_WARP0) {
  if (ST) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_ST_CTRL));
  else asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_CTRL));   // whole warpgroup, before the roles split
  if (warp == 0) {
    // ===================== producer: z tile (slices) -> staging ring =====================
    {
      if (lane == 0 && resident) {
        // the operand image stays in the two ring slots for the life of the CTA
        for (int b = 0; b < nchunks * ns; ++b) {
          const uint8_t* src = p.bimg + (size_t)b * L.bchunk_bytes;
          tc::mbar_arrive_expect_tx_a(BAR(B_B_FULL, b), L.bchunk_bytes);
          for (uint32_t off = 0; off < L.bchunk_bytes; off += 16384) {
            const uint32_t n = min(16384u, L.bchunk_bytes - off);
            tc::bulk_g2s_a(smem0 + L.bimg + (uint32_t)b * L.bchunk_bytes + off, src + off, n, BAR(B_B_FULL, b));
          }
        }
      }
      uint32_t js = 0;   // running slice counter of the staging ring
      STAT_DECL(1);
      for (int64_t it = 0; it < my_tiles; ++it) {
        const int64_t tile = tile_of(it);
        const int64_t row0 = tile * TM;
        const int rows = (int)max((int64_t)0, min((int64_t)TM, p.N - row0));
        for (int sl = 0; sl < ns; ++sl, ++js) {
          const int s = L.nstage == 2 ? (int)(js & 1u) : 0;
          const uint32_t ph = L.nstage == 2 ? (js >> 1) & 1u : js & 1u;
          { STAT_T0(); wait_or_trap(BAR(B_STAGE_EMPTY, s), ph ^ 1u, err_out, ERR_STAGE_EMPTY); STAT_ADD(0); }
          if (ns == 1) {
            if (lane == 0) {   // the whole tile is one contiguous block
              const uint32_t bytes = (uint32_t)rows * D * (uint32_t)sizeof(ZT);
              if (PAIR && rows == 0) tc::mbar_arrive_a(BAR(B_STAGE_FULL, s));   // the pair's tile past the end: nothing to load
              else {
                tc::mbar_arrive_expect_tx_a(BAR(B_STAGE_FULL, s), bytes);
                if (TRAIN) tc::bulk_g2s_keep_a(smem0 + L.stage[s], static_cast<const ZT*>(p.z) + row0 * D, bytes, BAR(B_STAGE_FULL, s));
                else tc::bulk_g2s_a(smem0 + L.stage[s], static_cast<const ZT*>(p.z) + row0 * D, bytes, BAR(B_STAGE_FULL, s));
              }
            }
          } else {
            // one 2-D TMA load per slice: box (ds columns, 128 rows) at (sl * ds, row0); rows past N arrive as zeros and
            // the barrier counts the whole box.  (As one bulk copy per 128- / 256-byte row segment — 128 per slice — this
            // was the bound of the sliced shapes: 2.1x the filter time at K = 512, e_dim 512.)
            if (lane == 0) {
              tc::mbar_arrive_expect_tx_a(BAR(B_STAGE_FULL, s), (uint32_t)TM * ds * (uint32_t)sizeof(ZT));
              if (TRAIN) tc::tma_load_2d_keep_a(smem0 + L.stage[s], &p.ztile, sl * ds, (int)row0, BAR(B_STAGE_FULL, s));
              else tc::tma_load_2d_a(smem0 + L.stage[s], &p.ztile, sl * ds, (int)row0, BAR(B_STAGE_FULL, s));
            }
          }
          __syncwarp();
        }
      }
      STAT_FLUSH(1, 0);
    }
  } else if (warp == BLOAD_WARP) {
    // ===================== codebook streamer: (chunk, slice) blocks of the operand image from L2 -> ring of L.nslots slots =====================
    if (lane == 0 && !resident) {
      uint32_t slot = 0, ph = 0;   // ring position: slot index and the phase bit of its barriers
      const uint32_t leader_bfull = PAIR ? tc::map_to_cta(BAR(B_B_FULL, 0), 0) : 0u;
      for (int64_t it = 0; it < my_tiles; ++it) {
        for (int c = 0; c < nchunks; ++c) {
          for (int sl = 0; sl < ns; ++sl) {
            wait_or_trap(BAR(B_B_EMPTY, slot), ph ^ 1u, err_out, ERR_B_FULL);
            const uint32_t bytes = sl == ns - 1 ? L.bchunk_bytes : L.bslice_bytes;   // the fold columns ride with the last slice
            // (pair kernel: block (c, sl) is stored as two half blocks, this CTA streams its own)
            if (PAIR) {
              // block (c, sl) is stored as two half blocks; each CTA streams its own half into its own ring slot with one 2-D
              // TMA load that completes on the LEADER's barrier (cta_group::2), which therefore counts both halves
              if (crank == 0) tc::mbar_arrive_expect_tx_a(BAR(B_B_FULL, slot), 2u * bytes);
              const int row = (int)(((size_t)((c * ns + sl) * 2 + (int)crank) * L.bchunk_bytes) >> 10);
              tc::tma_load_2d_pair_a(smem0 + L.bimg + slot * L.bchunk_bytes, &p.bmap[sl == ns - 1 ? 1 : 0], 0, row, leader_bfull + 8u * slot);
              if (++slot == L.nslots) { slot = 0; ph ^= 1u; }
              continue;
            }
            const uint8_t* src = p.bimg + (size_t)(c * ns + sl) * L.bchunk_bytes;
            tc::mbar_arrive_expect_tx_a(BAR(B_B_FULL, slot), bytes);
            for (uint32_t off = 0; off < bytes; off += 16384) {
              const uint32_t n = min(16384u, bytes - off);
              tc::bulk_g2s_a(smem0 + L.bimg + slot * L.bchunk_bytes + off, src + off, n, BAR(B_B_FULL, slot));
            }
            if (++slot == L.nslots) { slot = 0; ph ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp; lane 0 issues) =====================
    // (the completion relay described below now runs in warp 3)
    // In order per chunk: wait for the accumulator stage (named barrier, epilogue -> MMA), issue, wait for
    // the completion mbarrier of this chunk's tcgen05.commit and relay it to the 12 epilogue warps through a
    // named barrier, so that only this warp ever polls.  The next chunk is issued after the relay: with
    // two TMEM stages and an epilogue that takes longer per chunk than the MMAs, the tensor pipe is
    // never the one waited for.
    if (PAIR && crank != 0) {
      // ---- peer CTA of a pair: forward "A image of this tile written" to the leader's mbarrier (the freed accumulator stages
      // are announced by the filter warps themselves, the ring slots by the TMA loads)
      const uint32_t peer_bars = tc::map_to_cta(bar0, 0);   // the leader's barrier struct (same offsets)
#define PEER_BAR(id, i) (peer_bars + 8u * (uint32_t)((id) + (i)))
      for (int64_t it = 0; it < my_tiles; ++it) {
        nb_sync(NB_A_FULL + (int)(it & 1), NB_A_THREADS);                     // converters: fence.proxy.async + bar.arrive
        if (lane == 0) tc::mbar_arrive_remote(PEER_BAR(B_PEER_A_FULL, it & 1));
      }
#undef PEER_BAR
    } else {
      if (resident) for (int b = 0; b < nchunks * ns; ++b) wait_or_trap(BAR(B_B_FULL, b), 0, err_out, ERR_B_FULL);
      const uint32_t b_lbo = (PAIR ? 128u : 256u) * 16u, b_sbo = 128;
      const uint32_t a_lbo = A_CHUNK_BYTES, a_sbo = 128;
      // descriptors are (address >> 4) in the low bits: advancing by one k-step (two 8-wide k-chunks)
      // is a constant add that never carries out of the 14-bit address field
      const uint64_t a_step = (uint64_t)((2u * a_lbo) >> 4), b_step = (uint64_t)((2u * b_lbo) >> 4);
      // descriptors from the un-laundered window address: warp-uniform values the compiler keeps in uniform
      // registers, so each tcgen05.mma issues without a per-lane operand broadcast loop
      const uint32_t sbase = tc::smem_u32(smem);
      const uint64_t a_desc0 = tc::make_smem_desc(sbase + L.a_img[0], a_lbo, a_sbo);
      const uint64_t a_desc1 = tc::make_smem_desc(sbase + L.a_img[1], a_lbo, a_sbo);
      const uint64_t b_desc0 = tc::make_smem_desc(sbase + L.bimg, b_lbo, b_sbo);
      const uint32_t barbase = tc::smem_u32(ctl.bars);
      uint32_t q = 0;           // accumulator chunks consumed so far
      uint32_t rslot = 0, rph = 0;   // ring position of the next operand block (slot, phase bit)
      STAT_DECL(6);   // [3..5]: ring slot full (local), the peer's half, the peer's accumulator stage
#ifdef DVQ_TC_STATS
      const long long mma_t0 = clock64();
#endif
      for (int64_t it = 0; it < my_tiles; ++it) {
        const int a = L.a_bufs == 2 ? (int)(it & 1) : 0;
        { STAT_T0(); nb_sync(NB_A_FULL + (int)(it & 1), NB_A_THREADS); STAT_ADD(0); }
        if (PAIR) wait_or_trap_cluster(BAR(B_PEER_A_FULL, it & 1), (uint32_t)((it >> 1) & 1), err_out, ERR_PEER_A_FULL);
        TRACE(0, 0, 0);
        for (int c = 0; c < nchunks; ++c, ++q) {
          const uint32_t t = q & 1u;
          if (q >= 2) {
            STAT_T0(); nb_sync(NB_ACC_EMPTY + (int)t, NB_ACC_THREADS);
            STAT_ADD(1);
            if (PAIR) { STAT_T0(); wait_or_trap_cluster(BAR(B_PEER_ACC_EMPTY, t), ((q >> 1) & 1u) ^ 1u, err_out, ERR_PEER_ACC_EMPTY); STAT_ADD(5); }
          }
          tc::tc_fence_after();
          TRACE(0, 1, c & 1);
          const int n = min(256, K - c * 256);
          const uint32_t idesc = tc::make_idesc_f16(PAIR ? 256 : 128, n, 0);
          const uint32_t d_tmem = tmem_base + t * 256u;
          for (int sl = 0; sl < ns; ++sl) {
            const uint32_t bslot = resident ? (uint32_t)(c * ns + sl) : rslot;
            if (PAIR) { STAT_T0(); wait_or_trap_cluster(BAR(B_B_FULL, bslot), rph, err_out, ERR_B_FULL); STAT_ADD(3); }   // both halves (the peer's TMA completes here too)
            else if (!resident) { STAT_T0(); wait_or_trap(BAR(B_B_FULL, bslot), rph, err_out, ERR_B_FULL); STAT_ADD(3); }
            tc::tc_fence_after();
            if (tc::elect_one()) {
              const uint64_t bc = b_desc0 + (uint64_t)((bslot * L.bchunk_bytes) >> 4);
              uint64_t ad = (a ? a_desc1 : a_desc0) + (uint64_t)(sl * nk) * a_step, bd = bc;
              uint32_t acc = sl > 0 ? 1u : 0u;
#pragma unroll
              for (int j = 0; j < nk; ++j) {   // zh . eh, one slice
                if (PAIR) tc::umma_f16_pair(d_tmem, ad, bd, idesc, acc); else
                tc::umma_f16(d_tmem, ad, bd, idesc, acc);
#ifdef DVQ_KO_MMA2   // timing model of a half-rate MMA kind (kind::tf32 straight from the staged fp32 tile): every k-step twice
                tc::umma_f16(d_tmem, ad, bd, idesc, 1);
#endif
                acc = 1; ad += a_step; bd += b_step;
              }
              if (USE_ZL) {   // single-slice shapes only (see vq_tc_supported)
                bd = bc;
#pragma unroll
                for (int j = 0; j < nk; ++j) {   // zl . eh  (A holds -zl: negate-A bit 13 of the descriptor)
                  tc::umma_f16(d_tmem, ad, bd, idesc | (1u << 13), 1);
                  ad += a_step; bd += b_step;
                }
              }
              if (PAIR) {   // the same sequence on the pair; every completion goes to both CTAs' barriers
                if (sl == ns - 1) {
                  tc::umma_f16_pair(d_tmem, ad, bd, idesc, 1);
                  tc::umma_commit_pair_a(barbase + 8u * (B_ACC_FULL + t));
                  if (c == nchunks - 1) tc::umma_commit_pair_a(barbase + 8u * (uint32_t)(B_A_EMPTY + a));
                }
                tc::umma_commit_pair_a(barbase + 8u * (B_B_EMPTY + bslot));
              } else {
              if (sl == ns - 1) {
                tc::umma_f16(d_tmem, ad, bd, idesc, 1);   // fold columns: they follow the last slice in A and in the ring slot
                tc::umma_commit_a(barbase + 8u * (B_ACC_FULL + t));
                if (c == nchunks - 1) tc::umma_commit_a(barbase + 8u * (uint32_t)(B_A_EMPTY + a));  // every MMA of this tile done: A image free
              }
              if (!resident) tc::umma_commit_a(barbase + 8u * (B_B_EMPTY + bslot));   // ring slot free once these MMAs have read it
              }
            }
            if (!resident && ++rslot == L.nslots) { rslot = 0; rph ^= 1u; }
            __syncwarp();
          }
          TRACE(0, 2, c & 1);
          // Streamed codebooks: the completion of this chunk is awaited and relayed by warp 3, so that the next
          // chunk's MMAs are issued while these execute (+2-3 % at K = 16 384).  Resident image (two chunks per
          // tile): this warp relays itself — the extra hop measured ~1.5 % slower there.
#ifndef DVQ_ACC_MBAR
          if (resident) {
            wait_or_trap(BAR(B_ACC_FULL, t), (q >> 1) & 1u, err_out, ERR_ACC_FULL);
            TRACE(0, 3, c & 1);
            tc::tc_fence_before();
            nb_arrive(NB_ACC_FULL_HLP + (int)t, NB_ACC_HLP_THREADS);
            nb_arrive(NB_ACC_FULL_OWN + (int)t, NB_ACC_OWN_THREADS);
          }
#endif
        }
      }
#ifdef DVQ_TC_STATS
      stat_acc[2] = clock64() - mma_t0;
      if ((threadIdx.x & 31) == 0) for (int i = 3; i < 6; ++i) atomicAdd(p.stats + 11 + i, (unsigned long long)stat_acc[i]);
#endif
      STAT_FLUSH(3, 1);
    }
  } else {
    // ===================== relay (warp 3, streamed codebooks): tcgen05.commit mbarrier of a chunk -> named barriers of the filter warps =====================
    // Only this warp polls the completion mbarrier; the filter warps sleep in bar.sync.  A stage's barrier cannot
    // be committed again before this relay: the MMAs of chunk q + 2 wait for the filter warps to release the
    // stage, and those wait for this relay of chunk q.
    for (int64_t q = 0; q < (resident ? 0 : total_chunks); ++q) {
      const uint32_t t = (uint32_t)(q & 1);
      wait_or_trap(BAR(B_ACC_FULL, t), (uint32_t)((q >> 1) & 1), err_out, ERR_ACC_FULL);
      tc::tc_fence_before();
      nb_arrive(NB_ACC_FULL_HLP + (int)t, NB_ACC_HLP_THREADS);
      nb_arrive(NB_ACC_FULL_OWN + (int)t, NB_ACC_OWN_THREADS);
    }
  }
  } else if (warp < EPI_WARP0) {
    // ===================== converters: thread <-> tile row =====================
    if (ST) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_ST_SIDE));
    const int r = (warp - CONV_WARP0) * 32 + lane;
    const CbMeta cb = *p.cb;
    if (cb.magic != cb_magic(K, D, PAIR)) {   // DVQ_CODEBOOK_CACHED without a preparation of this shape in the workspace: fail loudly
      *err_out = ERR_NOT_PREPARED;
      __threadfence_system();
      __trap();
    }
    STAT_DECL(3);
#ifdef DVQ_TC_STATS
    const long long conv_t0 = clock64();
#endif
    const int nvs = ds / 4;   // float4 per row of one slice
    uint32_t js = 0;          // running slice counter of the staging ring
    auto convert_tile = [&](int64_t it) {
      const int64_t tile = tile_of(it);
      const int a = L.a_bufs == 2 ? (int)(it & 1) : 0;
      const uint32_t aph = L.a_bufs == 2 ? (uint32_t)((it >> 1) & 1) : (uint32_t)(it & 1);   // phase of B_A_EMPTY[a] this tile waits past
      const int rows = (int)max((int64_t)0, min((int64_t)TM, p.N - tile * TM));
      // squared norm of the row from the staged slice (lane-rotated conflict-free 128-bit reads).  Single slice: the row's
      // norm.  Sliced e_dim: the scale is needed before the first slice is converted, so it comes from an ESTIMATE — the
      // first slice's norm times the number of slices — and the true norm is accumulated while the slices are converted
      // (every bound below uses the true one; a row whose scaled norm then falls outside [2^8, 2^13] goes to the exact
      // kernel).  FP16's relative precision does not depend on the scale, so the estimate costs no accuracy; it replaces a
      // pre-pass kernel that read all of z once more.
      float nsq = 0.f;
      bool finite = true;
      {
        const int s = L.nstage == 2 ? (int)(js & 1u) : 0;
        { STAT_T0(); wait_or_trap(BAR(B_STAGE_FULL, s), L.nstage == 2 ? (js >> 1) & 1u : js & 1u, err_out, ERR_STAGE_FULL); STAT_ADD(0); }
        if (warp == CONV_WARP0) TRACE(3, 0, 0);
        const ZRaw* src = reinterpret_cast<const ZRaw*>(smem + L.stage[s]) + (size_t)r * nvs;
#ifdef DVQ_KO_NORM   // knock-out (timing experiment, wrong results): skip the norm pass
        if (r < rows) nsq = 64.f;
        if (false) {
#else
        if (r < rows) {
#endif
          // two packed (FFMA2) accumulator pairs: half the issued instructions and four short dependency chains
          uint64_t n01 = pack_f32x2(0.f, 0.f), n23 = n01;
          for (int i = 0; i < nvs; ++i) {
            const int c4 = (i + lane) & (nvs - 1);
            const float4 v = zup(src[c4]);
            const uint64_t v01 = pack_f32x2(v.x, v.y), v23 = pack_f32x2(v.z, v.w);
            n01 = ffma2(v01, v01, n01); n23 = ffma2(v23, v23, n23);
          }
          float q0, q1, q2, q3;
          unpack_f32x2(n01, q0, q1); unpack_f32x2(n23, q2, q3);
          nsq = (q0 + q1) + (q2 + q3);
          if (ns > 1) nsq *= (float)ns;
        }
      }
      if (r < rows) finite = (nsq < 1e30f);   // false for inf / nan too
      // scales and bounds
      const float zn = sqrtf(nsq) * (1.f + 1e-4f);
      const bool tiny = !(nsq > 1e-30f);
      int ex = (int)((__float_as_uint(zn) >> 23) & 255u) - 127;         // zn in [2^ex, 2^(ex+1))
      float s_n = exp2f((float)(10 - ex));                              // s_n*zn in [2^10, 2^11)
      const int rexp = cb.half_E - ex + 8;                              // fold scale r_n*2^8 = 2^rexp
      bool degenerate = (r < rows) && (tiny || !finite || cb.degenerate || rexp > 15 || rexp < -14);
      if (degenerate || r >= rows) s_n = 0.f;
      uint64_t rsq2 = pack_f32x2(0.f, 0.f);   // !USE_ZL: exact squared norm of the residual z' - zh that the product drops (even / odd partial sums)
      uint64_t nacc2 = pack_f32x2(0.f, 0.f);  // sliced e_dim: squared norm of the scaled row z', accumulated slice by slice
      const uint64_t s_n2 = pack_f32x2(s_n, s_n);
      if (warp == CONV_WARP0) TRACE(3, 1, 0);
      { STAT_T0(); wait_or_trap(BAR(B_A_EMPTY, a), aph ^ 1u, err_out, ERR_A_EMPTY); STAT_ADD(1); }
      if (warp == CONV_WARP0) TRACE(3, 2, 0);
      // convert slice by slice and write the A image
      uint8_t* aimg = smem + L.a_img[a] + (r >> 3) * 128 + (r & 7) * 16;
      for (int sl = 0; sl < ns; ++sl, ++js) {
        const int s = L.nstage == 2 ? (int)(js & 1u) : 0;
        if (sl > 0) { STAT_T0(); wait_or_trap(BAR(B_STAGE_FULL, s), L.nstage == 2 ? (js >> 1) & 1u : js & 1u, err_out, ERR_STAGE_FULL); STAT_ADD(0); }
        const ZRaw* src = reinterpret_cast<const ZRaw*>(smem + L.stage[s]) + (size_t)r * nvs;
        uint8_t* aslice = aimg + (size_t)(sl * (nvs / 2)) * A_CHUNK_BYTES;
#ifdef DVQ_KO_CONV   // knock-out: skip the FP16 conversion of the tile (the A image keeps stale data)
        for (int i = 0; i < 0; ++i) {
#else
        for (int i = 0; i < nvs / 2; ++i) {
#endif
          const int c8 = (i + lane) & (nvs / 2 - 1);                       // 8-wide k-chunk
          float4 v0, v1;
          stage_ld8(src, c8, v0, v1);
          // scale by the power-of-two s_n, two elements per FMUL2 (exact)
          const uint64_t xp[4] = {fmul2(pack_f32x2(v0.x, v0.y), s_n2), fmul2(pack_f32x2(v0.z, v0.w), s_n2),
                                  fmul2(pack_f32x2(v1.x, v1.y), s_n2), fmul2(pack_f32x2(v1.z, v1.w), s_n2)};
          if (ns > 1) nacc2 = ffma2(xp[3], xp[3], ffma2(xp[2], xp[2], ffma2(xp[1], xp[1], ffma2(xp[0], xp[0], nacc2))));
          // hi = fp16(x); with USE_ZL the second term is stored NEGATED, nl = fp16(hi - x) (one FHADD each, no
          // unpack) and the MMA issuer sets the A-negate bit of the instruction descriptor for the zl.eh products
          __half2 hi[4], lo[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float x0, x1;
            unpack_f32x2(xp[e], x0, x1);
            hi[e] = __floats2half2_rn(x0, x1);
            const uint32_t hb = *reinterpret_cast<const uint32_t*>(&hi[e]);
            const float r0 = half_minus_float(hb & 0xffffu, x0), r1 = half_minus_float(hb >> 16, x1);   // exact
            if (USE_ZL) lo[e] = __floats2half2_rn(r0, r1);
            else { const uint64_t rp = pack_f32x2(r0, r1); rsq2 = ffma2(rp, rp, rsq2); }
          }
          *reinterpret_cast<uint4*>(aslice + (size_t)c8 * A_CHUNK_BYTES) = *reinterpret_cast<uint4*>(hi);
          if (USE_ZL) *reinterpret_cast<uint4*>(aslice + (size_t)(nvs / 2 + c8) * A_CHUNK_BYTES) = *reinterpret_cast<uint4*>(lo);
        }
        warp_arrive(BAR(B_STAGE_EMPTY, s));       // staging slot may be refilled
      }
      // scaled norm bound: s_n * ||z|| from the exact norm (single slice) or the accumulated one (sliced; checked against
      // the window the fold columns and the indicator arithmetic were laid out for)
      float zs = s_n * zn;
      if (ns > 1) {
        float a0, a1;
        unpack_f32x2(nacc2, a0, a1);
        const float zt = sqrtf(a0 + a1) * (1.f + 1e-4f);
        if (s_n != 0.f && !(zt >= 256.f && zt <= 8192.f)) degenerate = true;   // (also inf / nan)
        zs = (s_n == 0.f) ? 0.f : fminf(zt, 8192.f);
      }
      const float f0a = __half2float(__float2half_ru(2.f * zs * (1.f + 1.f / 128.f)));
      const float fr = (s_n == 0.f) ? 0.f : exp2f((float)rexp);
      const float bias2 = 2.f * f0a * cb.b0;
      float eps = zs * cb.delta_max * (1.f + 1.f / 64.f)
                + bias2 * ((float)((USE_ZL ? 2 : 1) * ns * nk + 3) * (1.f / 1048576.f))   // tensor-core FP32 accumulation
                + 16.f * fr * (1.f / 256.f);                                              // ee rounding (r_n = fr / 256)
      if (USE_ZL) eps += (zs * (1.f / 4194304.f) + sqrtf((float)D) * (1.f / 33554432.f)) * cb.eh_norm_bound;   // zl rounding
      if (!USE_ZL) {
        float rs0, rs1;
        unpack_f32x2(rsq2, rs0, rs1);
        eps += sqrtf(rs0 + rs1) * (1.f + 1e-4f) * cb.eh_norm_bound;
      }
      float band = 2.f * eps * (1.f + 1.f / 16.f);
      if (degenerate) band = -1.f;    // marks "send to the exact kernel"
      const int kfold = (USE_ZL ? 2 : 1) * ns * (nvs / 2);   // fold k-chunks follow the zh (and zl) chunks
      {
        __half2 f[4];
        f[0] = __floats2half2_rn(f0a, fr);
        f[1] = __floats2half2_rn(fr, fr);
        f[2] = __floats2half2_rn(0.f, 0.f);
        f[3] = f[2];
        *reinterpret_cast<uint4*>(aimg + (size_t)kfold * A_CHUNK_BYTES) = *reinterpret_cast<uint4*>(f);
        f[0] = f[2]; f[1] = f[2];
        *reinterpret_cast<uint4*>(aimg + (size_t)(kfold + 1) * A_CHUNK_BYTES) = *reinterpret_cast<uint4*>(f);
      }
      reinterpret_cast<float*>(smem + L.meta)[(it & (META_SLOTS - 1)) * TM + r] = band;
      tc::fence_proxy_async_smem();           // A image visible to the tensor core (async proxy)
      nb_arrive(NB_A_FULL + (int)(it & 1), NB_A_THREADS);
      if (warp == CONV_WARP0) TRACE(3, 3, 0);
    };
    if (!CE) {
      for (int64_t it = 0; it < my_tiles; ++it) convert_tile(it);
    } else {
      // The converters stay one tile ahead of the MMAs (double-buffered A image) and spend the rest of a tile as
      // the fourth filter warp of their TMEM lane quarter: convert tile it + 1, then filter tile it as helper
      // EPQX - 1.  While they convert, the accumulator chunks they have not read yet stay occupied — a few
      // thousand cycles per tile against the tens of chunks a streamed codebook has.
      uint32_t q = 0;
      if (my_tiles > 0) convert_tile(0);
      for (int64_t it = 0; it < my_tiles; ++it) {
        if (it + 1 < my_tiles) convert_tile(it + 1);
        RowState st;
        float band = 0.f;
        filter_tile(it, q, EPQX - 1, r, st, band);
        helper_handoff(it, EPQX - 1, r, st);
      }
    }
#ifdef DVQ_TC_STATS
    stat_acc[2] = clock64() - conv_t0;
    if (warp != CONV_WARP0) { stat_acc[0] = stat_acc[1] = stat_acc[2] = 0; }
#endif
    STAT_FLUSH(3, 4);
  } else if (warp < GATHER_WARP0) {
    // ===================== epilogue: TMEM -> (min, ambiguity) per row =====================
    if (ST) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_ST_EPI));
    const int w = warp - EPI_WARP0;
    const int quarter = warp & 3;       // TMEM lanes this warp may access: 32*(warp_id % 4)
    const int wq = w >> 2;              // 0 = owner of these rows, 1..EPQ-1 = helpers (they split the columns)
    const int r = quarter * 32 + lane;  // tile row == TMEM lane
    uint32_t q = 0;
    STAT_DECL(5);
#ifdef DVQ_TC_STATS
    const long long epi_t0 = clock64();
#endif
    for (int64_t it = 0; it < my_tiles; ++it) {
      const int64_t tile = tile_of(it);
      const int64_t row0 = tile * TM;
      const int rows = (int)max((int64_t)0, min((int64_t)TM, p.N - row0));
      const int slot = (int)(it & 1);
      RowState st;
      float band = 0.f;
      filter_tile(it, q, wq, r, st, band);
      float* fin_base = reinterpret_cast<float*>(smem + L.fin);   // single slot: phase flips every tile
      if (wq > 0) {
        helper_handoff(it, wq, r, st);
      } else {
        { STAT_T0(); nb_sync(NB_FIN_FULL, NB_FIN_THREADS); STAT_ADD(2); }
        if (w == 0) TRACE(1, 2, 0);
        // merge the helpers' states: keep the smaller minimum; the loser's minimum either falls inside
        // the winner's band (ambiguous) or voids the loser's count entirely
        float m1 = st.m1;
        int cnt = st.cnt;
        int col = row_state_col(st);
        uint32_t cand = st.cand;
        bool flag = false;
#pragma unroll
        for (int h = 0; h < EPQX - 1; ++h) {
          const float* fin_key = fin_base + h * 4 * TM;
          const float ko = fin_key[r];
          const int co = reinterpret_cast<const int*>(fin_key + TM)[r];
          const int no = reinterpret_cast<const int*>(fin_key + 2 * TM)[r];
          const uint32_t cando = reinterpret_cast<const uint32_t*>(fin_key + 3 * TM)[r];
          if (ko < m1) {
            flag = (m1 - ko <= band);
            cand = flag ? cand_union<LIST>(cand, cando) : cando;      // an improvement beyond the band voids the old candidates
            m1 = ko; col = co; cnt = no;
          } else if (ko - m1 <= band) {
            flag = true;
            cand = cand_union<LIST>(cand, cando);
          }
        }
        if (it + 1 < my_tiles) nb_arrive(NB_FIN_EMPTY, NB_FIN_THREADS);
        flag = flag || (cnt > 0);
        if (band < 0.f) { flag = true; cand = LIST ? CAND_LIST_OVERFLOW : CAND_MASK_ALL; }   // degenerate row: every code is a candidate
        const bool valid = r < rows;
        flag = flag && valid;
        if (it >= 2) { STAT_T0(); nb_sync(NB_SIDX_EMPTY + slot, NB_SIDX_THREADS); STAT_ADD(3); }
        // code for the gather warps: byte offset of the code row in E, or — sign bit set — "undecided" with the
        // candidate-group mask in the low 31 bits (the gather warps append such rows to the refine list; the
        // exact kernel rewrites their z_q row and accounts their SSE / histogram contribution)
        reinterpret_cast<int*>(smem + L.sidx)[slot * TM + r] = flag ? (int)(cand | CAND_UNDECIDED) : col * D * 4;
        nb_arrive(NB_SIDX_FULL + slot, NB_SIDX_THREADS);
        if (w == 0) TRACE(1, 3, 0);
        if (valid && !flag) {
          p.idx[row0 + r] = (int64_t)col;          // 32 lanes x 8 B: one coalesced 256-byte store per warp
          if (TRAIN) {
            if (L.hist_in_smem) atomicAdd(reinterpret_cast<int*>(smem + L.hist) + col, 1);
            else atomicAdd(p.hist + col, 1ull);   // large codebooks: contention is low, shared memory is full
          }
        }
      }
    }
#ifdef DVQ_TC_STATS
    stat_acc[4] = clock64() - epi_t0;
    if (w != 0 && w != 4) { for (int i = 0; i < 5; ++i) stat_acc[i] = 0; }
    if (w == 4) { stat_acc[0] = 0; stat_acc[4] = 0; }   // w == 4: first helper warp
#endif
    STAT_FLUSH(5, 7);
  } else {
    // ===================== gather: z_q, idx, SSE, histogram for the decided rows =====================
    if (ST) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_ST_SIDE));
    else asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_GATHER));
    const int gw = warp - GATHER_WARP0;
    const int nv = D / 4;                              // float4 slots per row (power of two)
    const int rows_per_warp = TM / GATHER_WARPS;
    // lane -> (row, float4 column): a row is covered by lpr = min(nv, 32) lanes in `parts` = nv / lpr
    // passes; one warp-step covers rps = 32 / lpr rows.  All index math is shifts / loop-invariant
    // pointer bumps (immediates when e_dim is a template constant).
    const int lpr = nv < 32 ? nv : 32;
    const int lpr_shift = 31 - __clz(lpr);
    const int parts = nv / lpr;
    const int rps = 32 >> lpr_shift;
    const int c4_lane = lane & (lpr - 1), rsub = lane >> lpr_shift;
    const int nsteps = rows_per_warp / rps;            // row-steps per warp per tile (per part)
    const int rbase = gw * rows_per_warp + rsub;
    double sse_acc = 0.0;
    constexpr bool PREFETCH_Z = !ST;                   // request the first batch's z rows before the codes arrive (needs ~16 more registers)
    constexpr int UH = ST ? 2 : 4;                            // row-steps per batch; two batches in flight per lane (x2 loads in train mode)
    STAT_DECL(2);
#ifdef DVQ_TC_STATS
    const long long g_t0 = clock64();
#endif
    for (int64_t it = 0; it < my_tiles; ++it) {
      const int64_t tile = tile_of(it);
      const int64_t row0 = tile * TM;
      const int rows = (int)max((int64_t)0, min((int64_t)TM, p.N - row0));
      const int slot = (int)(it & 1);
      // Two batches of UH row-steps are kept in flight (software pipeline: the loads of batch b + 1 are issued
      // before batch b is consumed), and the z rows of the first batch — they do not depend on the codes — are
      // requested before this tile's codes arrive, so that only one L2 round trip per tile is exposed.
      float4 eA[UH], eB[UH];
      ZRaw zA[UH], zB[UH];
      int kA[UH], kB[UH];
      const bool full_tile = rows == TM;
      const bool piped = full_tile && (nsteps % (2 * UH)) == 0;
      const ZT* zp0 = static_cast<const ZT*>(p.z) + (row0 + rbase) * D + c4_lane * 4;
      if (TRAIN && piped && PREFETCH_Z) {
#pragma unroll
        for (int u = 0; u < UH; ++u) zA[u] = zraw_ldcs(zp0 + (int64_t)(u * rps) * D);
      }
      { STAT_T0(); nb_sync(NB_SIDX_FULL + slot, NB_SIDX_THREADS); STAT_ADD(0); }
      if (gw == 0) TRACE(4, 0, 0);
      const int* sp = reinterpret_cast<const int*>(smem + L.sidx) + slot * TM + rbase;
      {
        // undecided rows of this warp's 32 rows -> list for the candidate refine kernel (one atomic per warp that
        // has any).  LIST mode: rows with more than three candidate sub-chunks (and degenerate rows) go to a second
        // list, stored downwards from the end of the same buffer, that the exact FP32 tile kernel re-evaluates
        // against the whole codebook (a one-warp scan of a large codebook would take milliseconds).
        const int code = reinterpret_cast<const int*>(smem + L.sidx)[slot * TM + gw * rows_per_warp + lane];
        const bool und = code < 0 && lane < rows_per_warp && gw * rows_per_warp + lane < rows;
        const bool ovf = LIST && und && ((uint32_t)code & CAND_LIST_OVERFLOW) == CAND_LIST_OVERFLOW;
        const unsigned bal = __ballot_sync(0xffffffffu, und && !ovf);
        if (bal) {
          int base = 0;
          if (lane == 0) base = atomicAdd(p.counters + CNT_LISTED, __popc(bal));
          base = __shfl_sync(0xffffffffu, base, 0);
          if (und && !ovf) {
            const int pos = base + __popc(bal & ((1u << lane) - 1u));
            p.row_list[pos] = (int)(row0 + gw * rows_per_warp + lane);
            p.cand_list[pos] = (int)((uint32_t)code & ~CAND_UNDECIDED);
          }
        }
        if (LIST) {
          const unsigned bal2 = __ballot_sync(0xffffffffu, ovf);
          if (bal2) {
            int base = 0;
            if (lane == 0) base = atomicAdd(p.counters + CNT_OVF, __popc(bal2));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (ovf) p.row_list[p.N - 1 - (base + __popc(bal2 & ((1u << lane) - 1u)))] = (int)(row0 + gw * rows_per_warp + lane);
          }
        }
      }
      float lsse = 0.f;
#pragma unroll 1
#ifdef DVQ_KO_GATHER   // knock-out: no code gather, no z re-read, no z_q store
      for (int part = 0; part < 0; ++part) {
#else
      for (int part = 0; part < parts; ++part) {
#endif
        const int c4 = (part << 5) | c4_lane;
        const char* ec = reinterpret_cast<const char*>(p.E + c4 * 4);
        const ZT* zp = static_cast<const ZT*>(p.z) + (row0 + rbase) * D + c4 * 4;
        ZT* op = static_cast<ZT*>(p.zq) + (row0 + rbase) * D + c4 * 4;
        if (piped) {
          // fast path: no per-row checks
          auto issue = [&](int t0, float4 (&e4)[UH], ZRaw (&z4)[UH], int (&kk)[UH], bool have_z) {
#pragma unroll
            for (int u = 0; u < UH; ++u) kk[u] = sp[(t0 + u) * rps];
#pragma unroll
            for (int u = 0; u < UH; ++u) {
              e4[u] = __ldg(reinterpret_cast<const float4*>(ec + (uint32_t)max(kk[u], 0)));   // undecided: any valid row
              if (TRAIN && !have_z) z4[u] = zraw_ldcs(zp + (int64_t)((t0 + u) * rps) * D);   // last use of this tile
            }
          };
          auto finish = [&](int t0, const float4 (&e4)[UH], const ZRaw (&z4)[UH], const int (&kk)[UH]) {
#pragma unroll
            for (int u = 0; u < UH; ++u) {
              float4 o4 = e4[u];
              if (TRAIN) {
                // packed FP32 (FADD2 / FMUL2 / FFMA2): d = fl(e - z), z_q = fl(z + d), two elements per instruction,
                // each half an ordinary IEEE operation (bit-identical to the scalar form, no contraction)
                const uint64_t e01 = pack_f32x2(e4[u].x, e4[u].y), e23 = pack_f32x2(e4[u].z, e4[u].w);
                const float4 zu = zup(z4[u]);
                const uint64_t z01 = pack_f32x2(zu.x, zu.y), z23 = pack_f32x2(zu.z, zu.w);
                const uint64_t d01 = fsub2(e01, z01), d23 = fsub2(e23, z23);
                const uint64_t s2 = ffma2(d23, d23, fmul2(d01, d01));
                float s0, s1;
                unpack_f32x2(s2, s0, s1);
                lsse = fmaf(kk[u] < 0 ? 0.f : 1.f, s0 + s1, lsse);      // undecided rows are accounted by the exact kernel
                unpack_f32x2(fadd2(z01, d01), o4.x, o4.y);
                unpack_f32x2(fadd2(z23, d23), o4.z, o4.w);
              }
              zstcs4(op + (int64_t)((t0 + u) * rps) * D, o4);   // streaming: never re-read
            }
          };
          issue(0, eA, zA, kA, PREFETCH_Z && part == 0);   // part 0: the z rows of the first batch were requested before the barrier
#pragma unroll 1
          for (int t0 = 0; t0 < nsteps; t0 += 2 * UH) {
            issue(t0 + UH, eB, zB, kB, false);
            finish(t0, eA, zA, kA);
            if (t0 + 2 * UH < nsteps) issue(t0 + 2 * UH, eA, zA, kA, false);
            finish(t0 + UH, eB, zB, kB);
          }
        } else {
#pragma unroll 1
          for (int t = 0; t < nsteps; ++t) {            // last (partial) tile or odd step counts
            const int ro = t * rps;
            if (rbase + ro >= rows) continue;
            const int kv = sp[ro];
            const float4 e1 = __ldg(reinterpret_cast<const float4*>(ec + (uint32_t)max(kv, 0)));
            float4 o4 = e1;
            if (TRAIN) {
              const float4 z1 = zldcs4(zp + (int64_t)ro * D);
              const float dx = __fsub_rn(e1.x, z1.x), dy = __fsub_rn(e1.y, z1.y);
              const float dz = __fsub_rn(e1.z, z1.z), dw = __fsub_rn(e1.w, z1.w);
              const float ss = fmaf(dw, dw, fmaf(dz, dz, fmaf(dy, dy, dx * dx)));
              lsse = fmaf(kv < 0 ? 0.f : 1.f, ss, lsse);
              o4 = make_float4(__fadd_rn(z1.x, dx), __fadd_rn(z1.y, dy), __fadd_rn(z1.z, dz), __fadd_rn(z1.w, dw));
            }
            zstcs4(op + (int64_t)ro * D, o4);
          }
        }
      }
      if (gw == 0) TRACE(4, 1, 0);
      if (it + 2 < my_tiles) nb_arrive(NB_SIDX_EMPTY + slot, NB_SIDX_THREADS);
      sse_acc += (double)lsse;
    }
#ifdef DVQ_TC_STATS
    stat_acc[1] = clock64() - g_t0;
    if (gw != 0) { stat_acc[0] = stat_acc[1] = 0; }
#endif
    STAT_FLUSH(2, 12);
    // ---- CTA total of the squared error ----
    if (TRAIN) {
      sse_acc = warp_sum(sse_acc);
      if (lane == 0 && sse_acc != 0.0) atomicAdd(p.sse, sse_acc);
    }
  }

  tc::tc_fence_before();
  __syncthreads();
  if (TRAIN && L.hist_in_smem) {   // shared-memory histogram (filled by the epilogue warps) -> global, once per CTA
    const int* shist = reinterpret_cast<const int*>(smem + L.hist);
    for (int k = tid; k < K; k += NTHREADS) {
      const int hcount = shist[k];
      if (hcount) atomicAdd(p.hist + k, (unsigned long long)hcount);
    }
  }
  if (PAIR) {   // no CTA leaves (or frees its TMEM) while the pair's MMAs or remote arrives may still touch it
    tc::tc_fence_before();
    tc::cluster_sync_all();
    tc::tc_fence_after();
  }
  if (warp == 1) {
    if (PAIR) tc::tmem_dealloc_pair(tmem_base, 512);
    else tc::tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace

// z [N, D] fp32 / bf16 row-major as a 2-D tensor map with box (ds columns, TM rows), no swizzle: a slice of a row tile lands as
// [row][ds elements], the layout the converter warps read
static int encode_ztile(CUtensorMap* map, const void* z, int64_t N, int D, int ds, bool zbf) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                               const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    DVQ_CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (!fn || qres != cudaDriverEntryPointSuccess) return fail(DVQ_ERR_CUDA, "cuTensorMapEncodeTiled is not available in this driver");
    encode = reinterpret_cast<EncodeFn>(fn);
  }
  const cuuint64_t dims[2] = {(cuuint64_t)D, (cuuint64_t)N};
  const cuuint64_t strides[1] = {(cuuint64_t)D * (zbf ? 2u : 4u)};
  const cuuint32_t box[2] = {(cuuint32_t)ds, (cuuint32_t)TM};
  const cuuint32_t estr[2] = {1u, 1u};
  const CUresult r = encode(map, zbf ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(z), dims, strides,
                            box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(DVQ_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for z [%lld, %d]", (int)r, (long long)N, D);
  return DVQ_OK;
}

// the operand image as a [bytes / 1024, 256] int32 tensor, box = (256, rows): one half block lands densely in its ring slot
static int encode_bimg(CUtensorMap* map, const uint8_t* bimg, size_t image_bytes, uint32_t box_rows) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                               const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    DVQ_CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (!fn || qres != cudaDriverEntryPointSuccess) return fail(DVQ_ERR_CUDA, "cuTensorMapEncodeTiled is not available in this driver");
    encode = reinterpret_cast<EncodeFn>(fn);
  }
  const cuuint64_t dims[2] = {256, (cuuint64_t)(image_bytes / 1024)};
  const cuuint64_t strides[1] = {1024};
  const cuuint32_t box[2] = {256, box_rows};
  const cuuint32_t estr[2] = {1u, 1u};
  const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_INT32, 2, const_cast<uint8_t*>(bimg), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(DVQ_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for the operand image (%zu bytes, box rows %u)", (int)r, image_bytes, box_rows);
  return DVQ_OK;
}

bool vq_tc_supported(int64_t N, int K, int D) {
  if (N <= 0 || N > 2147483647LL - 256) return false;
  if (D < 16 || D > 512 || (D & (D - 1)) != 0) return false;   // power of two: index math is masks/shifts
  if (USE_ZL && D > DSLICE) return false;
  if (K % 32 != 0 || K < 32 || K > 32704) return false;   // list-mode candidate entries are 10 bits (sub-chunk index + 1 <= 1023)
  return smem_layout(K, D).total <= SMEM_LIMIT;
}

// dvq_debug_tc_image_offset: byte offset of (code k, column d; d in [D, D + 16) = fold columns) in the global operand image of
// either layout, and the image size (host-only; tests/test_cabi_symbols.py checks that the maps are injective and in range)
long long vq_tc_image_offset(int k, int d, int K, int D, int pair, long long* image_bytes) {
  const SmemLayout L1 = smem_layout(K, D);
  if (image_bytes) *image_bytes = (long long)((K + 255) / 256) * L1.ns * L1.bchunk_bytes;
  return (long long)bimg_offset(k, d, D, K, pair != 0);
}

// CTA-pair kernel (cta_group::2) for this call?  Streamed codebooks only.  Measured at N = 16.8M against the single-CTA
// kernel, whole call (profiles/README.md): e_dim 512 1.05x (K = 512) .. 1.67x (K = 16 384); e_dim 256 1.11-1.27x from
// K = 2048 on, 0.93x at K = 1024; e_dim 128 1.06-1.09x from K = 2048 on, 0.91x at K = 512; e_dim 64 0.98-1.00x (one slice
// per chunk: the accumulator hand-off between the SMs costs what the halved operand stream saves).  Hence: e_dim 512
// always, e_dim 128 / 256 from K = 2048 on.  DVQ_TC_PAIR=0 turns it off, DVQ_TC_PAIR=1 selects it for every streamed shape.
bool vq_tc_pair_selected(int64_t N, int K, int D) {
  static const char* pair_env = getenv("DVQ_TC_PAIR");
  if (pair_env && pair_env[0] == '0') return false;
  if (!vq_tc_supported(N, K, D)) return false;
  const SmemLayout L1 = smem_layout(K, D);
  if (((K + 255) / 256) * (int)L1.ns <= 2) return false;                 // resident image: the single-CTA kernel
  if (!(pair_env && pair_env[0] == '1') && !(D >= 512 || (D >= 128 && K >= 2048))) return false;
  if (smem_layout(K, D, 0, true).total > SMEM_LIMIT) return false;
  return N > TM;                                                         // at least two tiles
}

// dvq_debug_tc_pair_layout: out8 = { CTA-pair kernel selected for (N, K, D) (0/1), slice width, slices, A images, ring
// slots, z staging slots, dynamic shared memory, codes per ring slot } of the pair layout (host-only)
void vq_tc_pair_layout_info(int64_t N, int K, int D, int* out8, int zbytes) {
  for (int i = 0; i < 8; ++i) out8[i] = 0;
  if (!vq_tc_supported(N > 0 ? N : 1, K, D)) return;
  const SmemLayout L = smem_layout(K, D, 0, true, zbytes);
  out8[0] = vq_tc_pair_selected(N, K, D) ? 1 : 0;
  out8[1] = (int)L.ds; out8[2] = (int)L.ns; out8[3] = (int)L.a_bufs; out8[4] = (int)L.nslots; out8[5] = (int)L.nstage;
  out8[6] = (int)L.total + 128; out8[7] = (int)L.bcodes;
}

void vq_tc_layout_info(int K, int D, int* out8, int zbytes) {
  const bool shape_ok = D >= 16 && D <= 512 && (D & (D - 1)) == 0 && K % 32 == 0 && K >= 32 && K <= 32704;
  for (int i = 0; i < 8; ++i) out8[i] = 0;
  if (!shape_ok) return;
  const SmemLayout L = smem_layout(K, D, 0, false, zbytes);
  out8[0] = L.total <= SMEM_LIMIT ? 1 : 0;
  out8[1] = (int)L.ds; out8[2] = (int)L.ns; out8[3] = (int)L.a_bufs; out8[4] = (int)L.nslots; out8[5] = (int)L.nstage;
  out8[6] = (int)L.total + 128; out8[7] = (int)L.hist_in_smem;
}

size_t vq_tc_operand_bytes(int K, int D) {
  const SmemLayout L = smem_layout(K, D);
  return align_up(sizeof(CbMeta), 256) + align_up((size_t)((K + 255) / 256) * L.ns * L.bchunk_bytes, 256);
}

int launch_vq_tc(const void* z, const float* E, const float* ee, int64_t N, int K, int D, int train, void* z_q,
                 int64_t* idx, unsigned long long* hist, double* sse, void* bop, int* counters, int* row_list,
                 int* cand_list, int* zero_ints, int zero_n, bool codebook_cached, bool zbf, cudaStream_t s) {
  DeviceProps dp;
  int rc = device_props(&dp);
  if (rc) return rc;
  if ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(E) | reinterpret_cast<uintptr_t>(z_q)) % 16 != 0)
    return fail(DVQ_ERR_BAD_ALIGN, "tcgen05 path needs 16-byte aligned z / E / z_q");
  CbMeta* cb = static_cast<CbMeta*>(bop);
  uint8_t* bimg = static_cast<uint8_t*>(bop) + align_up(sizeof(CbMeta), 256);
  static const char* lay_env = getenv("DVQ_TC_LAYOUT");   // experiment: "a st sl" digits, e.g. 123 = 1 A image, 2 staging slots, 3 ring slots
  int ovr = lay_env ? atoi(lay_env) : 0;
  const int zbytes = zbf ? 2 : 4;
  if (ovr && (((K + 255) / 256) * (D / slice_width(D)) <= 2 || smem_layout(K, D, ovr, false, zbytes).total > SMEM_LIMIT || ovr / 100 < 1 || ovr / 100 > 2 ||
              ovr / 10 % 10 < 1 || ovr / 10 % 10 > 2 || ovr % 10 < 2 || ovr % 10 > MAX_BSLOTS_SOLO))
    ovr = 0;   // resident images keep their layout; impossible requests are ignored
  // CTA-pair kernel (cta_group::2) for streamed codebooks: on by default, DVQ_TC_PAIR=0 selects the single-CTA kernel (A/B runs).
  // It needs an even number of SMs to pair up and at least one full pair of tiles.
  static const char* ce_env = getenv("DVQ_TC_CE");
  static const char* st_env = getenv("DVQ_TC_ST");
  int pair_ovr = lay_env ? atoi(lay_env) : 0;   // the pair kernel accepts rings of up to MAX_BSLOTS slots
  if (pair_ovr && (pair_ovr / 100 < 1 || pair_ovr / 100 > 2 || pair_ovr / 10 % 10 < 1 || pair_ovr / 10 % 10 > 2 || pair_ovr % 10 < 2 || pair_ovr % 10 > MAX_BSLOTS ||
                   smem_layout(K, D, pair_ovr, true, zbytes).total > SMEM_LIMIT))
    pair_ovr = 0;
  const SmemLayout L1 = smem_layout(K, D, ovr, false, zbytes);
  const bool streamed = ((K + 255) / 256) * (int)L1.ns > 2;
  const bool pair = vq_tc_pair_selected(N, K, D) && dp.sm_count >= 2;   // chosen on (N, K, D) alone, whatever the z type
  const SmemLayout L = pair ? smem_layout(K, D, pair_ovr, true, zbytes) : L1;
  const size_t image_bytes = (size_t)((K + 255) / 256) * L1.ns * L1.bchunk_bytes;   // the same for both image layouts
  if (codebook_cached) {
    // DVQ_CODEBOOK_CACHED: CbMeta and the operand image in `bop` are those of this codebook; only the per-call
    // counters and bin tables are reset
    tc_reset_kernel<<<1, 256, 0, s>>>(counters, zero_ints, zero_n);
    DVQ_CUDA_CHECK(cudaGetLastError());
    count_launch();
  } else {
    tc_cb_stats_kernel<<<1, 256, 0, s>>>(ee, K, D, cb, counters, zero_ints, zero_n, pair);
    DVQ_CUDA_CHECK(cudaGetLastError());
    DVQ_CUDA_CHECK(cudaMemsetAsync(bimg, 0, image_bytes, s));
    tc_cb_image_kernel<<<(K * 32 + 255) / 256, 256, 0, s>>>(E, ee, K, D, cb, bimg, pair);
    DVQ_CUDA_CHECK(cudaGetLastError());
    count_launch(2);
  }

  TcParams p;
  memset(&p.ztile, 0, sizeof(p.ztile));
  if (D > DSLICE) {
    rc = encode_ztile(&p.ztile, z, N, D, (int)L.ds, zbf);
    if (rc) return rc;
  }
  memset(p.bmap, 0, sizeof(p.bmap));
  if (pair) {
    rc = encode_bimg(&p.bmap[0], bimg, image_bytes, L.bslice_bytes / 1024);
    if (!rc) rc = encode_bimg(&p.bmap[1], bimg, image_bytes, L.bchunk_bytes / 1024);
    if (rc) return rc;
  }
  p.z = z; p.E = E; p.bimg = bimg; p.cb = cb; p.N = N; p.K = K; p.D = D; p.train = train;
  p.zq = z_q; p.idx = idx; p.hist = hist; p.sse = sse; p.counters = counters; p.row_list = row_list; p.cand_list = cand_list;
  p.layout_ovr = pair ? pair_ovr : ovr;
  p.stats = reinterpret_cast<unsigned long long*>(counters + CNT_STATS);
  p.ntiles = (N + TM - 1) / TM;
  const size_t smem = L.total + 128;
  int64_t grid = p.ntiles < dp.sm_count ? p.ntiles : dp.sm_count;
  if (pair) {   // clusters of two CTAs: one per tile pair, at most one per TPC
    const int64_t units = (p.ntiles + 1) / 2;
    grid = 2 * (units < dp.sm_count / 2 ? units : dp.sm_count / 2);
  }
  // Converters join the filter as a fourth warp per TMEM lane quarter (DVQ_TC_CE=1; needs a streamed codebook and a
  // double-buffered A image).  It paid +4 % at e_dim 64, K >= 4096 while the filter was the bound; with the list-mode
  // early-out the filter is cheap and the variant is 5 % behind the default there, so it is not selected automatically.
  // (the bf16 kernels are instantiated without the CE / ST experiment variants: a bf16 call ignores DVQ_TC_CE / DVQ_TC_ST)
  const bool ce = !zbf && streamed && L.a_bufs == 2 && ce_env && ce_env[0] == '1';
#define DVQ_LAUNCH_TC(DT_, TR_, LS_, CE_, ST_, ZT_)                                                                         \
  do {                                                                                                                 \
    DVQ_CUDA_CHECK(cudaFuncSetAttribute(vq_tc_kernel<DT_, TR_, LS_, CE_, ST_, false, ZT_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    vq_tc_kernel<DT_, TR_, LS_, CE_, ST_, false, ZT_><<<(unsigned)grid, NTHREADS, smem, s>>>(p);                           \
  } while (0)
#define DVQ_LAUNCH_TC_PAIR(TR_, LS_, CE_, ST_, ZT_)                                                                         \
  do {                                                                                                                 \
    DVQ_CUDA_CHECK(cudaFuncSetAttribute(vq_tc_kernel<0, TR_, LS_, CE_, ST_, true, ZT_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    cudaLaunchConfig_t cfg = {};                                                                                       \
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(NTHREADS); cfg.dynamicSmemBytes = smem; cfg.stream = s;     \
    cudaLaunchAttribute at[1];                                                                                         \
    at[0].id = cudaLaunchAttributeClusterDimension;                                                                    \
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;                                 \
    cfg.attrs = at; cfg.numAttrs = 1;                                                                                  \
    DVQ_CUDA_CHECK(cudaLaunchKernelEx(&cfg, vq_tc_kernel<0, TR_, LS_, CE_, ST_, true, ZT_>, p));                        \
  } while (0)
#define DVQ_LAUNCH_TC_GENERIC(TR_, LS_)                                      \
  do {                                                                       \
    if (pair && st) DVQ_LAUNCH_TC_PAIR(TR_, LS_, false, true, float);        \
    else if (pair && ce) DVQ_LAUNCH_TC_PAIR(TR_, LS_, true, false, float);   \
    else if (pair) DVQ_LAUNCH_TC_PAIR(TR_, LS_, false, false, float);        \
    else if (st) DVQ_LAUNCH_TC(0, TR_, LS_, false, true, float);             \
    else if (ce) DVQ_LAUNCH_TC(0, TR_, LS_, true, false, float);             \
    else DVQ_LAUNCH_TC(0, TR_, LS_, false, false, float);                    \
  } while (0)
#define DVQ_LAUNCH_TC_GENERIC_BF16(TR_, LS_)                                 \
  do {                                                                       \
    if (pair) DVQ_LAUNCH_TC_PAIR(TR_, LS_, false, false, __nv_bfloat16);     \
    else DVQ_LAUNCH_TC(0, TR_, LS_, false, false, __nv_bfloat16);            \
  } while (0)
  // two-sub-chunk filter with the epilogue-heavy register split (DVQ_TC_ST=1; streamed codebooks only).  Measured
  // within +-2 % of the default at every K >= 2048 shape of the sweep, so it is not selected automatically.
  const bool st = !zbf && streamed && st_env && st_env[0] == '1';
  const bool list = cand_list_mode(K);
  if (zbf) {
    if (D == 64 && !list && !streamed) {
      if (train) DVQ_LAUNCH_TC(64, true, false, false, false, __nv_bfloat16); else DVQ_LAUNCH_TC(64, false, false, false, false, __nv_bfloat16);
    } else if (!list) {
      if (train) DVQ_LAUNCH_TC_GENERIC_BF16(true, false); else DVQ_LAUNCH_TC_GENERIC_BF16(false, false);
    } else {
      if (train) DVQ_LAUNCH_TC_GENERIC_BF16(true, true); else DVQ_LAUNCH_TC_GENERIC_BF16(false, true);
    }
  } else if (D == 64 && !list && !streamed) {
    if (train) DVQ_LAUNCH_TC(64, true, false, false, false, float); else DVQ_LAUNCH_TC(64, false, false, false, false, float);
  } else if (!list) {
    if (train) DVQ_LAUNCH_TC_GENERIC(true, false); else DVQ_LAUNCH_TC_GENERIC(false, false);
  } else {
    if (train) DVQ_LAUNCH_TC_GENERIC(true, true); else DVQ_LAUNCH_TC_GENERIC(false, true);
  }
#undef DVQ_LAUNCH_TC_GENERIC_BF16
#undef DVQ_LAUNCH_TC_GENERIC
#undef DVQ_LAUNCH_TC_PAIR
#undef DVQ_LAUNCH_TC
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

}  // namespace dvq
