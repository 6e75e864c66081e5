// tcgen05 GEMM with fused epilogues for the GatedPixelCNN prior's row-cached sampler (SURVEY §8f-1;
// network/pixelcnn/models.py:65-88 gated layer, :176-197 generate).  Every contraction of the sampler — the masked
// vertical / horizontal convolutions (one K-segment per kernel tap), vertical-to-horizontal and residual 1x1
// convolutions, the two 1x1 convolutions of the output head — is one launch of this kernel:
//
//     C[m, n] = sum over segments s of  A_s[m + shift_s, :] . W_s[:, n]        (FP16 operands, FP32 accumulation in TMEM)
//
// Activations live in HBM as UMMA operand IMAGES (FP16, K-major, no swizzle): rows in tiles of 128, a tile stored
// [K/8][128 rows][8 halfs], so a 64-wide K slice of a tile is 16 KB contiguous = ONE bulk copy (TMA engine) straight
// into the shared-memory operand slot, and a thread of the epilogue (thread = row) writes the next layer's operand
// with coalesced 16-byte stores.  Rows of a grid row are ordered column-major (m = column * B + b), so a convolution
// tap at column offset t is a whole-tile shift of t * B / 128 tiles: no im2col copy, no shift-add pass; taps that fall
// outside the grid are skipped per tile.  Weights are packed once into images [n-tile][K/8][256][8].
//
// Pipeline (one persistent CTA per SM, 6 warps): warp 0 producer (bulk copies into a 4-stage ring of 16 KB A + 32 KB B
// slices), warp 1 MMA issuer (tcgen05.mma M=128 N=256 K=16, two 256-column accumulator stages in TMEM so the MMAs of
// tile t+1 overlap the epilogue of tile t), warps 2-5 epilogue (thread = row, tcgen05.ld 32 columns at a time).
// Epilogues: GATE  tanh(a + cond_a) * sigmoid(b + cond_b) -> FP16 image (+ the raw pre-activation image for the
//                  vertical-to-horizontal convolution); an output tile holds 128 'a' and the matching 128 'b' columns;
//            RES   acc + bias (+ residual FP32 image) -> FP32 image and FP16 image;   RELU -> FP16 image;
//            LOGITS acc + bias -> FP32 row-major [rows, N].
// Roofline: tensor pipe; 128x256 tiles streamed from L2 have 85 flop/B, so L2 bandwidth caps the kernel near half of
// the BF16/FP16 peak (measured in profiles/).
#include <cuda_fp16.h>
#include <string.h>

#include "dvq_common.cuh"
#include "tc_prims.cuh"

namespace dvq {
namespace {

constexpr int PTM = 128, PTN = 256, PKS = 64, PSTAGES = 4;
constexpr uint32_t A_SLICE = (PKS / 8) * PTM * 16;      // 16 KB
constexpr uint32_t B_SLICE = (PKS / 8) * PTN * 16;      // 32 KB
constexpr uint32_t STAGE_BYTES = A_SLICE + B_SLICE;
constexpr int PC_THREADS = 192;
constexpr int MAX_SEG = 12;

enum PcMode { PC_GATE = 0, PC_RES = 1, PC_RELU = 2, PC_LOGITS = 3 };

struct PcSeg {
  const uint8_t* a_img;   // activation image (FP16), tiles of 128 rows
  const uint8_t* w_img;   // weight image [n-tile][ks/8][256][8] halfs
  int a_kd;               // K width of the activation image (tile stride = a_kd * 256 bytes)
  int ks;                 // K length of this segment (multiple of 64), read from column 0 of the image
  int tile_shift;         // source tile = output tile + tile_shift
  int col_shift;          // valid iff 0 <= grid column + col_shift < ncols_src
};

struct PcParams {
  PcSeg seg[MAX_SEG];
  int nseg, m_tiles, n_tiles, tiles_per_col, ncols_src, mode;
  const float* bias;          // [n_tiles * 256] in tile column order
  const uint8_t* cond_img;    // GATE: FP16 image [Bp, 2d] of cond[label] (natural a | b feature order), or nullptr
  uint8_t* out_img;           // FP16 output image (K width out_kd), GATE / RES / RELU
  uint8_t* pre_img;           // GATE: raw pre-activation image (K width 2 * out_kd) or nullptr
  float* res_img;             // RES: FP32 image [K/4][128][4] per tile, read (if res_in) and written
  float* logits;              // LOGITS: row-major [m_tiles * 128, n_tiles * 256]
  int out_kd, res_in, d_gate; // d_gate: number of gated features (column offset of the 'b' half in cond / pre images)
  int* err;
};

__device__ __forceinline__ float tanh_fast(float x) {
  float r;
  asm("tanh.approx.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ float2 unpack_f16x2(uint32_t v) {
  const __half2 h = *reinterpret_cast<const __half2*>(&v);
  return __half22float2(h);
}

// segment s contributes to the tiles of grid column col (the producer, MMA and epilogue warps all decide with this)
__device__ __forceinline__ bool seg_valid(const PcParams& p, int s, int col) {
  const int sc = col + p.seg[s].col_shift;
  return sc >= 0 && sc < p.ncols_src;
}

__global__ void __launch_bounds__(PC_THREADS, 1) pcnn_gemm_kernel(const __grid_constant__ PcParams p) {
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_full[PSTAGES], bar_empty[PSTAGES], bar_acc_full[2], bar_acc_empty[2];
  __shared__ uint32_t tmem_slot;
  __shared__ int serr;
  __shared__ float sbias[2][PTN];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    serr = 0;
    for (int i = 0; i < PSTAGES; ++i) { tc::mbar_init(&bar_full[i], 1); tc::mbar_init(&bar_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { tc::mbar_init(&bar_acc_full[i], 1); tc::mbar_init(&bar_acc_empty[i], 4); }
    tc::fence_barrier_init();
  }
  if (warp == 1) tc::tmem_alloc(&tmem_slot, 512);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = tmem_slot;
  volatile int* errw = &serr;
  const int ntiles = p.m_tiles * p.n_tiles;
  const uint32_t sbase = tc::smem_u32(smem);

  if (warp == 0) {
    // ===================== producer =====================
    if (lane == 0) {
      uint32_t it = 0;
      bool ok = true;
      for (int tile = blockIdx.x; ok && tile < ntiles; tile += gridDim.x) {
        const int mt = tile / p.n_tiles, nt = tile - mt * p.n_tiles;
        const int col = mt / p.tiles_per_col;
        for (int s = 0; ok && s < p.nseg; ++s) {
          if (!seg_valid(p, s, col)) continue;
          const PcSeg& sg = p.seg[s];
          const uint8_t* a = sg.a_img + (size_t)(mt + sg.tile_shift) * sg.a_kd * 256;
          const uint8_t* w = sg.w_img + (size_t)nt * sg.ks * 512;
          for (int k0 = 0; k0 < sg.ks; k0 += PKS, ++it) {
            const uint32_t st = it % PSTAGES, ph = (it / PSTAGES) & 1u;
            if (!tc::mbar_wait(&bar_empty[st], ph ^ 1u, errw, 1)) { ok = false; break; }
            tc::mbar_arrive_expect_tx(&bar_full[st], STAGE_BYTES);
            uint8_t* dst = smem + st * STAGE_BYTES;
            tc::bulk_g2s(dst, a + (size_t)(k0 / 8) * 2048, A_SLICE, &bar_full[st]);
            tc::bulk_g2s(dst + A_SLICE, w + (size_t)(k0 / 8) * 4096, B_SLICE / 2, &bar_full[st]);
            tc::bulk_g2s(dst + A_SLICE + B_SLICE / 2, w + (size_t)(k0 / 8) * 4096 + B_SLICE / 2, B_SLICE / 2, &bar_full[st]);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const uint32_t idesc = tc::make_idesc_f16(PTM, PTN, 0);
    uint32_t it = 0, q = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++q) {
      const int mt = tile / p.n_tiles;
      const int col = mt / p.tiles_per_col;
      const uint32_t t = q & 1u;
      if (!tc::mbar_wait(&bar_acc_empty[t], ((q >> 1) & 1u) ^ 1u, errw, 2)) break;
      tc::tc_fence_after();
      uint32_t acc = 0;
      for (int s = 0; s < p.nseg; ++s) {
        if (!seg_valid(p, s, col)) continue;
        const PcSeg& sg = p.seg[s];
        for (int k0 = 0; k0 < sg.ks; k0 += PKS, ++it) {
          const uint32_t st = it % PSTAGES, ph = (it / PSTAGES) & 1u;
          if (!tc::mbar_wait(&bar_full[st], ph, errw, 3)) { acc = 0xffffffffu; break; }
          tc::tc_fence_after();
          if (tc::elect_one()) {
            uint64_t ad = tc::make_smem_desc(sbase + st * STAGE_BYTES, PTM * 16, 128);
            uint64_t bd = tc::make_smem_desc(sbase + st * STAGE_BYTES + A_SLICE, PTN * 16, 128);
#pragma unroll
            for (int j = 0; j < PKS / 16; ++j) {
              tc::umma_f16(tmem + t * PTN, ad, bd, idesc, acc);
              acc = 1u;
              ad += (uint64_t)((2 * PTM * 16) >> 4); bd += (uint64_t)((2 * PTN * 16) >> 4);
            }
            tc::umma_commit(&bar_empty[st]);      // the slot is free once these MMAs have read it
          }
          acc = 1u;
          __syncwarp();
        }
        if (acc == 0xffffffffu) break;
      }
      if (acc == 0xffffffffu) break;
      if (tc::elect_one()) tc::umma_commit(&bar_acc_full[t]);
      __syncwarp();
    }
  } else {
    // ===================== epilogue: thread = row =====================
    const int ew = warp - 2;                            // 0..3
    const int quarter = warp & 3;                       // TMEM lanes this warp may access
    const int r = quarter * 32 + lane;                  // row inside the tile
    const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
    uint32_t q = 0, live_bits = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++q) {
      const int mt = tile / p.n_tiles, nt = tile - mt * p.n_tiles;
      const uint32_t t = q & 1u;
      // A tile with no valid segment got no MMA: its TMEM stage still holds an earlier tile and is cleared below.  Lane k
      // decides for the CTA's tile q + k, 32 tiles at a time, so the test stays off the per-tile path.
      if ((q & 31u) == 0) {
        const long long lt = tile + (long long)lane * gridDim.x;
        bool live = false;
        if (lt < ntiles)
          for (int s = 0; s < p.nseg && !live; ++s) live = seg_valid(p, s, (int)lt / p.n_tiles / p.tiles_per_col);
        live_bits = __ballot_sync(0xffffffffu, live);
      }
      // bias of this tile -> shared memory (the four epilogue warps: 2 floats per thread)
      {
        const int et = ew * 32 + lane;
        sbias[t][et] = __ldg(p.bias + (size_t)nt * PTN + et);
        sbias[t][et + 128] = __ldg(p.bias + (size_t)nt * PTN + et + 128);
        asm volatile("bar.sync 1, 128;" ::: "memory");
      }
      if (!tc::mbar_wait(&bar_acc_full[t], (q >> 1) & 1u, errw, 4)) break;
      tc::tc_fence_after();
      const uint32_t tbase = tmem + lane_addr + t * PTN;
      if (!((live_bits >> (q & 31u)) & 1u)) {
        for (int c = 0; c < PTN; c += 32) tc::tmem_st32_zero(tbase + (uint32_t)c);
        tc::tmem_st_wait();
      }
      const float* bs = sbias[t];
      if (p.mode == PC_GATE) {
        const int f0 = nt * 128;                        // first gated feature of this tile
        const size_t out_tile = (size_t)mt * p.out_kd * 256;
        const size_t pre_tile = (size_t)mt * p.out_kd * 512;
        const size_t cond_tile = (size_t)(mt % p.tiles_per_col) * p.d_gate * 512;
#pragma unroll 1
        for (int g = 0; g < 4; ++g) {
          uint32_t va[32], vb[32];
          tc::tmem_ld32(tbase + (uint32_t)(g * 32), va);
          tc::tmem_ld32(tbase + 128u + (uint32_t)(g * 32), vb);
          tc::tmem_ld_wait_dep32(va);
          tc::tmem_ld_wait_dep32(vb);
#pragma unroll
          for (int c8 = 0; c8 < 4; ++c8) {              // 8 features -> one 16-byte chunk of the output image
            const int f = f0 + g * 32 + c8 * 8;
            uint4 ca = make_uint4(0u, 0u, 0u, 0u), cb = ca;
            if (p.cond_img) {
              ca = __ldg(reinterpret_cast<const uint4*>(p.cond_img + cond_tile + (size_t)(f >> 3) * 2048 + r * 16));
              cb = __ldg(reinterpret_cast<const uint4*>(p.cond_img + cond_tile + (size_t)((p.d_gate + f) >> 3) * 2048 + r * 16));
            }
            const uint32_t cav[4] = {ca.x, ca.y, ca.z, ca.w}, cbv[4] = {cb.x, cb.y, cb.z, cb.w};
            uint32_t og[4], pa[4], pb[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int j = c8 * 8 + e * 2;
              const float a0 = __uint_as_float(va[j]) + bs[g * 32 + j], a1 = __uint_as_float(va[j + 1]) + bs[g * 32 + j + 1];
              const float b0 = __uint_as_float(vb[j]) + bs[128 + g * 32 + j], b1 = __uint_as_float(vb[j + 1]) + bs[128 + g * 32 + j + 1];
              pa[e] = pack_f16x2(a0, a1);
              pb[e] = pack_f16x2(b0, b1);
              const float2 fa = unpack_f16x2(cav[e]), fb = unpack_f16x2(cbv[e]);
              // tanh(a) * sigmoid(b), sigmoid(x) = 0.5 * tanh(x / 2) + 0.5
              const float g0 = tanh_fast(a0 + fa.x) * fmaf(0.5f, tanh_fast(0.5f * (b0 + fb.x)), 0.5f);
              const float g1 = tanh_fast(a1 + fa.y) * fmaf(0.5f, tanh_fast(0.5f * (b1 + fb.y)), 0.5f);
              og[e] = pack_f16x2(g0, g1);
            }
            *reinterpret_cast<uint4*>(p.out_img + out_tile + (size_t)(f >> 3) * 2048 + r * 16) = make_uint4(og[0], og[1], og[2], og[3]);
            if (p.pre_img) {
              *reinterpret_cast<uint4*>(p.pre_img + pre_tile + (size_t)(f >> 3) * 2048 + r * 16) = make_uint4(pa[0], pa[1], pa[2], pa[3]);
              *reinterpret_cast<uint4*>(p.pre_img + pre_tile + (size_t)((p.d_gate + f) >> 3) * 2048 + r * 16) = make_uint4(pb[0], pb[1], pb[2], pb[3]);
            }
          }
        }
      } else {
        const int f0 = nt * PTN;
#pragma unroll 1
        for (int g = 0; g < 8; ++g) {
          uint32_t v[32];
          tc::tmem_ld32(tbase + (uint32_t)(g * 32), v);
          tc::tmem_ld_wait_dep32(v);
          float x[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) x[j] = __uint_as_float(v[j]) + bs[g * 32 + j];
          if (p.mode == PC_LOGITS) {
            float* dst = p.logits + ((size_t)mt * PTM + r) * ((size_t)p.n_tiles * PTN) + f0 + g * 32;
#pragma unroll
            for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(dst + j) = make_float4(x[j], x[j + 1], x[j + 2], x[j + 3]);
          } else {
            if (p.mode == PC_RES) {
              float* rt = p.res_img + (size_t)mt * p.out_kd * 128;
#pragma unroll
              for (int c4 = 0; c4 < 8; ++c4) {
                float4* rp = reinterpret_cast<float4*>(rt + (size_t)((f0 + g * 32 + c4 * 4) >> 2) * 512 + r * 4);
                if (p.res_in) {
                  const float4 o = *rp;
                  x[c4 * 4] += o.x; x[c4 * 4 + 1] += o.y; x[c4 * 4 + 2] += o.z; x[c4 * 4 + 3] += o.w;
                }
                *rp = make_float4(x[c4 * 4], x[c4 * 4 + 1], x[c4 * 4 + 2], x[c4 * 4 + 3]);
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) x[j] = fmaxf(x[j], 0.f);
            }
            const size_t out_tile = (size_t)mt * p.out_kd * 256;
#pragma unroll
            for (int c8 = 0; c8 < 4; ++c8) {
              const int f = f0 + g * 32 + c8 * 8;
              *reinterpret_cast<uint4*>(p.out_img + out_tile + (size_t)(f >> 3) * 2048 + r * 16) =
                  make_uint4(pack_f16x2(x[c8 * 8], x[c8 * 8 + 1]), pack_f16x2(x[c8 * 8 + 2], x[c8 * 8 + 3]),
                             pack_f16x2(x[c8 * 8 + 4], x[c8 * 8 + 5]), pack_f16x2(x[c8 * 8 + 6], x[c8 * 8 + 7]));
            }
          }
        }
      }
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&bar_acc_empty[t]);
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (tid == 0 && serr != 0 && p.err) *p.err = serr;
  if (warp == 1) tc::tmem_dealloc(tmem, 512);
}

// indices of one grid row -> the embedding rows as FP16 operand image (+ FP32 residual image), rows m = column * Bp + b
__global__ void pcnn_embed_kernel(const int64_t* __restrict__ x, int x_stride, int W, int B, int Bp, const float* __restrict__ emb,
                                  int n_emb, int d, uint8_t* __restrict__ img16, float* __restrict__ img32) {
  const int chunks = d / 8;
  const int64_t total = (int64_t)W * Bp * chunks;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(i & 127);
    const int64_t rest = i >> 7;
    const int ch = (int)(rest % chunks);
    const int64_t tile = rest / chunks;
    const int64_t m = tile * 128 + r;
    const int c = (int)(m / Bp), b = (int)(m - (int64_t)c * Bp);
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (b < B) {
      int64_t k = x[(int64_t)b * x_stride + c];
      k = k < 0 ? 0 : (k >= n_emb ? n_emb - 1 : k);
      const float4 lo = ldg4(emb + k * d + ch * 8), hi = ldg4(emb + k * d + ch * 8 + 4);
      v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w; v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
    }
    *reinterpret_cast<uint4*>(img16 + (size_t)tile * d * 256 + (size_t)ch * 2048 + r * 16) =
        make_uint4(pack_f16x2(v[0], v[1]), pack_f16x2(v[2], v[3]), pack_f16x2(v[4], v[5]), pack_f16x2(v[6], v[7]));
    if (img32) {
      float* t32 = img32 + (size_t)tile * d * 128;
      *reinterpret_cast<float4*>(t32 + (size_t)(ch * 2) * 512 + r * 4) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(t32 + (size_t)(ch * 2 + 1) * 512 + r * 4) = make_float4(v[4], v[5], v[6], v[7]);
    }
  }
}

// table[label[b], :] (FP32 [n_rows, kd]) -> FP16 image [Bp, kd] (the class-conditional term of a gated layer)
__global__ void pcnn_rows_to_image_kernel(const int64_t* __restrict__ label, int B, int Bp, const float* __restrict__ table, int n_rows,
                                          int kd, uint8_t* __restrict__ img16) {
  const int chunks = kd / 8;
  const int64_t total = (int64_t)Bp * chunks;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(i & 127);
    const int64_t rest = i >> 7;
    const int ch = (int)(rest % chunks);
    const int64_t tile = rest / chunks;
    const int b = (int)(tile * 128 + r);
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (b < B) {
      int64_t k = label[b];
      k = k < 0 ? 0 : (k >= n_rows ? n_rows - 1 : k);
      const float4 lo = ldg4(table + k * kd + ch * 8), hi = ldg4(table + k * kd + ch * 8 + 4);
      v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w; v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
    }
    *reinterpret_cast<uint4*>(img16 + (size_t)tile * kd * 256 + (size_t)ch * 2048 + r * 16) =
        make_uint4(pack_f16x2(v[0], v[1]), pack_f16x2(v[2], v[3]), pack_f16x2(v[4], v[5]), pack_f16x2(v[6], v[7]));
  }
}

}  // namespace

int launch_pcnn_gemm(const DvqPcnnGemm* g, cudaStream_t s) {
  if (!g) return fail(DVQ_ERR_BAD_ARG, "gemm descriptor is NULL");
  if (g->nseg <= 0 || g->nseg > MAX_SEG) return fail(DVQ_ERR_BAD_SHAPE, "1..%d K-segments per launch", MAX_SEG);
  if (g->m_tiles <= 0 || g->n_tiles <= 0 || g->tiles_per_col <= 0) return fail(DVQ_ERR_BAD_SHAPE, "empty tile grid");
  if (g->mode < 0 || g->mode > 3) return fail(DVQ_ERR_BAD_ARG, "unknown epilogue mode");
  DeviceProps dp;
  int rc = device_props(&dp);
  if (rc) return rc;
  PcParams p;
  memset(&p, 0, sizeof(p));
  for (int i = 0; i < g->nseg; ++i) {
    const DvqPcnnSeg& sg = g->seg[i];
    if (!sg.a_img || !sg.w_img || sg.ks <= 0 || sg.ks % PKS || sg.a_kd < sg.ks || sg.a_kd % 8)
      return fail(DVQ_ERR_BAD_SHAPE, "segment %d: K must be a positive multiple of 64 within the image width", i);
    if ((reinterpret_cast<uintptr_t>(sg.a_img) | reinterpret_cast<uintptr_t>(sg.w_img)) % 16)
      return fail(DVQ_ERR_BAD_ALIGN, "segment %d: images need 16-byte alignment", i);
    p.seg[i].a_img = static_cast<const uint8_t*>(sg.a_img); p.seg[i].w_img = static_cast<const uint8_t*>(sg.w_img);
    p.seg[i].a_kd = sg.a_kd; p.seg[i].ks = sg.ks; p.seg[i].tile_shift = sg.tile_shift; p.seg[i].col_shift = sg.col_shift;
  }
  p.nseg = g->nseg; p.m_tiles = g->m_tiles; p.n_tiles = g->n_tiles; p.tiles_per_col = g->tiles_per_col; p.ncols_src = g->ncols_src;
  p.mode = g->mode; p.bias = g->bias; p.cond_img = static_cast<const uint8_t*>(g->cond_img); p.out_img = static_cast<uint8_t*>(g->out_img);
  p.pre_img = static_cast<uint8_t*>(g->pre_img); p.res_img = g->res_img; p.logits = g->logits; p.out_kd = g->out_kd; p.res_in = g->res_in;
  p.d_gate = g->d_gate; p.err = g->err;
  if (!p.bias) return fail(DVQ_ERR_BAD_ARG, "bias is NULL");
  if (p.mode == PC_LOGITS ? !p.logits : !p.out_img) return fail(DVQ_ERR_BAD_ARG, "output buffer is NULL");
  if (p.mode == PC_RES && !p.res_img) return fail(DVQ_ERR_BAD_ARG, "RES mode needs the FP32 residual image");
  const int ntiles = p.m_tiles * p.n_tiles;
  const int grid = ntiles < dp.sm_count ? ntiles : dp.sm_count;
  const size_t smem = (size_t)PSTAGES * STAGE_BYTES + 128;
  // the opt-in applies to the current device only; set once per device, not per launch (hundreds per sample grid)
  static bool attr_set[64] = {};
  if (!attr_set[dp.ordinal]) {
    DVQ_CUDA_CHECK(cudaFuncSetAttribute(pcnn_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set[dp.ordinal] = true;
  }
  pcnn_gemm_kernel<<<grid, PC_THREADS, smem, s>>>(p);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

int launch_pcnn_embed(const int64_t* x, int x_stride, int W, int B, int Bp, const float* emb, int n_emb, int d, void* img16,
                      float* img32, cudaStream_t s) {
  const int64_t total = (int64_t)W * Bp * (d / 8);
  int64_t blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  pcnn_embed_kernel<<<(unsigned)blocks, 256, 0, s>>>(x, x_stride, W, B, Bp, emb, n_emb, d, static_cast<uint8_t*>(img16), img32);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

int launch_pcnn_rows_to_image(const int64_t* label, int B, int Bp, const float* table, int n_rows, int kd, void* img16, cudaStream_t s) {
  const int64_t total = (int64_t)Bp * (kd / 8);
  int64_t blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  pcnn_rows_to_image_kernel<<<(unsigned)blocks, 256, 0, s>>>(label, B, Bp, table, n_rows, kd, static_cast<uint8_t*>(img16));
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

}  // namespace dvq
