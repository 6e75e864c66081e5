// Exact FP32 CUDA-core VQ kernel: fused distance + first-argmin + codebook gather +
// straight-through / SSE / usage histogram.  Replaces network/vqvae/quantizer.py:36-43,56-60
// without materialising the N x K distance matrix.
//
// Role in the design: the always-correct path for any (N, K, D).
//
// Numerics (SURVEY §0.4): the contract of vq_exact.cuh — the reference's structure, the winner is the lowest
// index among exact FP32 ties.
//
// Tiling: CTA = 256 threads, 128 rows x 128 codes x 16-wide D chunks; each thread owns an
// 8x8 register tile split 4+4 (rows ty*4.., 64+ty*4..; codes tx*4.., 64+tx*4..) so every
// shared-memory read is a conflict-free 128-bit load.  Roofline: FP32 FMA pipe
// (2*N*K*D flop); it is the *fallback*, the tensor path is the fast one.
#include <type_traits>

#include "vq_exact.cuh"

namespace dvq {

namespace {
constexpr int BM = 128;
constexpr int BN = 128;
constexpr int BK = 16;
constexpr int LDT = 132;  // padded leading dim (floats); multiple of 4 keeps float4 reads aligned
constexpr int NTHREADS = 256;

// T = float (codebook, fp32 z) or __nv_bfloat16 (DVQ_Z_BF16 z, upcast exactly)
template <bool VEC, typename T>
__device__ __forceinline__ float4 load4(const T* __restrict__ base, int64_t row, int D, int k) {
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (row < 0) return v;
  const T* p = base + row * (int64_t)D + k;
  if (VEC) {
    if (k < D) v = zldg4(p);
  } else {
    if (k + 0 < D) v.x = zf(__ldg(p + 0));
    if (k + 1 < D) v.y = zf(__ldg(p + 1));
    if (k + 2 < D) v.z = zf(__ldg(p + 2));
    if (k + 3 < D) v.w = zf(__ldg(p + 3));
  }
  return v;
}

template <bool VEC, typename ZT>
__global__ void __launch_bounds__(NTHREADS, 2)
vq_simt_kernel(const ZT* __restrict__ z, const float* __restrict__ E, const float* __restrict__ ee,
               int64_t N, int K, int D, int train, ZT* __restrict__ zq, int64_t* __restrict__ idx_out,
               unsigned long long* __restrict__ hist, double* __restrict__ sse) {
  __shared__ __align__(16) float zs[BK][LDT];
  __shared__ __align__(16) float es[BK][LDT];
  __shared__ int64_t srow[BM];
  __shared__ int sidx[BM];
  __shared__ __align__(16) float szz[BM];
  __shared__ double ssum[NTHREADS / 32];

  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int lrow = tid >> 2;       // loader: tile row (and +64)
  const int lk = (tid & 3) * 4;    // loader: offset inside the 16-wide D chunk
  const int warp = tid >> 5, lane = tid & 31;

  const int64_t ntiles = (N + BM - 1) / BM;

  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    if (tid < BM) {
      const int64_t r = tile * BM + tid;
      srow[tid] = r < N ? r : (int64_t)-1;
    }
    __syncthreads();
    const int64_t grow0 = srow[lrow], grow1 = srow[lrow + 64];

    // ||z_row||^2: one warp per row, lane-strided fmaf partials + shuffle tree (row stays in L2
    // for the main loop below)
    for (int r = warp; r < BM; r += NTHREADS / 32) {
      const int64_t grow = srow[r];
      float s2 = grow >= 0 ? sq_partial_ldg(z + grow * (int64_t)D, D, lane) : 0.f;
      s2 = warp_sum(s2);
      if (lane == 0) szz[r] = s2;
    }

    float best[8];
    int bidx[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { best[i] = INFINITY; bidx[i] = 0; }

    for (int kt = 0; kt < K; kt += BN) {
      float acc[8][8];
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

      const int64_t c0 = (kt + lrow < K) ? (int64_t)(kt + lrow) : -1;
      const int64_t c1 = (kt + lrow + 64 < K) ? (int64_t)(kt + lrow + 64) : -1;
      float4 pz0 = load4<VEC>(z, grow0, D, lk), pz1 = load4<VEC>(z, grow1, D, lk);
      float4 pe0 = load4<VEC>(E, c0, D, lk), pe1 = load4<VEC>(E, c1, D, lk);

      for (int d0 = 0; d0 < D; d0 += BK) {
        __syncthreads();  // everyone finished reading the previous chunk
        zs[lk + 0][lrow] = pz0.x; zs[lk + 1][lrow] = pz0.y; zs[lk + 2][lrow] = pz0.z; zs[lk + 3][lrow] = pz0.w;
        zs[lk + 0][lrow + 64] = pz1.x; zs[lk + 1][lrow + 64] = pz1.y; zs[lk + 2][lrow + 64] = pz1.z; zs[lk + 3][lrow + 64] = pz1.w;
        es[lk + 0][lrow] = pe0.x; es[lk + 1][lrow] = pe0.y; es[lk + 2][lrow] = pe0.z; es[lk + 3][lrow] = pe0.w;
        es[lk + 0][lrow + 64] = pe1.x; es[lk + 1][lrow + 64] = pe1.y; es[lk + 2][lrow + 64] = pe1.z; es[lk + 3][lrow + 64] = pe1.w;
        __syncthreads();
        if (d0 + BK < D) {  // register prefetch of the next chunk overlaps the FMAs below
          pz0 = load4<VEC>(z, grow0, D, d0 + BK + lk); pz1 = load4<VEC>(z, grow1, D, d0 + BK + lk);
          pe0 = load4<VEC>(E, c0, D, d0 + BK + lk);    pe1 = load4<VEC>(E, c1, D, d0 + BK + lk);
        }
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
          const float4 a0 = *reinterpret_cast<const float4*>(&zs[kk][ty * 4]);
          const float4 a1 = *reinterpret_cast<const float4*>(&zs[kk][64 + ty * 4]);
          const float4 b0 = *reinterpret_cast<const float4*>(&es[kk][tx * 4]);
          const float4 b1 = *reinterpret_cast<const float4*>(&es[kk][64 + tx * 4]);
          const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
          const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
          for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
      }
      // distance + running first-argmin for this code tile (codes visited in ascending order)
      float zz[8];
      {
        const float4 q0 = *reinterpret_cast<const float4*>(&szz[ty * 4]);
        const float4 q1 = *reinterpret_cast<const float4*>(&szz[64 + ty * 4]);
        zz[0] = q0.x; zz[1] = q0.y; zz[2] = q0.z; zz[3] = q0.w; zz[4] = q1.x; zz[5] = q1.y; zz[6] = q1.z; zz[7] = q1.w;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int c = kt + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
        if (c < K) {
          const float eev = __ldg(ee + c);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float dist = exact_dist(acc[i][j], zz[i], eev);
            if (dist < best[i]) { best[i] = dist; bidx[i] = c; }
          }
        }
      }
    }

    // combine the 16 threads (tx) that share each row: lexicographic (distance, index) minimum
#pragma unroll
    for (int i = 0; i < 8; ++i) {
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) {
        const float od = __shfl_xor_sync(0xffffffffu, best[i], o);
        const int oi = __shfl_xor_sync(0xffffffffu, bidx[i], o);
        if (od < best[i] || (od == best[i] && oi < bidx[i])) { best[i] = od; bidx[i] = oi; }
      }
    }
    if (tx == 0) {
#pragma unroll
      for (int i = 0; i < 8; ++i) sidx[(i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4))] = bidx[i];
    }
    __syncthreads();

    // gather / straight-through / SSE / histogram: one warp per row, 128-bit accesses
    double lsse = 0.0;
    for (int r = warp; r < BM; r += NTHREADS / 32) {
      const int64_t grow = srow[r];
      if (grow < 0) continue;
      const int k = sidx[r];
      const float* erow = E + (int64_t)k * D;
      const ZT* zrow = z + grow * (int64_t)D;
      ZT* orow = zq + grow * (int64_t)D;
      if (VEC) {
        for (int c = lane * 4; c < D; c += 128) {
          float4 o4 = ldg4(erow + c);
          if (train) o4 = st_step4(o4, zldg4(zrow + c), lsse);
          zst4(orow + c, o4);
        }
      } else {
        for (int c = lane; c < D; c += 32) {
          float o1 = __ldg(erow + c);
          if (train) o1 = st_step1(o1, zf(__ldg(zrow + c)), lsse);
          zst1(orow + c, o1);
        }
      }
      if (lane == 0) {
        idx_out[grow] = (int64_t)k;
        if (train) atomicAdd(hist + k, 1ull);
      }
    }
    if (train) {
      lsse = warp_sum(lsse);
      if (lane == 0) ssum[warp] = lsse;
      __syncthreads();
      if (tid == 0) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < NTHREADS / 32; ++w) t += ssum[w];
        atomicAdd(sse, t);
      }
    }
    __syncthreads();  // srow / sidx / ssum are rewritten by the next tile
  }
}

__global__ void code_norms_kernel(const float* __restrict__ E, int K, int D, float* __restrict__ ee) {
  // one warp per code: lane-strided fmaf partials, then a shuffle tree
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= K) return;
  const float s = warp_sum(sq_partial_ldg(E + (int64_t)warp * D, D, lane));
  if (lane == 0) ee[warp] = s;
}
}  // namespace

int launch_code_norms(const float* E, int K, int D, float* ee, cudaStream_t s) {
  const int threads = 256;
  const int blocks = (K * 32 + threads - 1) / threads;
  code_norms_kernel<<<blocks, threads, 0, s>>>(E, K, D, ee);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

int launch_vq_simt(const VqCall& c) {
  const int64_t tiles = (c.N + BM - 1) / BM;
  int64_t grid = (int64_t)c.sm_count * 2;
  if (tiles < grid) grid = tiles;
  if (grid < 1) grid = 1;
  // 128-bit codebook loads; z / z_q rows move 4 elements at a time (16 bytes fp32, 8 bytes bf16)
  const bool vec = (c.D % 4 == 0) && reinterpret_cast<uintptr_t>(c.E) % 16 == 0 &&
                   (reinterpret_cast<uintptr_t>(c.z) | reinterpret_cast<uintptr_t>(c.z_q)) % (c.zbf ? 8 : 16) == 0;
  with_z_type(c, [&](auto z, auto z_q) {
    using ZT = std::remove_pointer_t<decltype(z_q)>;
    auto kern = vec ? vq_simt_kernel<true, ZT> : vq_simt_kernel<false, ZT>;
    kern<<<(unsigned)grid, NTHREADS, 0, c.s>>>(z, c.E, c.ee, c.N, c.K, c.D, c.train, z_q, c.idx, c.hist, c.sse);
    return DVQ_OK;
  });
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

}  // namespace dvq
