// HBM-bound tail kernels of the VQ path: optional one-hot materialisation
// (quantizer.py:40-42), the scalar finalisation of loss / perplexity (:56-57, :63-64) and the
// index -> embedding gather behind get_emb (:68-75).
#include "dvq_common.cuh"

namespace dvq {
namespace {

// min_encodings [N,K] fp32: every element written exactly once with coalesced 128-bit stores
// (algorithmic bytes: 4*N*K written + 8*N read).
__global__ void onehot_kernel_v4(const int64_t* __restrict__ idx, int64_t N, int K, float* __restrict__ out) {
  const int kv = K >> 2;
  const int64_t total = N * (int64_t)kv;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / kv;
    const int col = (int)(i - row * kv) << 2;
    const int k = (int)__ldg(idx + row);
    float4 v;
    v.x = (col + 0 == k) ? 1.f : 0.f;
    v.y = (col + 1 == k) ? 1.f : 0.f;
    v.z = (col + 2 == k) ? 1.f : 0.f;
    v.w = (col + 3 == k) ? 1.f : 0.f;
    __stcs(reinterpret_cast<float4*>(out) + i, v);  // streaming store: never re-read
  }
}
__global__ void onehot_kernel_s(const int64_t* __restrict__ idx, int64_t N, int K, float* __restrict__ out) {
  const int64_t total = N * (int64_t)K;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / K;
    const int col = (int)(i - row * K);
    out[i] = (col == (int)__ldg(idx + row)) ? 1.f : 0.f;
  }
}

__global__ void finalize_kernel(const unsigned long long* __restrict__ hist, const double* __restrict__ sse,
                                int64_t N_arg, int K, int D, float al, float beta, float* __restrict__ loss,
                                float* __restrict__ ppl) {
  __shared__ double red[32];
  __shared__ double s_n;
  // N_arg == 0: the global row count is the histogram total (every row is counted exactly once), so a
  // row-sharded caller needs no second collective for it
  if (N_arg > 0) {
    if (threadIdx.x == 0) s_n = (double)N_arg;
  } else {
    double c = 0.0;
    for (int k = threadIdx.x; k < K; k += blockDim.x) c += (double)hist[k];
    c = warp_sum(c);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
      s_n = t;
    }
  }
  __syncthreads();
  const double n = s_n;
  double s = 0.0;
  const double inv_n = 1.0 / n;
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    const double p = (double)hist[k] * inv_n;
    s += p * log(p + 1e-10);
  }
  s = warp_sum(s);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
    *ppl = (float)exp(-t);
    const float m = (float)(*sse / (n * (double)D));
    *loss = __fadd_rn(__fmul_rn(al, m), __fmul_rn(beta, m));
  }
}

// out[n,:] = E[idx[n],:]; half-warp or full-warp per row depending on D, 128-bit accesses.
template <bool VEC>
__global__ void gather_kernel(const float* __restrict__ E, const int64_t* __restrict__ idx, int64_t N, int K,
                              int D, float* __restrict__ out, int* __restrict__ oob) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t row = warp0; row < N; row += nwarps) {
    const int64_t k = __ldg(idx + row);
    const bool ok = (k >= 0 && k < K);
    if (!ok && lane == 0 && oob) atomicExch(oob, 1);
    const float* src = E + (ok ? k : 0) * (int64_t)D;
    float* dst = out + row * (int64_t)D;
    if (VEC) {
      for (int c = lane * 4; c < D; c += 128) {
        float4 v = ok ? ldg4(src + c) : make_float4(0.f, 0.f, 0.f, 0.f);
        *reinterpret_cast<float4*>(dst + c) = v;
      }
    } else {
      for (int c = lane; c < D; c += 32) dst[c] = ok ? __ldg(src + c) : 0.f;
    }
  }
}

// Backward of the VQ forward (autograd of network/vqvae/quantizer.py:56-60; SURVEY §8f-3), one pass over the rows:
//   dz[n,:]      = g_zq[n,:] + (g_loss * al   * 2 / (rows * D)) * (z[n,:] - E[idx[n],:])        (straight-through + commitment)
//   dE[idx[n],:] +=          (g_loss * beta * 2 / (rows * D)) * (E[idx[n],:] - z[n,:])        (codebook term, scatter-add)
// g_loss and rows are DEVICE scalars (rows = the all-reduced histogram total on a row-sharded run: no host sync).
// A warp covers a row with 128-bit accesses; the scatter-add is a vector reduction (red.global.add.v4.f32).
__device__ __forceinline__ void red_add_v4(float* addr, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
// ZT = __nv_bfloat16 (DVQ_Z_BF16): z, g_zq and dz are bf16 rows, the arithmetic is the same fp32 on the upcast values and dz is
// rounded once when stored.
template <bool HAS_GZQ, bool WANT_DZ, bool WANT_DE, typename ZT>
__global__ void vq_backward_kernel(const ZT* __restrict__ z, const float* __restrict__ E, const int64_t* __restrict__ idx,
                                   const ZT* __restrict__ g_zq, const float* __restrict__ g_loss, const float* __restrict__ rows,
                                   int64_t N, int D, float al, float beta, ZT* __restrict__ dz, float* __restrict__ dE) {
  const float scale = 2.0f * __ldg(g_loss) / (__ldg(rows) * (float)D);
  const float sz = scale * al, se = scale * beta;
  const int nv = D >> 2;
  const int64_t total = N * (int64_t)nv;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / nv;
    const int c = (int)(i - row * nv) << 2;
    const int64_t k = __ldg(idx + row);
    const float4 z4 = zldcs4(z + row * D + c);
    const float4 e4 = ldg4(E + k * D + c);
    const float4 d4 = make_float4(z4.x - e4.x, z4.y - e4.y, z4.z - e4.z, z4.w - e4.w);
    if (WANT_DZ) {
      float4 o = make_float4(sz * d4.x, sz * d4.y, sz * d4.z, sz * d4.w);
      if (HAS_GZQ) {
        const float4 g4 = zldcs4(g_zq + row * D + c);
        o.x += g4.x; o.y += g4.y; o.z += g4.z; o.w += g4.w;
      }
      zstcs4(dz + row * D + c, o);
    }
    if (WANT_DE) red_add_v4(dE + k * D + c, make_float4(-se * d4.x, -se * d4.y, -se * d4.z, -se * d4.w));
  }
}

// Grouped get_emb (gen_net.py:101-106: six part codebooks, one index each): out[n, g * D .. g * D + D) = E_g[codes[n, g], :]
// for every group in ONE launch, written straight into the concatenated decoder input (row pitch out_stride floats).
struct GatherMultiParams {
  const float* E[8];
  int G;
};
__global__ void gather_multi_kernel(const GatherMultiParams gp, const int64_t* __restrict__ codes, int64_t N, int K, int D,
                                    float* __restrict__ out, int64_t out_stride, int* __restrict__ oob) {
  const int nv = D >> 2;
  const int64_t total = N * gp.G * (int64_t)nv;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % nv) << 2;
    const int64_t ng = i / nv;
    const int g = (int)(ng % gp.G);
    const int64_t n = ng / gp.G;
    const int64_t k = __ldg(codes + n * gp.G + g);
    const bool ok = k >= 0 && k < K;
    if (!ok && oob) atomicExch(oob, 1);
    const float4 v = ok ? ldg4(gp.E[g] + k * D + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    *reinterpret_cast<float4*>(out + n * out_stride + (int64_t)g * D + c) = v;
  }
}

// sums[k,:] += sum over the rows assigned to code k of z[n,:]  (the per-code input sums of an EMA codebook update)
template <typename ZT>
__global__ void vq_code_sums_kernel(const ZT* __restrict__ z, const int64_t* __restrict__ idx, int64_t N, int D,
                                    float* __restrict__ sums) {
  const int nv = D >> 2;
  const int64_t total = N * (int64_t)nv;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / nv;
    const int c = (int)(i - row * nv) << 2;
    red_add_v4(sums + __ldg(idx + row) * D + c, zldcs4(z + row * D + c));
  }
}
}  // namespace

int launch_vq_backward(const void* z, const float* E, const int64_t* idx, const void* g_zq, const float* g_loss,
                       const float* rows, int64_t N, int D, float al, float beta, void* dz, float* dE, bool zbf, cudaStream_t s) {
  if (N == 0 || (!dz && !dE)) return DVQ_OK;
  DeviceProps dp;
  int rc = device_props(&dp);
  if (rc) return rc;
  const int threads = 256;
  int64_t blocks = (N * (D / 4) + threads - 1) / threads;
  if (blocks > (int64_t)dp.sm_count * 16) blocks = (int64_t)dp.sm_count * 16;
#define DVQ_BWD(G_, Z_, E_, T_)                                                                                    \
  vq_backward_kernel<G_, Z_, E_, T_><<<(unsigned)blocks, threads, 0, s>>>(static_cast<const T_*>(z), E, idx,        \
      static_cast<const T_*>(g_zq), g_loss, rows, N, D, al, beta, static_cast<T_*>(dz), dE)
#define DVQ_BWD_T(T_)                                                                                              \
  do {                                                                                                             \
    if (dz && dE) { if (g_zq) DVQ_BWD(true, true, true, T_); else DVQ_BWD(false, true, true, T_); }                 \
    else if (dz) { if (g_zq) DVQ_BWD(true, true, false, T_); else DVQ_BWD(false, true, false, T_); }                \
    else DVQ_BWD(false, false, true, T_);                                                                          \
  } while (0)
  if (zbf) DVQ_BWD_T(__nv_bfloat16);
  else DVQ_BWD_T(float);
#undef DVQ_BWD_T
#undef DVQ_BWD
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

int launch_gather_multi(const float* const* E, int G, const int64_t* codes, int64_t N, int K, int D, float* out, int64_t out_stride,
                        int* oob, cudaStream_t s) {
  if (N == 0) return DVQ_OK;
  DeviceProps dp;
  int rc = device_props(&dp);
  if (rc) return rc;
  GatherMultiParams gp;
  gp.G = G;
  for (int g = 0; g < 8; ++g) gp.E[g] = g < G ? E[g] : nullptr;
  const int threads = 256;
  int64_t blocks = (N * G * (D / 4) + threads - 1) / threads;
  if (blocks > (int64_t)dp.sm_count * 16) blocks = (int64_t)dp.sm_count * 16;
  gather_multi_kernel<<<(unsigned)blocks, threads, 0, s>>>(gp, codes, N, K, D, out, out_stride, oob);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

int launch_vq_code_sums(const void* z, const int64_t* idx, int64_t N, int D, float* sums, bool zbf, cudaStream_t s) {
  if (N == 0) return DVQ_OK;
  DeviceProps dp;
  int rc = device_props(&dp);
  if (rc) return rc;
  const int threads = 256;
  int64_t blocks = (N * (D / 4) + threads - 1) / threads;
  if (blocks > (int64_t)dp.sm_count * 16) blocks = (int64_t)dp.sm_count * 16;
  if (zbf) vq_code_sums_kernel<__nv_bfloat16><<<(unsigned)blocks, threads, 0, s>>>(static_cast<const __nv_bfloat16*>(z), idx, N, D, sums);
  else vq_code_sums_kernel<float><<<(unsigned)blocks, threads, 0, s>>>(static_cast<const float*>(z), idx, N, D, sums);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

int launch_onehot(const int64_t* idx, int64_t N, int K, float* onehot, cudaStream_t s) {
  if (N == 0) return DVQ_OK;
  DeviceProps dp;
  int rc = device_props(&dp);
  if (rc) return rc;
  const int threads = 256;
  const int blocks = dp.sm_count * 8;
  if (K % 4 == 0 && reinterpret_cast<uintptr_t>(onehot) % 16 == 0)
    onehot_kernel_v4<<<blocks, threads, 0, s>>>(idx, N, K, onehot);
  else
    onehot_kernel_s<<<blocks, threads, 0, s>>>(idx, N, K, onehot);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

int launch_finalize(const unsigned long long* hist, const double* sse, int64_t N, int K, int D, float al,
                    float beta, float* loss, float* ppl, cudaStream_t s) {
  finalize_kernel<<<1, 256, 0, s>>>(hist, sse, N, K, D, al, beta, loss, ppl);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

int launch_gather(const float* E, const int64_t* idx, int64_t N, int K, int D, float* out, int* oob,
                  cudaStream_t s) {
  if (N == 0) return DVQ_OK;
  DeviceProps dp;
  int rc = device_props(&dp);
  if (rc) return rc;
  const int threads = 256;
  int64_t blocks = (N * 32 + threads - 1) / threads;
  if (blocks > (int64_t)dp.sm_count * 16) blocks = (int64_t)dp.sm_count * 16;
  const bool vec = (D % 4 == 0) && ((reinterpret_cast<uintptr_t>(E) | reinterpret_cast<uintptr_t>(out)) % 16 == 0);
  if (vec)
    gather_kernel<true><<<(unsigned)blocks, threads, 0, s>>>(E, idx, N, K, D, out, oob);
  else
    gather_kernel<false><<<(unsigned)blocks, threads, 0, s>>>(E, idx, N, K, D, out, oob);
  DVQ_CUDA_CHECK(cudaGetLastError());
  count_launch();
  return DVQ_OK;
}

}  // namespace dvq
