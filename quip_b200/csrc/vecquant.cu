// Signature-compatible stand-ins for the reference's absent `quant_cuda` extension:
//
//     quant_cuda.vecquant3matmul(vec, mat, mul, scales, zeros)      quant.py:229-230
//     quant_cuda.vecquant4matmul(vec, mat, mul, scales, zeros)      zeroShot/models/quant.py:207-208
//
// i.e. mul[n] += sum_k (scales[n] * code[k][n] - zeros[n]) * vec[k] for ONE token, fp32 in and out, on the
// REFERENCE's packed layout (Quant3Linear.pack, quant.py:192-220: int32 (K*3/32, N), 32 codes per 3 rows;
// Quant4Linear, zeroShot/models/quant.py:193-199: int32 (K/8, N), 8 codes per row; 2-bit: the natural extension,
// 16 codes per row).  A checkpoint packed by the reference therefore runs without conversion.  The native path
// (quip_qlinear_forward) is the fast one; this kernel is plain HBM streaming: a thread owns one output column, a warp
// reads 128 contiguous bytes per packed row, the token sits in shared memory, K is split over the grid and the
// partial sums are added to `mul` with one atomic per thread (in-place accumulate, as the reference's call does).
#include "common.cuh"

namespace quip {

namespace {

constexpr int VQ_THREADS = 256;
constexpr int VQ_GROUP_K = 32;            // codes per "group": 3 rows (3-bit), 4 rows (4-bit), 2 rows (2-bit)

template <int BITS>
__device__ __forceinline__ float group_dot(const uint32_t* w, const float* xs) {
  float acc = 0.f;
  if constexpr (BITS == 3) {
    const uint32_t w0 = w[0], w1 = w[1], w2 = w[2];
#pragma unroll
    for (int j = 0; j < 10; ++j) acc = fmaf((float)((w0 >> (3 * j)) & 7u), xs[j], acc);
    acc = fmaf((float)((w0 >> 30) | ((w1 & 1u) << 2)), xs[10], acc);
#pragma unroll
    for (int j = 0; j < 10; ++j) acc = fmaf((float)((w1 >> (3 * j + 1)) & 7u), xs[11 + j], acc);
    acc = fmaf((float)((w1 >> 31) | ((w2 & 3u) << 1)), xs[21], acc);
#pragma unroll
    for (int j = 0; j < 10; ++j) acc = fmaf((float)((w2 >> (3 * j + 2)) & 7u), xs[22 + j], acc);
  } else if constexpr (BITS == 4) {
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc = fmaf((float)((w[r] >> (4 * j)) & 15u), xs[8 * r + j], acc);
  } else {
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
      for (int j = 0; j < 16; ++j) acc = fmaf((float)((w[r] >> (2 * j)) & 3u), xs[16 * r + j], acc);
  }
  return acc;
}

// grid (ceil(N / VQ_THREADS), ksplit); each CTA covers groups [g0, g1) of 32 k
template <int BITS>
__global__ void __launch_bounds__(VQ_THREADS)
vecquant_kernel(const float* __restrict__ vec, const uint32_t* __restrict__ mat, float* __restrict__ mul,
                const float* __restrict__ scales, const float* __restrict__ zeros, int K, int N, int groups_per_cta) {
  constexpr int ROWS = BITS == 3 ? 3 : (BITS == 4 ? 4 : 2);
  extern __shared__ float xs[];                               // this CTA's k range of the token, then its sum
  const int ngroups = K / VQ_GROUP_K;
  const int g0 = blockIdx.y * groups_per_cta, g1 = min(ngroups, g0 + groups_per_cta);
  if (g0 >= g1) return;
  const int nk = (g1 - g0) * VQ_GROUP_K;
  float part = 0.f;
  for (int i = threadIdx.x; i < nk; i += VQ_THREADS) {
    const float v = vec[g0 * VQ_GROUP_K + i];
    xs[i] = v;
    part += v;
  }
  __shared__ float red[VQ_THREADS / 32];
#pragma unroll
  for (int o = 16; o; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
  __syncthreads();
  float xsum = 0.f;
#pragma unroll
  for (int w = 0; w < VQ_THREADS / 32; ++w) xsum += red[w];
  const int n = blockIdx.x * VQ_THREADS + threadIdx.x;
  if (n >= N) return;
  const uint32_t* col = mat + (size_t)g0 * ROWS * N + n;
  float dot = 0.f;
  int g = g0;
  for (; g + 4 <= g1; g += 4) {                               // 4 groups = up to 16 independent loads in flight
    uint32_t w[4][ROWS];
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int r = 0; r < ROWS; ++r) w[u][r] = __ldg(col + (size_t)((g - g0 + u) * ROWS + r) * N);
#pragma unroll
    for (int u = 0; u < 4; ++u) dot += group_dot<BITS>(w[u], xs + (g - g0 + u) * VQ_GROUP_K);
  }
  for (; g < g1; ++g) {
    uint32_t w[ROWS];
#pragma unroll
    for (int r = 0; r < ROWS; ++r) w[r] = __ldg(col + (size_t)((g - g0) * ROWS + r) * N);
    dot += group_dot<BITS>(w, xs + (g - g0) * VQ_GROUP_K);
  }
  atomicAdd(mul + n, scales[n] * dot - zeros[n] * xsum);
}

}  // namespace

}  // namespace quip

using namespace quip;

extern "C" int quip_vecquant_matmul(const float* vec, const int32_t* mat, float* mul, const float* scales,
                                    const float* zeros, int32_t K, int32_t N, int32_t bits, void* stream) {
  QUIP_CHECK_ARG(vec && mat && mul && scales && zeros, "quip_vecquant_matmul: null pointer");
  QUIP_CHECK_ARG(bits >= 2 && bits <= 4, "quip_vecquant_matmul: bits must be 2, 3 or 4 (got %d)", bits);
  QUIP_CHECK_ARG(K > 0 && K % 32 == 0 && N > 0, "quip_vecquant_matmul: K=%d must be a positive multiple of 32, N=%d positive", K, N);
  const int ngroups = K / VQ_GROUP_K;
  const int col_ctas = ceil_div(N, VQ_THREADS);
  int ksplit = ceil_div(4 * num_sms(), col_ctas);             // ~4 CTAs per SM
  if (ksplit > ngroups) ksplit = ngroups;
  int per = ceil_div(ngroups, ksplit);
  per = (per + 3) & ~3;                                       // whole unrolled iterations
  if ((size_t)per * VQ_GROUP_K * sizeof(float) > 40 * 1024) per = (40 * 1024 / (VQ_GROUP_K * sizeof(float))) & ~3;
  ksplit = ceil_div(ngroups, per);
  const size_t smem = (size_t)per * VQ_GROUP_K * sizeof(float);
  dim3 grid((unsigned)col_ctas, (unsigned)ksplit);
  cudaStream_t s = (cudaStream_t)stream;
  const uint32_t* m = reinterpret_cast<const uint32_t*>(mat);
  auto kern = bits == 3 ? vecquant_kernel<3> : (bits == 4 ? vecquant_kernel<4> : vecquant_kernel<2>);
  return launch("vecquant_kernel", kern, grid, VQ_THREADS, smem, s, false, vec, m, mul, scales, zeros, K, N, per);
}
