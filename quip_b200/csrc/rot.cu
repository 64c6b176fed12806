// Incoherence un-projection kernels: the structured U / V "butterfly" multiply of reference
// method.py:46-67, applied to activations at run time instead of being folded into a dense fp16
// weight at quantization time (method.py:195-214).
//
//   gather_kernel      out[m][l] = in[m][idx[l]] * scale[idx[l]] (+ bias[l])   -- p_in gather (V),
//                      p_in scatter written as a gather (U), 1/scaleWH (method.py:147-154), bias
//   rowsum_kernel      xsum[m] = sum_k x[m][k]  (fp32; feeds the asymmetric-grid epilogue term)
//   pass_small_kernel  one block-diagonal pass, block size p <= 64, mma.sync m16n8k16 with the factor
//                      held as B fragments in registers; contiguous or strided blocks
//   pass_big_kernel    one block-diagonal pass, contiguous blocks with p > 64 (e.g. 688 for 11008):
//                      a tiled mma.sync GEMM per block, cp.async double-buffered
//   pass_simple_kernel any p / stride, CUDA cores, fp32: the always-correct fallback and cross-check
//
// Data layout: activations (M, n) fp16 row-major in the side's *layout order* (DESIGN.md); factors
// fp16 [nblk or 1][p][p] row-major with out_i = sum_j f[i][j] in_j.
#include "common.cuh"

namespace quip {

int g_gather_rows = 0;        // quip_config("gather_rows", R)
int g_fewtok = 1;              // quip_config("fewtok", 0): route <= 8 tokens through the many-token kernels
int g_pass_min_tiles = 4;     // quip_config("pass_min_tiles", t): token tiles per CTA in the small-block passes

// ----------------------------------------------------------------------------------------------
// R rows per CTA share one read of the index vector (4 bytes/feature, twice the fp16 row itself)
template <int R>
__global__ void __launch_bounds__(256) gather_kernel(const __half* __restrict__ in, __half* __restrict__ out,
                                                     int64_t M, int n, const int32_t* __restrict__ idx,
                                                     const float* __restrict__ scale,
                                                     const __half* __restrict__ bias) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __half* rows = reinterpret_cast<__half*>(smem_raw);            // [R][n]
  const int64_t m0 = (int64_t)blockIdx.x * R;
  const int nr = (int)((M - m0) < R ? (M - m0) : R);
  const int cpr = n / 8;
  for (int c = threadIdx.x; c < nr * cpr; c += blockDim.x)
    reinterpret_cast<uint4*>(rows)[c] = ldg_nc_v4(in + m0 * n + (int64_t)c * 8);
  __syncthreads();
  for (int c = threadIdx.x; c < cpr; c += blockDim.x) {
    const int l0 = c * 8;
    int src[8];
    float sc[8], bs[8];
    if (idx) {
      const int4 a = *reinterpret_cast<const int4*>(idx + l0), b = *reinterpret_cast<const int4*>(idx + l0 + 4);
      src[0] = a.x; src[1] = a.y; src[2] = a.z; src[3] = a.w; src[4] = b.x; src[5] = b.y; src[6] = b.z; src[7] = b.w;
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) src[i] = l0 + i;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      sc[i] = scale ? scale[src[i]] : 1.f;
      bs[i] = bias ? __half2float(bias[l0 + i]) : 0.f;
    }
    for (int r = 0; r < nr; ++r) {
      __align__(16) __half v[8];
      const __half* row = rows + (size_t)r * n;
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = __float2half_rn(fmaf(__half2float(row[src[i]]), sc[i], bs[i]));
      *reinterpret_cast<uint4*>(out + (m0 + r) * n + l0) = *reinterpret_cast<const uint4*>(v);
    }
  }
}

__global__ void __launch_bounds__(256) rowsum_kernel(const __half* __restrict__ x, float* __restrict__ xsum,
                                                     int64_t M, int K) {
  int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int64_t m = (int64_t)blockIdx.x * 8 + warp;
  if (m >= M) return;
  const uint4* src = reinterpret_cast<const uint4*>(x + m * K);
  float acc = 0.f;
  for (int c = lane; c < K / 8; c += 32) {
    uint4 v = src[c];
    const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float2 f = __half22float2(h[i]);
      acc += f.x + f.y;
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) xsum[m] = acc;
}

// ----------------------------------------------------------------------------------------------
// generic fallback: one CTA per token row
__global__ void __launch_bounds__(256) pass_simple_kernel(const __half* __restrict__ in, __half* __restrict__ out,
                                                          const __half* __restrict__ F, int n, int p, int nblk,
                                                          int strided, int shared) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* v = reinterpret_cast<float*>(smem_raw);
  const int64_t m = blockIdx.x;
  for (int c = threadIdx.x; c < n; c += blockDim.x) v[c] = __half2float(in[m * n + c]);
  __syncthreads();
  for (int o = threadIdx.x; o < n; o += blockDim.x) {
    int b, i;
    if (strided) { b = o % nblk; i = o / nblk; } else { b = o / p; i = o % p; }
    const __half* f = F + ((int64_t)(shared ? 0 : b) * p + i) * p;
    float acc = 0.f;
    for (int j = 0; j < p; ++j) {
      int pos = strided ? (j * nblk + b) : (b * p + j);
      acc = fmaf(__half2float(f[j]), v[pos], acc);
    }
    out[m * n + o] = __float2half_rn(acc);
  }
}

// ----------------------------------------------------------------------------------------------
// small blocks (p <= 64): one warp owns BPW blocks, its factors live in registers as B fragments,
// the CTA streams 16-token tiles of its GB = 8*BPW blocks through shared memory.
template <int P>
struct SmallCfg {
  static constexpr int BPW = 64 / P >= 1 ? 64 / P : 1;   // blocks per warp (P=48 -> 1)
  static constexpr int GB = 8 * BPW;                     // blocks per CTA
  static constexpr int LD = P + 8;                       // smem row stride (halves)
  static constexpr int KS = P / 16, NT = P / 8;
  static constexpr int TILE = GB * 16 * LD;              // halves
};

template <int P>
__global__ void __launch_bounds__(256)
pass_small_kernel(const __half* __restrict__ in, __half* __restrict__ out, const __half* __restrict__ F,
                  int64_t M, int n, int p, int nblk, int strided, int shared, int tok_chunk, int vec) {
  using C = SmallCfg<P>;
  __shared__ __align__(16) __half T[C::TILE];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int b0 = blockIdx.x * C::GB;          // first block of this CTA
  const int64_t m_begin = (int64_t)blockIdx.y * tok_chunk;
  const int64_t m_end = m_begin + tok_chunk < M ? m_begin + tok_chunk : M;

  // factor -> B fragments.  b0: (k = 2t,2t+1 ; n = g), b1: (k = 2t+8,2t+9 ; n = g); k = j, n = i
  uint32_t bf[C::BPW][C::KS][C::NT][2];
#pragma unroll
  for (int bb = 0; bb < C::BPW; ++bb) {
    int blk = b0 + warp * C::BPW + bb;
    const __half* f = F + (int64_t)(shared ? 0 : (blk < nblk ? blk : 0)) * p * p;
#pragma unroll
    for (int ks = 0; ks < C::KS; ++ks)
#pragma unroll
      for (int nt = 0; nt < C::NT; ++nt)
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          int i = nt * 8 + g, j = ks * 16 + 2 * t + 8 * r;
          __half lo = __float2half(0.f), hi = lo;
          if (blk < nblk && i < p) {
            if (j < p) lo = f[(int64_t)i * p + j];
            if (j + 1 < p) hi = f[(int64_t)i * p + j + 1];
          }
          bf[bb][ks][nt][r] = (uint32_t)__half_as_ushort(lo) | ((uint32_t)__half_as_ushort(hi) << 16);
        }
  }

  const int span = C::GB * p;                  // contiguous case: columns per token in this CTA's tile
  for (int64_t m0 = m_begin; m0 < m_end; m0 += 16) {
    // ---- global -> shared, T[blk_local][tok][j], zero padded ----
    if (vec) {
      if (!strided) {
        const int cpt = span / 8;             // 16-byte chunks per token
        for (int c = tid; c < 16 * cpt; c += 256) {
          int tok = c / cpt, q = c % cpt;
          int col = b0 * p + q * 8;
          int bl = (q * 8) / p, j = (q * 8) % p;
          uint4 v = make_uint4(0, 0, 0, 0);
          if (m0 + tok < m_end && col < n) v = *reinterpret_cast<const uint4*>(in + (m0 + tok) * n + col);
          *reinterpret_cast<uint4*>(&T[(bl * 16 + tok) * C::LD + j]) = v;
        }
      } else {
        constexpr int CG = C::GB / 8;         // chunks of 8 blocks per (tok, j)
        for (int c = tid; c < 16 * p * CG; c += 256) {
          int c8 = c % CG, j = (c / CG) % p, tok = c / (CG * p);
          int blk = b0 + c8 * 8;
          uint4 v = make_uint4(0, 0, 0, 0);
          if (m0 + tok < m_end && blk < nblk)
            v = *reinterpret_cast<const uint4*>(in + (m0 + tok) * n + (int64_t)j * nblk + blk);
          const __half* h = reinterpret_cast<const __half*>(&v);
#pragma unroll
          for (int i = 0; i < 8; ++i) T[((c8 * 8 + i) * 16 + tok) * C::LD + j] = h[i];
        }
      }
    } else {
      for (int c = tid; c < 16 * C::GB * p; c += 256) {
        int j, bl, tok;
        if (!strided) { j = c % p; bl = (c / p) % C::GB; tok = c / (p * C::GB); }
        else { bl = c % C::GB; j = (c / C::GB) % p; tok = c / (C::GB * p); }
        int blk = b0 + bl;
        __half v = __float2half(0.f);
        if (m0 + tok < m_end && blk < nblk)
          v = in[(m0 + tok) * n + (strided ? (int64_t)j * nblk + blk : (int64_t)blk * p + j)];
        T[(bl * 16 + tok) * C::LD + j] = v;
      }
    }
    if (P != p) {                               // zero the padding columns j in [p, P)
      const int padw = P - p;
      for (int c = tid; c < C::GB * 16 * padw; c += 256)
        T[(c / padw) * C::LD + p + c % padw] = __float2half(0.f);
    }
    __syncthreads();

    // ---- per warp: D[tok][i] = sum_j A[tok][j] F[i][j], written back in place ----
#pragma unroll
    for (int bb = 0; bb < C::BPW; ++bb) {
      __half* tile = &T[((warp * C::BPW + bb) * 16) * C::LD];
      uint32_t a[C::KS][4];
#pragma unroll
      for (int ks = 0; ks < C::KS; ++ks) {
        a[ks][0] = *reinterpret_cast<const uint32_t*>(&tile[g * C::LD + ks * 16 + 2 * t]);
        a[ks][1] = *reinterpret_cast<const uint32_t*>(&tile[(g + 8) * C::LD + ks * 16 + 2 * t]);
        a[ks][2] = *reinterpret_cast<const uint32_t*>(&tile[g * C::LD + ks * 16 + 2 * t + 8]);
        a[ks][3] = *reinterpret_cast<const uint32_t*>(&tile[(g + 8) * C::LD + ks * 16 + 2 * t + 8]);
      }
      __syncwarp();
#pragma unroll
      for (int nt = 0; nt < C::NT; ++nt) {
        float d[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int ks = 0; ks < C::KS; ++ks) mma16816(d, a[ks], bf[bb][ks][nt]);
        *reinterpret_cast<__half2*>(&tile[g * C::LD + nt * 8 + 2 * t]) = __floats2half2_rn(d[0], d[1]);
        *reinterpret_cast<__half2*>(&tile[(g + 8) * C::LD + nt * 8 + 2 * t]) = __floats2half2_rn(d[2], d[3]);
      }
    }
    __syncthreads();

    // ---- shared -> global (same index map as the load) ----
    if (vec) {
      if (!strided) {
        const int cpt = span / 8;
        for (int c = tid; c < 16 * cpt; c += 256) {
          int tok = c / cpt, q = c % cpt;
          int col = b0 * p + q * 8;
          int bl = (q * 8) / p, j = (q * 8) % p;
          if (m0 + tok < m_end && col < n)
            *reinterpret_cast<uint4*>(out + (m0 + tok) * n + col) =
                *reinterpret_cast<const uint4*>(&T[(bl * 16 + tok) * C::LD + j]);
        }
      } else {
        constexpr int CG = C::GB / 8;
        for (int c = tid; c < 16 * p * CG; c += 256) {
          int c8 = c % CG, j = (c / CG) % p, tok = c / (CG * p);
          int blk = b0 + c8 * 8;
          if (m0 + tok < m_end && blk < nblk) {
            __align__(16) __half h[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) h[i] = T[((c8 * 8 + i) * 16 + tok) * C::LD + j];
            *reinterpret_cast<uint4*>(out + (m0 + tok) * n + (int64_t)j * nblk + blk) =
                *reinterpret_cast<const uint4*>(h);
          }
        }
      }
    } else {
      for (int c = tid; c < 16 * C::GB * p; c += 256) {
        int j, bl, tok;
        if (!strided) { j = c % p; bl = (c / p) % C::GB; tok = c / (p * C::GB); }
        else { bl = c % C::GB; j = (c / C::GB) % p; tok = c / (C::GB * p); }
        int blk = b0 + bl;
        if (m0 + tok < m_end && blk < nblk)
          out[(m0 + tok) * n + (strided ? (int64_t)j * nblk + blk : (int64_t)blk * p + j)] =
              T[(bl * 16 + tok) * C::LD + j];
      }
    }
    __syncthreads();
  }
}

// ----------------------------------------------------------------------------------------------
// big contiguous blocks (p > 64, p % 8 == 0): per block a GEMM  D[tok][i] = sum_j A[tok][j] F[i][j]
// CTA tile 128 tok x 128 i, BK = 32, 8 warps as 2 (tok) x 4 (i), each warp 64 x 32.
constexpr int BIG_BM = 128, BIG_BN = 128, BIG_BK = 32, BIG_LD = BIG_BK + 8, BIG_STAGES = 3;

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, bool valid) {
  uint32_t s = smem_u32(smem);
  int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gmem), "r"(sz));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* p) {
  uint32_t s = smem_u32(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(s));
}

__global__ void __launch_bounds__(256)
pass_big_kernel(const __half* __restrict__ in, __half* __restrict__ out, const __half* __restrict__ F,
                int64_t M, int n, int p, int shared) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __half* As = reinterpret_cast<__half*>(smem_raw);                     // [STAGES][BM][LD]
  __half* Bs = As + BIG_STAGES * BIG_BM * BIG_LD;                       // [STAGES][BN][LD]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wm = warp >> 2, wn = warp & 3;                              // 2 x 4
  const int blk = blockIdx.z;
  const int64_t m0 = (int64_t)blockIdx.y * BIG_BM;
  const int i0 = blockIdx.x * BIG_BN;
  const __half* Ablk = in + (int64_t)blk * p;                           // + m*n + j
  const __half* Fblk = F + (int64_t)(shared ? 0 : blk) * p * p;         // + i*p + j
  const int nk = (p + BIG_BK - 1) / BIG_BK;

  auto load_stage = [&](int stage, int kc) {
    const int j0 = kc * BIG_BK;
    // A: 128 rows x 4 chunks; B: 128 rows x 4 chunks -> 1024 chunks, 4 per thread
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      int c = tid + r * 256;
      int row = c >> 2, q = c & 3;
      bool va = (m0 + row < M) && (j0 + q * 8 < p);
      const __half* ga = Ablk + (va ? ((m0 + row) * n + j0 + q * 8) : 0);
      cp_async16(&As[(stage * BIG_BM + row) * BIG_LD + q * 8], ga, va);
      bool vb = (i0 + row < p) && (j0 + q * 8 < p);
      const __half* gb = Fblk + (vb ? ((int64_t)(i0 + row) * p + j0 + q * 8) : 0);
      cp_async16(&Bs[(stage * BIG_BN + row) * BIG_LD + q * 8], gb, vb);
    }
  };

  float acc[4][4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[a][b][c] = 0.f;

#pragma unroll
  for (int s = 0; s < BIG_STAGES - 1; ++s) {
    if (s < nk) load_stage(s, s);
    cp_async_commit();
  }
  for (int kc = 0; kc < nk; ++kc) {
    cp_async_wait<BIG_STAGES - 2>();
    __syncthreads();
    {
      int nxt = kc + BIG_STAGES - 1;
      if (nxt < nk) load_stage(nxt % BIG_STAGES, nxt);
      cp_async_commit();
    }
    const __half* A = &As[(kc % BIG_STAGES) * BIG_BM * BIG_LD];
    const __half* B = &Bs[(kc % BIG_STAGES) * BIG_BN * BIG_LD];
#pragma unroll
    for (int ks = 0; ks < BIG_BK / 16; ++ks) {
      uint32_t af[4][4], bfr[4][2];
#pragma unroll
      for (int mt = 0; mt < 4; ++mt) {
        // x4: matrices (rows 0-7,k0-7) (rows 8-15,k0-7) (rows 0-7,k8-15) (rows 8-15,k8-15) = a0..a3
        int row = wm * 64 + mt * 16 + (lane & 15);
        int col = ks * 16 + (lane >> 4) * 8;
        ldmatrix_x4(af[mt], &A[row * BIG_LD + col]);
      }
#pragma unroll
      for (int np = 0; np < 2; ++np) {
        // two n-tiles per x4: (n 0-7,k0-7) (n 0-7,k8-15) (n 8-15,k0-7) (n 8-15,k8-15)
        uint32_t r[4];
        int row = wn * 32 + np * 16 + (lane & 7) + ((lane >> 4) << 3);
        int col = ks * 16 + ((lane >> 3) & 1) * 8;
        ldmatrix_x4(r, &B[row * BIG_LD + col]);
        bfr[np * 2][0] = r[0]; bfr[np * 2][1] = r[1];
        bfr[np * 2 + 1][0] = r[2]; bfr[np * 2 + 1][1] = r[3];
      }
#pragma unroll
      for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) mma16816(acc[mt][nt], af[mt], bfr[nt]);
    }
  }
  cp_async_wait<0>();

  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      int i = i0 + wn * 32 + nt * 8 + 2 * t;
      if (i >= p) continue;                    // p even -> i+1 < p too
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        int64_t m = m0 + wm * 64 + mt * 16 + g + 8 * h;
        if (m < M)
          *reinterpret_cast<__half2*>(out + m * n + (int64_t)blk * p + i) =
              __floats2half2_rn(acc[mt][nt][2 * h], acc[mt][nt][2 * h + 1]);
      }
    }
}

}  // namespace quip

using namespace quip;

template <int R>
static int launch_gather(const __half* in, __half* out, int64_t M, int n, const int32_t* idx, const float* scale,
                         const __half* bias, cudaStream_t s) {
  return launch("gather_kernel", gather_kernel<R>, ceil_div(M, R), 256, (size_t)R * n * sizeof(__half), s, false, in, out,
                M, n, idx, scale, bias);
}

extern "C" int quip_gather(const void* in, void* out, int64_t M, int32_t n, const int32_t* idx,
                           const float* scale, const void* bias, void* stream) {
  QUIP_CHECK_ARG(in && out && M > 0 && n > 0 && n % 8 == 0, "gather: bad arguments (M=%lld n=%d)", (long long)M, n);
  QUIP_CHECK_ARG(in != out, "gather cannot run in place");
  QUIP_CHECK_ARG((size_t)n * sizeof(__half) <= 200 * 1024, "gather: n=%d too large", n);
  cudaStream_t s = (cudaStream_t)stream;
  const __half* i = (const __half*)in;
  __half* o = (__half*)out;
  const __half* b = (const __half*)bias;
  if (g_fewtok && M <= g_fewtok_max_m) return gather_fewtok(i, o, M, n, idx, scale, b, s);
  // rows per CTA: share the index vector across rows, but keep several waves of CTAs so that one CTA's load
  // phase overlaps another's permute phase
  const size_t row = (size_t)n * sizeof(__half);
  int R = g_gather_rows > 0 ? g_gather_rows : 4;
  while (R > 1 && (M < (int64_t)R * 592 || R * row > 96 * 1024)) R >>= 1;
  if (R >= 8) return launch_gather<8>(i, o, M, n, idx, scale, b, s);
  if (R >= 4) return launch_gather<4>(i, o, M, n, idx, scale, b, s);
  if (R >= 2) return launch_gather<2>(i, o, M, n, idx, scale, b, s);
  return launch_gather<1>(i, o, M, n, idx, scale, b, s);
}

extern "C" int quip_rowsum(const void* x, float* xsum, int64_t M, int32_t K, void* stream) {
  QUIP_CHECK_ARG(x && xsum && M > 0 && K > 0 && K % 8 == 0, "rowsum: bad arguments");
  return launch("rowsum_kernel", rowsum_kernel, ceil_div(M, 8), 256, 0, (cudaStream_t)stream, false, (const __half*)x, xsum,
                M, K);
}

template <int P>
static int launch_small(const QuipPass* ps, const __half* in, __half* out, int64_t M, int n, cudaStream_t s) {
  using C = SmallCfg<P>;
  int groups = ceil_div(ps->nblk, C::GB);
  // aim for >= ~2 waves of CTAs while keeping the register-resident factors amortised over many tiles
  int tok_chunk = 512;
  while (tok_chunk > 16 && (int64_t)groups * ceil_div(M, tok_chunk) < 296) tok_chunk >>= 1;
  int vec = ps->strided ? (ps->nblk % 8 == 0) : (ps->p % 8 == 0 && n % 8 == 0);
  dim3 grid(groups, ceil_div(M, tok_chunk));
  return launch("pass_small_kernel", pass_small_kernel<P>, grid, 256, 0, s, false, in, out, (const __half*)ps->factors, M, n,
                ps->p, ps->nblk, ps->strided, ps->shared, tok_chunk, vec);
}

extern "C" int quip_rot_pass(const QuipPass* ps, const void* in_, void* out_, int64_t M, int32_t n, int impl,
                             void* stream) {
  QUIP_CHECK_ARG(ps && in_ && out_ && ps->factors, "rot_pass: null pointer");
  QUIP_CHECK_ARG(M > 0 && n > 0 && ps->p > 0 && ps->nblk > 0 && (int64_t)ps->p * ps->nblk == n,
                 "rot_pass: p*nblk != n (p=%d nblk=%d n=%d)", ps->p, ps->nblk, n);
  QUIP_CHECK_ARG(in_ != out_, "rot_pass cannot run in place");
  cudaStream_t s = (cudaStream_t)stream;
  const __half* in = (const __half*)in_;
  __half* out = (__half*)out_;
  const int p = ps->p;
  if (impl == 0 && g_fewtok && pass_fewtok_ok(ps, M, n))
    return pass_fewtok(ps, in, out, M, n, nullptr, nullptr, nullptr, nullptr, s);
  bool small_ok = p <= 64;
  bool big_ok = p > 64 && !ps->strided && p % 8 == 0 && n % 8 == 0;
  if (impl != 1 && small_ok) {
    bool handled = false;
    if (int e = launch_small_fast(ps, in, out, M, n, s, &handled)) return e;
    if (handled) return QUIP_OK;
    if (p <= 16) return launch_small<16>(ps, in, out, M, n, s);
    if (p <= 32) return launch_small<32>(ps, in, out, M, n, s);
    if (p <= 48) return launch_small<48>(ps, in, out, M, n, s);
    return launch_small<64>(ps, in, out, M, n, s);
  }
  if (impl != 1 && impl != 3 && big_ok && M > 32 && ((((uintptr_t)in | (uintptr_t)out | (uintptr_t)ps->factors) & 15) == 0))
    return pass_big_tc(ps, in, out, M, n, s);      // tcgen05: the 688x688 blocks of an 11008 side are real GEMMs
  if (impl != 1 && big_ok) {
    const size_t smem = (size_t)BIG_STAGES * (BIG_BM + BIG_BN) * BIG_LD * sizeof(__half);
    const dim3 grid(ceil_div(p, BIG_BN), ceil_div(M, BIG_BM), ps->nblk);
    return launch("pass_big_kernel", pass_big_kernel, grid, 256, smem, s, false, in, out, (const __half*)ps->factors, M, n, p,
                  ps->shared);
  }
  if (impl == 2) {
    set_error("rot_pass: no tensor-core kernel for p=%d strided=%d", p, ps->strided);
    return QUIP_ERR_UNSUPPORTED;
  }
  size_t smem = (size_t)n * sizeof(float);
  QUIP_CHECK_ARG(smem <= 200 * 1024, "rot_pass: n=%d too large for the generic kernel", n);
  return launch("pass_simple_kernel", pass_simple_kernel, (unsigned)M, 256, smem, s, false, in, out, (const __half*)ps->factors,
                n, p, ps->nblk, ps->strided, ps->shared);
}
