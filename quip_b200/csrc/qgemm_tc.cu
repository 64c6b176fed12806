// Packed-integer x fp16 GEMM on the 5th-generation tensor cores (tcgen05 + TMEM), for many tokens
// (the reference's eval loop calls every Linear with M = 2048: opt.py:262-264, llama.py:226-227).
//
//   D[n][m] (TMEM, fp32) = sum_k A[n][k] * B[m][k]
//     A = packed weights, 128 output rows per tile, expanded to fp16 d=(c-cbar)/2^bits by the
//         producer warps and written straight into the 128B-swizzled K-major operand layout
//         (generic-proxy st.shared + fence.proxy.async), never touching HBM as fp16;
//     B = activations x2 (M,K) fp16, BN tokens per tile, staged by TMA (cp.async.bulk.tensor, 128B
//         swizzle, out-of-bounds rows zero-filled so ragged M needs no special case);
//   epilogue: z[m][n] = P_n * D + R_n * xsum[m] (+ bias_n) -> fp16, straight from tcgen05.ld registers.
//
// Warp roles (448 threads, one persistent CTA per SM, static tile schedule):
//   warp 0      TMA producer            warp 1      TMEM alloc + MMA issuer (one lane)
//   warps 2-5   epilogue (TMEM lane quarter = warp % 4)
//   warps 6-13  weight producers (2 groups of 4 alternating k super-blocks): 128-bit loads of packed
//               words -> registers -> fp16 -> smem
// Pipelines: smem ring full[s]/empty[s] (TMA + 4 producer warps -> MMA -> tcgen05.commit), and a
// double-buffered TMEM accumulator tmem_full[a]/tmem_empty[a] (MMA -> epilogue).
#include "tc_common.cuh"

namespace quip {

template <int BN>
struct TcCfg {
  static constexpr int A_BYTES = TC_BM * TC_BK * 2;            // 16 KB
  static constexpr int B_BYTES = BN * TC_BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = (200 * 1024) / STAGE_BYTES;    // 256 -> 4, 128 -> 6
  static constexpr int TMEM_COLS = 2 * BN;                     // double-buffered accumulator
  static constexpr size_t SMEM = (size_t)STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/ + 8192 /*epilogue*/;
};

// DENSE = false: A is the packed matrix (N rows, K columns), expanded by the producer warps.
// DENSE = true : block-diagonal pass with big blocks -- `nblk` independent GEMMs out_b = in_b . F_b^T, A = fp16
//                factor F_b (N = K = p) fetched by TMA (3-D map, rows/cols beyond p zero-filled), B = the
//                block's p contiguous activation columns, output written to the same columns.
template <int BITS, int BN, bool DENSE>
__global__ void __launch_bounds__(TC_THREADS, 1)
qgemm_tc_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_a,
                const uint32_t* __restrict__ q, const float* __restrict__ scales, const float* __restrict__ zeros,
                const __half* __restrict__ bias, const float* __restrict__ xsum, __half* __restrict__ z, int M, int K,
                int N, int symmetric, int nblk, int shared_factor) {
  using C = TcCfg<BN>;
  extern __shared__ unsigned char smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  unsigned char* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_gen + (size_t)C::STAGES * C::STAGE_BYTES);
  uint64_t* full = bars;                       // [STAGES]
  uint64_t* empty = bars + C::STAGES;          // [STAGES]
  uint64_t* tmem_full = empty + C::STAGES;     // [2]
  uint64_t* tmem_empty = tmem_full + 2;        // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  __half* epi_stage = reinterpret_cast<__half*>(smem_gen + (size_t)C::STAGES * C::STAGE_BYTES + 256);   // 4 x 2 KB

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // packed GEMM: 128 output rows (MMA M) x BN tokens (MMA N).  DENSE pass: 128 TOKENS (MMA M) x BN factor rows
  // (MMA N), so every epilogue thread owns one token row and stores 64 contiguous bytes per 32 columns.
  const int tiles_n = DENSE ? (N + BN - 1) / BN : (N + TC_BM - 1) / TC_BM;
  const int tiles_m = DENSE ? (M + TC_BM - 1) / TC_BM : (M + BN - 1) / BN;
  const int per_blk = tiles_n * tiles_m;
  const int num_tiles = per_blk * nblk;
  const int KB = (K + TC_BK - 1) / TC_BK;
  const int KSB = K >> 7;
  const int64_t ldz = (int64_t)N * nblk;       // output row pitch (== N for the packed GEMM)

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_x) : "memory");
    if (DENSE) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_a) : "memory");
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(&full[s], DENSE ? 1 : 1 + 4);  // TMA producer (+ 4 weight-producer warps)
      mbar_init(&empty[s], 1);                 // one tcgen05.commit
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], 4);            // 4 epilogue warps
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)C::TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================= TMA producer: activation tiles =================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int blk = tile / per_blk, rr = tile % per_blk;
        const int m0 = (rr / tiles_n) * (DENSE ? TC_BM : BN), n0 = (rr % tiles_n) * (DENSE ? BN : TC_BM);
        for (int kb = 0; kb < KB; ++kb) {
          mbar_wait(&empty[s], ph ^ 1u);
          mbar_arrive_expect_tx(&full[s], DENSE ? C::STAGE_BYTES : C::B_BYTES);
          unsigned char* stage = smem_gen + (size_t)s * C::STAGE_BYTES;
          if (DENSE) {
            tma_load_2d(stage, &tmap_x, &full[s], blk * K + kb * TC_BK, m0);                     // A: 128 tokens
            tma_load_3d(stage + C::A_BYTES, &tmap_a, &full[s], kb * TC_BK, n0, shared_factor ? 0 : blk);   // B: BN factor rows
          } else {
            tma_load_2d(stage + C::A_BYTES, &tmap_x, &full[s], kb * TC_BK, m0);
          }
          if (++s == C::STAGES) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    const uint32_t idesc = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
    int s = 0;
    uint32_t ph = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int as = it & 1;
      const uint32_t aph = (uint32_t)(it >> 1) & 1u;
      mbar_wait(&tmem_empty[as], aph ^ 1u);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + (uint32_t)(as * BN);
      for (int kb = 0; kb < KB; ++kb) {
        mbar_wait(&full[s], ph);
        tc_fence_after();
        if (lane == 0) {
          const uint32_t a_addr = smem_base + (uint32_t)(s * C::STAGE_BYTES);
          const uint64_t adesc = make_sw128_desc(a_addr);
          const uint64_t bdesc = make_sw128_desc(a_addr + C::A_BYTES);
#pragma unroll
          for (int k = 0; k < TC_BK / 16; ++k)     // +32 bytes along K inside the swizzle atom = +2 encoded
            umma_f16_ss(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) ? 1u : 0u);
          umma_commit(&empty[s]);                  // frees the stage once these MMAs have read it
          if (kb == KB - 1) umma_commit(&tmem_full[as]);
        }
        __syncwarp();
        if (++s == C::STAGES) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp < 6) {
    // ================= epilogue: TMEM -> registers -> z =================
    const int quarter = warp & 3;
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int as = it & 1;
      const uint32_t aph = (uint32_t)(it >> 1) & 1u;
      const int blk = tile / per_blk, rr = tile % per_blk;
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(as * BN);
      if constexpr (DENSE) {
        const int m = (rr / tiles_n) * TC_BM + quarter * 32 + lane;          // this thread's token
        const int i0 = (rr % tiles_n) * BN;                                  // first factor row of the tile
        __half* zrow = z + (int64_t)m * ldz + (int64_t)blk * N;
        mbar_wait(&tmem_full[as], aph);
        tc_fence_after();
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 32) {
          uint32_t r[32];
          tmem_ld32(taddr + (uint32_t)c0, r);
          tmem_ld_wait();
          const int i = i0 + c0;
          if (m < M && i < N) {
            if (i + 32 <= N) {
#pragma unroll
              for (int v4 = 0; v4 < 4; ++v4) {
                uint4 o;
                uint32_t* ow = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
                for (int h = 0; h < 4; ++h) {
                  __half2 hv = __floats2half2_rn(__uint_as_float(r[8 * v4 + 2 * h]), __uint_as_float(r[8 * v4 + 2 * h + 1]));
                  ow[h] = *reinterpret_cast<uint32_t*>(&hv);
                }
                *reinterpret_cast<uint4*>(zrow + i + 8 * v4) = o;
              }
            } else {
#pragma unroll
              for (int c = 0; c < 32; ++c)
                if (i + c < N) zrow[i + c] = __float2half_rn(__uint_as_float(r[c]));
            }
          }
        }
      } else {
        const int n = (rr % tiles_n) * TC_BM + quarter * 32 + lane;
        const int m0 = (rr / tiles_n) * BN;
        float Pn = 1.f, Rn = 0.f, bn = 0.f;
        if (n < N) {
          float sc = scales[n];
          Pn = sc * (float)(1 << BITS);
          if (!symmetric) Rn = sc * (0.5f * (float)((1 << BITS) - 1)) - zeros[n];
          if (bias) bn = __half2float(bias[n]);
        }
        __half* stage = epi_stage + (warp - 2) * EPI_STAGE_HALVES;
        const int n_warp = (rr % tiles_n) * TC_BM + quarter * 32;
        mbar_wait(&tmem_full[as], aph);
        tc_fence_after();
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 32) {
          uint32_t r[32];
          tmem_ld32(taddr + (uint32_t)c0, r);
          tmem_ld_wait();
          float v[32];
#pragma unroll
          for (int c = 0; c < 32; ++c) {
            v[c] = Pn * __uint_as_float(r[c]) + bn;
            if (!symmetric) {
              const int m = m0 + c0 + c;
              v[c] += Rn * (m < M ? __ldg(&xsum[m]) : 0.f);
            }
          }
          epilogue_store_chunk(stage, v, z, ldz, m0 + c0, M, n_warp, N, lane);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[as]);
    }
  } else if (!DENSE) {
    // ================= weight producers: packed words -> fp16 operand tile =================
    const int pw = (warp - 6) & 3, grp = (warp - 6) >> 2;
    weight_producer_loop<BITS, C::STAGES, C::STAGE_BYTES>(
        pw, grp, lane, q, KSB, N, empty, smem_base, (int)blockIdx.x, (int)gridDim.x, num_tiles,
        [&](int tile) { return ((tile % per_blk) % tiles_n) * (TC_BM / 16); },
        [&](int s) { mbar_arrive(&full[s]); });
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)C::TMEM_COLS)
                 : "memory");
  }
}

// ---- host side ---------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (PFN_encodeTiled)p;
  }
  return fn;
}

// activations (rows, cols) fp16 row-major -> 2-D map, box {64 cols, box_rows}, 128B swizzle, zero OOB fill
int make_act_map(CUtensorMap* tmap, const void* x, int64_t rows, int64_t cols, int box_rows) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return QUIP_ERR_CUDA;
  }
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * sizeof(__half)};
  cuuint32_t box[2] = {(cuuint32_t)TC_BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, (void*)x, dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (ptr=%p rows=%lld cols=%lld)", (int)r, x,
              (long long)rows, (long long)cols);
    return QUIP_ERR_CUDA;
  }
  return QUIP_OK;
}

template <int BITS, int BN>
static int launch_tc(const QuipLinearDesc* d, const __half* x, const float* xsum, const __half* bias, __half* z,
                     int M, cudaStream_t s) {
  using C = TcCfg<BN>;
  CUtensorMap tmap;
  if (int e = make_act_map(&tmap, x, M, d->K, BN)) return e;
  const int grid = std::min(ceil_div(d->N, TC_BM) * ceil_div(M, BN), num_sms());
  return launch("qgemm_tc_kernel", qgemm_tc_kernel<BITS, BN, false>, grid, TC_THREADS, C::SMEM, s, false, tmap, tmap,
                reinterpret_cast<const uint32_t*>(d->qweight), d->scales, d->zeros, bias, xsum, z, M, d->K, d->N,
                (d->flags & QUIP_FLAG_SYMMETRIC) ? 1 : 0, 1, 0);
}

// block-diagonal pass with big contiguous blocks on the tensor cores (see DENSE in the kernel)
template <int BN>
static int launch_tc_dense(const QuipPass* ps, const __half* in, __half* out, int M, int n, cudaStream_t s) {
  using C = TcCfg<BN>;
  PFN_encodeTiled enc = get_encode();
  CUtensorMap tmx, tma;
  if (int e = make_act_map(&tmx, in, M, n, TC_BM)) return e;       // 128 tokens per tile (MMA M)
  const int p = ps->p;
  cuuint64_t dims[3] = {(cuuint64_t)p, (cuuint64_t)p, (cuuint64_t)(ps->shared ? 1 : ps->nblk)};
  cuuint64_t strides[2] = {(cuuint64_t)p * sizeof(__half), (cuuint64_t)p * p * sizeof(__half)};
  cuuint32_t box[3] = {(cuuint32_t)TC_BK, (cuuint32_t)BN, 1};       // BN factor rows per tile (MMA N)
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(&tma, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, (void*)ps->factors, dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (factors) failed with CUresult %d (p=%d nblk=%d)", (int)r, p, ps->nblk);
    return QUIP_ERR_CUDA;
  }
  const int grid = std::min(ceil_div(p, BN) * ceil_div(M, TC_BM) * ps->nblk, num_sms());
  return launch("qgemm_tc_kernel<dense>", qgemm_tc_kernel<2, BN, true>, grid, TC_THREADS, C::SMEM, s, false, tmx, tma,
                nullptr, nullptr, nullptr, nullptr, nullptr, out, M, p, p, 1, ps->nblk, ps->shared ? 1 : 0);
}

int pass_big_tc(const QuipPass* ps, const __half* in, __half* out, int64_t M, int n, cudaStream_t s) {
  QUIP_CHECK_ARG(!ps->strided && ps->p % 8 == 0 && n % 8 == 0, "tcgen05 pass needs contiguous blocks, p %% 8 == 0");
  QUIP_CHECK_ARG((((uintptr_t)in | (uintptr_t)out | (uintptr_t)ps->factors) & 15) == 0, "tcgen05 pass: unaligned pointer");
  return ps->p > 128 ? launch_tc_dense<256>(ps, in, out, (int)M, n, s) : launch_tc_dense<128>(ps, in, out, (int)M, n, s);
}

int qgemm_tc(const QuipLinearDesc* d, const __half* x, const float* xsum, const __half* bias, __half* z, int M,
             cudaStream_t s) {
  QUIP_CHECK_ARG(((uintptr_t)x & 15) == 0, "tcgen05 path needs 16-byte aligned activations");
  const bool wide = M > 128;
#define QUIP_TC(B)                                                            \
  if (d->bits == B)                                                           \
    return wide ? launch_tc<B, 256>(d, x, xsum, bias, z, M, s) : launch_tc<B, 128>(d, x, xsum, bias, z, M, s);
  QUIP_TC(2) QUIP_TC(3) QUIP_TC(4)
#undef QUIP_TC
  set_error("tcgen05 kernel: unsupported bits=%d", d->bits);
  return QUIP_ERR_UNSUPPORTED;
}

}  // namespace quip
