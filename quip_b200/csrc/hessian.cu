// Calibration Hessian H += X^T X on the tensor cores (SURVEY section 8(f) rank 2).
//
// Reference: QuantMethod.add_batch (method.py:98-120) casts the (tokens, features) activations of a Linear to float64 and
// adds inp @ inp.T to a float64 H; post_batch (method.py:122-123) divides by the batch count and rounds to float32.  A
// float64 GEMM per batch per Linear is the bulk of calibration time.  The activations are fp16, so every product
// x[t][i] * x[t][j] is EXACT in float32 (11 + 11 significant bits); only the sum needs care.  This kernel therefore
//   * multiplies on the fp16 tensor cores with float32 accumulation (mma.sync.m16n8k16) over chunks of HS_CHUNK tokens
//     -- at most 256 exact products per accumulator, relative error <= 256 * 2^-24 of the chunk's sum, and
//   * carries the running total in the caller's float64 H: each CTA owns one 128 x 128 tile of the UPPER block triangle
//     (tiles ti <= tj; the caller mirrors once at the end), so the read-modify-write needs no atomics.
// The float32 H the reference finally keeps (post_batch) has 2^-24 relative precision itself; measured against the float64
// GEMM the result agrees to ~1e-7 (tests/test_gpu_quantize.py).
//
// Operands: X (T, K) fp16 row-major is staged in shared memory as it lies in HBM ([token][feature], rows padded to 272
// bytes so that the eight row addresses of an ldmatrix hit distinct banks); both MMA operands want two consecutive TOKENS
// per register, i.e. the transposed tile, which ldmatrix.trans delivers.
#include "common.cuh"

namespace quip {

namespace {

constexpr int HS_TILE = 128;            // features per tile side
constexpr int HS_TOK = 32;              // tokens per pipeline stage
constexpr int HS_CHUNK = 256;           // tokens summed in float32 before the float64 carry
constexpr int HS_LD = HS_TILE + 8;      // padded row, in halves
constexpr int HS_THREADS = 256;         // 8 warps: 2 (i) x 4 (j), warp tile 64 x 32
constexpr int HS_STAGES = 3;

__device__ __forceinline__ void cp_async16(void* smem, const void* g, bool valid) {
  const int sz = valid ? 16 : 0;        // src-size 0: zero fill (tokens / features beyond the matrix)
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem)), "l"(g), "r"(sz) : "memory");
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t (&r)[4], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(smem_u32(p)));
}

// grid: one CTA per tile (ti <= tj) of the upper block triangle; H (K, K) float64 row-major, lower block triangle untouched
__global__ void __launch_bounds__(HS_THREADS)
hessian_syrk_kernel(const __half* __restrict__ X, double* __restrict__ H, int T, int K, int ntile) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __half* sI = reinterpret_cast<__half*>(smem_raw);                         // [STAGES][HS_TOK][HS_LD]
  __half* sJ = sI + HS_STAGES * HS_TOK * HS_LD;
  // linear index -> (ti, tj), ti <= tj
  int ti = 0, rem = blockIdx.x;
  while (rem >= ntile - ti) { rem -= ntile - ti; ++ti; }
  const int tj = ti + rem;
  const int i0 = ti * HS_TILE, j0 = tj * HS_TILE;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wi = warp >> 2, wj = warp & 3;                                   // warp tile: rows wi*64.., cols wj*32..
  const int g = lane >> 2, t4 = lane & 3;

  auto load_stage = [&](int stage, int tok0) {
    // 2 tiles x HS_TOK rows x 16 chunks of 16 bytes = 1024 chunks, 4 per thread
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int idx = tid + c * HS_THREADS;
      const int which = idx >> 9, r = (idx >> 4) & (HS_TOK - 1), ch = idx & 15;
      const int f0 = (which ? j0 : i0) + ch * 8, tok = tok0 + r;
      const bool ok = tok < T && f0 < K;                                     // K % 8 == 0: a chunk is inside or outside
      __half* dst = (which ? sJ : sI) + (stage * HS_TOK + r) * HS_LD + ch * 8;
      cp_async16(dst, X + (size_t)(ok ? tok : 0) * K + (ok ? f0 : 0), ok);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };

  const int nstage_total = (T + HS_TOK - 1) / HS_TOK;
  float acc[4][4][4];
  auto zero_acc = [&]() {
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[a][b][c] = 0.f;
  };
  auto carry = [&]() {
    // acc[a][b]: rows i0 + wi*64 + a*16 + g (+8), cols j0 + wj*32 + b*8 + 2*t4 (+1)
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int i = i0 + wi * 64 + a * 16 + g + (c >> 1) * 8, j = j0 + wj * 32 + b * 8 + 2 * t4 + (c & 1);
          if (i < K && j < K) H[(size_t)i * K + j] += (double)acc[a][b][c];
        }
  };

  zero_acc();
  for (int s = 0; s < HS_STAGES - 1; ++s) {
    if (s < nstage_total) load_stage(s, s * HS_TOK);
    else asm volatile("cp.async.commit_group;" ::: "memory");
  }
  for (int st = 0; st < nstage_total; ++st) {
    asm volatile("cp.async.wait_group %0;" ::"n"(HS_STAGES - 2) : "memory");
    __syncthreads();
    if (st + HS_STAGES - 1 < nstage_total) load_stage((st + HS_STAGES - 1) % HS_STAGES, (st + HS_STAGES - 1) * HS_TOK);
    else asm volatile("cp.async.commit_group;" ::: "memory");
    const __half* bI = sI + (st % HS_STAGES) * HS_TOK * HS_LD;
    const __half* bJ = sJ + (st % HS_STAGES) * HS_TOK * HS_LD;
#pragma unroll
    for (int k0 = 0; k0 < HS_TOK; k0 += 16) {
      // A fragments (rows = features i, k = tokens): x4.trans matrices (i 0-7, t 0-7), (i 8-15, t 0-7), (i 0-7, t 8-15), (i 8-15, t 8-15)
      uint32_t af[4][4];
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const int mtx = lane >> 3, r = lane & 7;
        const __half* p = bI + (k0 + (mtx >> 1) * 8 + r) * HS_LD + wi * 64 + a * 16 + (mtx & 1) * 8;
        ldsm_x4_trans(af[a], p);
      }
      // B fragments (k = tokens, n = features j): per pair of n-tiles one x4.trans: (t 0-7, j 0-7), (t 8-15, j 0-7), (t 0-7, j 8-15), (t 8-15, j 8-15)
      uint32_t bfr[2][4];
#pragma unroll
      for (int bp = 0; bp < 2; ++bp) {
        const int mtx = lane >> 3, r = lane & 7;
        const __half* p = bJ + (k0 + (mtx & 1) * 8 + r) * HS_LD + wj * 32 + bp * 16 + (mtx >> 1) * 8;
        ldsm_x4_trans(bfr[bp], p);
      }
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const uint32_t bb[2] = {bfr[b >> 1][(b & 1) * 2], bfr[b >> 1][(b & 1) * 2 + 1]};
          mma16816(acc[a][b], af[a], bb);
        }
    }
    if (((st + 1) * HS_TOK) % HS_CHUNK == 0 || st + 1 == nstage_total) {
      carry();
      zero_acc();
    }
  }
}

}  // namespace

}  // namespace quip

using namespace quip;

extern "C" int quip_hessian_accumulate(const void* x, double* H, int64_t tokens, int32_t K, void* stream) {
  QUIP_CHECK_ARG(x && H, "quip_hessian_accumulate: null pointer");
  QUIP_CHECK_ARG(tokens >= 0 && tokens < (1ll << 31) && K > 0 && K % 8 == 0, "quip_hessian_accumulate: K=%d must be a positive multiple of 8", K);
  QUIP_CHECK_ARG((reinterpret_cast<uintptr_t>(x) & 15) == 0, "quip_hessian_accumulate: activations must be 16-byte aligned");
  if (tokens == 0) return QUIP_OK;
  const int ntile = ceil_div(K, HS_TILE);
  const int64_t nct = (int64_t)ntile * (ntile + 1) / 2;
  const size_t smem = (size_t)2 * HS_STAGES * HS_TOK * HS_LD * sizeof(__half);
  return launch("hessian_syrk_kernel", hessian_syrk_kernel, (unsigned)nct, HS_THREADS, smem, (cudaStream_t)stream, false,
                (const __half*)x, H, (int)tokens, K, ntile);
}
