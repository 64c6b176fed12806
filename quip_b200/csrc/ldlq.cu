// LDLQ adaptive rounding on the GPU: the quantisation-time hot loop of the reference (SURVEY section 8(f) rank 1).
//
// Reference: round_ldl (vector_balance.py:155-199) visits the d columns last to first, each step a GEMV launch
//     w_hat[:, i] = clamp(floor(w[:, i] + (w[:, i:] - w_hat[:, i:]) @ L[i:, i] + 1/2), 0, 2^b - 1)
// and round_ldl_block (:218-257) regroups it in blocks of 128 columns; the greedy passes (:185-199, blocked :259-286)
// are d more sequential column steps each.  The m output rows never interact, so here
//   * the feedback of all FINISHED blocks enters through one GEMM per block (host side, torch / cuBLAS fp32:
//     base = w[:, blk] + err[:, done] @ L[done, blk]), and
//   * the sequential part -- the <= 128 columns inside a block -- runs in ONE kernel launch: a group of LANES threads per
//     row, the block's triangle of L (or square of H for the greedy pass) in shared memory, the row's running errors
//     in shared memory, the column loop inside the kernel.  ~10^4 launches per layer become d / 128.
// Data is column-major ("transposed": element (row r, column j) at [j * ld + r]) so that a warp's rows are contiguous.
//
// Arithmetic is float32 like the reference's; the dot product of a step is summed in a fixed order (LANES partial
// sums over interleaved columns, then a butterfly), so results are deterministic, but the order differs from the
// reference's GEMV: a rounding decision can flip where w + feedback lands within ~1e-6 of a half-integer.
#include "common.cuh"

namespace quip {

namespace {

constexpr int LQ_BLOCK = 128;         // columns per block (vector_balance.py:222 blocksize)
constexpr int LQ_LANES = 4;           // threads cooperating on one row
constexpr int LQ_ROWS = 64;           // rows per CTA
constexpr int LQ_THREADS = LQ_ROWS * LQ_LANES;
constexpr int LQ_LD = LQ_ROWS + 8;   // row pitch of the per-column error / s arrays: the 4 lanes of a row read 4 consecutive
                                      // columns, 8 rows per warp -> bank 8 * lane + row, conflict-free (pitch 64: 4-way)

__device__ __forceinline__ float lane_sum(float v) {
#pragma unroll
  for (int o = LQ_LANES / 2; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// One block of columns, LDLQ step.
//   baseT (cnt, ld): w[:, blk] + feedback of the finished blocks      wT (cnt, ld): w[:, blk]
//   Lb (cnt, cnt) row-major: L[blk, blk] - I (strictly lower part used: Lb[j'][j], j' > j)
//   qT (cnt, ld) out: rounded values (integers as float)               errT (cnt, ld) out: w - q
__global__ void __launch_bounds__(LQ_THREADS)
ldlq_block_kernel(const float* __restrict__ baseT, const float* __restrict__ wT, const float* __restrict__ Lb,
                  float* __restrict__ qT, float* __restrict__ errT, int m, int ld, int cnt, float top) {
  extern __shared__ float sm[];
  float* Ls = sm;                                 // [cnt][cnt + 1] transposed: Ls[j * (cnt+1) + j'] = Lb[j'][j]
  float* E = sm + cnt * (cnt + 1);                // [cnt][LQ_LD]: errors of the columns already rounded
  const int tid = threadIdx.x, lane = tid % LQ_LANES, rl = tid / LQ_LANES;
  const int row = blockIdx.x * LQ_ROWS + rl;
  for (int i = tid; i < cnt * cnt; i += LQ_THREADS) {
    const int jp = i / cnt, j = i - jp * cnt;
    Ls[j * (cnt + 1) + jp] = Lb[i];
  }
  __syncthreads();
  const bool live = row < m;
  for (int j = cnt - 1; j >= 0; --j) {
    // feedback of the in-block columns j' > j, split over the lanes of the row (j' = j + 1 + lane, + LANES, ...)
    float acc0 = 0.f, acc1 = 0.f;
    const float* lrow = Ls + j * (cnt + 1);
    int jp = j + 1 + lane;
    for (; jp + LQ_LANES < cnt; jp += 2 * LQ_LANES) {
      acc0 = fmaf(E[jp * LQ_LD + rl], lrow[jp], acc0);
      acc1 = fmaf(E[(jp + LQ_LANES) * LQ_LD + rl], lrow[jp + LQ_LANES], acc1);
    }
    if (jp < cnt) acc0 = fmaf(E[jp * LQ_LD + rl], lrow[jp], acc0);
    const float fb = lane_sum(acc0 + acc1);
    float e = 0.f;
    if (live && lane == 0) {
      const float w = wT[(size_t)j * ld + row];
      const float v = baseT[(size_t)j * ld + row] + fb;
      const float q = fminf(fmaxf(floorf(v + 0.5f), 0.f), top);
      e = w - q;
      qT[(size_t)j * ld + row] = q;
      errT[(size_t)j * ld + row] = e;
    }
    if (lane == 0) E[j * LQ_LD + rl] = e;
    __syncwarp();                                 // the LANES threads of a row sit in one warp
  }
}

// One block of columns, one greedy coordinate-descent sweep (vector_balance.py:267-283).
//   preT (cnt, ld): s[:, outside the block] @ Hn[outside, blk]   (S0 @ H0 + S2 @ H2)
//   Hb (cnt, cnt) row-major: Hn[blk, blk] (symmetric)
//   wrT / sT (cnt, ld) in-out: current values and s = wr - w of the block's columns
__global__ void __launch_bounds__(LQ_THREADS)
greedy_block_kernel(const float* __restrict__ preT, const float* __restrict__ Hb, float* __restrict__ wrT,
                    float* __restrict__ sT, int m, int ld, int cnt) {
  extern __shared__ float sm[];
  float* Hs = sm;                                 // [cnt][cnt + 1]: Hs[i * (cnt+1) + j] = Hb[j][i] (= Hb[i][j])
  float* S = sm + cnt * (cnt + 1);                // [cnt][LQ_LD]: the row's s over the block, updated in place
  const int tid = threadIdx.x, lane = tid % LQ_LANES, rl = tid / LQ_LANES;
  const int row = blockIdx.x * LQ_ROWS + rl;
  const bool live = row < m;
  for (int i = tid; i < cnt * cnt; i += LQ_THREADS) {
    const int j = i / cnt, c = i - j * cnt;
    Hs[c * (cnt + 1) + j] = Hb[i];
  }
  for (int i = tid; i < cnt * LQ_ROWS; i += LQ_THREADS) {
    const int j = i / LQ_ROWS, r = i - j * LQ_ROWS, gr = blockIdx.x * LQ_ROWS + r;
    S[j * LQ_LD + r] = gr < m ? sT[(size_t)j * ld + gr] : 0.f;
  }
  __syncthreads();
  for (int i = cnt - 1; i >= 0; --i) {
    float acc0 = 0.f, acc1 = 0.f;
    const float* hrow = Hs + i * (cnt + 1);
    int j = lane;
    for (; j + LQ_LANES < cnt; j += 2 * LQ_LANES) {
      acc0 = fmaf(S[j * LQ_LD + rl], hrow[j], acc0);
      acc1 = fmaf(S[(j + LQ_LANES) * LQ_LD + rl], hrow[j + LQ_LANES], acc1);
    }
    if (j < cnt) acc0 = fmaf(S[j * LQ_LD + rl], hrow[j], acc0);
    const float dot = lane_sum(acc0 + acc1);
    if (lane == 0) {
      float snew = S[i * LQ_LD + rl];
      if (live) {
        const float hs = preT[(size_t)i * ld + row] + dot;
        const float cur = wrT[(size_t)i * ld + row];
        const float move = cur - rintf(cur - hs / hrow[i]);                  // torch.round: half to even
        wrT[(size_t)i * ld + row] = cur - move;
        snew -= move;
        sT[(size_t)i * ld + row] = snew;
      }
      S[i * LQ_LD + rl] = snew;
    }
    __syncwarp();
  }
}

size_t lq_smem(int cnt) { return ((size_t)cnt * (cnt + 1) + (size_t)cnt * LQ_LD) * sizeof(float); }

}  // namespace

}  // namespace quip

using namespace quip;

extern "C" int quip_ldlq_block(const float* baseT, const float* wT, const float* Lb, float* qT, float* errT, int64_t m,
                               int64_t ld, int32_t cnt, int32_t bits, void* stream) {
  QUIP_CHECK_ARG(baseT && wT && Lb && qT && errT, "quip_ldlq_block: null pointer");
  QUIP_CHECK_ARG(cnt >= 1 && cnt <= LQ_BLOCK && m >= 1 && ld >= m && m < (1ll << 31), "quip_ldlq_block: bad sizes (cnt=%d)", cnt);
  QUIP_CHECK_ARG(bits >= 1 && bits <= 8, "quip_ldlq_block: bits out of range");
  return launch("ldlq_block_kernel", ldlq_block_kernel, (unsigned)ceil_div(m, LQ_ROWS), LQ_THREADS, lq_smem(cnt),
                (cudaStream_t)stream, false, baseT, wT, Lb, qT, errT, (int)m, (int)ld, cnt, (float)((1 << bits) - 1));
}

extern "C" int quip_greedy_block(const float* preT, const float* Hb, float* wrT, float* sT, int64_t m, int64_t ld,
                                 int32_t cnt, void* stream) {
  QUIP_CHECK_ARG(preT && Hb && wrT && sT, "quip_greedy_block: null pointer");
  QUIP_CHECK_ARG(cnt >= 1 && cnt <= LQ_BLOCK && m >= 1 && ld >= m && m < (1ll << 31), "quip_greedy_block: bad sizes (cnt=%d)", cnt);
  return launch("greedy_block_kernel", greedy_block_kernel, (unsigned)ceil_div(m, LQ_ROWS), LQ_THREADS, lq_smem(cnt),
                (cudaStream_t)stream, false, preT, Hb, wrT, sT, (int)m, (int)ld, cnt);
}
