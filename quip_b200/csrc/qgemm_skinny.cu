// Packed-integer x fp16 contraction for few tokens (M <= 32): the HBM-bound regime of the path
// (decode; reference Quant3Linear.forward is M == 1 only, quant.py:222-233, calling the absent
// quant_cuda.vecquant3matmul).  The packed words are streamed with coalesced 128-bit loads straight
// into registers, expanded to fp16 in registers (1 shift + 1 LOP3 + 1 HADD2 per pair of codes) in
// exactly the A-fragment order of mma.sync.m16n8k16, and contracted against token fragments read
// from shared memory; fp32 accumulation.  Weights are the "M" side of the MMA (16 output rows),
// tokens the "N" side (8 per tile).
//
//   z[m][n] = P_n * sum_k x[m][k] d[n][k] + R_n * sum_k x[m][k]  (+ bias_n),
//   d = (code - cbar)/2^bits,  P_n = scales_n 2^bits,  R_n = scales_n cbar - zeros_n.
//
// Grid: x = tiles of RBC*16 output rows, y = K splits.  Each warp walks the k super-blocks of its
// CTA's K range (stride 8 warps) for all RBC row blocks; the 8 warps are reduced through shared
// memory, K splits through an fp32 workspace where the last CTA to arrive (per row tile) sums the
// partials in a fixed order and applies the epilogue.
#include "common.cuh"

namespace quip {

constexpr int SK_WARPS = 8;
constexpr int SK_XPAD = 32;          // halves; makes the 8-lane LDS.128 phases conflict-free

template <int BITS>
struct SbRegs {
  uint32_t w[BITS == 2 ? 4 : (BITS == 3 ? 6 : 8)];
};

template <int BITS>
__device__ __forceinline__ void load_sb(const uint32_t* __restrict__ base, int lane, SbRegs<BITS>& r) {
  if constexpr (BITS == 2) {
    uint4 v = ldg_nc_v4(base + lane * 4);
    r.w[0] = v.x; r.w[1] = v.y; r.w[2] = v.z; r.w[3] = v.w;
  } else if constexpr (BITS == 4) {
    uint4 a = ldg_nc_v4(base + lane * 4), b = ldg_nc_v4(base + 128 + lane * 4);
    r.w[0] = a.x; r.w[1] = a.y; r.w[2] = a.z; r.w[3] = a.w;
    r.w[4] = b.x; r.w[5] = b.y; r.w[6] = b.z; r.w[7] = b.w;
  } else {
    uint4 a = ldg_nc_v4(base + lane * 4);
    uint2 b = ldg_nc_v2(base + 128 + lane * 2);
    r.w[0] = a.x; r.w[1] = a.y; r.w[2] = a.z; r.w[3] = a.w;
    r.w[4] = b.x; r.w[5] = b.y;
  }
}

template <int BITS, int CH>
__device__ __forceinline__ void expand_sb_chunk(const SbRegs<BITS>& r, uint32_t (&h)[8]) {
  if constexpr (BITS == 2) expand_chunk<2>(r.w[CH], 0u, h);
  else if constexpr (BITS == 4) expand_chunk<4>(r.w[2 * CH], r.w[2 * CH + 1], h);
  else expand_chunk<3, (CH & 1)>(r.w[CH], r.w[4 + (CH >> 1)], h);
}

template <int BITS, int NT8, int RBC>
__global__ void __launch_bounds__(SK_WARPS * 32)
qgemm_skinny_kernel(const uint32_t* __restrict__ q, const __half* __restrict__ x, const float* __restrict__ scales,
                    const float* __restrict__ zeros, const __half* __restrict__ bias, __half* __restrict__ z,
                    int M, int K, int N, int ksb_per_split, int symmetric, float* __restrict__ part,
                    int* __restrict__ counters) {
  constexpr int TOK = 8 * NT8, ROWS = 16 * RBC, RLD = ROWS + 8;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int KSB = K >> 7;                                 // k super-blocks in the matrix
  const int ksb0 = blockIdx.y * ksb_per_split;
  const int ksb1 = min(KSB, ksb0 + ksb_per_split);
  const int kslice = (ksb1 - ksb0) * 128;
  const int xld = ksb_per_split * 128 + SK_XPAD;
  __half* xs = reinterpret_cast<__half*>(smem_raw);                                // [TOK][xld]
  float* red = reinterpret_cast<float*>(smem_raw + (size_t)TOK * xld * sizeof(__half));   // [8][TOK][RLD]
  float* xsum_s = red + SK_WARPS * TOK * RLD;                                      // [TOK]
  __shared__ int s_last;

  // ---- stage the activations of this K range once per CTA: xs[tok][k] ----
  {
    const int cpr = kslice / 8;
    for (int c = tid; c < TOK * cpr; c += SK_WARPS * 32) {
      int tok = c / cpr, qd = c % cpr;
      uint4 v = make_uint4(0, 0, 0, 0);
      if (tok < M) v = *reinterpret_cast<const uint4*>(x + (int64_t)tok * K + ksb0 * 128 + qd * 8);
      *reinterpret_cast<uint4*>(&xs[tok * xld + qd * 8]) = v;
    }
  }
  __syncthreads();
  if (!symmetric) {   // partial row sums of x over this K range (fp32), one warp per token round-robin
    for (int tok = warp; tok < TOK; tok += SK_WARPS) {
      float a = 0.f;
      for (int k = lane; k < kslice; k += 32) a += __half2float(xs[tok * xld + k]);
#pragma unroll
      for (int o = 16; o; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
      if (lane == 0) xsum_s[tok] = a;
    }
  }

  const int NRB = N >> 4;
  const int ntiles = (NRB + RBC - 1) / RBC;               // row tiles in the matrix
  const int nk = ksb1 - ksb0;
  const int rounds = (nk + SK_WARPS - 1) / SK_WARPS;      // k iterations per warp per row tile (lockstep)
  const int nsplit = gridDim.y;
  const bool direct = nsplit == 1;

  // software pipeline over the flattened (row tile, k round) sequence: the packed words of step i+1 are
  // in flight while step i is expanded and multiplied
  SbRegs<BITS> cur[RBC], nxt[RBC];
  auto fetch = [&](int tile, int round, SbRegs<BITS> (&dst)[RBC]) {
    const int ksb = ksb0 + round * SK_WARPS + warp;
    const int kk = min(ksb, ksb1 - 1);
#pragma unroll
    for (int r = 0; r < RBC; ++r) {
      int rb = min(tile * RBC + r, NRB - 1);              // tail tile: re-read a valid block, masked at the store
      load_sb<BITS>(q + ((int64_t)rb * KSB + kk) * sb_words(BITS), lane, dst[r]);
    }
  };

  int tile = blockIdx.x;
  if (tile < ntiles) fetch(tile, 0, cur);
  for (; tile < ntiles; tile += gridDim.x) {
    float acc[RBC][NT8][4];
#pragma unroll
    for (int a = 0; a < RBC; ++a)
#pragma unroll
      for (int b = 0; b < NT8; ++b)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[a][b][c] = 0.f;

    for (int round = 0; round < rounds; ++round) {
      // prefetch the next step (next k round, or the first round of this CTA's next row tile)
      {
        int nt = tile, nr = round + 1;
        if (nr == rounds) { nr = 0; nt = tile + gridDim.x; }
        if (nt < ntiles) fetch(nt, nr, nxt);
      }
      const int ksb = ksb0 + round * SK_WARPS + warp;
      if (ksb < ksb1) {
        const __half* xk = xs + (ksb - ksb0) * 128 + 8 * t;
        auto do_chunk = [&](auto chc) {
          constexpr int CH = decltype(chc)::value;
          uint32_t xb[NT8][4];
#pragma unroll
          for (int nt = 0; nt < NT8; ++nt) {
            uint4 v = *reinterpret_cast<const uint4*>(xk + (nt * 8 + g) * xld + CH * 32);
            xb[nt][0] = v.x; xb[nt][1] = v.y; xb[nt][2] = v.z; xb[nt][3] = v.w;
          }
#pragma unroll
          for (int r = 0; r < RBC; ++r) {
            uint32_t h[8];
            expand_sb_chunk<BITS, CH>(cur[r], h);
#pragma unroll
            for (int s = 0; s < 2; ++s) {
              uint32_t a[4] = {h[4 * s], h[4 * s + 1], h[4 * s + 2], h[4 * s + 3]};
#pragma unroll
              for (int nt = 0; nt < NT8; ++nt) {
                uint32_t b[2] = {xb[nt][2 * s], xb[nt][2 * s + 1]};
                mma16816(acc[r][nt], a, b);
              }
            }
          }
        };
        do_chunk(std::integral_constant<int, 0>{});
        do_chunk(std::integral_constant<int, 1>{});
        do_chunk(std::integral_constant<int, 2>{});
        do_chunk(std::integral_constant<int, 3>{});
      }
#pragma unroll
      for (int r = 0; r < RBC; ++r) cur[r] = nxt[r];
    }

    // ---- reduce the 8 warps: red[warp][tok][row] ----
#pragma unroll
    for (int r = 0; r < RBC; ++r)
#pragma unroll
      for (int nt = 0; nt < NT8; ++nt) {
        float* b = red + (warp * TOK + nt * 8 + 2 * t) * RLD + r * 16 + g;
        b[0] = acc[r][nt][0];
        b[RLD] = acc[r][nt][1];
        b[8] = acc[r][nt][2];
        b[RLD + 8] = acc[r][nt][3];
      }
    __syncthreads();

    const int n0 = tile * ROWS;
    for (int e = tid; e < TOK * ROWS; e += SK_WARPS * 32) {
      int tok = e / ROWS, r = e % ROWS;
      int n = n0 + r;
      if (tok >= M || n >= N) continue;
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < SK_WARPS; ++w) s += red[(w * TOK + tok) * RLD + r];
      float sc = scales[n];
      float v = sc * (float)(1 << BITS) * s;
      if (!symmetric) v += (sc * (0.5f * (float)((1 << BITS) - 1)) - zeros[n]) * xsum_s[tok];
      if (direct) {
        if (bias) v += __half2float(bias[n]);
        z[(int64_t)tok * N + n] = __float2half_rn(v);
      } else {
        part[((int64_t)blockIdx.y * M + tok) * N + n] = v;
      }
    }
    if (!direct) {
      // ---- K splits: the last CTA to finish this row tile sums the partials in split order ----
      __threadfence();
      __syncthreads();
      if (tid == 0) {
        int prev = atomicAdd(&counters[tile], 1);
        s_last = (prev == nsplit - 1);
        if (s_last) counters[tile] = 0;                   // leave the header zeroed for the next call
      }
      __syncthreads();
      if (s_last) {
        __threadfence();
        for (int e = tid; e < TOK * ROWS; e += SK_WARPS * 32) {
          int tok = e / ROWS, r = e % ROWS;
          int n = n0 + r;
          if (tok >= M || n >= N) continue;
          float v = 0.f;
          for (int sp = 0; sp < nsplit; ++sp) v += __ldcg(&part[((int64_t)sp * M + tok) * N + n]);
          if (bias) v += __half2float(bias[n]);
          z[(int64_t)tok * N + n] = __float2half_rn(v);
        }
      }
    }
    __syncthreads();                                      // red[] is reused by the next row tile
  }
}

template <int BITS, int NT8, int RBC>
static int launch_skinny(const QuipLinearDesc* d, const __half* x, const __half* bias, __half* z, int M,
                         int ksplit, float* part, int* counters, cudaStream_t s) {
  const int KSB = d->K / 128;
  const int per = ceil_div(KSB, ksplit);
  ksplit = ceil_div(KSB, per);
  constexpr int TOK = 8 * NT8, ROWS = 16 * RBC, RLD = ROWS + 8;
  size_t smem = (size_t)TOK * (per * 128 + SK_XPAD) * sizeof(__half) +
                (size_t)(SK_WARPS * TOK * RLD + TOK) * sizeof(float);
  QUIP_CHECK_ARG(smem <= 220 * 1024, "skinny kernel: K slice too large (%zu B of shared memory)", smem);
  // persistent in the row dimension: ~2 CTAs per SM in total, each looping over row tiles with its K slice of
  // the activations staged once
  int tiles = ceil_div(d->N, ROWS);
  QUIP_CHECK_ARG(ksplit == 1 || tiles <= 4096, "skinny kernel: too many row tiles (%d) for split-K counters", tiles);
  int gx = ceil_div(2 * num_sms(), ksplit);
  if (gx > tiles) gx = tiles;
  if (gx < 1) gx = 1;
  return launch("qgemm_skinny_kernel", qgemm_skinny_kernel<BITS, NT8, RBC>, dim3(gx, ksplit), SK_WARPS * 32, smem, s, false,
                reinterpret_cast<const uint32_t*>(d->qweight), x, d->scales, d->zeros, bias, z, M, d->K, d->N, per,
                (d->flags & QUIP_FLAG_SYMMETRIC) ? 1 : 0, part, counters);
}

// Heuristic split.  Every K split costs a round trip of fp32 partials (write, fence, counter, the last CTA reads them all), and
// that -- not the staging of the activations -- is what the kernel waits for at 9..32 tokens: on 4096 x 4096 with 32 tokens
// 8 splits take 36.6 us, 2 splits 17.0 us; with 16 tokens 15.7 against 10.3-10.8 us (profiles/mb_skinny_r02.json).  So: just
// enough splits for about one CTA per SM, K slices of at least 512, and as many more as the staged activations of M tokens
// need to fit shared memory (K = 28672 with 32 tokens: 16 slices).
int skinny_pick_ksplit(int N, int K, int rows_per_cta, int M) {
  int tiles = ceil_div(N, rows_per_cta);
  int ksb = K / 128;
  int ks = 1;
  while (tiles * ks < 128 && ksb / (ks * 2) >= 4) ks *= 2;
  const int tok = M <= 8 ? 8 : (M <= 16 ? 16 : 32);
  auto smem = [&](int k) {
    return (size_t)tok * (ceil_div(ksb, k) * 128 + SK_XPAD) * sizeof(__half) + (size_t)(SK_WARPS * tok * 72 + tok) * sizeof(float);
  };
  while (smem(ks) > 216 * 1024 && ks < ksb) ks *= 2;
  return ks;
}

size_t skinny_workspace_bytes(int N, int M, int ksplit) {
  return ksplit > 1 ? (size_t)ksplit * M * N * sizeof(float) : 0;
}

int qgemm_skinny(const QuipLinearDesc* d, const __half* x, const __half* bias, __half* z, int M, int ksplit,
                 float* part, int* counters, cudaStream_t s) {
  QUIP_CHECK_ARG(M >= 1 && M <= 32, "skinny kernel handles 1..32 tokens (got %d)", M);
#define QUIP_SK(B, T)                                                                         \
  if (d->bits == B && M <= 8 * T)                                                             \
    return launch_skinny<B, T, 4>(d, x, bias, z, M, ksplit, part, counters, s);
  QUIP_SK(2, 1) QUIP_SK(2, 2) QUIP_SK(2, 4)
  QUIP_SK(3, 1) QUIP_SK(3, 2) QUIP_SK(3, 4)
  QUIP_SK(4, 1) QUIP_SK(4, 2) QUIP_SK(4, 4)
#undef QUIP_SK
  set_error("skinny kernel: unsupported bits=%d", d->bits);
  return QUIP_ERR_UNSUPPORTED;
}

}  // namespace quip
