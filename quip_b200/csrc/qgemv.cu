// Packed-integer x fp16 contraction for a handful of tokens (decode, M <= 8): the HBM-bound regime
// of the path (reference Quant3Linear.forward is M == 1 only, quant.py:222-233, on the absent
// quant_cuda.vecquant3matmul).  Speed of light is one pass over the packed words at ~6.5 TB/s, i.e. an
// SM has ~22 cycles per 512-byte super-block: the limits are (1) instructions per weight on the ALU
// pipe (LOP3/SHF retire one warp-instruction per 2 cycles per SM sub-partition) and on the legacy tensor
// pipe (every mma.sync shape retires one per 8 cycles per sub-partition -- tools/mma_rate.cu), and
// (2) dependent round trips to memory.  Two datapaths share one skeleton:
//
// * qgemv_i8_kernel (2-/4-bit, up to 5 tokens): integer tensor cores, IMMA.16832.  The codes are used as
//   they are -- four ANDs turn one packed word into the four A registers (common.cuh) -- and a token is
//   split once per CTA into three balanced signed bytes of round(x 2^22/amax), three B columns.  Sums of
//   products are exact in int32; 5 ALU instructions and 1-2 MMAs per 16 weights x 32 lanes.
//       y[m][n] = scales_n s_m (65536 I_hi + 256 I_mid + I_lo) - zeros_n S_m + bias_n,  s_m = amax_m / 2^22.
//
// * qgemv_kernel (fp16, HMMA.16816; 6-8 tokens and 3-bit).  The usual "mask, OR exponent, subtract" costs
//   1.4 instructions per weight; here the subtraction is dropped: a pair of codes is masked in place
//   inside the fp16 mantissa wherever one shift per row leaves it, which reads as 1 + c/4^(e+1) with
//   e in {0,2} depending on the bit offset.  The token operand of that k position is pre-scaled by 4^(e-2)
//   once per CTA when the activations are staged, so every product is 4^(e-2) x_k + c_k x_k / 64 and
//       sum_k A_k B_k = T_m + (1/64) sum_k c_k x_k,      T_m = sum_k 4^(e(k)-2) x_k  (per token),
//   exact in the fp32 accumulator (the offset costs at most 6 of its 24 bits).  4 shifts (two of them IMADs on
//   the FMA pipe) + 8 LOP3 per 16 weights.  4-bit likewise; 3-bit keeps the recentring expansion.
//   T_m and the plain row sum S_m fall out of one extra MMA per k-step against a constant A fragment
//   (rows 0-7 ones, rows 8-15 4^(2-e)) during a CTA's first row tile.
//       y[m][n] = scales_n (A1 (acc - T_m) + A2 S_m) - zeros_n S_m + bias_n,
//       (A1, A2) = (64, 0) / (8, 3.5) / (256, 0) for 2 / 3 / 4 bits.
//
// Skeleton.  A CTA owns RBC row blocks over the *whole* K (its warps split the k super-blocks), so the only
// reduction is through shared memory: no split-K partials, counters or fences.  The packed words are
// requested before anything else (they do not depend on the previous kernel: with programmatic dependent
// launch they are in flight while it drains), then the tokens are staged.
//
// Three kernels carry the int8 datapath, one per regime (routing in qgemv() below):
//   qgemv_i8_tma_kernel     a single layer (all latency): bulk-copy ring + consumer warps + epilogue warp
//   qgemv_i8_kernel         its register-ring (LDG) sibling, used when K x tokens leaves no room for the ring
//   qgemv_i8_stream_kernel  >= 32 row blocks per SM (stacked / grouped matrices): barrier-free streaming,
//                           78 % of the HBM peak at one token
#include "tc_common.cuh"

namespace quip {

constexpr int GV_WARPS = 8;
constexpr int GV_XPAD = 32;            // halves; makes the 8-lane LDS.128 phases conflict-free

int g_gv_rbc = 0;                      // quip_config("gv_rbc", r): row blocks per CTA tile (0 = heuristic)
int g_gv_int = 1;                      // quip_config("gv_int", 0): fp16 tensor path for every token count
int g_gv_tma = 1;                      // quip_config("gv_tma", 0): register-ring variant of the int8 path
int g_gv_cw = 16;                      // quip_config("gv_cw", 8|16): consumer warps of the bulk-copy kernel
int g_gv_stream = 32;                  // quip_config("gv_stream", r): streaming kernel when N/16 >= r * SMs (0: never)
int g_gv_persist = 1;                  // quip_config("gv_persist", 0): one CTA per row tile instead of a persistent grid

template <int BITS>
struct Gv {
  static constexpr int kWords = BITS == 2 ? 4 : (BITS == 3 ? 6 : 8);
  static constexpr bool kRaw = BITS != 3;                       // offset-free expansion + prescaled tokens
  static constexpr float kA1 = BITS == 2 ? 64.f : (BITS == 3 ? 8.f : 256.f);
  static constexpr float kA2 = BITS == 3 ? 3.5f : 0.f;
};

// fp16x2 constants
constexpr uint32_t H2_ONE = 0x3C003C00u, H2_SIXTEENTH = 0x2C002C00u, H2_SIXTEEN = 0x4C004C00u;

// token scale 4^(e-2) of k pair u (pos 2u, 2u+1 of a lane's 8 k) and its inverse
template <int BITS>
__device__ __forceinline__ constexpr uint32_t gv_scale(int u) {
  if (BITS == 2) return u < 2 ? H2_ONE : H2_SIXTEENTH;
  if (BITS == 4) return (u & 1) ? H2_SIXTEENTH : H2_ONE;
  return H2_ONE;
}
template <int BITS>
__device__ __forceinline__ constexpr uint32_t gv_inv_scale(int u) {
  if (BITS == 2) return u < 2 ? H2_ONE : H2_SIXTEEN;
  if (BITS == 4) return (u & 1) ? H2_SIXTEEN : H2_ONE;
  return H2_ONE;
}

// (a & mask) | c in ONE LOP3: c must live in a register (a LOP3 encodes a single immediate), which the
// compiler will not do on its own for a constant -- it emits an AND and an OR, doubling the ALU work.
__device__ __forceinline__ uint32_t and_or(uint32_t a, uint32_t mask, uint32_t c) {
  uint32_t d;
  asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(d) : "r"(a), "r"(mask), "r"(c));
  return d;
}
__device__ __forceinline__ uint32_t opaque_u32(uint32_t v) {   // a constant the optimiser cannot see through
  uint32_t d;
  asm("mov.b32 %0, %1;" : "=r"(d) : "r"(v));
  return d;
}

__device__ __forceinline__ uint32_t hmul2_u32(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("mul.rn.f16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}

template <int BITS>
struct GvRegs {
  uint32_t w[Gv<BITS>::kWords];
};

template <int BITS>
__device__ __forceinline__ void gv_load(const uint32_t* __restrict__ base, int lane, GvRegs<BITS>& r) {
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

// chunk CH of a lane -> h[2u + r] (k pair u, row half r).  2-/4-bit: 1 + c/2^BITS/4^e, no recentring.
// 2-bit half-word (slot2): row g pairs at bits 0 (u0), 4 (u2), 8 (u1), 12 (u3), row g+8 two bits higher.
// w<<4 / w<<2 put u0 on mantissa bit 4 (e = 2) and u2 on bit 8 (e = 0) for the two rows, w>>4 / w>>6 do the
// same for u1 / u3.  Bits that cross the half-word boundary land outside every mask.
template <int BITS, int CH>
__device__ __forceinline__ void gv_expand(const GvRegs<BITS>& r, uint32_t one, uint32_t (&h)[8]) {
  if constexpr (BITS == 2) {
    const uint32_t w = r.w[CH];
    const uint32_t b0 = w << 4, b1 = w << 2, b2 = w >> 4, b3 = w >> 6;
    h[0] = and_or(b0, 0x00300030u, one); h[1] = and_or(b1, 0x00300030u, one);   // u=0: e=2
    h[2] = and_or(b2, 0x00300030u, one); h[3] = and_or(b3, 0x00300030u, one);   // u=1: e=2
    h[4] = and_or(b0, 0x03000300u, one); h[5] = and_or(b1, 0x03000300u, one);   // u=2: e=0
    h[6] = and_or(b2, 0x03000300u, one); h[7] = and_or(b3, 0x03000300u, one);   // u=3: e=0
  } else if constexpr (BITS == 4) {
    // half-word nibbles (slot4): u%2 = 0 at bits 0 (row g) / 4 (row g+8), u%2 = 1 at 8 / 12.
    // w<<2, w>>2 -> field at bits 2-5 (e = 2); w>>2, w>>6 -> bits 6-9 (e = 0).
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const uint32_t w = r.w[2 * CH + i];
      const uint32_t c0 = w << 2, c1 = w >> 2, c2 = w >> 6;
      h[4 * i + 0] = and_or(c0, 0x003C003Cu, one); h[4 * i + 1] = and_or(c1, 0x003C003Cu, one);
      h[4 * i + 2] = and_or(c1, 0x03C003C0u, one); h[4 * i + 3] = and_or(c2, 0x03C003C0u, one);
    }
  } else {
    expand_chunk<3, (CH & 1)>(r.w[CH], r.w[4 + (CH >> 1)], h);
  }
}

template <int BITS, int NT8, int RBC, int D>
__global__ void __launch_bounds__(GV_WARPS * 32)
qgemv_kernel(const uint32_t* __restrict__ q, const __half* __restrict__ x, const float* __restrict__ scales,
             const float* __restrict__ zeros, const __half* __restrict__ bias, __half* __restrict__ z, int M, int K,
             int N) {
  constexpr int TOK = 8 * NT8, ROWS = 16 * RBC, RLD = ROWS + 4, W = GV_WARPS;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int KSB = K >> 7, NRB = N >> 4;
  const int ntiles = (NRB + RBC - 1) / RBC;
  const int xld = K + GV_XPAD;
  __half* xs = reinterpret_cast<__half*>(smem_raw);                                        // [M][xld]
  float* red = reinterpret_cast<float*>(smem_raw + (((size_t)M * xld * sizeof(__half) + 15) & ~(size_t)15));  // [2][W][TOK][RLD]
  float* red_st = red + 2 * W * TOK * RLD;                                                 // [W][2][TOK]: S, T

  const int nround = (KSB - warp + W - 1) / W;            // k super-blocks of this warp: ks = warp + W*round
  const int nround_pad = ((KSB + W - 1) / W + D - 1) / D * D;   // same for every warp; slot = round % D

  // ---- the ring: slot d holds step (tile, round) with round % D == d ----
  GvRegs<BITS> ring[D][RBC];
  auto fetch = [&](int tile, int round, GvRegs<BITS> (&dst)[RBC]) {
    if (tile < ntiles && round < nround) {
      const int ks = warp + W * round;
#pragma unroll
      for (int r = 0; r < RBC; ++r) {
        const int rb = min(tile * RBC + r, NRB - 1);      // tail tile: re-read a valid block, masked at the store
        gv_load<BITS>(q + ((int64_t)rb * KSB + ks) * sb_words(BITS), lane, dst[r]);
      }
    }
  };
  int tile = blockIdx.x;
#pragma unroll
  for (int d = 0; d < D; ++d) {                           // weights first: independent of the previous kernel
    int ft = tile, fr = d;
    if (fr >= nround_pad) { fr -= nround_pad; ft += gridDim.x; }
    fetch(ft, fr, ring[d]);
  }
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");

  // ---- stage the tokens once per CTA, pre-scaled per k position ----
  {
    const int cpr = K >> 3;
    for (int tok = 0; tok < M; ++tok) {
      const uint4* src = reinterpret_cast<const uint4*>(x + (int64_t)tok * K);
      uint4* dst = reinterpret_cast<uint4*>(xs + (size_t)tok * xld);
      for (int c = tid; c < cpr; c += W * 32) {
        uint4 v = src[c];
        if constexpr (Gv<BITS>::kRaw) {
          if (gv_scale<BITS>(1) != H2_ONE) v.y = hmul2_u32(v.y, gv_scale<BITS>(1));
          if (gv_scale<BITS>(2) != H2_ONE) v.z = hmul2_u32(v.z, gv_scale<BITS>(2));
          if (gv_scale<BITS>(3) != H2_ONE) v.w = hmul2_u32(v.w, gv_scale<BITS>(3));
        }
        dst[c] = v;
      }
    }
  }
  __syncthreads();

  const uint32_t one = opaque_u32(H2_ONE);
  // constant A fragments of the token-sum MMA, k-steps 0 and 1: {row g, row g+8} x {k pair 2s, 2s+1}
  const uint32_t cst[2][4] = {
      {one, opaque_u32(gv_inv_scale<BITS>(0)), one, opaque_u32(gv_inv_scale<BITS>(1))},
      {one, opaque_u32(gv_inv_scale<BITS>(2)), one, opaque_u32(gv_inv_scale<BITS>(3))}};
  // epilogue ownership: thread -> output row erow of the tile, tokens etok + j*ETS
  constexpr int ETS = (W * 32) / ROWS;                     // tokens covered per pass of the CTA
  constexpr int EPT = (TOK + ETS - 1) / ETS;               // passes
  const int erow = tid % ROWS, etok = tid / ROWS;
  float S[EPT], T[EPT];
  bool first = true;
  int parity = 0;
  for (; tile < ntiles; tile += gridDim.x) {
    // this tile's dequantisation parameters: requested now, used after the k loop
    float e_sc = 0.f, e_ze = 0.f, e_bi = 0.f;
    {
      const int n = tile * ROWS + erow;
      if (n < N && etok < M) {
        e_sc = __ldg(scales + n);
        e_ze = __ldg(zeros + n);
        if (bias) e_bi = __half2float(__ldg(bias + n));
      }
    }
    float acc[RBC][NT8][4];
    float acc_st[NT8][4];
#pragma unroll
    for (int b = 0; b < NT8; ++b)
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        acc_st[b][c] = 0.f;
#pragma unroll
        for (int a = 0; a < RBC; ++a) acc[a][b][c] = 0.f;
      }

    // FIRST (compile time): this CTA's first row tile also accumulates the token sums
    auto run_tile = [&](auto first_c) {
      constexpr bool FIRST = decltype(first_c)::value;
      for (int round0 = 0; round0 < nround_pad; round0 += D) {
#pragma unroll
        for (int d = 0; d < D; ++d) {
          const int round = round0 + d;
          if (round < nround) {
            const int ks = warp + W * round;
            const __half* xk = xs + ks * 128 + 8 * t;
            auto do_chunk = [&](auto chc) {
              constexpr int CH = decltype(chc)::value;
              uint32_t xb[NT8][4];
#pragma unroll
              for (int nt = 0; nt < NT8; ++nt) {
                // token columns >= M re-read the last real token: their results are never stored
                const uint4 v = *reinterpret_cast<const uint4*>(xk + (size_t)min(nt * 8 + g, M - 1) * xld + CH * 32);
                xb[nt][0] = v.x; xb[nt][1] = v.y; xb[nt][2] = v.z; xb[nt][3] = v.w;
              }
#pragma unroll
              for (int r = 0; r < RBC; ++r) {
                uint32_t h[8];
                gv_expand<BITS, CH>(ring[d][r], one, h);
#pragma unroll
                for (int s = 0; s < 2; ++s) {
                  const uint32_t a[4] = {h[4 * s], h[4 * s + 1], h[4 * s + 2], h[4 * s + 3]};
#pragma unroll
                  for (int nt = 0; nt < NT8; ++nt) {
                    const uint32_t b[2] = {xb[nt][2 * s], xb[nt][2 * s + 1]};
                    mma16816(acc[r][nt], a, b);
                  }
                }
              }
              if constexpr (FIRST) {
                // token sums on the tensor pipe, one MMA per k-step: rows 0-7 of the constant A tile are ones
                // (-> T, the sum of the pre-scaled tokens), rows 8-15 undo the scale (-> S, the plain sum)
#pragma unroll
                for (int s = 0; s < 2; ++s)
#pragma unroll
                  for (int nt = 0; nt < NT8; ++nt) {
                    const uint32_t b[2] = {xb[nt][2 * s], xb[nt][2 * s + 1]};
                    mma16816(acc_st[nt], cst[s], b);
                  }
              }
            };
            do_chunk(std::integral_constant<int, 0>{});
            do_chunk(std::integral_constant<int, 1>{});
            do_chunk(std::integral_constant<int, 2>{});
            do_chunk(std::integral_constant<int, 3>{});
          }
          // refill this slot with the step D ahead (possibly in this CTA's next row tile)
          int ft = tile, fr = round + D;
          if (fr >= nround_pad) { fr -= nround_pad; ft += gridDim.x; }
          fetch(ft, fr, ring[d]);
        }
      }
    };
    if (first) run_tile(std::true_type{});
    else run_tile(std::false_type{});

    // ---- reduce the warps (each covered different k): red[tile parity][warp][tok][row] ----
    float* redp = red + (parity ? W * TOK * RLD : 0);
#pragma unroll
    for (int r = 0; r < RBC; ++r)
#pragma unroll
      for (int nt = 0; nt < NT8; ++nt) {
        float* b = redp + (warp * TOK + nt * 8 + 2 * t) * RLD + r * 16 + g;
        b[0] = acc[r][nt][0];
        b[RLD] = acc[r][nt][1];
        b[8] = acc[r][nt][2];
        b[RLD + 8] = acc[r][nt][3];
      }
    if (first && g == 0) {
#pragma unroll
      for (int nt = 0; nt < NT8; ++nt) {
        float* b = red_st + warp * 2 * TOK + nt * 8 + 2 * t;
        b[0] = acc_st[nt][2]; b[1] = acc_st[nt][3];          // rows 8-15: S
        b[TOK] = acc_st[nt][0]; b[TOK + 1] = acc_st[nt][1];  // rows 0-7: T
      }
    }
    __syncthreads();      // the only barrier of a tile: red[] alternates, so the next tile's writes cannot race

    if (first) {          // every epilogue thread keeps the sums of its own tokens for all later tiles
#pragma unroll
      for (int j = 0; j < EPT; ++j) {
        const int tok = etok + j * ETS;
        float s = 0.f, tt = 0.f;
        if (tok < M) {
#pragma unroll
          for (int w = 0; w < W; ++w) {
            s += red_st[w * 2 * TOK + tok];
            tt += red_st[w * 2 * TOK + TOK + tok];
          }
        }
        S[j] = s;
        T[j] = Gv<BITS>::kRaw ? tt : 0.f;
      }
    }
    {
      const int n = tile * ROWS + erow;
#pragma unroll
      for (int j = 0; j < EPT; ++j) {
        const int tok = etok + j * ETS;
        if (tok < M && n < N) {
          float s = 0.f;
#pragma unroll
          for (int w = 0; w < W; ++w) s += redp[(w * TOK + tok) * RLD + erow];
          float v = e_sc * (Gv<BITS>::kA1 * (s - T[j]) + Gv<BITS>::kA2 * S[j]) - e_ze * S[j] + e_bi;
          z[(int64_t)tok * N + n] = __float2half_rn(v);
        }
      }
    }
    first = false;
    parity ^= 1;
  }
}

// ---------------------------------------------------------------------------------------------
// int8 tensor-core path
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void imma16832(int (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile(
      "mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+r"(d[0]), "+r"(d[1]), "+r"(d[2]), "+r"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

constexpr int GV_LIMBS = 3;            // bytes per token value: round(x * 2^22 / amax) in balanced base 256
constexpr float GV_QMAX = 4194304.f;   // 2^22: the top limb stays within +-64

// A registers of chunk CH: rows g (a0, a2) and g+8 (a1, a3; scaled by 4 / 16, undone in the epilogue)
template <int BITS, int CH>
__device__ __forceinline__ void gv_expand_i8(const GvRegs<BITS>& r, uint32_t (&a)[4]) {
  if constexpr (BITS == 2) {
    const uint32_t w = r.w[CH], w4 = w >> 4;
    a[0] = w & 0x03030303u; a[1] = w & 0x0C0C0C0Cu; a[2] = w4 & 0x03030303u; a[3] = w4 & 0x0C0C0C0Cu;
  } else {
    const uint32_t w0 = r.w[2 * CH], w1 = r.w[2 * CH + 1];
    a[0] = w0 & 0x0F0F0F0Fu; a[1] = w0 & 0xF0F0F0F0u; a[2] = w1 & 0x0F0F0F0Fu; a[3] = w1 & 0xF0F0F0F0u;
  }
}

template <int BITS, int NT8, int RBC, int D>
__global__ void __launch_bounds__(GV_WARPS * 32)
qgemv_i8_kernel(const uint32_t* __restrict__ q, const __half* __restrict__ x, const float* __restrict__ scales,
                const float* __restrict__ zeros, const __half* __restrict__ bias, __half* __restrict__ z, int M, int K,
                int N) {
  constexpr int COLS = 8 * NT8, ROWS = 16 * RBC, RLD = ROWS + 4, W = GV_WARPS;
  constexpr float HI_ROW_SCALE = BITS == 2 ? 0.25f : 0.0625f;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int KSB = K >> 7, NRB = N >> 4;
  const int ntiles = (NRB + RBC - 1) / RBC;
  const int ncol = GV_LIMBS * M;                          // B columns in use: 3 per token
  const int lld = K + 32;                                 // bytes; LDS.64 phases conflict-free
  int8_t* limbs = reinterpret_cast<int8_t*>(smem_raw);                                     // [ncol][lld], slot order
  int* red = reinterpret_cast<int*>(smem_raw + (((size_t)ncol * lld + 15) & ~(size_t)15));  // [2][W][COLS][RLD]
  float* tokf = reinterpret_cast<float*>(red + 2 * W * COLS * RLD);                        // [M][2]: s_m, S_m
  float* wred = tokf + 2 * 8;                                                              // [W][2] scratch

  const int nround = (KSB - warp + W - 1) / W;
  const int nround_pad = ((KSB + W - 1) / W + D - 1) / D * D;
  GvRegs<BITS> ring[D][RBC];
  auto fetch = [&](int tile, int round, GvRegs<BITS> (&dst)[RBC]) {
    if (tile < ntiles && round < nround) {
      const int ks = warp + W * round;
#pragma unroll
      for (int r = 0; r < RBC; ++r) {
        const int rb = min(tile * RBC + r, NRB - 1);
        gv_load<BITS>(q + ((int64_t)rb * KSB + ks) * sb_words(BITS), lane, dst[r]);
      }
    }
  };
  int tile = blockIdx.x;
#pragma unroll
  for (int d = 0; d < D; ++d) {                           // weights first: independent of the previous kernel
    int ft = tile, fr = d;
    if (fr >= nround_pad) { fr -= nround_pad; ft += gridDim.x; }
    fetch(ft, fr, ring[d]);
  }
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");

  // ---- tokens -> three signed bytes each, once per CTA ----
  const int cpr = K >> 3;
  for (int tok = 0; tok < M; ++tok) {
    const uint4* src = reinterpret_cast<const uint4*>(x + (int64_t)tok * K);
    float amax = 0.f, sum = 0.f;
    for (int c = tid; c < cpr; c += W * 32) {
      const uint4 v = src[c];
      const __half2* h2 = reinterpret_cast<const __half2*>(&v);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 f = __half22float2(h2[i]);
        amax = fmaxf(amax, fmaxf(fabsf(f.x), fabsf(f.y)));
        sum += f.x + f.y;
      }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
      sum += __shfl_xor_sync(0xffffffffu, sum, o);
    }
    if (lane == 0) { wred[2 * warp] = amax; wred[2 * warp + 1] = sum; }
    __syncthreads();
    amax = 0.f; sum = 0.f;
#pragma unroll
    for (int w = 0; w < W; ++w) { amax = fmaxf(amax, wred[2 * w]); sum += wred[2 * w + 1]; }   // same order everywhere
    const float inv = amax > 0.f ? GV_QMAX / amax : 0.f;
    if (tid == 0) { tokf[2 * tok] = amax / GV_QMAX; tokf[2 * tok + 1] = sum; }
    for (int c = tid; c < cpr; c += W * 32) {
      const uint4 v = src[c];                             // second read hits L1/L2
      const __half2* h2 = reinterpret_cast<const __half2*>(&v);
      int qv[8];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 f = __half22float2(h2[i]);
        qv[2 * i] = __float2int_rn(f.x * inv);
        qv[2 * i + 1] = __float2int_rn(f.y * inv);
      }
      // balanced limbs, stored in slot order: byte s of a run <- k offset {0,2,1,3,4,6,5,7}[s]
      uint32_t lb[GV_LIMBS][2] = {};
#pragma unroll
      for (int sidx = 0; sidx < 8; ++sidx) {
        constexpr int PI[8] = {0, 2, 1, 3, 4, 6, 5, 7};
        int v0 = qv[PI[sidx]];
        const int lo = (int)(int8_t)(v0 & 0xFF);
        v0 = (v0 - lo) >> 8;
        const int mid = (int)(int8_t)(v0 & 0xFF);
        const int hi = (v0 - mid) >> 8;
        lb[0][sidx >> 2] |= (uint32_t)(hi & 0xFF) << (8 * (sidx & 3));
        lb[1][sidx >> 2] |= (uint32_t)(mid & 0xFF) << (8 * (sidx & 3));
        lb[2][sidx >> 2] |= (uint32_t)(lo & 0xFF) << (8 * (sidx & 3));
      }
#pragma unroll
      for (int l = 0; l < GV_LIMBS; ++l)
        *reinterpret_cast<uint2*>(limbs + (size_t)(GV_LIMBS * tok + l) * lld + 8 * c) = make_uint2(lb[l][0], lb[l][1]);
    }
    __syncthreads();                                      // wred reuse; also publishes the limbs
  }

  constexpr int ETS = (W * 32) / ROWS;
  constexpr int EPT = (8 + ETS - 1) / ETS;                // tokens (<= 8 ever) per epilogue thread
  const int erow = tid % ROWS, etok = tid / ROWS;
  int parity = 0;
  for (; tile < ntiles; tile += gridDim.x) {
    float e_sc = 0.f, e_ze = 0.f, e_bi = 0.f;
    {
      const int n = tile * ROWS + erow;
      if (n < N && etok < M) {
        e_sc = __ldg(scales + n);
        e_ze = __ldg(zeros + n);
        if (bias) e_bi = __half2float(__ldg(bias + n));
      }
    }
    int acc[RBC][NT8][4];
#pragma unroll
    for (int a = 0; a < RBC; ++a)
#pragma unroll
      for (int b = 0; b < NT8; ++b)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[a][b][c] = 0;

    for (int round0 = 0; round0 < nround_pad; round0 += D) {
#pragma unroll
      for (int d = 0; d < D; ++d) {
        const int round = round0 + d;
        if (round < nround) {
          const int ks = warp + W * round;
          const int8_t* lk = limbs + ks * 128 + 8 * t;
          auto do_chunk = [&](auto chc) {
            constexpr int CH = decltype(chc)::value;
            uint32_t xb[NT8][2];
#pragma unroll
            for (int nt = 0; nt < NT8; ++nt) {
              // columns beyond the last limb re-read it: their results are never stored
              const uint2 v = *reinterpret_cast<const uint2*>(lk + (size_t)min(nt * 8 + g, ncol - 1) * lld + CH * 32);
              xb[nt][0] = v.x; xb[nt][1] = v.y;
            }
#pragma unroll
            for (int r = 0; r < RBC; ++r) {
              uint32_t a[4];
              gv_expand_i8<BITS, CH>(ring[d][r], a);
#pragma unroll
              for (int nt = 0; nt < NT8; ++nt) imma16832(acc[r][nt], a, xb[nt]);
            }
          };
          do_chunk(std::integral_constant<int, 0>{});
          do_chunk(std::integral_constant<int, 1>{});
          do_chunk(std::integral_constant<int, 2>{});
          do_chunk(std::integral_constant<int, 3>{});
        }
        int ft = tile, fr = round + D;
        if (fr >= nround_pad) { fr -= nround_pad; ft += gridDim.x; }
        fetch(ft, fr, ring[d]);
      }
    }

    // ---- reduce the warps: integer sums, order-independent ----
    int* redp = red + (parity ? W * COLS * RLD : 0);
#pragma unroll
    for (int r = 0; r < RBC; ++r)
#pragma unroll
      for (int nt = 0; nt < NT8; ++nt) {
        int* b = redp + (warp * COLS + nt * 8 + 2 * t) * RLD + r * 16 + g;
        b[0] = acc[r][nt][0];
        b[RLD] = acc[r][nt][1];
        b[8] = acc[r][nt][2];
        b[RLD + 8] = acc[r][nt][3];
      }
    __syncthreads();
    {
      const int n = tile * ROWS + erow;
      const float rs = (erow & 8) ? HI_ROW_SCALE : 1.f;   // rows g+8 were masked in place, 4x / 16x too large
#pragma unroll
      for (int j = 0; j < EPT; ++j) {
        const int tok = etok + j * ETS;
        if (tok < M && n < N) {
          float limb[GV_LIMBS];
#pragma unroll
          for (int l = 0; l < GV_LIMBS; ++l) {
            int sacc = 0;
#pragma unroll
            for (int w = 0; w < W; ++w) sacc += redp[(w * COLS + GV_LIMBS * tok + l) * RLD + erow];
            limb[l] = (float)sacc;
          }
          const float dot = tokf[2 * tok] * rs * (65536.f * limb[0] + 256.f * limb[1] + limb[2]);   // sum_k c x
          const float v = e_sc * dot - e_ze * tokf[2 * tok + 1] + e_bi;
          z[(int64_t)tok * N + n] = __float2half_rn(v);
        }
      }
    }
    parity ^= 1;
  }
}

// ---------------------------------------------------------------------------------------------
// int8 path, bulk-copy fed and warp specialised (the default).  The register ring above ties the bytes in
// flight to the progress of the very warps that consume them: a warp that waits (barrier, epilogue, a slow
// neighbour) stops requesting, and the profile shows every warp stalled on its own loads at 40 % of HBM.
// Here one producer thread streams the packed words with cp.async.bulk (1-D TMA) into a shared-memory ring
// of 16-KiB stages, up to ~190 KiB in flight per SM whatever the consumers do; eight consumer warps take
// their super-blocks of a stage with one conflict-free LDS.128 each; a ninth warp owns the epilogue, fed
// through a double-buffered reduction buffer with its own mbarrier pair, so consumer warps never wait for
// one another: producer -> consumers -> epilogue are three decoupled stages.
//   stage  = up to 32 consecutive super-blocks of one row block (K <= 4096: its whole k run)
//   tile   = RBC row blocks x all their stages; static tile -> CTA schedule (tile = blockIdx + i * grid)
// ---------------------------------------------------------------------------------------------
constexpr int gt_threads(int cw) { return (cw + 2) * 32; }   // consumer warps + producer warp + epilogue warp
constexpr int GT_STAGE_SB = 32;                    // super-blocks per ring stage

__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
template <int CW>
__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 1, %0;" ::"n"(CW * 32) : "memory"); }

template <int BITS>
__device__ __forceinline__ void gv_lds(const uint32_t* sb, int lane, GvRegs<BITS>& r) {
  const uint4 a = *reinterpret_cast<const uint4*>(sb + lane * 4);
  r.w[0] = a.x; r.w[1] = a.y; r.w[2] = a.z; r.w[3] = a.w;
  if constexpr (BITS == 4) {
    const uint4 b = *reinterpret_cast<const uint4*>(sb + 128 + lane * 4);
    r.w[4] = b.x; r.w[5] = b.y; r.w[6] = b.z; r.w[7] = b.w;
  }
}

// Tokens -> three balanced signed bytes of round(x * 2^22 / amax) each, in slot order, once per CTA; also s_m and the
// plain row sum S_m (tokf).  Called by the W consumer warps only (named barrier 1).
template <int W>
__device__ __forceinline__ void gv_quantize_tokens(const __half* __restrict__ x, int M, int K, int8_t* limbs, int lld,
                                                   float* tokf, float* wred, int ctid, int warp, int lane) {
  const int cpr = K >> 3;
  // ---- tokens -> three signed bytes each, once per CTA (the ring fills meanwhile) ----
  // one sweep for the maxima and sums of all tokens (a single barrier), one sweep to quantise
  constexpr int MAXTOK = 5;
  {
    float amax[MAXTOK], sum[MAXTOK];
#pragma unroll
    for (int tok = 0; tok < MAXTOK; ++tok) { amax[tok] = 0.f; sum[tok] = 0.f; }
    for (int c = ctid; c < cpr; c += W * 32) {
#pragma unroll
      for (int tok = 0; tok < MAXTOK; ++tok) {
        if (tok < M) {
          const uint4 v = *reinterpret_cast<const uint4*>(x + (int64_t)tok * K + 8 * c);
          const __half2* h2 = reinterpret_cast<const __half2*>(&v);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float2 f = __half22float2(h2[i]);
            amax[tok] = fmaxf(amax[tok], fmaxf(fabsf(f.x), fabsf(f.y)));
            sum[tok] += f.x + f.y;
          }
        }
      }
    }
#pragma unroll
    for (int tok = 0; tok < MAXTOK; ++tok) {
      if (tok < M) {
#pragma unroll
        for (int o = 16; o; o >>= 1) {
          amax[tok] = fmaxf(amax[tok], __shfl_xor_sync(0xffffffffu, amax[tok], o));
          sum[tok] += __shfl_xor_sync(0xffffffffu, sum[tok], o);
        }
        if (lane == 0) { wred[(2 * tok) * W + warp] = amax[tok]; wred[(2 * tok + 1) * W + warp] = sum[tok]; }
      }
    }
  }
  consumer_sync<W>();
  float inv[MAXTOK];
#pragma unroll
  for (int tok = 0; tok < MAXTOK; ++tok) {
    inv[tok] = 0.f;
    if (tok < M) {
      float amax = 0.f, sum = 0.f;
#pragma unroll
      for (int w = 0; w < W; ++w) { amax = fmaxf(amax, wred[(2 * tok) * W + w]); sum += wred[(2 * tok + 1) * W + w]; }
      inv[tok] = amax > 0.f ? GV_QMAX / amax : 0.f;
      if (ctid == 0) { tokf[2 * tok] = amax / GV_QMAX; tokf[2 * tok + 1] = sum; }
    }
  }
  for (int c = ctid; c < cpr; c += W * 32) {
#pragma unroll
    for (int tok = 0; tok < MAXTOK; ++tok) {
      if (tok < M) {
        const uint4 v = *reinterpret_cast<const uint4*>(x + (int64_t)tok * K + 8 * c);   // second read hits L1/L2
        const __half2* h2 = reinterpret_cast<const __half2*>(&v);
        int qv[8];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float2 f = __half22float2(h2[i]);
          qv[2 * i] = __float2int_rn(f.x * inv[tok]);
          qv[2 * i + 1] = __float2int_rn(f.y * inv[tok]);
        }
        uint32_t lb[GV_LIMBS][2] = {};
#pragma unroll
        for (int sidx = 0; sidx < 8; ++sidx) {
          constexpr int PI[8] = {0, 2, 1, 3, 4, 6, 5, 7};
          int v0 = qv[PI[sidx]];
          const int lo = (int)(int8_t)(v0 & 0xFF);
          v0 = (v0 - lo) >> 8;
          const int mid = (int)(int8_t)(v0 & 0xFF);
          const int hi = (v0 - mid) >> 8;
          lb[0][sidx >> 2] |= (uint32_t)(hi & 0xFF) << (8 * (sidx & 3));
          lb[1][sidx >> 2] |= (uint32_t)(mid & 0xFF) << (8 * (sidx & 3));
          lb[2][sidx >> 2] |= (uint32_t)(lo & 0xFF) << (8 * (sidx & 3));
        }
#pragma unroll
        for (int l = 0; l < GV_LIMBS; ++l)
          *reinterpret_cast<uint2*>(limbs + (size_t)(GV_LIMBS * tok + l) * lld + 8 * c) = make_uint2(lb[l][0], lb[l][1]);
      }
    }
  }
  consumer_sync<W>();

}

template <int BITS, int NT8, int RBC, int CW>
__global__ void __launch_bounds__(gt_threads(CW))
qgemv_i8_tma_kernel(const uint32_t* __restrict__ q, const __half* __restrict__ x, const float* __restrict__ scales,
                    const float* __restrict__ zeros, const __half* __restrict__ bias, __half* __restrict__ z, int M,
                    int K, int N, int NS) {
  constexpr int COLS = 8 * NT8, ROWS = 16 * RBC, RLD = ROWS + 4, W = CW;
  constexpr float HI_ROW_SCALE = BITS == 2 ? 0.25f : 0.0625f;
  constexpr uint32_t STAGE_BYTES = GT_STAGE_SB * sb_words(BITS) * 4;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int KSB = K >> 7, NRB = N >> 4;
  const int ntiles = (NRB + RBC - 1) / RBC;
  const int npiece = (KSB + GT_STAGE_SB - 1) / GT_STAGE_SB;
  const int SP = (KSB + npiece - 1) / npiece;             // super-blocks per stage (last piece may be shorter)
  const int ncol = GV_LIMBS * M;
  const int lld = K + 32;

  unsigned char* ring = smem_raw;                                                          // [NS][STAGE_BYTES]
  int8_t* limbs = reinterpret_cast<int8_t*>(ring + (size_t)NS * STAGE_BYTES);              // [ncol][lld]
  int* red = reinterpret_cast<int*>(reinterpret_cast<unsigned char*>(limbs) + (((size_t)ncol * lld + 15) & ~(size_t)15));
  float* tokf = reinterpret_cast<float*>(red + 2 * W * COLS * RLD);                        // [8][2]: s_m, S_m
  float* wred = tokf + 16;                                                                 // [2 * 5 tokens][W]
  uint64_t* full = reinterpret_cast<uint64_t*>(wred + 10 * W);                             // [NS]
  uint64_t* empty = full + NS;                                                             // [NS]
  uint64_t* red_full = empty + NS;                                                         // [2]
  uint64_t* red_empty = red_full + 2;                                                      // [2]

  if (tid == 0) {
    for (int i = 0; i < NS; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], W); }
    for (int i = 0; i < 2; ++i) { mbar_init(&red_full[i], W); mbar_init(&red_empty[i], 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (warp == W) {
    // ===================== producer: one thread, runs ahead by the whole ring =====================
    if (lane == 0) {
      int slot = 0;
      uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
        for (int piece = 0; piece < npiece; ++piece) {
          const int sb0 = piece * SP;
          const uint32_t bytes = (uint32_t)(min(KSB, sb0 + SP) - sb0) * sb_words(BITS) * 4u;
#pragma unroll
          for (int r = 0; r < RBC; ++r) {
            mbar_wait(&empty[slot], ph ^ 1u);
            const int rb = min(tile * RBC + r, NRB - 1);
            mbar_arrive_expect_tx(&full[slot], bytes);
            bulk_load_1d(ring + (size_t)slot * STAGE_BYTES, q + ((int64_t)rb * KSB + sb0) * sb_words(BITS), bytes,
                         &full[slot]);
            if (++slot == NS) { slot = 0; ph ^= 1u; }
          }
        }
    }
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    return;
  }
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");      // x is read, z written only after the previous kernel

  if (warp == W + 1) {
    // ===================== epilogue warp =====================
    uint32_t tcount = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tcount) {
      const int parity = (int)(tcount & 1u);
      const uint32_t ph = (tcount >> 1) & 1u;
      const int* redp = red + (parity ? W * COLS * RLD : 0);
      // this tile's dequantisation parameters travel while the consumers are still multiplying
      constexpr int OPL = (5 * ROWS + 31) / 32;           // outputs per lane at the most tokens this path takes
      float e_sc[OPL], e_ze[OPL], e_bi[OPL];
#pragma unroll
      for (int j = 0; j < OPL; ++j) {
        const int o = lane + 32 * j, n = tile * ROWS + o % ROWS;
        e_sc[j] = e_ze[j] = e_bi[j] = 0.f;
        if (o < M * ROWS && n < N) {
          e_sc[j] = __ldg(scales + n);
          e_ze[j] = __ldg(zeros + n);
          if (bias) e_bi[j] = __half2float(__ldg(bias + n));
        }
      }
      mbar_wait(&red_full[parity], ph);
#pragma unroll
      for (int j = 0; j < OPL; ++j) {
        const int o = lane + 32 * j, tok = o / ROWS, row = o % ROWS, n = tile * ROWS + row;
        if (o < M * ROWS && n < N) {
          float limb[GV_LIMBS];
#pragma unroll
          for (int l = 0; l < GV_LIMBS; ++l) {
            int sacc = 0;
#pragma unroll
            for (int w = 0; w < W; ++w) sacc += redp[(w * COLS + GV_LIMBS * tok + l) * RLD + row];
            limb[l] = (float)sacc;
          }
          const float rs = (row & 8) ? HI_ROW_SCALE : 1.f;
          const float dot = tokf[2 * tok] * rs * (65536.f * limb[0] + 256.f * limb[1] + limb[2]);
          z[(int64_t)tok * N + n] = __float2half_rn(e_sc[j] * dot - e_ze[j] * tokf[2 * tok + 1] + e_bi[j]);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&red_empty[parity]);
    }
    return;
  }

  // ===================== consumer warps =====================
  // ---- tokens -> three signed bytes each, once per CTA (the ring fills meanwhile) ----
  gv_quantize_tokens<W>(x, M, K, limbs, lld, tokf, wred, tid, warp, lane);

  int slot = 0;                                           // ring position, advanced like the producer's
  uint32_t ph = 0, tcount = 0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tcount) {
    // two accumulator chains per (row block, column group): chunks 0,2 and 1,3 -- an IMMA waits ~30 cycles for
    // the one it accumulates onto, and with a handful of warps per scheduler that latency is the whole budget
    int acc[RBC][NT8][2][4];
#pragma unroll
    for (int a = 0; a < RBC; ++a)
#pragma unroll
      for (int b = 0; b < NT8; ++b)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[a][b][0][c] = acc[a][b][1][c] = 0;

    for (int piece = 0; piece < npiece; ++piece) {
      const int sb0 = piece * SP;
      const int nsb = min(KSB, sb0 + SP) - sb0;
      const unsigned char* stage[RBC];
      uint64_t* done[RBC];
#pragma unroll
      for (int r = 0; r < RBC; ++r) {
        mbar_wait(&full[slot], ph);
        stage[r] = ring + (size_t)slot * STAGE_BYTES;
        done[r] = &empty[slot];
        if (++slot == NS) { slot = 0; ph ^= 1u; }
      }
      GvRegs<BITS> cur[RBC], nxt[RBC];
      if (warp < nsb) {
#pragma unroll
        for (int r = 0; r < RBC; ++r)
          gv_lds<BITS>(reinterpret_cast<const uint32_t*>(stage[r]) + (size_t)warp * sb_words(BITS), lane, cur[r]);
      }
      for (int i = warp; i < nsb; i += W) {
        if (i + W < nsb) {                                // next super-block's words travel under this one's math
#pragma unroll
          for (int r = 0; r < RBC; ++r)
            gv_lds<BITS>(reinterpret_cast<const uint32_t*>(stage[r]) + (size_t)(i + W) * sb_words(BITS), lane, nxt[r]);
        }
        const int8_t* lk = limbs + (sb0 + i) * 128 + 8 * t;
        uint32_t xb[4][NT8][2];
#pragma unroll
        for (int ch = 0; ch < 4; ++ch)
#pragma unroll
          for (int nt = 0; nt < NT8; ++nt) {
            const uint2 v = *reinterpret_cast<const uint2*>(lk + (size_t)min(nt * 8 + g, ncol - 1) * lld + ch * 32);
            xb[ch][nt][0] = v.x; xb[ch][nt][1] = v.y;
          }
        auto do_chunk = [&](auto chc) {
          constexpr int CH = decltype(chc)::value;
#pragma unroll
          for (int r = 0; r < RBC; ++r) {
            uint32_t a[4];
            gv_expand_i8<BITS, CH>(cur[r], a);
#pragma unroll
            for (int nt = 0; nt < NT8; ++nt) imma16832(acc[r][nt][CH & 1], a, xb[CH][nt]);
          }
        };
        do_chunk(std::integral_constant<int, 0>{});
        do_chunk(std::integral_constant<int, 1>{});
        do_chunk(std::integral_constant<int, 2>{});
        do_chunk(std::integral_constant<int, 3>{});
#pragma unroll
        for (int r = 0; r < RBC; ++r) cur[r] = nxt[r];
      }
      __syncwarp();
      if (lane == 0) {
#pragma unroll
        for (int r = 0; r < RBC; ++r) mbar_arrive(done[r]);
      }
    }

    // ---- hand the partial sums to the epilogue warp ----
    const int parity = (int)(tcount & 1u);
    mbar_wait(&red_empty[parity], ((tcount >> 1) & 1u) ^ 1u);
    int* redp = red + (parity ? W * COLS * RLD : 0);
#pragma unroll
    for (int r = 0; r < RBC; ++r)
#pragma unroll
      for (int nt = 0; nt < NT8; ++nt) {
        int* b = redp + (warp * COLS + nt * 8 + 2 * t) * RLD + r * 16 + g;
        b[0] = acc[r][nt][0][0] + acc[r][nt][1][0];
        b[RLD] = acc[r][nt][0][1] + acc[r][nt][1][1];
        b[8] = acc[r][nt][0][2] + acc[r][nt][1][2];
        b[RLD + 8] = acc[r][nt][0][3] + acc[r][nt][1][3];
      }
    __syncwarp();
    if (lane == 0) mbar_arrive(&red_full[parity]);
  }
}

template <int BITS, int NT8, int RBC, int D>
static int launch_gv(const QuipLinearDesc* d, const __half* x, const __half* bias, __half* z, int M, cudaStream_t s) {
  constexpr int TOK = 8 * NT8, ROWS = 16 * RBC, RLD = ROWS + 4;
  const size_t xs_bytes = ((size_t)M * (d->K + GV_XPAD) * sizeof(__half) + 15) & ~(size_t)15;
  const size_t smem = xs_bytes + (size_t)(2 * GV_WARPS * TOK * RLD + GV_WARPS * 2 * TOK) * sizeof(float);
  auto kern = qgemv_kernel<BITS, NT8, RBC, D>;
  int grid = ceil_div(d->N / 16, RBC);
  if (g_gv_persist) grid = std::min(grid, blocks_per_sm((const void*)kern, GV_WARPS * 32, smem) * num_sms());
  return launch("qgemv_kernel", kern, grid, GV_WARPS * 32, smem, s, false, reinterpret_cast<const uint32_t*>(d->qweight),
                x, d->scales, d->zeros, bias, z, M, d->K, d->N);
}

template <int BITS, int NT8, int RBC, int D>
static int launch_gv_i8(const QuipLinearDesc* d, const __half* x, const __half* bias, __half* z, int M, cudaStream_t s) {
  constexpr int COLS = 8 * NT8, ROWS = 16 * RBC, RLD = ROWS + 4;
  const size_t limb_bytes = ((size_t)GV_LIMBS * M * (d->K + 32) + 15) & ~(size_t)15;
  const size_t smem = limb_bytes + (size_t)(2 * GV_WARPS * COLS * RLD) * sizeof(int) + (size_t)(16 + 2 * GV_WARPS) * sizeof(float);
  auto kern = qgemv_i8_kernel<BITS, NT8, RBC, D>;
  int grid = ceil_div(d->N / 16, RBC);
  if (g_gv_persist) grid = std::min(grid, blocks_per_sm((const void*)kern, GV_WARPS * 32, smem) * num_sms());
  return launch("qgemv_i8_kernel", kern, grid, GV_WARPS * 32, smem, s, false,
                reinterpret_cast<const uint32_t*>(d->qweight), x, d->scales, d->zeros, bias, z, M, d->K, d->N);
}

// ---------------------------------------------------------------------------------------------
// int8 path, streaming variant for very many row blocks (stacked / grouped matrices, >= 32 row blocks per SM):
// every warp owns whole row blocks and streams their k run straight from global memory into a register ring
// (8 x 512 B in flight per warp, 24 warps per SM), accumulates alone and writes its 16 x M outputs itself.  No
// shared-memory ring, no producer, no barrier after the token prologue: the same shape as a plain read loop
// (tools/read_bw.cu: 6.7-7.0 TB/s read-only on this GPU) with ~33 instructions of math per 512 bytes.
// Measured on a 352256 x 4096 matrix, one token: 5.15 TB/s = 78 % of the HBM copy peak (2-bit), 6.7 TB/s
// (4-bit); the cooperative bulk-copy kernel above stays at 3.8 TB/s there (its ring alone, math removed, moves
// 4.4 TB/s) but is the faster one for a single layer, where nothing is steady and latency is everything
// (4096 x 4096: 4.1 us against 8.7 us).
// ---------------------------------------------------------------------------------------------
constexpr int GS_WARPS = 8;            // per CTA; 3 CTAs per SM
constexpr int GS_D = 8;                // super-blocks in flight per warp

template <int BITS, int NT8>
__global__ void __launch_bounds__(GS_WARPS * 32, 3)
qgemv_i8_stream_kernel(const uint32_t* __restrict__ q, const __half* __restrict__ x, const float* __restrict__ scales,
                       const float* __restrict__ zeros, const __half* __restrict__ bias, __half* __restrict__ z, int M,
                       int K, int N) {
  constexpr int W = GS_WARPS, D = BITS == 2 ? GS_D : GS_D / 2;
  constexpr float HI_ROW_SCALE = BITS == 2 ? 0.25f : 0.0625f;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int KSB = K >> 7, NRB = N >> 4;
  const int ncol = GV_LIMBS * M;
  const int lld = K + 32;
  const int warps_total = gridDim.x * W;
  const int nsb_pad = (KSB + D - 1) / D * D;              // slot = sb % D, the same in every row block

  int8_t* limbs = reinterpret_cast<int8_t*>(smem_raw);
  float* tokf = reinterpret_cast<float*>(smem_raw + (((size_t)ncol * lld + 15) & ~(size_t)15));
  float* wred = tokf + 16;

  // ---- the ring: slot d holds super-block sb (sb % D == d) of the current or the next row block ----
  GvRegs<BITS> ring[D];
  const int rb0 = blockIdx.x * W + warp;
  auto fetch = [&](int rb, int sb, GvRegs<BITS>& dst) {
    if (rb < NRB && sb < KSB) gv_load<BITS>(q + ((int64_t)rb * KSB + sb) * sb_words(BITS), lane, dst);
  };
#pragma unroll
  for (int d = 0; d < D; ++d) fetch(rb0, d, ring[d]);     // weights first: independent of the previous kernel
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");

  gv_quantize_tokens<W>(x, M, K, limbs, lld, tokf, wred, tid, warp, lane);

  for (int rb = rb0; rb < NRB; rb += warps_total) {
    const int n0 = rb * 16 + g;
    const float sc0 = __ldg(scales + n0), sc1 = __ldg(scales + n0 + 8);
    const float ze0 = __ldg(zeros + n0), ze1 = __ldg(zeros + n0 + 8);
    const float bi0 = bias ? __half2float(__ldg(bias + n0)) : 0.f, bi1 = bias ? __half2float(__ldg(bias + n0 + 8)) : 0.f;
    int acc[NT8][2][4];
#pragma unroll
    for (int b = 0; b < NT8; ++b)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[b][0][c] = acc[b][1][c] = 0;

    for (int sb0 = 0; sb0 < nsb_pad; sb0 += D) {
#pragma unroll
      for (int d = 0; d < D; ++d) {
        const int sb = sb0 + d;
        if (sb < KSB) {
          const int8_t* lk = limbs + sb * 128 + 8 * t;
          uint32_t xb[4][NT8][2];
#pragma unroll
          for (int ch = 0; ch < 4; ++ch)
#pragma unroll
            for (int nt = 0; nt < NT8; ++nt) {
              const uint2 v = *reinterpret_cast<const uint2*>(lk + (size_t)min(nt * 8 + g, ncol - 1) * lld + ch * 32);
              xb[ch][nt][0] = v.x; xb[ch][nt][1] = v.y;
            }
          auto do_chunk = [&](auto chc) {
            constexpr int CH = decltype(chc)::value;
            uint32_t a[4];
            gv_expand_i8<BITS, CH>(ring[d], a);
#pragma unroll
            for (int nt = 0; nt < NT8; ++nt) imma16832(acc[nt][CH & 1], a, xb[CH][nt]);
          };
          do_chunk(std::integral_constant<int, 0>{});
          do_chunk(std::integral_constant<int, 1>{});
          do_chunk(std::integral_constant<int, 2>{});
          do_chunk(std::integral_constant<int, 3>{});
        }
        // refill the slot with the super-block D ahead, possibly in this warp's next row block
        int frb = rb, fsb = sb + D;
        if (fsb >= nsb_pad) { fsb -= nsb_pad; frb += warps_total; }
        fetch(frb, fsb, ring[d]);
      }
    }

    // ---- epilogue inside the warp: limb column c of a token sits in lane t = (c % 8) / 2, register c % 2 ----
#pragma unroll
    for (int tok = 0; tok < (NT8 == 1 ? 2 : 5); ++tok) {
      if (tok < M) {
        float dot0 = 0.f, dot1 = 0.f;                     // rows g and g+8
#pragma unroll
        for (int l = 0; l < GV_LIMBS; ++l) {
          const int col = GV_LIMBS * tok + l, nt = col >> 3, cc = col & 7, st = cc >> 1, reg = cc & 1;
          const int v0 = acc[nt][0][reg] + acc[nt][1][reg], v1 = acc[nt][0][2 + reg] + acc[nt][1][2 + reg];
          const float f0 = (float)__shfl_sync(0xffffffffu, v0, 4 * g + st);
          const float f1 = (float)__shfl_sync(0xffffffffu, v1, 4 * g + st);
          const float wgt = l == 0 ? 65536.f : (l == 1 ? 256.f : 1.f);
          dot0 += wgt * f0;
          dot1 += wgt * f1;
        }
        if (t == 0) {
          const float sm = tokf[2 * tok], S = tokf[2 * tok + 1];
          z[(int64_t)tok * N + n0] = __float2half_rn(sc0 * (sm * dot0) - ze0 * S + bi0);
          z[(int64_t)tok * N + n0 + 8] = __float2half_rn(sc1 * (sm * HI_ROW_SCALE * dot1) - ze1 * S + bi1);
        }
      }
    }
  }
}

template <int BITS, int NT8>
static int launch_gv_i8_stream(const QuipLinearDesc* d, const __half* x, const __half* bias, __half* z, int M,
                               cudaStream_t s) {
  const size_t limb_bytes = ((size_t)GV_LIMBS * M * (d->K + 32) + 15) & ~(size_t)15;
  const size_t smem = limb_bytes + (size_t)(16 + 10 * GS_WARPS) * sizeof(float);
  auto kern = qgemv_i8_stream_kernel<BITS, NT8>;
  const int grid = std::min(blocks_per_sm((const void*)kern, GS_WARPS * 32, smem) * num_sms(), ceil_div(d->N / 16, GS_WARPS));
  return launch("qgemv_i8_stream_kernel", kern, grid, GS_WARPS * 32, smem, s, true,
                reinterpret_cast<const uint32_t*>(d->qweight), x, d->scales, d->zeros, bias, z, M, d->K, d->N);
}

static bool gv_stream_fits(int K, int M) {
  return (size_t)GV_LIMBS * M * (K + 32) + 1024 <= (size_t)48 * 1024;      // four CTAs per SM
}

template <int BITS, int NT8, int RBC, int CW>
static int launch_gv_i8_tma(const QuipLinearDesc* d, const __half* x, const __half* bias, __half* z, int M,
                            cudaStream_t s) {
  constexpr int COLS = 8 * NT8, ROWS = 16 * RBC, RLD = ROWS + 4;
  constexpr size_t STAGE_BYTES = (size_t)GT_STAGE_SB * sb_words(BITS) * 4;
  const size_t limb_bytes = ((size_t)GV_LIMBS * M * (d->K + 32) + 15) & ~(size_t)15;
  const size_t fixed = limb_bytes + (size_t)(2 * CW * COLS * RLD) * sizeof(int) + (size_t)(16 + 10 * CW) * sizeof(float);
  const size_t budget = 227 * 1024 - 256;
  int ns = fixed + 64 < budget ? (int)((budget - fixed - 64) / (STAGE_BYTES + 16)) : 0;
  if (ns > 12) ns = 12;
  QUIP_CHECK_ARG(ns >= 2 * RBC, "qgemv: K=%d with %d tokens leaves no room for the weight ring", d->K, M);
  const size_t smem = (size_t)ns * STAGE_BYTES + fixed + (size_t)(2 * ns + 4) * sizeof(uint64_t);
  const int grid = std::min(ceil_div(d->N / 16, RBC), num_sms());
  return launch("qgemv_i8_tma_kernel", qgemv_i8_tma_kernel<BITS, NT8, RBC, CW>, grid, gt_threads(CW), smem, s, true,
                reinterpret_cast<const uint32_t*>(d->qweight), x, d->scales, d->zeros, bias, z, M, d->K, d->N, ns);
}

// does the bulk-copy kernel have room for at least a minimal ring next to the token bytes?
static bool gv_tma_fits(int K, int M, int bits, int nt8, int rbc, int cw) {
  const size_t stage = (size_t)GT_STAGE_SB * sb_words(bits) * 4;
  const size_t fixed = (size_t)GV_LIMBS * M * (K + 32) + (size_t)(2 * cw * 8 * nt8 * (16 * rbc + 4)) * 4 + 1024;
  return fixed + (size_t)(2 * rbc + 2) * (stage + 16) <= (size_t)227 * 1024 - 256;
}

// shared memory of the register-ring int8 kernel (three token bytes per k + reduction buffers)
static bool gv_i8_ldg_fits(int K, int M, int nt8) {
  const size_t smem = (size_t)GV_LIMBS * M * (K + 32) + (size_t)(2 * GV_WARPS * 8 * nt8 * 36) * sizeof(int) + 1024;
  return smem <= (size_t)227 * 1024 - 256;
}
// ... and of the fp16 kernel (one fp16 per k per token)
static bool gv_f16_fits(int K, int M) {
  const size_t smem = (size_t)M * (K + GV_XPAD) * sizeof(__half) +
                      (size_t)(2 * GV_WARPS * 8 * 36 + GV_WARPS * 16) * sizeof(float) + 16;
  return smem <= 200 * 1024;
}

// Can a whole-K kernel take M tokens of this K?  (Llama-2-70B's down_proj, K = 28672, fits three tokens; above
// that the caller uses the split-K kernel.)
bool qgemv_fits(int K, int M, int bits) {
  if (M > 8 || K < 128 * GV_WARPS) return false;
  if (g_gv_int && bits != 3 && M <= 5 && (gv_i8_ldg_fits(K, M, M <= 2 ? 1 : 2) || gv_tma_fits(K, M, bits, M <= 2 ? 1 : 2, 1, 8)))
    return true;
  return gv_f16_fits(K, M);
}

int qgemv(const QuipLinearDesc* d, const __half* x, const __half* bias, __half* z, int M, cudaStream_t s) {
  QUIP_CHECK_ARG(M >= 1 && M <= 8, "qgemv handles 1..8 tokens (got %d)", M);
  QUIP_CHECK_ARG(qgemv_fits(d->K, M, d->bits), "qgemv: K=%d with %d tokens does not fit shared memory", d->K, M);
  int rbc = g_gv_rbc;
  if (rbc != 1 && rbc != 2) rbc = (d->N / 16 >= 4 * num_sms()) ? 2 : 1;
  if (g_gv_int && d->bits != 3 && M <= 5) {
    const int nt8 = M <= 2 ? 1 : 2;
    if (g_gv_tma && g_gv_stream && d->N / 16 >= g_gv_stream * num_sms() && gv_stream_fits(d->K, M)) {
      // many row blocks per warp slot (stacked / grouped matrices): every warp streams whole row blocks
      if (d->bits == 2 && nt8 == 1) return launch_gv_i8_stream<2, 1>(d, x, bias, z, M, s);
      if (d->bits == 2 && nt8 == 2) return launch_gv_i8_stream<2, 2>(d, x, bias, z, M, s);
      if (d->bits == 4 && nt8 == 1) return launch_gv_i8_stream<4, 1>(d, x, bias, z, M, s);
      if (d->bits == 4 && nt8 == 2) return launch_gv_i8_stream<4, 2>(d, x, bias, z, M, s);
    }
    if (g_gv_tma) {
      int trbc = g_gv_rbc;
      if (trbc != 1 && trbc != 2) trbc = 2;
      int cw = g_gv_cw == 8 ? 8 : 16;
      if (cw == 16 && !gv_tma_fits(d->K, M, d->bits, nt8, trbc, 16)) cw = 8;      // smaller reduction buffers
      if (trbc == 2 && !gv_tma_fits(d->K, M, d->bits, nt8, 2, cw)) trbc = 1;
      if (gv_tma_fits(d->K, M, d->bits, nt8, trbc, cw)) {
#define QUIP_GVT(B, T)                                                                      \
  if (d->bits == B && nt8 == T) {                                                           \
    if (cw == 8) {                                                                          \
      if (trbc == 2) return launch_gv_i8_tma<B, T, 2, 8>(d, x, bias, z, M, s);              \
      return launch_gv_i8_tma<B, T, 1, 8>(d, x, bias, z, M, s);                             \
    }                                                                                       \
    if (trbc == 2) return launch_gv_i8_tma<B, T, 2, 16>(d, x, bias, z, M, s);               \
    return launch_gv_i8_tma<B, T, 1, 16>(d, x, bias, z, M, s);                              \
  }
        QUIP_GVT(2, 1) QUIP_GVT(2, 2) QUIP_GVT(4, 1) QUIP_GVT(4, 2)
#undef QUIP_GVT
      }
    }
#define QUIP_GVI(B, T, DD)                                                                  \
  if (d->bits == B && nt8 == T && gv_i8_ldg_fits(d->K, M, T)) {                             \
    if (rbc == 2) return launch_gv_i8<B, T, 2, DD>(d, x, bias, z, M, s);                    \
    return launch_gv_i8<B, T, 1, 2 * DD>(d, x, bias, z, M, s);                              \
  }
    QUIP_GVI(2, 1, 4) QUIP_GVI(2, 2, 4) QUIP_GVI(4, 1, 2) QUIP_GVI(4, 2, 2)
#undef QUIP_GVI
  }
#define QUIP_GV(B, DD)                                                                      \
  if (d->bits == B) {                                                                       \
    if (rbc == 2) return launch_gv<B, 1, 2, DD>(d, x, bias, z, M, s);                       \
    return launch_gv<B, 1, 1, 2 * DD>(d, x, bias, z, M, s);                                 \
  }
  QUIP_CHECK_ARG(gv_f16_fits(d->K, M), "qgemv: K=%d with %d tokens does not fit shared memory", d->K, M);
  QUIP_GV(2, 2) QUIP_GV(3, 2) QUIP_GV(4, 1)
#undef QUIP_GV
  set_error("qgemv: unsupported bits=%d", d->bits);
  return QUIP_ERR_UNSUPPORTED;
}

}  // namespace quip
