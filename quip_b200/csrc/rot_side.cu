// One whole incoherence side in one kernel, for many tokens (prefill / the eval loop's M = 2048):
//
//   K side:  x2 = pass1(pass0( (x * 1/s)[idx] )),  (+ the row sums of x2 the asymmetric epilogue needs)
//   N side:  y  = pass1(pass0(z))[idx] + bias
//
// (reference: one call of mul_ortho_butterfly, method.py:46-67, plus the scaleWH division of
// method.py:202-204 on the K side and the bias on the N side.)  As separate kernels -- gather, strided
// pass, contiguous pass -- each step is a full HBM round trip of the (M, n) activations: 96 MB and ~50 us per
// 4096-wide side at M = 2048, a third of the step.  Here a CTA keeps 16 token rows in shared memory for
// the whole side: x is read once and x2 written once; the factors (1 MiB per side) come from L2, stored a second
// time in tensor-core fragment order (QuipPass.factors_frag) so that a warp fetches 512 contiguous bytes per load
// -- read row-major, every fragment load touched eight cache lines and the load pipe, not the tensor pipe, set the pace.
//
// Shared-memory layout.  A side of n = PA * PB features is a PA x PB matrix per token (layout index
// l = a * PB + b).  The "strided" pass multiplies columns (blocks of PA features, stride PB) and the
// "contiguous" pass rows (blocks of PB).  A tensor-core A-fragment register wants two k-adjacent values
// of one token in one 32-bit word, and k runs along a in one pass and along b in the other.  So rows are
// stored in pairs: word (u, b) = { (a = 2u, b), (a = 2u+1, b) }.  The column pass reads and writes whole
// words (k pairs are a pairs); the row pass handles row blocks 2u and 2u+1 together, splits two words into
// the two blocks' fragments with one PRMT each, and packs its outputs back from the two blocks' accumulators.
// Both passes run in place (a block only touches its own column / row pair), with 32-bit accesses only.
#include "common.cuh"

namespace quip {

constexpr int SD_TOK = 16;             // token rows per CTA = the MMA M
constexpr int SD_WARPS = 16;

template <int PA, int PB>
struct SideCfg {
  static constexpr int N = PA * PB;
  static constexpr int SU = PB + 2;                                   // words per row pair (+2: column pass lanes t -> banks 2t)
  static constexpr int R0 = (PA / 2) * SU;
  static constexpr int R = R0 + ((8 - R0 % 32) + 32) % 32;            // words per token row, = 8 mod 32
  static constexpr size_t T_BYTES = (size_t)SD_TOK * R * 4;
  static constexpr size_t S_BYTES = (size_t)8 * N * sizeof(__half);   // eight staging rows (input gather)
  static constexpr size_t SMEM = T_BYTES + S_BYTES + SD_TOK * SD_WARPS * sizeof(float);
};

__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
  __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}

// factor words of n-tile nt, k pair j of one block in fragment order (include/quip_b200.h): one LDG.128 per lane,
// 512 contiguous bytes per warp
template <int P>
__device__ __forceinline__ uint4 frag_load(const uint4* __restrict__ blk, int nt, int j, int lane) {
  return __ldg(blk + (nt * (P / 32) + j) * 32 + lane);
}

// The passes run as a flat sequence of units (block, group of n-tiles) per warp; the factor words of unit i+1 are
// requested before the MMAs of unit i, across block boundaries, and the first unit of a pass is requested by the
// caller before the barrier (or the stage-in) that precedes the pass: the L2 latency is paid once per pass.

// ---- column pass: blocks b (PB of them), k = a (PA), factor F[b][i][a] ----
template <int PA, int PB>
struct ColPass {
  using C = SideCfg<PA, PB>;
  static constexpr int KS = PA / 16, J = PA / 32, NT = PA / 8, G = 4, GROUPS = NT / G;
  static constexpr int NBW = (PB + SD_WARPS - 1) / SD_WARPS;          // blocks per warp
  static constexpr int UNITS = NBW * GROUPS;
  uint4 bf[G][J];

  __device__ __forceinline__ void fetch(const uint4* __restrict__ F, int shared, int warp, int lane, int unit, uint4 (&dst)[G][J]) {
    const int b = warp + (unit / GROUPS) * SD_WARPS, grp = unit % GROUPS;
    if (unit < UNITS && b < PB) {
      const uint4* Fb = F + (size_t)(shared ? 0 : b) * (PA * PA / 8);
#pragma unroll
      for (int q = 0; q < G; ++q)
#pragma unroll
        for (int j = 0; j < J; ++j) dst[q][j] = frag_load<PA>(Fb, grp * G + q, j, lane);
    }
  }
  __device__ __forceinline__ void prefetch(const uint4* __restrict__ F, int shared, int warp, int lane) { fetch(F, shared, warp, lane, 0, bf); }

  __device__ __forceinline__ void run(uint32_t* T, const uint4* __restrict__ F, int shared, int warp, int lane) {
    const int g = lane >> 2, t = lane & 3;
    uint32_t a[KS][4];
#pragma unroll 1
    for (int unit = 0; unit < UNITS; ++unit) {
      const int b = warp + (unit / GROUPS) * SD_WARPS, grp = unit % GROUPS;
      uint4 nx[G][J];
      fetch(F, shared, warp, lane, unit + 1, nx);
      if (b < PB) {
        if (grp == 0) {
#pragma unroll
          for (int ks = 0; ks < KS; ++ks) {
            const uint32_t* w = T + g * C::R + (8 * ks + t) * C::SU + b;
            a[ks][0] = w[0];
            a[ks][1] = w[8 * C::R];
            a[ks][2] = w[4 * C::SU];
            a[ks][3] = w[8 * C::R + 4 * C::SU];
          }
        }
#pragma unroll
        for (int q = 0; q < G; ++q) {
          float c[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int j = 0; j < J; ++j) {
            const uint32_t b0[2] = {bf[q][j].x, bf[q][j].y}, b1[2] = {bf[q][j].z, bf[q][j].w};
            mma16816(c, a[2 * j], b0);
            mma16816(c, a[2 * j + 1], b1);
          }
          // outputs i = 8 nt + 2t, +1 of tokens g / g+8: one word each
          uint32_t* w = T + g * C::R + (4 * (grp * G + q) + t) * C::SU + b;
          w[0] = pack_h2(c[0], c[1]);
          w[8 * C::R] = pack_h2(c[2], c[3]);
        }
      }
#pragma unroll
      for (int q = 0; q < G; ++q)
#pragma unroll
        for (int j = 0; j < J; ++j) bf[q][j] = nx[q][j];
    }
  }
};

// ---- row pass: row blocks 2u, 2u+1 together, k = b (PB), factors F[a][i][b] ----
template <int PA, int PB>
struct RowPass {
  using C = SideCfg<PA, PB>;
  static constexpr int KS = PB / 16, J = PB / 32, NT = PB / 8, G = 2, GROUPS = NT / G;
  static constexpr int NUW = (PA / 2 + SD_WARPS - 1) / SD_WARPS;      // row pairs per warp
  static constexpr int UNITS = NUW * GROUPS;
  uint4 bf0[G][J], bf1[G][J];

  __device__ __forceinline__ void fetch(const uint4* __restrict__ F, int shared, int warp, int lane, int unit, uint4 (&d0)[G][J],
                                        uint4 (&d1)[G][J]) {
    const int u = warp + (unit / GROUPS) * SD_WARPS, grp = unit % GROUPS;
    if (unit < UNITS && u < PA / 2) {
      const uint4* F0 = F + (size_t)(shared ? 0 : 2 * u) * (PB * PB / 8);
      const uint4* F1 = F + (size_t)(shared ? 0 : 2 * u + 1) * (PB * PB / 8);
#pragma unroll
      for (int q = 0; q < G; ++q)
#pragma unroll
        for (int j = 0; j < J; ++j) {
          d0[q][j] = frag_load<PB>(F0, grp * G + q, j, lane);
          d1[q][j] = frag_load<PB>(F1, grp * G + q, j, lane);
        }
    }
  }
  __device__ __forceinline__ void prefetch(const uint4* __restrict__ F, int shared, int warp, int lane) { fetch(F, shared, warp, lane, 0, bf0, bf1); }

  __device__ __forceinline__ void run(uint32_t* T, const uint4* __restrict__ F, int shared, int warp, int lane) {
    const int g = lane >> 2, t = lane & 3;
    uint32_t a0[KS][4], a1[KS][4];                        // fragments of row block 2u / 2u+1
#pragma unroll 1
    for (int unit = 0; unit < UNITS; ++unit) {
      const int u = warp + (unit / GROUPS) * SD_WARPS, grp = unit % GROUPS;
      uint4 nx0[G][J], nx1[G][J];
      fetch(F, shared, warp, lane, unit + 1, nx0, nx1);
      if (u < PA / 2) {
        if (grp == 0) {
#pragma unroll
          for (int ks = 0; ks < KS; ++ks) {
            const uint32_t* w = T + g * C::R + u * C::SU + 16 * ks + 2 * t;
            const uint32_t w00 = w[0], w01 = w[1], w10 = w[8 * C::R], w11 = w[8 * C::R + 1];
            const uint32_t w20 = w[8], w21 = w[9], w30 = w[8 * C::R + 8], w31 = w[8 * C::R + 9];
            a0[ks][0] = __byte_perm(w00, w01, 0x5410); a1[ks][0] = __byte_perm(w00, w01, 0x7632);
            a0[ks][1] = __byte_perm(w10, w11, 0x5410); a1[ks][1] = __byte_perm(w10, w11, 0x7632);
            a0[ks][2] = __byte_perm(w20, w21, 0x5410); a1[ks][2] = __byte_perm(w20, w21, 0x7632);
            a0[ks][3] = __byte_perm(w30, w31, 0x5410); a1[ks][3] = __byte_perm(w30, w31, 0x7632);
          }
        }
#pragma unroll
        for (int q = 0; q < G; ++q) {
          float c0[4] = {0.f, 0.f, 0.f, 0.f}, c1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int j = 0; j < J; ++j) {
            const uint32_t p0[2] = {bf0[q][j].x, bf0[q][j].y}, p1[2] = {bf0[q][j].z, bf0[q][j].w};
            const uint32_t r0[2] = {bf1[q][j].x, bf1[q][j].y}, r1[2] = {bf1[q][j].z, bf1[q][j].w};
            mma16816(c0, a0[2 * j], p0);
            mma16816(c0, a0[2 * j + 1], p1);
            mma16816(c1, a1[2 * j], r0);
            mma16816(c1, a1[2 * j + 1], r1);
          }
          // outputs i = 8 nt + 2t, +1: word (u, i) = { block 2u, block 2u+1 }
          uint32_t* w = T + g * C::R + u * C::SU + 8 * (grp * G + q) + 2 * t;
          w[0] = pack_h2(c0[0], c1[0]);
          w[1] = pack_h2(c0[1], c1[1]);
          w[8 * C::R] = pack_h2(c0[2], c1[2]);
          w[8 * C::R + 1] = pack_h2(c0[3], c1[3]);
        }
      }
#pragma unroll
      for (int q = 0; q < G; ++q)
#pragma unroll
        for (int j = 0; j < J; ++j) { bf0[q][j] = nx0[q][j]; bf1[q][j] = nx1[q][j]; }
    }
  }
};

// half-word address of layout element l = a * PB + b inside a token row
template <int PA, int PB>
__device__ __forceinline__ int half_index(int l) {
  const int a = l / PB, b = l - a * PB;
  return 2 * ((a >> 1) * SideCfg<PA, PB>::SU + b) + (a & 1);
}

template <int PA, int PB>
__global__ void __launch_bounds__(SD_WARPS * 32)
side_fused_kernel(const __half* __restrict__ in, __half* __restrict__ out, int64_t M, const int32_t* __restrict__ in_idx,
                  const float* __restrict__ in_scale, const int32_t* __restrict__ out_idx,
                  const __half* __restrict__ out_bias, const uint4* __restrict__ F_col, int col_shared,
                  const uint4* __restrict__ F_row, int row_shared, int col_first, float* __restrict__ xsum) {
  using C = SideCfg<PA, PB>;
  constexpr int N = C::N, NTH = SD_WARPS * 32;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint32_t* T = reinterpret_cast<uint32_t*>(smem_raw);
  __half* T16 = reinterpret_cast<__half*>(smem_raw);
  __half* S = reinterpret_cast<__half*>(smem_raw + C::T_BYTES);        // [2][N] staging rows
  float* wsum = reinterpret_cast<float*>(smem_raw + C::T_BYTES + C::S_BYTES);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t m0 = (int64_t)blockIdx.x * SD_TOK;
  const int nr = (int)((M - m0) < SD_TOK ? (M - m0) : SD_TOK);

  // the first pass's first factor words travel under the stage-in
  ColPass<PA, PB> colp;
  RowPass<PA, PB> rowp;
  if (col_first) colp.prefetch(F_col, col_shared, warp, lane);
  else rowp.prefetch(F_row, row_shared, warp, lane);

  // ---------------- stage in ----------------
  if (in_idx || in_scale) {
    // gather: word (u, b) of a row <- x[idx[2u*PB + b]], x[idx[(2u+1)*PB + b]] (times 1/s), via a staged copy of the row
    constexpr int WPT = (N / 2 + NTH - 1) / NTH;           // words per thread per row
    int src0[WPT], src1[WPT];
    float sc0[WPT], sc1[WPT];
#pragma unroll
    for (int i = 0; i < WPT; ++i) {
      const int w = tid + i * NTH;
      src0[i] = src1[i] = 0; sc0[i] = sc1[i] = 1.f;
      if (w < N / 2) {
        const int u = w / PB, b = w - u * PB;
        const int l0 = (2 * u) * PB + b, l1 = l0 + PB;
        src0[i] = in_idx ? __ldg(in_idx + l0) : l0;
        src1[i] = in_idx ? __ldg(in_idx + l1) : l1;
        if (in_scale) { sc0[i] = __ldg(in_scale + src0[i]); sc1[i] = __ldg(in_scale + src1[i]); }
      }
    }
    // rows travel eight at a time (all requested at once), the second eight while the first are permuted
    constexpr int CHT = (N / 8 + NTH - 1) / NTH;           // 16-byte chunks per thread per row
    uint4 v[8][CHT];
    auto request = [&](int r0) {
#pragma unroll
      for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int i = 0; i < CHT; ++i) {
          const int c = tid + i * NTH;
          v[r][i] = make_uint4(0u, 0u, 0u, 0u);
          if (c < N / 8 && r0 + r < nr) v[r][i] = ldg_nc_v4(in + (m0 + r0 + r) * N + 8 * c);
        }
    };
    auto park = [&]() {
#pragma unroll
      for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int i = 0; i < CHT; ++i) {
          const int c = tid + i * NTH;
          if (c < N / 8) reinterpret_cast<uint4*>(S + (size_t)r * N)[c] = v[r][i];
        }
    };
    auto permute = [&](int r0) {
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const __half* row = S + (size_t)r * N;
#pragma unroll
        for (int i = 0; i < WPT; ++i) {
          const int w = tid + i * NTH;
          if (w < N / 2) {
            const int u = w / PB, b = w - u * PB;
            float v0 = __half2float(row[src0[i]]), v1 = __half2float(row[src1[i]]);
            if (in_scale) { v0 *= sc0[i]; v1 *= sc1[i]; }
            T[(r0 + r) * C::R + u * C::SU + b] = pack_h2(v0, v1);
          }
        }
      }
    };
    request(0);
    park();
    __syncthreads();
    request(8);
    permute(0);
    __syncthreads();
    park();
    __syncthreads();
    permute(8);
    __syncthreads();
  } else {
    // plain rows: a thread merges 8 features of rows 2u and 2u+1 into 8 words; all loads of a batch first
    constexpr int ITEMS = SD_TOK * (PA / 2) * (PB / 8), PER = (ITEMS + NTH - 1) / NTH, BATCH = PER < 4 ? PER : 4;
#pragma unroll 1
    for (int i0 = 0; i0 < PER; i0 += BATCH) {
      uint4 lo[BATCH], hi[BATCH];
#pragma unroll
      for (int i = 0; i < BATCH; ++i) {
        const int c = tid + (i0 + i) * NTH;
        const int r = c / ((PA / 2) * (PB / 8)), rem = c - r * ((PA / 2) * (PB / 8));
        const int u = rem / (PB / 8), b0 = (rem - u * (PB / 8)) * 8;
        lo[i] = hi[i] = make_uint4(0u, 0u, 0u, 0u);
        if (i0 + i < PER && c < ITEMS && r < nr) {
          lo[i] = ldg_nc_v4(in + (m0 + r) * N + (size_t)(2 * u) * PB + b0);
          hi[i] = ldg_nc_v4(in + (m0 + r) * N + (size_t)(2 * u + 1) * PB + b0);
        }
      }
#pragma unroll
      for (int i = 0; i < BATCH; ++i) {
        const int c = tid + (i0 + i) * NTH;
        if (i0 + i < PER && c < ITEMS) {
          const int r = c / ((PA / 2) * (PB / 8)), rem = c - r * ((PA / 2) * (PB / 8));
          const int u = rem / (PB / 8), b0 = (rem - u * (PB / 8)) * 8;
          uint32_t* w = T + r * C::R + u * C::SU + b0;
          w[0] = __byte_perm(lo[i].x, hi[i].x, 0x5410); w[1] = __byte_perm(lo[i].x, hi[i].x, 0x7632);
          w[2] = __byte_perm(lo[i].y, hi[i].y, 0x5410); w[3] = __byte_perm(lo[i].y, hi[i].y, 0x7632);
          w[4] = __byte_perm(lo[i].z, hi[i].z, 0x5410); w[5] = __byte_perm(lo[i].z, hi[i].z, 0x7632);
          w[6] = __byte_perm(lo[i].w, hi[i].w, 0x5410); w[7] = __byte_perm(lo[i].w, hi[i].w, 0x7632);
        }
      }
    }
    __syncthreads();
  }

  // ---------------- the two passes, in place ----------------
  if (col_first) {
    colp.run(T, F_col, col_shared, warp, lane);
    rowp.prefetch(F_row, row_shared, warp, lane);
    __syncthreads();
    rowp.run(T, F_row, row_shared, warp, lane);
  } else {
    rowp.run(T, F_row, row_shared, warp, lane);
    colp.prefetch(F_col, col_shared, warp, lane);
    __syncthreads();
    colp.run(T, F_col, col_shared, warp, lane);
  }
  __syncthreads();

  // ---------------- stage out ----------------
  if (out_idx || out_bias) {
    constexpr int CPT = (N / 8 + NTH - 1) / NTH;           // 8-feature chunks per thread per row
    int hidx[CPT][8];
    float bs[CPT][8];
#pragma unroll
    for (int i = 0; i < CPT; ++i) {
      const int c = tid + i * NTH;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        hidx[i][e] = 0; bs[i][e] = 0.f;
        if (c < N / 8) {
          const int j = 8 * c + e;
          hidx[i][e] = half_index<PA, PB>(out_idx ? __ldg(out_idx + j) : j);
          if (out_bias) bs[i][e] = __half2float(__ldg(out_bias + j));
        }
      }
    }
    for (int r = 0; r < nr; ++r) {
      const __half* row = T16 + (size_t)r * 2 * C::R;
#pragma unroll
      for (int i = 0; i < CPT; ++i) {
        const int c = tid + i * NTH;
        if (c < N / 8) {
          __align__(16) __half v[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) v[e] = __float2half_rn(__half2float(row[hidx[i][e]]) + bs[i][e]);
          *reinterpret_cast<uint4*>(out + (m0 + r) * N + 8 * c) = *reinterpret_cast<const uint4*>(v);
        }
      }
    }
  } else {
    constexpr int CPR = PA * (PB / 8);                      // 8-feature chunks per row
    for (int r = 0; r < nr; ++r) {
      float s = 0.f;
      for (int c = tid; c < CPR; c += NTH) {
        const int a = c / (PB / 8), b0 = (c - a * (PB / 8)) * 8;
        const uint32_t* w = T + r * C::R + (a >> 1) * C::SU + b0;
        const uint32_t sel = (a & 1) ? 0x7632u : 0x5410u;
        uint4 v;
        v.x = __byte_perm(w[0], w[1], sel); v.y = __byte_perm(w[2], w[3], sel);
        v.z = __byte_perm(w[4], w[5], sel); v.w = __byte_perm(w[6], w[7], sel);
        *reinterpret_cast<uint4*>(out + (m0 + r) * N + (size_t)a * PB + b0) = v;
        const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
        for (int e = 0; e < 4; ++e) { const float2 f = __half22float2(h[e]); s += f.x + f.y; }
      }
      if (xsum) {                                          // fixed-order reduction: lanes, then warps
#pragma unroll
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) wsum[r * SD_WARPS + warp] = s;
      }
    }
    if (xsum) {
      __syncthreads();
      if (tid < nr) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < SD_WARPS; ++w) s += wsum[tid * SD_WARPS + w];
        xsum[m0 + tid] = s;
      }
    }
  }
}

template <int PA, int PB>
static int launch_side(const __half* in, __half* out, int64_t M, const int32_t* in_idx, const float* in_scale,
                       const int32_t* out_idx, const __half* out_bias, const QuipPass* col, const QuipPass* row,
                       int col_first, float* xsum, cudaStream_t s) {
  return launch("side_fused_kernel", side_fused_kernel<PA, PB>, (unsigned)ceil_div(M, SD_TOK), SD_WARPS * 32,
                SideCfg<PA, PB>::SMEM, s, false, in, out, M, in_idx, in_scale, out_idx, out_bias,
                (const uint4*)col->factors_frag, col->shared, (const uint4*)row->factors_frag, row->shared, col_first, xsum);
}

// Can this side (two passes) run as one fused kernel?  One strided pass of p = PA over PB blocks and one contiguous
// pass of p = PB over PA blocks, for an instantiated (PA, PB).
bool side_fused_ok(const QuipSide* sd, int n) {
  if (sd->n != n || sd->npass != 2) return false;
  const QuipPass& p0 = sd->pass[0];
  const QuipPass& p1 = sd->pass[1];
  const QuipPass* col = p0.strided ? &p0 : (p1.strided ? &p1 : nullptr);
  const QuipPass* row = p0.strided ? &p1 : &p0;
  if (!col || row->strided) return false;
  if (col->p != row->nblk || col->nblk != row->p) return false;
  if (!col->factors_frag || !row->factors_frag) return false;      // the caller did not provide fragment-order factors
  const int PA = col->p, PB = row->p;
  return (PA == 64 && PB == 64) || (PA == 32 && PB == 64) || (PA == 64 && PB == 32);
}

// in -> out through a whole side.  K side: in_idx / in_scale (gather + 1/s before the passes), xsum optional.
// N side: out_idx / out_bias (gather + bias after the passes).
int side_fused(const QuipSide* sd, const __half* in, __half* out, int64_t M, const int32_t* in_idx, const float* in_scale,
               const int32_t* out_idx, const __half* out_bias, float* xsum, cudaStream_t s) {
  const QuipPass& p0 = sd->pass[0];
  const QuipPass* col = p0.strided ? &sd->pass[0] : &sd->pass[1];
  const QuipPass* row = p0.strided ? &sd->pass[1] : &sd->pass[0];
  const int col_first = p0.strided ? 1 : 0;
  const int PA = col->p, PB = row->p;
  if (PA == 64 && PB == 64) return launch_side<64, 64>(in, out, M, in_idx, in_scale, out_idx, out_bias, col, row, col_first, xsum, s);
  if (PA == 32 && PB == 64) return launch_side<32, 64>(in, out, M, in_idx, in_scale, out_idx, out_bias, col, row, col_first, xsum, s);
  if (PA == 64 && PB == 32) return launch_side<64, 32>(in, out, M, in_idx, in_scale, out_idx, out_bias, col, row, col_first, xsum, s);
  set_error("fused side: unsupported block sizes %d x %d", PA, PB);
  return QUIP_ERR_UNSUPPORTED;
}

}  // namespace quip
