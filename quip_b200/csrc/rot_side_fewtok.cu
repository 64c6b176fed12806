// A whole incoherence side for a handful of tokens (decode, M <= 8) in ONE launch, without a grid-wide barrier.
//
// One side is two block-diagonal passes (reference mul_ortho_butterfly, method.py:46-67): the outputs of the first pass
// are regrouped -- every block of the second pass takes exactly one output from each block of the first (the (p1, p2)
// view is multiplied along its columns, then along its rows).  As separate kernels (rot_fewtok.cu) the regrouping is a
// kernel boundary: 2.2 us of dependent launch latency per pass, four passes per QuantLinear, more than the time the bytes
// take.  Here the CTA that owns a block c1 of the SECOND pass computes its own inputs: input j of block c1 is output
// i_j of first-pass block c0_j, i.e. ONE ROW of that block's factor times the block's inputs,
//
//     t[j]    = sum_k F0[c0_j][i_j][k] * in[ src(pos0(c0_j, k)) ]              (p1 dot products of length p0)
//     out[j'] = sum_j F1[c1][j'][j] * t[j]                                     (the second pass's block itself)
//
// No factor byte is read twice across the grid (row i_j of block c0_j belongs to block c1 alone); only the token vector
// (n values per token) is read by every CTA, from L2.  Second-pass blocks wider than SF_ROWS rows are cut into row tiles:
// those CTAs repeat the (small) first-pass dots of their block -- for the 688 x 688 blocks of an 11008 side that is 22 KB
// of 16-wide rows from a 352 KB array that lives in L2.
//
// Latency, not bytes, is what a decode-time kernel pays for.  Before griddepcontrol.wait -- i.e. while the previous kernel
// is still running -- a CTA requests every factor row it will use (cp.async into shared memory) and reads the gather
// index; after the wait it stages the token vector (16-byte loads), regroups it into first-pass block order through a
// 16-bit copy of the index (padded rows: conflict-free), and both passes run out of shared memory: one dependent global
// round trip (the tokens) instead of one per pass.
//
// Arithmetic: fp16 factors and tokens, float32 products and sums in a fixed order, the intermediate t kept in float32
// (one fp16 rounding fewer than the two-kernel route), output rounded to fp16 once (+ bias after the rounding, as the
// stand-alone gather adds it).  Fusions: in_idx / in_scale (K side: gather + 1/s), out_inv / out_bias (N side).
#include "common.cuh"

namespace quip {

namespace {

constexpr int SF_THREADS = 1024;      // the work is a long chain of short dependent steps: many warps hide each other's latencies
constexpr int SF_PL = 8;              // lanes per output row in the second pass
constexpr int SF_MAXTOK = 8;
constexpr int SF_MLP = 8;             // independent 16-byte loads a thread keeps in flight in the staging loops
constexpr int SF_ROWS = 32;           // second-pass output rows per CTA when its blocks are wider than 64

struct SidePassArg {
  const __half* F;                    // [shared ? 1 : nblk][p][p] row-major
  int p, nblk, strided, shared;
};

__device__ __forceinline__ int pos_of(const SidePassArg& ps, int blk, int j) { return ps.strided ? j * ps.nblk + blk : blk * ps.p + j; }

__device__ __forceinline__ void cp_async16(void* smem, const void* g) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem)), "l"(g) : "memory");
}

// Shared-memory plan (bytes, every section 16-byte aligned); the same arithmetic on the host decides whether a side fits.
struct SfPlan {
  int xld;                 // padded length of one first-pass block in xs0 (p0 + 2 halves: conflict-free transposing stores)
  size_t f0, f1, ts, od, xs0, tmp, sidx, total;
};
__host__ __device__ inline SfPlan sf_plan(int n, int p0, int nblk0, int p1, int M, int ndots, int nout) {
  SfPlan pl;
  pl.xld = p0 + 2;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 15) & ~(size_t)15; return o; };
  pl.f0 = take((size_t)ndots * p0 * 2);            // the first-pass factor rows this CTA consumes
  pl.f1 = take((size_t)nout * p1 * 2);             // its second-pass rows
  pl.ts = take((size_t)ndots * M * 4);             // second-pass inputs, float
  pl.od = take((size_t)nout * 8);                  // destination index and bias of every output row of this CTA
  pl.xs0 = take((size_t)M * nblk0 * pl.xld * 2);   // tokens in first-pass block order
  pl.tmp = take((size_t)M * n * 2);                // tokens as they lie in memory
  pl.sidx = take((size_t)n * 2);                   // feature of layout position q (n < 65536)
  pl.total = off;
  return pl;
}

// grid.x = work items: (group of `blocks_per_cta` second-pass blocks) x (row tile rt)
template <int M>
__global__ void __launch_bounds__(SF_THREADS)
side_fewtok_kernel(const __half* __restrict__ in, __half* __restrict__ out, int n, SidePassArg P0, SidePassArg P1,
                   const int32_t* __restrict__ in_idx, const float* __restrict__ in_scale,
                   const int32_t* __restrict__ out_inv, const __half* __restrict__ out_bias, int rows_per_cta, int blocks_per_cta) {
  extern __shared__ __align__(16) unsigned char sm_raw[];
  const int p0 = P0.p, p1 = P1.p;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int rtiles = (p1 + rows_per_cta - 1) / rows_per_cta;
  const int item = blockIdx.x;
  const int c1_first = (item / rtiles) * blocks_per_cta, rt = item % rtiles;
  const int ndots = blocks_per_cta * p1;
  const int nrows = min(rows_per_cta, p1 - rt * rows_per_cta);
  const int nout = blocks_per_cta * nrows;                                        // a multiple of 16
  const SfPlan pl = sf_plan(n, p0, P0.nblk, p1, M, ndots, blocks_per_cta * rows_per_cta);
  __half* F0s = reinterpret_cast<__half*>(sm_raw + pl.f0);                         // [ndots][p0]
  __half* F1s = reinterpret_cast<__half*>(sm_raw + pl.f1);                         // [nout][p1]
  float* ts = reinterpret_cast<float*>(sm_raw + pl.ts);                            // [ndots][M]
  int* dst_s = reinterpret_cast<int*>(sm_raw + pl.od);                             // [nout]
  float* bias_s = reinterpret_cast<float*>(dst_s + blocks_per_cta * rows_per_cta); // [nout]
  __half* xs0 = reinterpret_cast<__half*>(sm_raw + pl.xs0);                        // [M][nblk0][xld]
  __half* tmp = reinterpret_cast<__half*>(sm_raw + pl.tmp);                        // [M][n]
  uint16_t* sidx = reinterpret_cast<uint16_t*>(sm_raw + pl.sidx);                  // [n]

  // Index arithmetic without divisions (they dominated the instruction count of a first version): the second-pass block c1
  // takes element c1 of EVERY first-pass block, so input j of block c1 is row i = c1 of first-pass block c0 = j
  // (nblk0 == p1, nblk1 == p0); loops are two-dimensional (warp x lane) instead of flat with / and %.
  constexpr int NW = SF_THREADS / 32;
  const bool multi = blocks_per_cta > 1;                                          // only for 16-wide second-pass blocks

  // ---- everything that does not depend on the previous kernel is requested now: this CTA's factor rows travel to
  // shared memory (cp.async) and the gather index is read while the previous kernel drains ----
  {
    const int cpr0 = p0 >> 3;                                                     // 16-byte pieces per first-pass row
    for (int d = warp; d < ndots; d += NW) {
      const int bl = multi ? d / p1 : 0, j = d - bl * p1, c1 = c1_first + bl;
      if (c1 < P1.nblk) {
        const __half* src = P0.F + ((size_t)(P0.shared ? 0 : j) * p0 + c1) * p0;  // row c1 of first-pass block j
        for (int pc = lane; pc < cpr0; pc += 32) cp_async16(F0s + (size_t)d * p0 + 8 * pc, src + 8 * pc);
      }
    }
    const int cpr1 = p1 >> 3;
    for (int o = warp; o < nout; o += NW) {
      const int bl = multi ? o / nrows : 0, r = rt * rows_per_cta + (o - bl * nrows), c1 = c1_first + bl;
      if (c1 < P1.nblk) {
        const __half* src = P1.F + ((size_t)(P1.shared ? 0 : c1) * p1 + r) * p1;
        for (int pc = lane; pc < cpr1; pc += 32) cp_async16(F1s + (size_t)o * p1 + 8 * pc, src + 8 * pc);
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    for (int o = tid; o < nout; o += SF_THREADS) {                                // where the outputs go (scatter index, bias)
      const int bl = multi ? o / nrows : 0, r = rt * rows_per_cta + (o - bl * nrows), c1 = c1_first + bl;
      int dst = 0;
      float bs = 0.f;
      if (c1 < P1.nblk) {
        const int pos = pos_of(P1, c1, r);
        dst = out_inv ? __ldg(out_inv + pos) : pos;
        bs = out_bias ? __half2float(__ldg(out_bias + dst)) : 0.f;
      }
      dst_s[o] = dst;
      bias_s[o] = bs;
    }
    // the index: 16-byte loads, SF_MLP of them in flight per thread (a plain loop would pay one memory latency per turn)
    for (int base = tid; base < (n >> 2); base += SF_THREADS * SF_MLP) {
      int4 v[SF_MLP];
#pragma unroll
      for (int u = 0; u < SF_MLP; ++u) {
        const int c = base + u * SF_THREADS;
        v[u] = make_int4(4 * c, 4 * c + 1, 4 * c + 2, 4 * c + 3);
        if (in_idx && c < (n >> 2)) v[u] = __ldg(reinterpret_cast<const int4*>(in_idx) + c);
      }
#pragma unroll
      for (int u = 0; u < SF_MLP; ++u) {
        const int c = base + u * SF_THREADS;
        if (c < (n >> 2)) *reinterpret_cast<uint2*>(sidx + 4 * c) = make_uint2((uint32_t)v[u].x | ((uint32_t)v[u].y << 16),
                                                                                (uint32_t)v[u].z | ((uint32_t)v[u].w << 16));
      }
    }
  }
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");

  // ---- the tokens: 16-byte loads in memory order (times 1/s, rounded as the stand-alone gather rounds) ... ----
  for (int base = tid; base < M * (n >> 3); base += SF_THREADS * SF_MLP) {
    uint4 v[SF_MLP];
#pragma unroll
    for (int u = 0; u < SF_MLP; ++u) {
      const int c = base + u * SF_THREADS;
      if (c < M * (n >> 3)) v[u] = *reinterpret_cast<const uint4*>(in + (size_t)c * 8);      // row m = c / (n/8), features 8 (c % (n/8))
    }
#pragma unroll
    for (int u = 0; u < SF_MLP; ++u) {
      const int c = base + u * SF_THREADS;
      if (c < M * (n >> 3)) {
        if (in_scale) {
          const int f0 = (c % (n >> 3)) * 8;
          __half* h = reinterpret_cast<__half*>(&v[u]);
#pragma unroll
          for (int e = 0; e < 8; ++e) h[e] = __float2half_rn(__half2float(h[e]) * __ldg(in_scale + f0 + e));
        }
        *reinterpret_cast<uint4*>(tmp + (size_t)c * 8) = v[u];
      }
    }
  }
  __syncthreads();
  // ---- ... then into first-pass block order: xs0[m][c0][k] = x[m][idx[pos0(c0, k)]]: consecutive lanes take consecutive
  // layout positions q (index reads conflict-free); the row padding makes the transposing stores conflict-free too ----
  if (P0.strided) {                                                               // q = k * nblk0 + c0
    for (int k = warp; k < p0; k += NW)
      for (int c0 = lane; c0 < P0.nblk; c0 += 32) {
        const int src = sidx[k * P0.nblk + c0];
#pragma unroll
        for (int m = 0; m < M; ++m) xs0[((size_t)m * P0.nblk + c0) * pl.xld + k] = tmp[(size_t)m * n + src];
      }
  } else {                                                                        // q = c0 * p0 + k
    for (int c0 = warp; c0 < P0.nblk; c0 += NW)
      for (int k = lane; k < p0; k += 32) {
        const int src = sidx[c0 * p0 + k];
#pragma unroll
        for (int m = 0; m < M; ++m) xs0[((size_t)m * P0.nblk + c0) * pl.xld + k] = tmp[(size_t)m * n + src];
      }
  }
  asm volatile("cp.async.wait_all;" ::: "memory");
  __syncthreads();

  // ---- first pass, only the rows this CTA's second-pass blocks consume: `lpd` lanes per dot product ----
  const int lpd = p0 >= 64 ? 32 : (p0 >= 32 ? 16 : 8);                            // p0 is a multiple of 16
  const int dpw = 32 / lpd, sub = lane / lpd, ll = lane - sub * lpd;
  for (int d0 = warp * dpw; d0 < ndots; d0 += NW * dpw) {
    const int d = d0 + sub;
    const int bl = multi ? d / p1 : 0, j = d - bl * p1, c1 = c1_first + bl;
    float acc[M];
#pragma unroll
    for (int m = 0; m < M; ++m) acc[m] = 0.f;
    if (d < ndots && c1 < P1.nblk) {
      const __half* frow = F0s + (size_t)d * p0;
      const __half* xb = xs0 + (size_t)j * pl.xld;                                // first-pass block c0 = j
#pragma unroll 4
      for (int k = 2 * ll; k < p0; k += 2 * lpd) {
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(frow + k));
#pragma unroll
        for (int m = 0; m < M; ++m) {
          const float2 x = __half22float2(*reinterpret_cast<const __half2*>(xb + (size_t)m * P0.nblk * pl.xld + k));
          acc[m] = fmaf(f.y, x.y, fmaf(f.x, x.x, acc[m]));
        }
      }
    }
#pragma unroll
    for (int m = 0; m < M; ++m) {
      for (int o = lpd >> 1; o; o >>= 1) acc[m] += __shfl_xor_sync(0xffffffffu, acc[m], o);
    }
    if (ll == 0 && d < ndots) {
#pragma unroll
      for (int m = 0; m < M; ++m) ts[(size_t)d * M + m] = acc[m];
    }
  }
  __syncthreads();

  // ---- second pass: rows [rt * rows_per_cta, ...) of each of this CTA's blocks, a group of 4 lanes per output row ----
  for (int o4 = tid; o4 < nout * SF_PL; o4 += SF_THREADS) {                       // nout * SF_PL is a multiple of 128: whole warps
    const int o = o4 / SF_PL, part = o4 % SF_PL;
    const int bl = multi ? o / nrows : 0, r = rt * rows_per_cta + (o - bl * nrows), c1 = c1_first + bl;
    float acc[M];
#pragma unroll
    for (int m = 0; m < M; ++m) acc[m] = 0.f;
    const bool live = c1 < P1.nblk;
    if (live) {
      const __half* frow = F1s + (size_t)o * p1;
      const float* tb = ts + (size_t)bl * p1 * M;
#pragma unroll 2
      for (int k = 8 * part; k < p1; k += 8 * SF_PL) {                            // 16-byte pieces of the row, interleaved over the lanes
        const uint4 v = *reinterpret_cast<const uint4*>(frow + k);
        const __half2* h2 = reinterpret_cast<const __half2*>(&v);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 f = __half22float2(h2[e]);
#pragma unroll
          for (int m = 0; m < M; ++m)
            acc[m] = fmaf(f.y, tb[(size_t)(k + 2 * e + 1) * M + m], fmaf(f.x, tb[(size_t)(k + 2 * e) * M + m], acc[m]));
        }
      }
    }
#pragma unroll
    for (int m = 0; m < M; ++m) {
#pragma unroll
      for (int sh = SF_PL / 2; sh; sh >>= 1) acc[m] += __shfl_xor_sync(0xffffffffu, acc[m], sh);
    }
    if (live && part == 0) {
      const int dst = dst_s[o];
      const float bs = bias_s[o];
#pragma unroll
      for (int m = 0; m < M; ++m) {
        const float v = out_bias ? __half2float(__float2half_rn(acc[m])) + bs : acc[m];
        out[(size_t)m * n + dst] = __float2half_rn(v);
      }
    }
  }
}

}  // namespace

constexpr size_t SF_SMEM_MAX = 224 * 1024;
static int sf_blocks_per_cta(int p1) { return p1 <= 16 ? 4 : 1; }
static int sf_rows_per_cta(int p1) { return p1 <= 64 ? p1 : (p1 > 512 ? SF_ROWS : 64); }
static size_t side_fewtok_smem(int n, const QuipPass& a, const QuipPass& b, int M) {
  const int bpc = sf_blocks_per_cta(b.p);
  return sf_plan(n, a.p, a.nblk, b.p, M, bpc * b.p, bpc * sf_rows_per_cta(b.p)).total;
}

// Can this side run as one few-token kernel?  Two passes whose blocks tile each other (p0 * nblk0 == p1 * nblk1 == n,
// one strided and one contiguous, nblk0 == p1), rows 16-byte aligned.
bool side_fewtok_ok(const QuipSide* sd, int n, int64_t M) {
  if (M < 1 || M > SF_MAXTOK || sd->n != n || sd->npass != 2) return false;
  const QuipPass& a = sd->pass[0];
  const QuipPass& b = sd->pass[1];
  if (a.strided == b.strided) return false;
  if ((int64_t)a.p * a.nblk != n || (int64_t)b.p * b.nblk != n || a.nblk != b.p || b.nblk != a.p) return false;
  if (a.p % 16 || b.p % 16) return false;
  if ((((uintptr_t)a.factors) | ((uintptr_t)b.factors)) & 15) return false;
  if (n >= 65536 || n % 8) return false;                       // 16-bit positions in shared memory, 16-byte token loads
  return side_fewtok_smem(n, a, b, (int)M) <= SF_SMEM_MAX;
}

int side_fewtok(const QuipSide* sd, const __half* in, __half* out, int64_t M, int n, const int32_t* in_idx,
                const float* in_scale, const int32_t* out_inv, const __half* out_bias, cudaStream_t s) {
  const QuipPass& a = sd->pass[0];
  const QuipPass& b = sd->pass[1];
  QUIP_CHECK_ARG((((uintptr_t)in | (uintptr_t)in_idx) & 15) == 0, "few-token side: tokens and index must be 16-byte aligned");
  SidePassArg P0{(const __half*)a.factors, a.p, a.nblk, a.strided, a.shared};
  SidePassArg P1{(const __half*)b.factors, b.p, b.nblk, b.strided, b.shared};
  // second-pass blocks up to 64 wide: whole blocks per CTA (four 16-wide ones together); wider: row tiles
  int blocks_per_cta = sf_blocks_per_cta(b.p);
  int rows_per_cta = sf_rows_per_cta(b.p);
  const int rtiles = ceil_div(b.p, rows_per_cta);
  const int items = ceil_div(b.nblk, blocks_per_cta) * rtiles;
  const size_t smem = side_fewtok_smem(n, a, b, (int)M);
  QUIP_CHECK_ARG(M >= 1 && M <= SF_MAXTOK, "few-token side: %lld tokens", (long long)M);
  static constexpr decltype(&side_fewtok_kernel<1>) kerns[SF_MAXTOK] = {
      side_fewtok_kernel<1>, side_fewtok_kernel<2>, side_fewtok_kernel<3>, side_fewtok_kernel<4>,
      side_fewtok_kernel<5>, side_fewtok_kernel<6>, side_fewtok_kernel<7>, side_fewtok_kernel<8>};
  return launch("side_fewtok_kernel", kerns[M - 1], (unsigned)items, SF_THREADS, smem, s, true, in, out, n, P0, P1, in_idx,
                in_scale, out_inv, out_bias, rows_per_cta, blocks_per_cta);
}

}  // namespace quip
