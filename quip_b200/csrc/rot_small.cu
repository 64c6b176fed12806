// Fast block-diagonal passes for small blocks (p <= 64, p % 8 == 0): the memory-bound half of the
// incoherence un-projection (reference method.py:58-63 applied to activations).
//
// Every warp owns BPW = 64/P blocks and keeps their p x p factors as mma.sync B fragments in registers
// for its whole lifetime; tokens stream through shared memory 16 at a time per MMA (tokens = MMA "M").
//
//   pass_contig_kernel   blocks contiguous in memory (pos = blk*p + j).  Warps are fully independent:
//                        each runs its own cp.async ring over 128-byte row segments, multiplies in
//                        place and stores its own rows -- no __syncthreads in the loop.
//   pass_strided_kernel  blocks strided (pos = j*nblk + blk).  The CTA's GB = 8*BPW adjacent blocks are
//                        loaded as 16-byte runs, transposed into per-block tiles in shared memory
//                        (2-byte scatter), multiplied, and written back through the inverse map; the
//                        next tile's global loads are in flight in registers during the math.
#include "common.cuh"

namespace quip {

template <int P>
struct FCfg {
  static constexpr int BPW = (64 / P) >= 1 ? (64 / P) : 1;
  static constexpr int LD = P + 8;
  static constexpr int KS = P / 16, NT = P / 8;
  static constexpr int TM = P >= 48 ? 32 : 16;      // tokens per tile
};

__device__ __forceinline__ void cp_async16s(void* smem, const void* gmem, bool valid) {
  uint32_t s = smem_u32(smem);
  int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gmem), "r"(sz));
}
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], const void* p) {
  uint32_t s = smem_u32(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(s));
}

// factor (p x p fp16 row-major, out_i = sum_j f[i][j] in_j) -> B fragments: b0 (k=2t,2t+1; n=g), b1 (k=2t+8,+9)
template <int P>
__device__ __forceinline__ void load_bfrags(const __half* __restrict__ f, int p, bool valid, int g, int t,
                                            uint32_t (&bf)[FCfg<P>::KS][FCfg<P>::NT][2]) {
  using C = FCfg<P>;
#pragma unroll
  for (int ks = 0; ks < C::KS; ++ks)
#pragma unroll
    for (int nt = 0; nt < C::NT; ++nt)
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int i = nt * 8 + g, j = ks * 16 + 2 * t + 8 * r;
        uint32_t v = 0;
        if (valid && i < p && j < p)            // p is even here, so j + 1 < p as well and the word is aligned
          v = __ldg(reinterpret_cast<const uint32_t*>(f + (int64_t)i * p + j));
        bf[ks][nt][r] = v;
      }
}

// D[tok][i] = sum_j A[tok][j] F[i][j] for one block tile (TM tokens), in place
template <int P, int TM>
__device__ __forceinline__ void mul_tile_inplace(__half* tile, const uint32_t (&bf)[FCfg<P>::KS][FCfg<P>::NT][2],
                                                 int lane) {
  using C = FCfg<P>;
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int mt = 0; mt < TM / 16; ++mt) {
    uint32_t a[C::KS][4];
#pragma unroll
    for (int ks = 0; ks < C::KS; ++ks)
      ldsm_x4(a[ks], &tile[(mt * 16 + (lane & 15)) * C::LD + ks * 16 + (lane >> 4) * 8]);
    __syncwarp();
#pragma unroll
    for (int nt = 0; nt < C::NT; ++nt) {
      float d[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int ks = 0; ks < C::KS; ++ks) mma16816(d, a[ks], bf[ks][nt]);
      *reinterpret_cast<__half2*>(&tile[(mt * 16 + g) * C::LD + nt * 8 + 2 * t]) = __floats2half2_rn(d[0], d[1]);
      *reinterpret_cast<__half2*>(&tile[(mt * 16 + g + 8) * C::LD + nt * 8 + 2 * t]) = __floats2half2_rn(d[2], d[3]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
constexpr int PC_WARPS = 4, PC_STAGES = 3;

template <int P, bool AFFINE>
__global__ void __launch_bounds__(PC_WARPS * 32)
pass_contig_kernel(const __half* __restrict__ in, __half* __restrict__ out, const __half* __restrict__ F, int64_t M,
                   int n, int p, int nblk, int shared, int tok_chunk) {
  using C = FCfg<P>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int TILE = C::BPW * C::TM * C::LD;                 // halves per stage per warp
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  __half* ring = reinterpret_cast<__half*>(smem_raw) + (size_t)warp * PC_STAGES * TILE;
  const int blk0 = (blockIdx.x * PC_WARPS + warp) * C::BPW;
  if (blk0 >= nblk) return;                                     // warps are independent: safe to leave
  const int64_t m_begin = (int64_t)blockIdx.y * tok_chunk;
  const int64_t m_end = m_begin + tok_chunk < M ? m_begin + tok_chunk : M;
  const int ntiles = (int)((m_end - m_begin + C::TM - 1) / C::TM);

  if (P != p) {                                                 // zero the padding columns once
    const int padw = P - p;
    for (int c = lane; c < PC_STAGES * C::BPW * C::TM * padw; c += 32)
      ring[(c / padw) * C::LD + p + c % padw] = __float2half(0.f);
  }
  const int w8 = C::BPW * p / 8;                                // 16-byte chunks per token row segment
  const int64_t col0 = (int64_t)blk0 * p;
  // The (token, chunk) -> address map is the same for every tile.  When 32 % w8 == 0 (p | 64) it is affine in
  // the per-lane step r (token += 32/w8, same chunk), so the divisions are resolved once; other block sizes
  // take the generic path.
  constexpr int MAXC = (C::TM * C::BPW * P / 8 + 31) / 32;      // chunks per lane per tile (upper bound)
  constexpr bool affine = AFFINE;                             // host guarantees 32 % w8 == 0
  const int tstep = affine ? 32 / w8 : 0;
  auto chunk = [&](int r, int& soff, int& goff, int& tok) -> bool {
    int c = lane + r * 32, q, bl, j;
    if (affine) {
      tok = lane / w8 + r * tstep; q = lane % w8;
    } else {
      if (c >= C::TM * w8) return false;
      tok = c / w8; q = c % w8;
    }
    if (tok >= C::TM) return false;
    bl = (q * 8) / p; j = (q * 8) % p;
    if (blk0 + bl >= nblk) return false;
    soff = (bl * C::TM + tok) * C::LD + j;
    goff = tok * n + q * 8;
    return true;
  };
  int s0 = 0, g0 = 0, t0 = 0;
  const bool ok0 = chunk(0, s0, g0, t0);

  auto issue = [&](int tile) {
    __half* dst = ring + (size_t)(tile % PC_STAGES) * TILE;
    const int64_t m0 = m_begin + (int64_t)tile * C::TM;
    const __half* src0 = in + m0 * n + col0;
#pragma unroll
    for (int r = 0; r < MAXC; ++r) {
      int so, go, tk;
      bool ok;
      if (affine) { ok = ok0 && (t0 + r * tstep < C::TM); so = s0 + r * tstep * C::LD; go = g0 + r * tstep * n; tk = t0 + r * tstep; }
      else ok = chunk(r, so, go, tk);
      if (!ok) continue;
      const bool valid = m0 + tk < m_end;
      cp_async16s(&dst[so], valid ? (src0 + go) : in, valid);
    }
  };

#pragma unroll
  for (int s = 0; s < PC_STAGES - 1; ++s) {
    if (s < ntiles) issue(s);
    asm volatile("cp.async.commit_group;");
  }
  uint32_t bf[C::BPW][C::KS][C::NT][2];                         // factors fetched while the first tiles are in flight
#pragma unroll
  for (int bb = 0; bb < C::BPW; ++bb)
    load_bfrags<P>(F + (int64_t)(shared ? 0 : min(blk0 + bb, nblk - 1)) * p * p, p, blk0 + bb < nblk, g, t, bf[bb]);
  for (int it = 0; it < ntiles; ++it) {
    asm volatile("cp.async.wait_group %0;" ::"n"(PC_STAGES - 2));
    __syncwarp();
    if (it + PC_STAGES - 1 < ntiles) issue(it + PC_STAGES - 1);
    asm volatile("cp.async.commit_group;");
    __half* tile = ring + (size_t)(it % PC_STAGES) * TILE;
#pragma unroll
    for (int bb = 0; bb < C::BPW; ++bb) mul_tile_inplace<P, C::TM>(tile + bb * C::TM * C::LD, bf[bb], lane);
    __syncwarp();
    const int64_t m0 = m_begin + (int64_t)it * C::TM;
    __half* dst0 = out + m0 * n + col0;
#pragma unroll
    for (int r = 0; r < MAXC; ++r) {
      int so, go, tk;
      bool ok;
      if (affine) { ok = ok0 && (t0 + r * tstep < C::TM); so = s0 + r * tstep * C::LD; go = g0 + r * tstep * n; tk = t0 + r * tstep; }
      else ok = chunk(r, so, go, tk);
      if (ok && m0 + tk < m_end) *reinterpret_cast<uint4*>(dst0 + go) = *reinterpret_cast<const uint4*>(&tile[so]);
    }
    __syncwarp();
  }
  asm volatile("cp.async.wait_group 0;");
}

// ------------------------------------------------------------------------------------------------
constexpr int PS_TM = 16;        // tokens per tile of the strided kernel (keeps the prefetch registers small)

template <int P, bool AFFINE, int W>
__global__ void __launch_bounds__(W * 32, (W == 16 ? 1 : 2))
pass_strided_kernel(const __half* __restrict__ in, __half* __restrict__ out, const __half* __restrict__ F, int64_t M,
                    int n, int p, int nblk, int shared, int tok_chunk) {
  using C = FCfg<P>;
  constexpr int GB = W * C::BPW;                         // blocks per CTA
  constexpr int CG = GB / 8;                                    // 16-byte chunks per (tok, j)
  constexpr int TILE = GB * PS_TM * C::LD;                      // halves per buffer
  // a "chunk" is two adjacent elements j, j+1 of 8 adjacent blocks for one token: two 16-byte global runs,
  // transposed with 32-bit shared-memory accesses (sub-word st/ld.shared are several times slower)
  constexpr int NCH = (PS_TM * (P / 2) * CG + W * 32 - 1) / (W * 32);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __half* T = reinterpret_cast<__half*>(smem_raw);              // [2][GB][TM][LD]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int b0 = blockIdx.x * GB;
  const int64_t m_begin = (int64_t)blockIdx.y * tok_chunk;
  const int64_t m_end = m_begin + tok_chunk < M ? m_begin + tok_chunk : M;
  const int ntiles = (int)((m_end - m_begin + PS_TM - 1) / PS_TM);
  const int hp = p / 2;                                         // p is even (p % 8 == 0)
  const int nchunks = PS_TM * hp * CG;

  if (P != p) {
    const int padw = P - p;
    for (int c = tid; c < 2 * GB * PS_TM * padw; c += W * 32)
      T[(c / padw) * C::LD + p + c % padw] = __float2half(0.f);
  }

  // per-thread chunk map (tile-invariant).  With (32 W) % (hp*CG) == 0 it is affine in r (token += 32W/(hp*CG),
  // same (j pair, block run)); other block sizes take the generic path with divisions.
  const int ppc = hp * CG;
  constexpr bool affine = AFFINE;
  const int tstep = affine ? (W * 32) / ppc : 0;
  auto chunk = [&](int r, int& soff, int& goff, int& tok) -> bool {
    int c8, jp;
    if (affine) {
      tok = tid / ppc + r * tstep; c8 = tid % CG; jp = (tid / CG) % hp;
    } else {
      const int c = tid + r * W * 32;
      if (c >= nchunks) return false;
      c8 = c % CG; jp = (c / CG) % hp; tok = c / ppc;
    }
    if (tok >= PS_TM) return false;
    const int blk = b0 + c8 * 8;
    if (blk >= nblk) return false;
    soff = ((c8 * 8) * PS_TM + tok) * C::LD + 2 * jp;            // even -> 4-byte aligned
    goff = tok * n + (2 * jp) * nblk + blk;
    return true;
  };
  int s0 = 0, g0 = 0, t0 = 0;
  const bool ok0 = chunk(0, s0, g0, t0);
#define QUIP_CHUNK(r, so, go, tk, ok)                                                                       \
  int so, go, tk;                                                                                          \
  bool ok;                                                                                                 \
  if (affine) { tk = t0 + (r) * tstep; ok = ok0 && tk < PS_TM; so = s0 + (r) * tstep * C::LD; go = g0 + (r) * tstep * n; } \
  else ok = chunk(r, so, go, tk);
  constexpr int BSTRIDE = PS_TM * C::LD;                        // smem distance between adjacent blocks' tiles

  uint4 pre[NCH][2];                                            // rows j and j+1 of each chunk
  auto prefetch = [&](int tile) {
    const int64_t m0 = m_begin + (int64_t)tile * PS_TM;
    const __half* src0 = in + m0 * n;
#pragma unroll
    for (int r = 0; r < NCH; ++r) {
      pre[r][0] = pre[r][1] = make_uint4(0, 0, 0, 0);
      QUIP_CHUNK(r, so, go, tk, ok)
      if (ok && m0 + tk < m_end) {
        pre[r][0] = ldg_nc_v4(src0 + go);
        pre[r][1] = ldg_nc_v4(src0 + go + nblk);
      }
    }
  };

  prefetch(0);                                                  // first tile in flight while the factors are fetched
  uint32_t bf[C::BPW][C::KS][C::NT][2];
#pragma unroll
  for (int bb = 0; bb < C::BPW; ++bb) {
    const int blk = b0 + warp * C::BPW + bb;
    load_bfrags<P>(F + (int64_t)(shared ? 0 : min(blk, nblk - 1)) * p * p, p, blk < nblk, g, t, bf[bb]);
  }
  for (int it = 0; it < ntiles; ++it) {
    __half* buf = T + (size_t)(it & 1) * TILE;
#pragma unroll
    for (int r = 0; r < NCH; ++r) {
      QUIP_CHUNK(r, so, go, tk, ok)
      if (ok) {
        const uint32_t* lo = reinterpret_cast<const uint32_t*>(&pre[r][0]);   // element j   of blocks 0..7
        const uint32_t* hi = reinterpret_cast<const uint32_t*>(&pre[r][1]);   // element j+1 of blocks 0..7
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          // blocks 2w and 2w+1: pack (j, j+1) of one block into a word
          *reinterpret_cast<uint32_t*>(&buf[so + (2 * w) * BSTRIDE]) = __byte_perm(lo[w], hi[w], 0x5410);
          *reinterpret_cast<uint32_t*>(&buf[so + (2 * w + 1) * BSTRIDE]) = __byte_perm(lo[w], hi[w], 0x7632);
        }
      }
    }
    __syncthreads();
    if (it + 1 < ntiles) prefetch(it + 1);
#pragma unroll
    for (int bb = 0; bb < C::BPW; ++bb)
      mul_tile_inplace<P, PS_TM>(buf + (size_t)((warp * C::BPW + bb) * PS_TM) * C::LD, bf[bb], lane);
    __syncthreads();
    const int64_t m0 = m_begin + (int64_t)it * PS_TM;
    __half* dst0 = out + m0 * n;
#pragma unroll
    for (int r = 0; r < NCH; ++r) {
      QUIP_CHUNK(r, so, go, tk, ok)
      if (ok && m0 + tk < m_end) {
        uint32_t lo[4], hi[4];
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          const uint32_t e = *reinterpret_cast<const uint32_t*>(&buf[so + (2 * w) * BSTRIDE]);      // block 2w  : (i, i+1)
          const uint32_t o = *reinterpret_cast<const uint32_t*>(&buf[so + (2 * w + 1) * BSTRIDE]);  // block 2w+1: (i, i+1)
          lo[w] = __byte_perm(e, o, 0x5410);      // row i  : blocks 2w, 2w+1
          hi[w] = __byte_perm(e, o, 0x7632);      // row i+1: blocks 2w, 2w+1
        }
        *reinterpret_cast<uint4*>(dst0 + go) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        *reinterpret_cast<uint4*>(dst0 + go + nblk) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
      }
    }
  }
#undef QUIP_CHUNK
}

// ------------------------------------------------------------------------------------------------
static int pick_tok_chunk(int64_t M, int gx, int tm) {
  // enough CTAs for ~2 per SM, but keep >= 4 tiles per CTA when M allows so the register-resident
  // factors are amortised
  int64_t want_gy = (296 + gx - 1) / gx;
  int64_t chunk = (M + want_gy - 1) / want_gy;
  if (chunk < (int64_t)g_pass_min_tiles * tm) chunk = (int64_t)g_pass_min_tiles * tm;
  chunk = (chunk + tm - 1) / tm * tm;
  return (int)(chunk < (int64_t)tm ? tm : chunk);
}

template <int P>
static int launch_fast(const QuipPass* ps, const __half* in, __half* out, int64_t M, int n, cudaStream_t s) {
  using C = FCfg<P>;
  const __half* F = (const __half*)ps->factors;
  if (!ps->strided) {
    const int gx = ceil_div(ps->nblk, PC_WARPS * C::BPW);
    const int tok_chunk = pick_tok_chunk(M, gx, C::TM);
    size_t smem = (size_t)PC_WARPS * PC_STAGES * C::BPW * C::TM * C::LD * sizeof(__half);
    const bool affine = (32 % (C::BPW * ps->p / 8)) == 0;
    auto kern = affine ? pass_contig_kernel<P, true> : pass_contig_kernel<P, false>;
    return launch("pass_contig_kernel", kern, dim3(gx, ceil_div(M, tok_chunk)), PC_WARPS * 32, smem, s, false, in, out, F, M,
                  n, ps->p, ps->nblk, ps->shared, tok_chunk);
  } else {
    // 64-wide blocks: 16 warps = 16 adjacent blocks per CTA, so the strided runs are full 32-byte sectors
    constexpr int W = (P == 64) ? 16 : 8;
    constexpr int GB = W * C::BPW;
    const int gx = ceil_div(ps->nblk, GB);
    const int tok_chunk = pick_tok_chunk(M, gx, PS_TM);
    size_t smem = (size_t)2 * GB * PS_TM * C::LD * sizeof(__half);
    const bool affine = ((W * 32) % ((ps->p / 2) * (GB / 8))) == 0;
    auto kern = affine ? pass_strided_kernel<P, true, W> : pass_strided_kernel<P, false, W>;
    return launch("pass_strided_kernel", kern, dim3(gx, ceil_div(M, tok_chunk)), W * 32, smem, s, false, in, out, F, M, n,
                  ps->p, ps->nblk, ps->shared, tok_chunk);
  }
}

// Fast path for p <= 64 when the 16-byte vector conditions hold; otherwise *handled stays false and the
// caller falls back to the generic kernels in rot.cu.
int launch_small_fast(const QuipPass* ps, const __half* in, __half* out, int64_t M, int n, cudaStream_t s,
                      bool* handled) {
  *handled = false;
  const int p = ps->p;
  if (p > 64 || p % 8 != 0 || n % 8 != 0) return QUIP_OK;
  if (ps->strided && ps->nblk % 8 != 0) return QUIP_OK;
  if (((uintptr_t)in & 15) || ((uintptr_t)out & 15) || ((uintptr_t)ps->factors & 3)) return QUIP_OK;
  *handled = true;
  if (p <= 16) return launch_fast<16>(ps, in, out, M, n, s);
  if (p <= 32) return launch_fast<32>(ps, in, out, M, n, s);
  if (p <= 48) return launch_fast<48>(ps, in, out, M, n, s);
  return launch_fast<64>(ps, in, out, M, n, s);
}

}  // namespace quip
