// Block-diagonal passes and the index/scale/bias gather for a handful of tokens (decode, M <= 8).
//
// With one token a pass of the incoherence transform (reference method.py:46-67, one stage of
// mul_ortho_butterfly) is a batch of matrix-vector products whose cost is reading the factors once:
// 0.5 MiB per pass at n = 4096, 15 MiB for the sixteen 688 x 688 blocks of an 11008 side -- more bytes
// than the packed weights they surround.  The many-token kernels (rot_small.cu, qgemm_tc.cu DENSE) keep
// factors resident and stream tokens; at M = 1 they run a handful of CTAs.  Here the roles flip, as in
// qgemv.cu: the factor is the streamed A operand of mma.sync.m16n8k16, read straight from its row-major
// array (a lane takes 8 bytes of rows g and g+8 per 16 k: full 32-byte sectors, no shared memory), the
// tokens are the 8-wide B operand.
//
// Task = (block, 16 output rows, k part): the k range of a row tile is cut into parts of at most
// FT_STEPS x 16 so that a warp requests everything it will ever read before its first MMA; the parts of a
// row tile sit in one CTA and are summed through shared memory in a fixed order.  All factor loads are
// issued before griddepcontrol.wait: under programmatic dependent launch they overlap the previous kernel.
#include "common.cuh"

namespace quip {

constexpr int FT_WARPS = 8;
constexpr int FT_STEPS = 12;           // k16 steps per task: 12 x (2 x 8 B) per lane in flight

constexpr int FT_XPT = 6;              // input elements staged per thread (covers 2 blocks of 688)

// Optional fusions (the few-token forward of api.cu uses both, saving two launches per QuantLinear):
//   in_idx / in_scale : the pass reads  in[m][in_idx[pos]] * in_scale[in_idx[pos]]  instead of in[m][pos]
//                       (the K-side gather + 1/s of quip_gather, rounded to fp16 exactly as it rounds)
//   out_inv / out_bias: the pass writes out[m][out_inv[pos]] = value + out_bias[out_inv[pos]]
//                       (the N-side gather y[j] = layout[idx[j]] + bias[j], out_inv = idx^-1)
//
// NG = groups of 8 tokens (the MMA's n): the factor fragments are loaded once and reused by every group, so 9..32
// tokens (batched decode) cost a few more MMAs per task, not more factor traffic.
template <int NG>
__global__ void __launch_bounds__(FT_WARPS * 32)
pass_fewtok_kernel(const __half* __restrict__ in, __half* __restrict__ out, const __half* __restrict__ F, int M, int n,
                   int p, int nblk, int strided, int shared, int kparts, int steps_per_part,
                   const int32_t* __restrict__ in_idx, const float* __restrict__ in_scale,
                   const int32_t* __restrict__ out_inv, const __half* __restrict__ out_bias, int nb_cta) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ float red[NG][FT_WARPS][16][9];
  __half* xs = reinterpret_cast<__half*>(smem_raw);        // [M][xld]: the input blocks this CTA multiplies
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int rtiles = p >> 4;                               // 16-row tiles per block
  const int groups_per_cta = FT_WARPS / kparts;            // (block, row tile) pairs per CTA
  const int grp = warp / kparts, part = warp % kparts;
  const int64_t task0 = (int64_t)blockIdx.x * groups_per_cta, task = task0 + grp;
  const bool live = task < (int64_t)nblk * rtiles;
  const int b = live ? (int)(task / rtiles) : 0, rt = live ? (int)(task % rtiles) : 0;
  const int b_first = (int)(task0 / rtiles);
  const int xld = nb_cta * p + 16;
  const int ksteps = p >> 4;
  const int s0 = part * steps_per_part, s1 = min(ksteps, s0 + steps_per_part);

  // ---- factor rows g and g+8 of this tile: everything requested up front (weights: no dependency) ----
  // Pairs of k16 steps are one 128-bit load per row: within a 32-wide k block a lane owns 8 consecutive k
  // (32u + 8t ..), the first four feeding the MMA of step 2u, the last four that of step 2u+1 (the token operand is
  // read with the same labelling).  A trailing odd step (p = 688 = 21 x 32 + 16) uses 64-bit loads of 4 consecutive k.
  const __half* frow = F + ((int64_t)(shared ? 0 : b) * p + rt * 16 + g) * p;
  constexpr int FT_PAIRS = FT_STEPS / 2;
  uint4 a_lo[FT_PAIRS], a_hi[FT_PAIRS];
  const int npair = live ? (s1 - s0) / 2 : 0;             // s0 is even (steps_per_part is)
  const bool tail = live && ((s1 - s0) & 1);
#pragma unroll
  for (int u = 0; u < FT_PAIRS; ++u) {
    a_lo[u] = make_uint4(0u, 0u, 0u, 0u);
    a_hi[u] = make_uint4(0u, 0u, 0u, 0u);
    if (u < npair) {
      a_lo[u] = ldg_nc_v4(frow + (s0 + 2 * u) * 16 + 8 * t);
      a_hi[u] = ldg_nc_v4(frow + (int64_t)8 * p + (s0 + 2 * u) * 16 + 8 * t);
    }
  }
  uint2 t_lo = make_uint2(0u, 0u), t_hi = make_uint2(0u, 0u);
  if (tail) {
    t_lo = ldg_nc_v2(frow + (s1 - 1) * 16 + 4 * t);
    t_hi = ldg_nc_v2(frow + (int64_t)8 * p + (s1 - 1) * 16 + 4 * t);
  }
  // ---- where this CTA's inputs and outputs live: index vectors are parameters too ----
  // plain contiguous input (no index, no scale): 8-byte copies after the wait; otherwise element by element
  const bool vec_in = !strided && !in_idx && !in_scale;
  const int b_last = min(nblk - 1, (int)((task0 + groups_per_cta - 1) / rtiles));
  int src[FT_XPT];
  float ssc[FT_XPT];
#pragma unroll
  for (int i = 0; i < FT_XPT; ++i) {
    const int e = tid + i * FT_WARPS * 32;
    src[i] = -1;
    ssc[i] = 1.f;
    if (!vec_in && e < nb_cta * p) {
      const int bl = e / p, j = e - bl * p, bb = b_first + bl;
      if (bb <= b_last) {
        const int pos = strided ? (j * nblk + bb) : (bb * p + j);
        src[i] = in_idx ? __ldg(in_idx + pos) : pos;
        if (in_scale) ssc[i] = __ldg(in_scale + src[i]);
      }
    }
  }
  int dst[2];
  float dbias[2];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int i = rt * 16 + g + 8 * h;
    const int pos = strided ? (i * nblk + b) : (b * p + i);
    dst[h] = (live && out_inv) ? __ldg(out_inv + pos) : pos;
    dbias[h] = (live && out_bias) ? __half2float(__ldg(out_bias + dst[h])) : 0.f;
  }
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");

  // ---- stage the tokens of this CTA's blocks ----
  if (vec_in) {
    const int nq = (b_last - b_first + 1) * p / 4;         // 8-byte groups per token (p % 16 == 0)
    for (int e = tid; e < nq * M; e += FT_WARPS * 32) {
      const int m = e / nq, qd = e - m * nq;
      *reinterpret_cast<uint2*>(xs + m * xld + 4 * qd) =
          *reinterpret_cast<const uint2*>(in + (int64_t)m * n + (int64_t)b_first * p + 4 * qd);
    }
  } else {
#pragma unroll
    for (int i = 0; i < FT_XPT; ++i) {
      const int e = tid + i * FT_WARPS * 32;
      if (src[i] >= 0) {
#pragma unroll 4
        for (int m = 0; m < M; ++m) {
          const float v = __half2float(__ldg(in + (int64_t)m * n + src[i]));
          xs[m * xld + e] = in_scale ? __float2half_rn(v * ssc[i]) : __float2half_rn(v);
        }
      }
    }
  }
  __syncthreads();

  // ---- tokens with the same k labelling; columns >= M re-read the last token ----
  const __half* xrow[NG];
#pragma unroll
  for (int q = 0; q < NG; ++q) xrow[q] = xs + min(8 * q + g, M - 1) * xld + (b - b_first) * p;
  float acc[NG][4];
#pragma unroll
  for (int q = 0; q < NG; ++q)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[q][c] = 0.f;
#pragma unroll
  for (int u = 0; u < FT_PAIRS; ++u) {
    if (u < npair) {
      // a lane's four consecutive k are MMA slots (2t, 2t+1, 2t+8, 2t+9) on both operands
      const uint32_t a0[4] = {a_lo[u].x, a_hi[u].x, a_lo[u].y, a_hi[u].y};
      const uint32_t a1[4] = {a_lo[u].z, a_hi[u].z, a_lo[u].w, a_hi[u].w};
#pragma unroll
      for (int q = 0; q < NG; ++q) {
        const uint4 v = *reinterpret_cast<const uint4*>(xrow[q] + (s0 + 2 * u) * 16 + 8 * t);
        const uint32_t b0[2] = {v.x, v.y}, b1[2] = {v.z, v.w};
        mma16816(acc[q], a0, b0);
        mma16816(acc[q], a1, b1);
      }
    }
  }
  if (tail) {
    const uint32_t a[4] = {t_lo.x, t_hi.x, t_lo.y, t_hi.y};
#pragma unroll
    for (int q = 0; q < NG; ++q) {
      const uint2 v = *reinterpret_cast<const uint2*>(xrow[q] + (s1 - 1) * 16 + 4 * t);
      const uint32_t bfrag[2] = {v.x, v.y};
      mma16816(acc[q], a, bfrag);
    }
  }

  // ---- sum the k parts in a fixed order, store rows g / g+8 for tokens 8q + 2t, 8q + 2t + 1 ----
  if (kparts > 1) {
#pragma unroll
    for (int q = 0; q < NG; ++q) {
      red[q][warp][g][2 * t] = acc[q][0]; red[q][warp][g][2 * t + 1] = acc[q][1];
      red[q][warp][g + 8][2 * t] = acc[q][2]; red[q][warp][g + 8][2 * t + 1] = acc[q][3];
    }
    __syncthreads();
    if (part != 0) return;
#pragma unroll
    for (int q = 0; q < NG; ++q) {
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[q][c] = 0.f;
      for (int w = 0; w < kparts; ++w) {
        acc[q][0] += red[q][warp + w][g][2 * t]; acc[q][1] += red[q][warp + w][g][2 * t + 1];
        acc[q][2] += red[q][warp + w][g + 8][2 * t]; acc[q][3] += red[q][warp + w][g + 8][2 * t + 1];
      }
    }
  }
  if (!live) return;
#pragma unroll
  for (int q = 0; q < NG; ++q)
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int tok = 8 * q + 2 * t + (c & 1), h = c >> 1;
      if (tok < M) {
        // fused bias: the pass result is rounded to fp16 first, as the stand-alone gather would read it
        const float v = out_bias ? __half2float(__float2half_rn(acc[q][c])) + dbias[h] : acc[q][c];
        out[(int64_t)tok * n + dst[h]] = __float2half_rn(v);
      }
    }
}

// out[m][l] = in[m][idx ? idx[l] : l] * (scale ? scale[src] : 1) + (bias ? bias[l] : 0), one thread per 8 outputs
// of one token: for a few tokens the grid is n/8 threads wide instead of one CTA per token row.
__global__ void __launch_bounds__(128)
gather_fewtok_kernel(const __half* __restrict__ in, __half* __restrict__ out, int M, int n, const int32_t* __restrict__ idx,
                     const float* __restrict__ scale, const __half* __restrict__ bias) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n / 8) return;
  const int l0 = c * 8;
  int src[8];
  float sc[8], bs[8];
  if (idx) {                                               // parameters first: they do not depend on the previous kernel
    const int4 a = *reinterpret_cast<const int4*>(idx + l0), b = *reinterpret_cast<const int4*>(idx + l0 + 4);
    src[0] = a.x; src[1] = a.y; src[2] = a.z; src[3] = a.w; src[4] = b.x; src[5] = b.y; src[6] = b.z; src[7] = b.w;
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i) src[i] = l0 + i;
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    sc[i] = scale ? __ldg(scale + src[i]) : 1.f;
    bs[i] = bias ? __half2float(__ldg(bias + l0 + i)) : 0.f;
  }
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  for (int m = 0; m < M; ++m) {
    __align__(16) __half v[8];
    const __half* row = in + (int64_t)m * n;
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __float2half_rn(fmaf(__half2float(__ldg(row + src[i])), sc[i], bs[i]));
    *reinterpret_cast<uint4*>(out + (int64_t)m * n + l0) = *reinterpret_cast<const uint4*>(v);
  }
}

int g_fewtok_max_m = 32;      // 9..32 tokens (batched decode) through the few-token kernels too; quip_config("fewtok_max_m", 8)
                              // sends them to the many-token route instead

bool pass_fewtok_ok(const QuipPass* ps, int64_t M, int n) {
  return M <= g_fewtok_max_m && M <= 32 && ps->p % 16 == 0 && ps->p >= 16 && (n % 8 == 0) && (((uintptr_t)ps->factors) & 15) == 0;
}

int pass_fewtok(const QuipPass* ps, const __half* in, __half* out, int64_t M, int n, const int32_t* in_idx,
                const float* in_scale, const int32_t* out_inv, const __half* out_bias, cudaStream_t s) {
  const int p = ps->p, ksteps = p / 16;
  int kparts = 1;
  while (kparts < FT_WARPS && ((ceil_div(ksteps, kparts) + 1) & ~1) > FT_STEPS) kparts *= 2;
  QUIP_CHECK_ARG(ceil_div(ksteps, kparts) <= FT_STEPS, "few-token pass: block size %d too large", p);
  int steps_per_part = ceil_div(ksteps, kparts);
  if (kparts > 1) steps_per_part = (steps_per_part + 1) & ~1;          // parts start on a 32-wide k block
  const int rtiles = p / 16;
  const int64_t groups = (int64_t)ps->nblk * rtiles;
  const int per_cta = FT_WARPS / kparts;
  int nb_cta = (per_cta + rtiles - 1) / rtiles + ((per_cta % rtiles) && (rtiles % per_cta) ? 1 : 0);   // blocks a CTA can touch
  if (nb_cta > ps->nblk) nb_cta = ps->nblk;
  QUIP_CHECK_ARG(nb_cta * p <= FT_XPT * FT_WARPS * 32, "few-token pass: %d blocks of %d per CTA exceed the staging budget", nb_cta, p);
  const size_t smem = (size_t)M * (nb_cta * p + 16) * sizeof(__half);
  QUIP_CHECK_ARG(smem <= 200 * 1024, "few-token pass: %zu bytes of token staging", smem);
  auto kern = M <= 8 ? pass_fewtok_kernel<1> : (M <= 16 ? pass_fewtok_kernel<2> : pass_fewtok_kernel<4>);
  return launch("pass_fewtok_kernel", kern, (unsigned)ceil_div(groups, per_cta), FT_WARPS * 32, smem, s, true, in, out,
                (const __half*)ps->factors, (int)M, n, p, ps->nblk, ps->strided, ps->shared, kparts, steps_per_part, in_idx,
                in_scale, out_inv, out_bias, nb_cta);
}

int gather_fewtok(const __half* in, __half* out, int64_t M, int n, const int32_t* idx, const float* scale,
                  const __half* bias, cudaStream_t s) {
  return launch("gather_fewtok_kernel", gather_fewtok_kernel, (unsigned)ceil_div(n / 8, 128), 128, 0, s, true, in, out,
                (int)M, n, idx, scale, bias);
}

}  // namespace quip
