// Glue kernels of the per-layer eval step: the elementwise work BETWEEN the packed linears of a Llama decoder layer
// (RMSNorm, residual add, rotary embedding, SiLU gate), each one HBM pass instead of the 5-8 torch launches the HF
// modules issue.  ncu launch list of the eval step (profiles/launches_r01.json): those torch launches are 27 % of the
// step (RMSNorm 8 launches ~105 us, rotary 9 launches ~260 us, silu*up 2 launches ~40 us per decoder layer at 2048
// tokens); the kernels below move the same bytes once: ~34 MB / 67 MB / 135 MB per call, i.e. 5-20 us at HBM speed.
//
// Rounding points follow the HF modules exactly (transformers modeling_llama: LlamaRMSNorm.forward,
// apply_rotary_pos_emb / rotate_half, LlamaMLP.forward with SiLU), so a layer built on these kernels differs from the
// HF layer only through the summation order of the fp32 mean of squares:
//   rmsnorm      s = fp16(x + r)           (the residual add `residual + hidden_states`, one fp16 rounding)
//                y = w * fp16(float(s) * rsqrt(mean(float(s)^2) + eps))       (weight * hidden.to(fp16): two roundings)
//   rope         out = fp16(fp16(q*cos) + fp16(rot(q)*sin)), rot(q) = cat(-q[h/2:], q[:h/2])   (three roundings)
//   silu_mul     out = fp16(fp16(g / (1 + exp(-g))) * u)                      (silu computed in fp32, two roundings)
// All are HBM-bound streaming kernels: 128-bit accesses, one CTA per row (rmsnorm) or a grid-stride loop sized to the
// SM count (rope, silu_mul).
#include "common.cuh"

namespace quip {

namespace {

constexpr int RN_MAXV = 4;          // 128-bit vectors of a row held in registers per thread

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

union H8 {
  uint4 v;
  __half2 h2[4];
  __half h[8];
};

// One CTA per row.  x, r, sum_out, y: (rows, d) fp16 contiguous; w: (d) fp16.  r / sum_out may be null.
__global__ void __launch_bounds__(1024) rmsnorm_kernel(const __half* __restrict__ x, const __half* __restrict__ r,
                                                       const __half* __restrict__ w, __half* __restrict__ sum_out,
                                                       __half* __restrict__ y, int d, float eps) {
  __shared__ float red[32];
  const int64_t row = blockIdx.x;
  const int nvec = d >> 3;
  const uint4* xr = reinterpret_cast<const uint4*>(x + row * d);
  const uint4* rr = r ? reinterpret_cast<const uint4*>(r + row * d) : nullptr;
  H8 v[RN_MAXV];
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < RN_MAXV; ++i) {
    const int c = threadIdx.x + i * blockDim.x;
    if (c < nvec) {
      v[i].v = xr[c];
      if (rr) {
        H8 t;
        t.v = rr[c];
#pragma unroll
        for (int j = 0; j < 4; ++j) v[i].h2[j] = __hadd2_rn(v[i].h2[j], t.h2[j]);
        if (sum_out) reinterpret_cast<uint4*>(sum_out + row * d)[c] = v[i].v;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = __half22float2(v[i].h2[j]);
        ss = fmaf(f.x, f.x, ss);
        ss = fmaf(f.y, f.y, ss);
      }
    }
  }
  ss = warp_sum(ss);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  if (lane == 0) red[warp] = ss;
  __syncthreads();
  float tot = (lane < nwarps) ? red[lane] : 0.f;
  tot = warp_sum(tot);
  const float inv = rsqrtf(tot / (float)d + eps);
  const uint4* wr = reinterpret_cast<const uint4*>(w);
  uint4* yr = reinterpret_cast<uint4*>(y + row * d);
#pragma unroll
  for (int i = 0; i < RN_MAXV; ++i) {
    const int c = threadIdx.x + i * blockDim.x;
    if (c < nvec) {
      H8 ww, o;
      ww.v = wr[c];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = __half22float2(v[i].h2[j]);
        const __half2 n = __floats2half2_rn(f.x * inv, f.y * inv);
        o.h2[j] = __hmul2_rn(ww.h2[j], n);
      }
      yr[c] = o.v;
    }
  }
}

// Rotary embedding in place on q (rows, nq*hd) and k (rows, nkv*hd); cos, sin: (rows, hd) fp16.
// One work item = 8 consecutive lanes i of the first half of a head and their partners i + hd/2.
__global__ void __launch_bounds__(256) rope_kernel(__half* __restrict__ q, __half* __restrict__ k,
                                                   const __half* __restrict__ cs, const __half* __restrict__ sn,
                                                   int64_t rows, int nq, int nkv, int hd) {
  const int hv = hd >> 4;                       // work items per head
  const int heads = nq + nkv;
  const int64_t total = rows * heads * hv;
  for (int64_t it = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; it < total; it += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(it % hv);
    const int64_t t = it / hv;
    const int head = (int)(t % heads);
    const int64_t row = t / heads;
    __half* base = head < nq ? q + (row * nq + head) * (int64_t)hd : k + (row * nkv + (head - nq)) * (int64_t)hd;
    const int half_hd = hd >> 1;
    H8 x1, x2, c1, c2, s1, s2, o1, o2;
    x1.v = *reinterpret_cast<const uint4*>(base + c * 8);
    x2.v = *reinterpret_cast<const uint4*>(base + half_hd + c * 8);
    c1.v = *reinterpret_cast<const uint4*>(cs + row * hd + c * 8);
    c2.v = *reinterpret_cast<const uint4*>(cs + row * hd + half_hd + c * 8);
    s1.v = *reinterpret_cast<const uint4*>(sn + row * hd + c * 8);
    s2.v = *reinterpret_cast<const uint4*>(sn + row * hd + half_hd + c * 8);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      // first half: x1*cos + (-x2)*sin ; second half: x2*cos + x1*sin   (every product and the sum rounded to fp16)
      o1.h2[j] = __hadd2_rn(__hmul2_rn(x1.h2[j], c1.h2[j]), __hmul2_rn(__hneg2(x2.h2[j]), s1.h2[j]));
      o2.h2[j] = __hadd2_rn(__hmul2_rn(x2.h2[j], c2.h2[j]), __hmul2_rn(x1.h2[j], s2.h2[j]));
    }
    *reinterpret_cast<uint4*>(base + c * 8) = o1.v;
    *reinterpret_cast<uint4*>(base + half_hd + c * 8) = o2.v;
  }
}

__global__ void __launch_bounds__(256) silu_mul_kernel(const __half* __restrict__ g, const __half* __restrict__ u,
                                                       __half* __restrict__ out, int64_t nvec) {
  for (int64_t it = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; it < nvec; it += (int64_t)gridDim.x * blockDim.x) {
    H8 a, b, o;
    a.v = ldg_nc_v4(reinterpret_cast<const uint4*>(g) + it);
    b.v = ldg_nc_v4(reinterpret_cast<const uint4*>(u) + it);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = __half22float2(a.h2[j]);
      const __half2 s = __floats2half2_rn(f.x / (1.0f + expf(-f.x)), f.y / (1.0f + expf(-f.y)));
      o.h2[j] = __hmul2_rn(s, b.h2[j]);
    }
    reinterpret_cast<uint4*>(out)[it] = o.v;
  }
}

// SiLU(gate) * up with the permutations of the three surrounding incoherence sides folded in:
//   out[r][l] = fp16(fp16(silu(G[r][ig[l]])) * U[r][iu[l]]),   idx[l] = ig[l] | iu[l] << 16
// G and U are the gate / up projections still in their U-side layout order (their output gathers skipped), out is the down
// projection's input already in its V-side layout order (its input gather skipped): ig = u_idx(gate)[v_idx(down)], iu
// likewise -- three gather kernels and silu_mul become one pass.  SG_ROWS token rows per CTA share the index loads; the rows
// sit in shared memory (16-byte loads), the permuted reads are 2-byte shared-memory accesses, the stores 16 bytes.
constexpr int SG_ROWS = 2;
constexpr int SG_THREADS = 512;

__global__ void __launch_bounds__(SG_THREADS)
silu_mul_gather_kernel(const __half* __restrict__ g, const __half* __restrict__ u, const uint32_t* __restrict__ idx,
                       __half* __restrict__ out, int64_t rows, int n, int rpc) {
  extern __shared__ __align__(16) unsigned char sg_raw[];
  __half* gs = reinterpret_cast<__half*>(sg_raw);                 // [rpc][n]   (rpc <= SG_ROWS token rows per CTA)
  __half* us = gs + (size_t)rpc * n;                              // [rpc][n]
  const int64_t r0 = (int64_t)blockIdx.x * rpc;
  const int nr = (int)((rows - r0) < rpc ? (rows - r0) : rpc);
  const int nvec = n >> 3;
  for (int c = threadIdx.x; c < nr * nvec; c += SG_THREADS) {
    const int r = c / nvec, v = c - r * nvec;
    reinterpret_cast<uint4*>(gs + (size_t)r * n)[v] = ldg_nc_v4(reinterpret_cast<const uint4*>(g + (r0 + r) * n) + v);
    reinterpret_cast<uint4*>(us + (size_t)r * n)[v] = ldg_nc_v4(reinterpret_cast<const uint4*>(u + (r0 + r) * n) + v);
  }
  __syncthreads();
  for (int v = threadIdx.x; v < nvec; v += SG_THREADS) {
    const uint4 i0 = __ldg(reinterpret_cast<const uint4*>(idx) + 2 * v), i1 = __ldg(reinterpret_cast<const uint4*>(idx) + 2 * v + 1);
    const uint32_t ii[8] = {i0.x, i0.y, i0.z, i0.w, i1.x, i1.y, i1.z, i1.w};
#pragma unroll
    for (int r = 0; r < SG_ROWS; ++r) {
      if (r < nr) {
        H8 o;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float gv = __half2float(gs[(size_t)r * n + (ii[e] & 0xFFFFu)]);
          const __half sv = __float2half_rn(gv / (1.0f + expf(-gv)));
          o.h[e] = __hmul(sv, us[(size_t)r * n + (ii[e] >> 16)]);
        }
        reinterpret_cast<uint4*>(out + (r0 + r) * n)[v] = o.v;
      }
    }
  }
}

int stream_grid(int64_t items, int threads) {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
  }
  const int64_t want = (items + threads - 1) / threads;
  const int64_t cap = (int64_t)sms * 8;                 // 8 CTAs of 256 threads per SM: one full wave, grid-stride beyond
  return (int)(want < cap ? (want > 0 ? want : 1) : cap);
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace

}  // namespace quip

using namespace quip;

extern "C" int quip_rmsnorm(const void* x, const void* residual, const void* weight, void* sum_out, void* y,
                            int64_t rows, int32_t d, float eps, void* stream) {
  QUIP_CHECK_ARG(x && weight && y, "quip_rmsnorm: null pointer");
  QUIP_CHECK_ARG(rows >= 0 && d > 0 && d % 8 == 0, "quip_rmsnorm: width %d is not a positive multiple of 8", d);
  QUIP_CHECK_ARG(rows < (1ll << 31), "quip_rmsnorm: too many rows");
  QUIP_CHECK_ARG(!sum_out || residual, "quip_rmsnorm: sum_out without a residual");
  QUIP_CHECK_ARG(aligned16(x) && aligned16(weight) && aligned16(y) && aligned16(residual) && aligned16(sum_out),
                 "quip_rmsnorm: pointers must be 16-byte aligned");
  if (rows == 0) return QUIP_OK;
  const int nvec = d / 8;
  int threads = ((nvec + RN_MAXV - 1) / RN_MAXV + 31) / 32 * 32;
  QUIP_CHECK_ARG(threads <= 1024, "quip_rmsnorm: width %d exceeds %d", d, 1024 * RN_MAXV * 8);
  return launch("rmsnorm_kernel", rmsnorm_kernel, (unsigned)rows, threads, 0, (cudaStream_t)stream, false, (const __half*)x,
                (const __half*)residual, (const __half*)weight, (__half*)sum_out, (__half*)y, d, eps);
}

extern "C" int quip_rope(void* q, void* k, const void* cos, const void* sin, int64_t rows, int32_t n_q_heads,
                         int32_t n_kv_heads, int32_t head_dim, void* stream) {
  QUIP_CHECK_ARG(q && cos && sin, "quip_rope: null pointer");
  QUIP_CHECK_ARG(n_q_heads > 0 && n_kv_heads >= 0 && (k || n_kv_heads == 0), "quip_rope: bad head counts");
  QUIP_CHECK_ARG(head_dim > 0 && head_dim % 16 == 0, "quip_rope: head_dim %d is not a multiple of 16", head_dim);
  QUIP_CHECK_ARG(aligned16(q) && aligned16(k) && aligned16(cos) && aligned16(sin), "quip_rope: pointers must be 16-byte aligned");
  if (rows <= 0) return QUIP_OK;
  const int64_t items = rows * (n_q_heads + n_kv_heads) * (head_dim / 16);
  return launch("rope_kernel", rope_kernel, stream_grid(items, 256), 256, 0, (cudaStream_t)stream, false, (__half*)q,
                (__half*)k, (const __half*)cos, (const __half*)sin, rows, n_q_heads, n_kv_heads, head_dim);
}

extern "C" int quip_silu_mul(const void* gate, const void* up, void* out, int64_t n, void* stream) {
  QUIP_CHECK_ARG(gate && up && out, "quip_silu_mul: null pointer");
  QUIP_CHECK_ARG(n >= 0 && n % 8 == 0, "quip_silu_mul: element count must be a multiple of 8");
  QUIP_CHECK_ARG(aligned16(gate) && aligned16(up) && aligned16(out), "quip_silu_mul: pointers must be 16-byte aligned");
  if (n == 0) return QUIP_OK;
  return launch("silu_mul_kernel", silu_mul_kernel, stream_grid(n / 8, 256), 256, 0, (cudaStream_t)stream, false,
                (const __half*)gate, (const __half*)up, (__half*)out, n / 8);
}

extern "C" int quip_silu_mul_gather(const void* gate, const void* up, const uint32_t* idx, void* out, int64_t rows, int32_t n,
                                    void* stream) {
  QUIP_CHECK_ARG(gate && up && idx && out, "quip_silu_mul_gather: null pointer");
  QUIP_CHECK_ARG(rows >= 0 && n > 0 && n % 8 == 0 && n < 65536, "quip_silu_mul_gather: width %d must be a multiple of 8 below 65536", n);
  QUIP_CHECK_ARG(aligned16(gate) && aligned16(up) && aligned16(idx) && aligned16(out), "quip_silu_mul_gather: pointers must be 16-byte aligned");
  QUIP_CHECK_ARG(gate != out && up != out, "quip_silu_mul_gather: out must not alias the inputs (it is a permutation)");
  if (rows == 0) return QUIP_OK;
  const int rpc = (size_t)2 * SG_ROWS * n * sizeof(__half) <= 110 * 1024 ? SG_ROWS : 1;      // two CTAs per SM when they fit
  const size_t smem = (size_t)2 * rpc * n * sizeof(__half);
  QUIP_CHECK_ARG(smem <= 220 * 1024, "quip_silu_mul_gather: width %d does not fit shared memory", n);
  return launch("silu_mul_gather_kernel", silu_mul_gather_kernel, (unsigned)ceil_div(rows, rpc), SG_THREADS, smem,
                (cudaStream_t)stream, false, (const __half*)gate, (const __half*)up, idx, (__half*)out, rows, n, rpc);
}
