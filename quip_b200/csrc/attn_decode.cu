// One decode step of attention for B sequences over the static KV cache (quip_b200/generate.py), flash-decoding style.
//
// Cache layout per layer: (B, n_kv_heads, max_len, head_dim) fp16.  Sequence b writes its new K / V row at pos[b] and
// attends to positions 0 .. pos[b]; only those rows are read, so the bytes moved are 2 * sum_b (pos[b]+1) * nkv * hd * 2
// plus q / out.  The G = nh / nkv query heads of a KV head are one CTA's work, so each K / V row is read once per group
// and never copied (GQA).
//
//   split kernel    grid (nsplit, nkv, B), AD_SPLIT positions per CTA.  Scores s = scale * q.k in fp32 (the row at
//                   pos[b] from k_new, not from the cache, so no CTA depends on another's cache write), the chunk's max m
//                   and l = sum exp(s - m), and the unnormalised o = sum exp(s - m) v, all fp32, to the workspace.  The
//                   CTA whose chunk holds pos[b] also writes k_new / v_new to the cache.  CTAs past pos[b] exit.
//   combine kernel  grid (nh, B): the chunks of a (sequence, head) merged in chunk order -- a fixed order, so the output
//                   is deterministic -- and rounded once to fp16.
// Every sum inside a CTA has a fixed order too (shuffle trees, then the row groups in index order).
#include "common.cuh"

namespace quip {

namespace {

constexpr int AD_SPLIT = 128;    // cache positions per split CTA
constexpr int AD_THREADS = 128;
constexpr int AD_ROWS = 4;       // K / V rows each thread has in flight

union H8 {
  uint4 v;
  __half2 h2[4];
};

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// A thread owns 8 consecutive dims (16 bytes) of a row: HD/8 lanes per row, AD_THREADS/(HD/8) rows per pass.
template <int HD, int G>
__global__ void __launch_bounds__(AD_THREADS)
attn_decode_split_kernel(const __half* __restrict__ q, const __half* __restrict__ k_new, const __half* __restrict__ v_new,
                         __half* __restrict__ k_cache, __half* __restrict__ v_cache, const int32_t* __restrict__ pos,
                         float scale, float* __restrict__ part_o, float* __restrict__ part_ml, int nkv, int max_len,
                         int nsplit) {
  constexpr int LPR = HD / 8;
  constexpr int RPP = AD_THREADS / LPR;
  __shared__ float s_p[G][AD_SPLIT];
  __shared__ __align__(16) float s_red[RPP][G * HD];
  __shared__ float s_ml[G][2];
  const int split = blockIdx.x, kvh = blockIdx.y, b = blockIdx.z;
  const int p = pos[b];
  const int t0 = split * AD_SPLIT;
  if (p < 0 || p >= max_len || t0 > p) return;
  const int n = min(AD_SPLIT, p + 1 - t0);
  const int nh = nkv * G;
  const int lane = threadIdx.x % LPR, rg = threadIdx.x / LPR;
  const size_t head = (size_t)b * nkv + kvh;
  __half* kc = k_cache + head * max_len * HD;
  __half* vc = v_cache + head * max_len * HD;
  const uint4 kn = *reinterpret_cast<const uint4*>(k_new + head * HD + lane * 8);
  const uint4 vn = *reinterpret_cast<const uint4*>(v_new + head * HD + lane * 8);
  if (p < t0 + AD_SPLIT && rg == 0) {              // the chunk holding pos[b] stores the new row
    *reinterpret_cast<uint4*>(kc + (size_t)p * HD + lane * 8) = kn;
    *reinterpret_cast<uint4*>(vc + (size_t)p * HD + lane * 8) = vn;
  }

  float qr[G][8];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    H8 t;
    t.v = *reinterpret_cast<const uint4*>(q + ((size_t)b * nh + kvh * G + g) * HD + lane * 8);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = __half22float2(t.h2[j]);
      qr[g][2 * j] = f.x * scale;
      qr[g][2 * j + 1] = f.y * scale;
    }
  }

  // scores
  for (int r0 = 0; r0 < n; r0 += RPP * AD_ROWS) {
    H8 kr[AD_ROWS];
#pragma unroll
    for (int i = 0; i < AD_ROWS; ++i) {
      const int r = r0 + i * RPP + rg, t = t0 + r;
      kr[i].v = make_uint4(0, 0, 0, 0);
      if (r < n) kr[i].v = t == p ? kn : ldg_nc_v4(kc + (size_t)t * HD + lane * 8);
    }
#pragma unroll
    for (int i = 0; i < AD_ROWS; ++i) {
      float d[G];
#pragma unroll
      for (int g = 0; g < G; ++g) {
        d[g] = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = __half22float2(kr[i].h2[j]);
          d[g] = fmaf(qr[g][2 * j], f.x, d[g]);
          d[g] = fmaf(qr[g][2 * j + 1], f.y, d[g]);
        }
#pragma unroll
        for (int o = LPR / 2; o > 0; o >>= 1) d[g] += __shfl_xor_sync(0xffffffffu, d[g], o);
      }
      const int r = r0 + i * RPP + rg;
      if (lane == 0 && r < n) {
#pragma unroll
        for (int g = 0; g < G; ++g) s_p[g][r] = d[g];
      }
    }
  }
  __syncthreads();

  // softmax numerators of the chunk, one warp per head
  const int warp = threadIdx.x >> 5, wl = threadIdx.x & 31;
  for (int g = warp; g < G; g += AD_THREADS / 32) {
    float m = -INFINITY;
    for (int r = wl; r < n; r += 32) m = fmaxf(m, s_p[g][r]);
    m = warp_max(m);
    float l = 0.f;
    for (int r = wl; r < n; r += 32) {
      const float e = expf(s_p[g][r] - m);
      s_p[g][r] = e;
      l += e;
    }
    l = warp_sum(l);
    if (wl == 0) {
      s_ml[g][0] = m;
      s_ml[g][1] = l;
    }
  }
  __syncthreads();

  // o = sum_r p[r] * v[r]
  float acc[G][8];
#pragma unroll
  for (int g = 0; g < G; ++g)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[g][j] = 0.f;
  for (int r0 = 0; r0 < n; r0 += RPP * AD_ROWS) {
    H8 vr[AD_ROWS];
#pragma unroll
    for (int i = 0; i < AD_ROWS; ++i) {
      const int r = r0 + i * RPP + rg, t = t0 + r;
      if (r < n) vr[i].v = t == p ? vn : ldg_nc_v4(vc + (size_t)t * HD + lane * 8);
    }
#pragma unroll
    for (int i = 0; i < AD_ROWS; ++i) {
      const int r = r0 + i * RPP + rg;
      if (r < n) {
#pragma unroll
        for (int g = 0; g < G; ++g) {
          const float w = s_p[g][r];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 f = __half22float2(vr[i].h2[j]);
            acc[g][2 * j] = fmaf(w, f.x, acc[g][2 * j]);
            acc[g][2 * j + 1] = fmaf(w, f.y, acc[g][2 * j + 1]);
          }
        }
      }
    }
  }
#pragma unroll
  for (int g = 0; g < G; ++g) {
    float4* dst = reinterpret_cast<float4*>(&s_red[rg][g * HD + lane * 8]);
    dst[0] = make_float4(acc[g][0], acc[g][1], acc[g][2], acc[g][3]);
    dst[1] = make_float4(acc[g][4], acc[g][5], acc[g][6], acc[g][7]);
  }
  __syncthreads();
  for (int e = threadIdx.x; e < G * HD; e += AD_THREADS) {
    float o = 0.f;
#pragma unroll
    for (int i = 0; i < RPP; ++i) o += s_red[i][e];
    const int g = e / HD, dd = e % HD;
    part_o[(((size_t)b * nh + kvh * G + g) * nsplit + split) * HD + dd] = o;
  }
  if (threadIdx.x < G) {
    float* ml = part_ml + (((size_t)b * nh + kvh * G + threadIdx.x) * nsplit + split) * 2;
    ml[0] = s_ml[threadIdx.x][0];
    ml[1] = s_ml[threadIdx.x][1];
  }
}

// grid (nh, B), one thread per dim
__global__ void __launch_bounds__(128)
attn_decode_combine_kernel(const float* __restrict__ part_o, const float* __restrict__ part_ml,
                           const int32_t* __restrict__ pos, __half* __restrict__ out, int nh, int hd, int max_len,
                           int nsplit) {
  const int h = blockIdx.x, b = blockIdx.y, d = threadIdx.x;
  const int p = pos[b];
  __half* dst = out + ((size_t)b * nh + h) * hd + d;
  if (p < 0 || p >= max_len) {                     // position outside the cache: nothing was computed
    *dst = __float2half_rn(NAN);
    return;
  }
  const int ns = p / AD_SPLIT + 1;
  const size_t row = (size_t)b * nh + h;
  const float* ml = part_ml + row * nsplit * 2;
  float m = -INFINITY;
  for (int s = 0; s < ns; ++s) m = fmaxf(m, ml[2 * s]);
  float l = 0.f, o = 0.f;
  for (int s = 0; s < ns; ++s) {
    const float w = expf(ml[2 * s] - m);
    l = fmaf(ml[2 * s + 1], w, l);
    o = fmaf(part_o[(row * nsplit + s) * hd + d], w, o);
  }
  *dst = __float2half_rn(o / l);
}

template <int HD, int G>
int launch_split(const __half* q, const __half* kn, const __half* vn, __half* kc, __half* vc, const int32_t* pos,
                 float scale, float* part_o, float* part_ml, int B, int nkv, int max_len, int nsplit, cudaStream_t s) {
  return launch("attn_decode_split_kernel", attn_decode_split_kernel<HD, G>, dim3(nsplit, nkv, B), AD_THREADS, 0, s,
                false, q, kn, vn, kc, vc, pos, scale, part_o, part_ml, nkv, max_len, nsplit);
}

template <int HD>
int split_for_group(int G, const __half* q, const __half* kn, const __half* vn, __half* kc, __half* vc,
                    const int32_t* pos, float scale, float* part_o, float* part_ml, int B, int nkv, int max_len,
                    int nsplit, cudaStream_t s) {
  switch (G) {
    case 1: return launch_split<HD, 1>(q, kn, vn, kc, vc, pos, scale, part_o, part_ml, B, nkv, max_len, nsplit, s);
    case 2: return launch_split<HD, 2>(q, kn, vn, kc, vc, pos, scale, part_o, part_ml, B, nkv, max_len, nsplit, s);
    case 4: return launch_split<HD, 4>(q, kn, vn, kc, vc, pos, scale, part_o, part_ml, B, nkv, max_len, nsplit, s);
    case 8: return launch_split<HD, 8>(q, kn, vn, kc, vc, pos, scale, part_o, part_ml, B, nkv, max_len, nsplit, s);
  }
  set_error("quip_decode_attention: %d query heads per KV head is not supported (1, 2, 4 or 8)", G);
  return QUIP_ERR_UNSUPPORTED;
}

size_t workspace_bytes(int64_t B, int64_t nh, int64_t max_len, int64_t hd) {
  const int64_t nsplit = (max_len + AD_SPLIT - 1) / AD_SPLIT;
  return (size_t)(B * nh * nsplit * (hd + 2)) * sizeof(float);
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace

}  // namespace quip

using namespace quip;

extern "C" int quip_decode_attention_workspace_bytes(int32_t batch, int32_t n_heads, int32_t max_len, int32_t head_dim,
                                                     size_t* out_bytes) {
  QUIP_CHECK_ARG(out_bytes, "quip_decode_attention_workspace_bytes: null pointer");
  QUIP_CHECK_ARG(batch > 0 && n_heads > 0 && max_len > 0 && head_dim > 0,
                 "quip_decode_attention_workspace_bytes: sizes must be positive");
  *out_bytes = workspace_bytes(batch, n_heads, max_len, head_dim);
  return QUIP_OK;
}

extern "C" int quip_decode_attention(const void* q, const void* k_new, const void* v_new, void* k_cache, void* v_cache,
                                     const int32_t* pos, int32_t batch, int32_t n_heads, int32_t n_kv_heads,
                                     int32_t max_len, int32_t head_dim, float scale, void* out, void* workspace,
                                     size_t workspace_bytes_, void* stream) {
  QUIP_CHECK_ARG(q && k_new && v_new && k_cache && v_cache && pos && out && workspace,
                 "quip_decode_attention: null pointer");
  QUIP_CHECK_ARG(batch > 0 && batch <= 65535 && n_kv_heads > 0 && n_kv_heads <= 65535 && max_len > 0,
                 "quip_decode_attention: bad sizes (batch %d, kv heads %d, max_len %d)", batch, n_kv_heads, max_len);
  QUIP_CHECK_ARG(n_heads > 0 && n_heads % n_kv_heads == 0,
                 "quip_decode_attention: %d query heads are not a multiple of %d KV heads", n_heads, n_kv_heads);
  QUIP_CHECK_ARG(aligned16(q) && aligned16(k_new) && aligned16(v_new) && aligned16(k_cache) && aligned16(v_cache) &&
                 aligned16(out) && aligned16(workspace), "quip_decode_attention: pointers must be 16-byte aligned");
  if (head_dim != 64 && head_dim != 128) {
    set_error("quip_decode_attention: head_dim %d is not supported (64 or 128)", head_dim);
    return QUIP_ERR_UNSUPPORTED;
  }
  const size_t need = workspace_bytes(batch, n_heads, max_len, head_dim);
  if (workspace_bytes_ < need) {
    set_error("quip_decode_attention: workspace of %zu bytes, %zu needed", workspace_bytes_, need);
    return QUIP_ERR_WORKSPACE;
  }
  const int nsplit = ceil_div(max_len, AD_SPLIT);
  float* part_o = static_cast<float*>(workspace);
  float* part_ml = part_o + (size_t)batch * n_heads * nsplit * head_dim;
  const int G = n_heads / n_kv_heads;
  cudaStream_t s = (cudaStream_t)stream;
  const __half *qh = (const __half*)q, *kn = (const __half*)k_new, *vn = (const __half*)v_new;
  __half *kc = (__half*)k_cache, *vc = (__half*)v_cache;
  const int rc = head_dim == 64
                     ? split_for_group<64>(G, qh, kn, vn, kc, vc, pos, scale, part_o, part_ml, batch, n_kv_heads, max_len, nsplit, s)
                     : split_for_group<128>(G, qh, kn, vn, kc, vc, pos, scale, part_o, part_ml, batch, n_kv_heads, max_len, nsplit, s);
  if (rc != QUIP_OK) return rc;
  return launch("attn_decode_combine_kernel", attn_decode_combine_kernel, dim3(n_heads, batch), head_dim, 0, s, false,
                (const float*)part_o, (const float*)part_ml, pos, (__half*)out, (int)n_heads, (int)head_dim, (int)max_len,
                nsplit);
}
