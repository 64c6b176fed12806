// GPU packers: codes (N,K) uint8 <-> native fragment-major layout, and readers for the
// reference's packed layouts.  Replaces the CPU/numpy loop of Quant3Linear.pack
// (reference quant.py:185-220; TODO "perform packing on GPU" at opt.py:302).
// Layout definition: oracle/packing.py (the checker) and DESIGN.md.
#include "common.cuh"

namespace quip {

// coordinates of element (n, k) inside the native layout
struct Coord {
  int64_t sb;     // super-block index
  int lane, ch, pos, hi_row;
};
__device__ __forceinline__ Coord coord_of(int n, int k, int K) {
  Coord c;
  int rb = n >> 4, r = n & 15;
  int g = r & 7;
  c.hi_row = r >> 3;
  int ks = k >> 7, kk = k & 127;
  c.ch = kk >> 5;
  int t = (kk & 31) >> 3;
  c.pos = kk & 7;
  c.lane = g * 4 + t;
  c.sb = (int64_t)rb * (K >> 7) + ks;
  return c;
}

// (word index, bit shift) of the main plane; for bits==3 this is the hi plane (code >> 1)
template <int BITS>
__device__ __forceinline__ void locate(const Coord& c, int64_t& word, int& shift) {
  int e = c.pos & 1;
  int64_t base = c.sb * sb_words(BITS);
  if (BITS == 4) {
    int w = c.pos >> 2;
    int jp = slot4((c.pos & 3) >> 1, c.hi_row);
    word = base + (c.ch >> 1) * 128 + c.lane * 4 + (c.ch & 1) * 2 + w;
    shift = 4 * jp + 16 * e;
  } else {
    int j = slot2(c.pos >> 1, c.hi_row);
    word = base + c.lane * 4 + c.ch;
    shift = 2 * j + 16 * e;
  }
}
__device__ __forceinline__ void locate_lo3(const Coord& c, int64_t& word, int& shift) {
  int j = slot2(c.pos >> 1, c.hi_row);
  word = c.sb * sb_words(3) + 128 + c.lane * 2 + (c.ch >> 1);
  shift = 8 * (c.ch & 1) + j + 16 * (c.pos & 1);
}

// One thread per (row n, 8 consecutive k): the 8 codes of one lane-run, i.e. one byte row.
// Threads OR their fields into the words with atomics-free ownership: a word is shared by rows
// g / g+8 and (bits=2) both halves, so build per-(sb,lane,ch) words in one thread instead.
template <int BITS>
__global__ void pack_kernel(const uint8_t* __restrict__ codes, int N, int K, uint32_t* __restrict__ q) {
  // one thread per (super-block, lane, chunk): owns rows {g, g+8} x 8 k = 16 codes
  int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = (int64_t)(N >> 4) * (K >> 7) * 32 * 4;
  if (tid >= total) return;
  int ch = tid & 3;
  int lane = (tid >> 2) & 31;
  int64_t sb = tid >> 7;
  int ks = sb % (K >> 7);
  int rb = sb / (K >> 7);
  int g = lane >> 2, t = lane & 3;
  int k0 = ks * 128 + ch * 32 + t * 8;
  uint32_t c[2][8];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const uint8_t* src = codes + (int64_t)(rb * 16 + g + 8 * h) * K + k0;
    uint2 v = *reinterpret_cast<const uint2*>(src);      // k0 % 8 == 0 and K % 128 == 0 -> aligned
    uint32_t w[2] = {v.x, v.y};
#pragma unroll
    for (int i = 0; i < 8; ++i) c[h][i] = (w[i >> 2] >> (8 * (i & 3))) & 0xFFu;
  }
  const uint32_t cm = (1u << BITS) - 1u;
  int64_t base = sb * sb_words(BITS);
  if (BITS == 2 || BITS == 3) {
    uint32_t w = 0, lo = 0;
#pragma unroll
    for (int pos = 0; pos < 8; ++pos)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        int j = slot2(pos >> 1, h);
        uint32_t code = c[h][pos] & cm;
        uint32_t top = BITS == 3 ? (code >> 1) : code;
        w |= top << (2 * j + 16 * (pos & 1));
        lo |= (code & 1u) << (j + 16 * (pos & 1));
      }
    q[base + lane * 4 + ch] = w;
    if (BITS == 3) {
      // lo word is shared by chunks (ch, ch^1): 8 pair slots each -> two threads write disjoint bit
      // ranges of the same word; combine with an atomic OR (buffer is zero-initialised by the caller)
      atomicOr(&q[base + 128 + lane * 2 + (ch >> 1)], lo << (8 * (ch & 1)));
    }
  } else {
    uint32_t w[2] = {0, 0};
#pragma unroll
    for (int pos = 0; pos < 8; ++pos)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        int jp = slot4((pos & 3) >> 1, h);
        w[pos >> 2] |= (c[h][pos] & cm) << (4 * jp + 16 * (pos & 1));
      }
    int64_t wi = base + (ch >> 1) * 128 + lane * 4 + (ch & 1) * 2;
    *reinterpret_cast<uint2*>(&q[wi]) = make_uint2(w[0], w[1]);
  }
}

template <int BITS>
__global__ void unpack_kernel(const uint32_t* __restrict__ q, int N, int K, uint8_t* __restrict__ codes) {
  int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= (int64_t)N * K) return;
  int n = tid / K, k = tid % K;
  Coord c = coord_of(n, k, K);
  int64_t word;
  int shift;
  locate<BITS>(c, word, shift);
  uint32_t code;
  if (BITS == 3) {
    code = ((q[word] >> shift) & 3u) << 1;
    locate_lo3(c, word, shift);
    code |= (q[word] >> shift) & 1u;
  } else {
    code = (q[word] >> shift) & ((1u << BITS) - 1u);
  }
  codes[tid] = (uint8_t)code;
}

// reference layouts: qweight (K*bits/32, N) int32, packed along K (quant.py:192-220,
// zeroShot/models/quant.py:193-199)
template <int BITS>
__global__ void convert_ref_kernel(const uint32_t* __restrict__ q, int K, int N, uint8_t* __restrict__ codes) {
  int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= (int64_t)N * K) return;
  int k = tid / N, n = tid % N;            // threads run along N: coalesced reads of the (rows, N) matrix
  uint32_t code;
  if (BITS == 4) {
    code = (q[(int64_t)(k >> 3) * N + n] >> (4 * (k & 7))) & 15u;
  } else if (BITS == 2) {
    code = (q[(int64_t)(k >> 4) * N + n] >> (2 * (k & 15))) & 3u;
  } else {
    int p = k & 31;
    const uint32_t* row = q + (int64_t)(k >> 5) * 3 * N + n;
    uint32_t r0 = row[0], r1 = row[N], r2 = row[2 * (int64_t)N];
    if (p < 10) code = (r0 >> (3 * p)) & 7u;
    else if (p == 10) code = (r0 >> 30) | ((r1 & 1u) << 2);
    else if (p < 21) code = (r1 >> (3 * (p - 11) + 1)) & 7u;
    else if (p == 21) code = (r1 >> 31) | ((r2 & 3u) << 1);
    else code = (r2 >> (3 * (p - 22) + 2)) & 7u;
  }
  codes[(int64_t)n * K + k] = (uint8_t)code;
}

}  // namespace quip

using namespace quip;

extern "C" size_t quip_packed_words(int32_t N, int32_t K, int32_t bits) {
  if (N <= 0 || K <= 0 || N % SB_ROWS || K % SB_K || bits < 2 || bits > 4) return 0;
  return (size_t)(N / SB_ROWS) * (K / SB_K) * sb_words(bits);
}

static int check_shape(int N, int K, int bits) {
  QUIP_CHECK_ARG(bits >= 2 && bits <= 4, "bits must be 2, 3 or 4 (got %d)", bits);
  QUIP_CHECK_ARG(N > 0 && N % SB_ROWS == 0, "N=%d must be a positive multiple of 16", N);
  QUIP_CHECK_ARG(K > 0 && K % SB_K == 0, "K=%d must be a positive multiple of 128", K);
  return QUIP_OK;
}

extern "C" int quip_pack_codes(const uint8_t* codes, int32_t N, int32_t K, int32_t bits, int32_t* qweight,
                               void* stream) {
  if (int e = check_shape(N, K, bits)) return e;
  QUIP_CHECK_ARG(codes && qweight, "null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  int64_t total = (int64_t)(N / 16) * (K / 128) * 128;
  int grid = ceil_div(total, 256);
  uint32_t* q = reinterpret_cast<uint32_t*>(qweight);
  if (bits == 3) QUIP_CUDA(cudaMemsetAsync(q, 0, quip_packed_words(N, K, 3) * 4, s));
  auto kern = bits == 2 ? pack_kernel<2> : (bits == 3 ? pack_kernel<3> : pack_kernel<4>);
  return launch("pack_kernel", kern, grid, 256, 0, s, false, codes, N, K, q);
}

extern "C" int quip_unpack_codes(const int32_t* qweight, int32_t N, int32_t K, int32_t bits, uint8_t* codes,
                                 void* stream) {
  if (int e = check_shape(N, K, bits)) return e;
  QUIP_CHECK_ARG(codes && qweight, "null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  int grid = ceil_div((int64_t)N * K, 256);
  const uint32_t* q = reinterpret_cast<const uint32_t*>(qweight);
  auto kern = bits == 2 ? unpack_kernel<2> : (bits == 3 ? unpack_kernel<3> : unpack_kernel<4>);
  return launch("unpack_kernel", kern, grid, 256, 0, s, false, q, N, K, codes);
}

extern "C" int quip_convert_ref(const int32_t* ref_qweight, int32_t K, int32_t N, int32_t bits, uint8_t* codes,
                                void* stream) {
  QUIP_CHECK_ARG(bits >= 2 && bits <= 4, "bits must be 2, 3 or 4 (got %d)", bits);
  QUIP_CHECK_ARG(N > 0 && K > 0 && K % 32 == 0, "reference layouts need K %% 32 == 0 (K=%d, N=%d)", K, N);
  QUIP_CHECK_ARG(codes && ref_qweight, "null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  int grid = ceil_div((int64_t)N * K, 256);
  const uint32_t* q = reinterpret_cast<const uint32_t*>(ref_qweight);
  auto kern = bits == 2 ? convert_ref_kernel<2> : (bits == 3 ? convert_ref_kernel<3> : convert_ref_kernel<4>);
  return launch("convert_ref_kernel", kern, grid, 256, 0, s, false, q, K, N, codes);
}
