// Shared helpers for the quip_b200 sm_100a kernels.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <algorithm>
#include <atomic>
#include <utility>

#include "../../include/quip_b200.h"

namespace quip {

// ---- error plumbing (thread-local message, C ABI returns codes) -------------
void set_error(const char* fmt, ...);

#define QUIP_CHECK_ARG(cond, ...)            \
  do {                                       \
    if (!(cond)) {                           \
      quip::set_error(__VA_ARGS__);          \
      return QUIP_ERR_ARG;                   \
    }                                        \
  } while (0)

#define QUIP_CUDA(expr)                                                                  \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess) {                                                             \
      quip::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__,  \
                      __LINE__);                                                         \
      return QUIP_ERR_CUDA;                                                              \
    }                                                                                    \
  } while (0)

// ---- kernel launches (api.cu) -----------------------------------------------------
extern std::atomic<int64_t> g_launches;   // quip_launch_count
extern int g_pdl;                         // quip_config("pdl")

// Raise kern's max-dynamic-shared-memory attribute on the current device to smem, once per (kernel, device) and size;
// the attribute is never lowered.
cudaError_t raise_smem_limit(const void* kern, size_t smem);
int num_sms();                                                     // of the current device
int blocks_per_sm(const void* kern, int threads, size_t smem);     // occupancy (>= 1), cached per kernel, device and shape

// Every kernel of the library starts here: kern<<<grid, block, smem, s>>>(args...), the shared-memory opt-in included,
// counted in quip_launch_count.  The arguments convert to the kernel's parameter types as in a call.  With pdl (and
// quip_config("pdl") on) the kernel may start while its predecessor in the stream drains (programmatic dependent
// launch); everything it does before griddepcontrol.wait must then be independent of that predecessor.
template <class... P, class... A>
int launch(const char* name, void (*kern)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, bool pdl,
           A&&... args) {
  cudaError_t e = raise_smem_limit((const void*)kern, smem);
  if (e == cudaSuccess) {
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cfg.attrs = attr;
    cfg.numAttrs = pdl && g_pdl ? 1 : 0;
    e = cudaLaunchKernelEx(&cfg, kern, std::forward<A>(args)...);
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("launch of %s failed: %s", name, cudaGetErrorString(e));
    return QUIP_ERR_CUDA;
  }
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return QUIP_OK;
}

// ---- entry points shared between the .cu files --------------------------------
// quip_config switches
extern int g_gather_rows, g_pass_min_tiles, g_fewtok;                     // rot.cu
extern int g_fewtok_max_m;                                                // rot_fewtok.cu: token count up to which the few-token kernels run
extern int g_gv_rbc, g_gv_persist, g_gv_int, g_gv_tma, g_gv_cw, g_gv_stream;  // qgemv.cu

// contractions (qgemm_skinny.cu, qgemv.cu, qgemm_tc.cu)
int qgemm_skinny(const QuipLinearDesc* d, const __half* x, const __half* bias, __half* z, int M, int ksplit,
                 float* part, int* counters, cudaStream_t s);
int skinny_pick_ksplit(int N, int K, int rows_per_cta, int M);
size_t skinny_workspace_bytes(int N, int M, int ksplit);
int qgemv(const QuipLinearDesc* d, const __half* x, const __half* bias, __half* z, int M, cudaStream_t s);
bool qgemv_fits(int K, int M, int bits);
int qgemm_tc(const QuipLinearDesc* d, const __half* x, const float* xsum, const __half* bias, __half* z, int M,
             cudaStream_t s);

// passes and gathers (rot_fewtok.cu, rot_small.cu, rot_side.cu, rot_side_fewtok.cu, qgemm_tc.cu)
bool pass_fewtok_ok(const QuipPass* ps, int64_t M, int n);
int pass_fewtok(const QuipPass* ps, const __half* in, __half* out, int64_t M, int n, const int32_t* in_idx,
                const float* in_scale, const int32_t* out_inv, const __half* out_bias, cudaStream_t s);
int gather_fewtok(const __half* in, __half* out, int64_t M, int n, const int32_t* idx, const float* scale,
                  const __half* bias, cudaStream_t s);
int launch_small_fast(const QuipPass* ps, const __half* in, __half* out, int64_t M, int n, cudaStream_t s, bool* handled);
int pass_big_tc(const QuipPass* ps, const __half* in, __half* out, int64_t M, int n, cudaStream_t s);
bool side_fused_ok(const QuipSide* sd, int n);
int side_fused(const QuipSide* sd, const __half* in, __half* out, int64_t M, const int32_t* in_idx, const float* in_scale,
               const int32_t* out_idx, const __half* out_bias, float* xsum, cudaStream_t s);
bool side_fewtok_ok(const QuipSide* sd, int n, int64_t M);   // both passes of a side in one launch, M <= 8
int side_fewtok(const QuipSide* sd, const __half* in, __half* out, int64_t M, int n, const int32_t* in_idx,
                const float* in_scale, const int32_t* out_inv, const __half* out_bias, cudaStream_t s);

constexpr int SB_ROWS = 16;   // super-block: 16 rows x 128 k  (oracle/packing.py)
constexpr int SB_K = 128;
__host__ __device__ constexpr int sb_words(int bits) { return bits == 2 ? 128 : (bits == 3 ? 192 : 256); }

static inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// ---- device helpers ---------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}

__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ uint2 ldg_nc_v2(const void* p) {
  uint2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  return r;
}

// mma.sync m16n8k16, fp16 inputs, fp32 accumulate (legacy tensor path; used by the
// HBM-bound skinny kernel and the small block-diagonal rotation passes)
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
      "{%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// ---- code -> fp16 "d = (c - cbar) / 2^bits" expansion ------------------------------
// A pair of codes sits at bits [lo, lo+q) and [16+lo, 16+lo+q) of a word.  One shift moves
// them to the top of the two fp16 mantissas, one LOP3 masks and ORs the exponent of 1.0, so the
// halves read 1 + c/2^q; one HADD2 recentres.  (c - cbar)/2^q is exact in fp16 for q <= 4.
template <int BITS>
struct Dq {
  static constexpr uint32_t kMask = BITS == 2 ? 0x03000300u : (BITS == 3 ? 0x03800380u : 0x03C003C0u);
  static constexpr uint32_t kOne = 0x3C003C00u;
  // -(1 + cbar/2^bits): 2-bit -1.375, 3-bit -1.4375, 4-bit -1.46875
  static constexpr uint32_t kNegCenter = BITS == 2 ? 0xBD80BD80u : (BITS == 3 ? 0xBDC0BDC0u : 0xBDE0BDE0u);
};

__device__ __forceinline__ uint32_t hadd2_u32(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("add.rn.f16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}

// pair at field offset `lo` (compile-time) of a plane with Q bits per code, destination mantissa bit DST
template <int LO, int DST>
__device__ __forceinline__ uint32_t shift_to(uint32_t w) {
  if constexpr (LO < DST) return w << (DST - LO);
  else if constexpr (LO > DST) return w >> (LO - DST);
  else return w;
}

// 2-bit word (8 pairs j at bits 2j / 16+2j) -> pair j as fp16x2 of d
template <int J>
__device__ __forceinline__ uint32_t dq2(uint32_t w) {
  uint32_t v = (shift_to<2 * J, 8>(w) & Dq<2>::kMask) | Dq<2>::kOne;
  return hadd2_u32(v, Dq<2>::kNegCenter);
}
// 4-bit word (4 pairs j at bits 4j / 16+4j)
template <int J>
__device__ __forceinline__ uint32_t dq4(uint32_t w) {
  uint32_t v = (shift_to<4 * J, 6>(w) & Dq<4>::kMask) | Dq<4>::kOne;
  return hadd2_u32(v, Dq<4>::kNegCenter);
}
// 3-bit: hi word as 2-bit (pair J), lo word holds pair JJ at bits JJ / 16+JJ
template <int J, int JJ>
__device__ __forceinline__ uint32_t dq3(uint32_t whi, uint32_t wlo) {
  uint32_t v = (shift_to<2 * J, 8>(whi) & 0x03000300u) | Dq<3>::kOne;
  v |= shift_to<JJ, 7>(wlo) & 0x00800080u;
  return hadd2_u32(v, Dq<3>::kNegCenter);
}

// Bit layout of one (lane, chunk) word group: 16 codes = rows {g, g+8} x the lane's 8 consecutive k.
// Three consumers read the same bits, each with the cheapest extraction its datapath allows:
//   * IMMA.16832 (qgemv.cu, 1-5 tokens): the four A registers are  w & 0x03030303, w & 0x0C0C0C0C,
//     (w>>4) & 0x03030303, (w>>4) & 0x0C0C0C0C  -- byte j of the word holds "slot" j (bits 0-1 row g,
//     2-3 row g+8) and slot 4+j (bits 4-5, 6-7);
//   * HMMA.16816 / tcgen05 (fp16): a register is a pair of codes of one row at the same offset of the low
//     and high half-word -- slots (j, j+2) -- so slot s stands for k offset {0,2,1,3,4,6,5,7}[s] and every
//     fp16x2 register holds two consecutive k.
// In half-word terms: pair (u = pos/2, row half r) sits at bit 2*slot2(u,r) of each half.  4-bit: word
// pos/4, nibble slot4(u%2, r) of each half (byte j: low nibble row g, high nibble row g+8).
__host__ __device__ constexpr int slot2(int u, int r) { return 2 * ((u & 1) * 2 + (u >> 1)) + r; }
__host__ __device__ constexpr int slot4(int uw, int r) { return 2 * uw + r; }

// Expand one (lane, chunk): 16 codes -> 8 fp16x2 registers h[2u + r] (k pair u, row half r).
// MMA step s (k positions 4s..4s+3) uses a0..a3 = h[4s..4s+3].
// words: bits=2 -> w[0]; bits=4 -> w[0] (pos 0-3), w[1] (pos 4-7); bits=3 -> w[0] hi, w[1] lo with LOSEL
template <int BITS, int LOSEL = 0>
__device__ __forceinline__ void expand_chunk(uint32_t w0, uint32_t w1, uint32_t (&h)[8]) {
  if constexpr (BITS == 2) {
    h[0] = dq2<slot2(0, 0)>(w0); h[1] = dq2<slot2(0, 1)>(w0); h[2] = dq2<slot2(1, 0)>(w0); h[3] = dq2<slot2(1, 1)>(w0);
    h[4] = dq2<slot2(2, 0)>(w0); h[5] = dq2<slot2(2, 1)>(w0); h[6] = dq2<slot2(3, 0)>(w0); h[7] = dq2<slot2(3, 1)>(w0);
  } else if constexpr (BITS == 4) {
    h[0] = dq4<slot4(0, 0)>(w0); h[1] = dq4<slot4(0, 1)>(w0); h[2] = dq4<slot4(1, 0)>(w0); h[3] = dq4<slot4(1, 1)>(w0);
    h[4] = dq4<slot4(0, 0)>(w1); h[5] = dq4<slot4(0, 1)>(w1); h[6] = dq4<slot4(1, 0)>(w1); h[7] = dq4<slot4(1, 1)>(w1);
  } else {
    constexpr int B = 8 * LOSEL;
    h[0] = dq3<slot2(0, 0), B + slot2(0, 0)>(w0, w1); h[1] = dq3<slot2(0, 1), B + slot2(0, 1)>(w0, w1);
    h[2] = dq3<slot2(1, 0), B + slot2(1, 0)>(w0, w1); h[3] = dq3<slot2(1, 1), B + slot2(1, 1)>(w0, w1);
    h[4] = dq3<slot2(2, 0), B + slot2(2, 0)>(w0, w1); h[5] = dq3<slot2(2, 1), B + slot2(2, 1)>(w0, w1);
    h[6] = dq3<slot2(3, 0), B + slot2(3, 0)>(w0, w1); h[7] = dq3<slot2(3, 1), B + slot2(3, 1)>(w0, w1);
  }
}

}  // namespace quip
