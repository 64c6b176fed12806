/*
 * quip_b200 -- C ABI of the B200-native packed QuantLinear path.
 *
 * This is the boundary the reference's FFI for this path would bind.  The
 * reference (Cornell-RelaxML/QuIP) has exactly one native call site on the
 * path, the absent `quant_cuda` extension:
 *
 *     quant_cuda.vecquant3matmul(x, qweight, y, scales, zeros)   quant.py:229-230
 *     quant_cuda.vecquant4matmul(x, qweight, y, scales, zeros)   zeroShot/models/quant.py:207-208
 *
 * i.e. "y += (scales*code - zeros) . x" on a packed-integer matrix, called from
 * Quant3Linear.forward (quant.py:222-233).  quip_qlinear_forward() replaces that
 * call and, in the same launch sequence, the work the reference folds into its
 * dense fp16 weight at quantization time (method.py:195-214): the scaleWH
 * rescale and the U / V incoherence un-projection.  quip_pack_codes() replaces
 * the CPU/numpy packer Quant3Linear.pack (quant.py:185-220, TODO at opt.py:302);
 * quip_convert_ref() reads the reference's own 3-/4-bit layouts.
 *
 * Conventions: plain pointers and sizes, no torch types.  All data pointers are
 * DEVICE pointers unless a parameter says "host"; the caller owns every buffer;
 * calls are asynchronous on the `stream` handle (a cudaStream_t cast to void*);
 * no internal allocation -- scratch comes from the caller-provided workspace.
 * Every function returns 0 on success and a non-zero code on error, with a
 * human-readable message available from quip_last_error() (thread-local).
 * There is no CPU fallback: on a machine without an sm_100 device the launch
 * entry points return QUIP_ERR_CUDA.
 */
#ifndef QUIP_B200_H_
#define QUIP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QUIP_ABI_VERSION 2

enum {
  QUIP_OK = 0,
  QUIP_ERR_ARG = 1,        /* bad shape / null pointer / unsupported bits */
  QUIP_ERR_WORKSPACE = 2,  /* workspace too small */
  QUIP_ERR_CUDA = 3,       /* CUDA runtime / driver error (message has the detail) */
  QUIP_ERR_UNSUPPORTED = 4
};

/* One block-diagonal pass of a butterfly (reference method.py:58-63).
 * A side of size n is viewed as nblk blocks of p elements; block b is
 * multiplied by its own (or the shared) p x p factor:
 *     out[pos(b,i)] = sum_j factors[b or 0][i][j] * in[pos(b,j)]
 * pos(b,j) = b*p + j (strided == 0) or j*nblk + b (strided == 1). */
typedef struct {
  int32_t p;
  int32_t nblk;
  int32_t strided;
  int32_t shared;          /* 1: a single factor for every block (method.py:38-39, "noblock") */
  const void* factors;     /* fp16 [shared ? 1 : nblk][p][p], row-major */
  const void* factors_frag;/* optional copy of the same factors in tensor-core fragment order, or NULL.  Only read by
                              the one-kernel sides of the many-token forward (p in {32, 64}); without it those sides run
                              as separate gather / pass kernels with the same result.  Word
                              (((blk*(p/8) + nt)*(p/32) + j)*32 + lane)*4 + q  holds  F[blk][8nt + lane/4][k0], [k0+1]
                              with k0 = 32j + 16(q/2) + 8(q%2) + 2(lane%4): one 128-bit load per lane is two k-steps
                              of mma.m16n8k16 B fragments. */
} QuipPass;

/* One incoherence side: V acts on the K input features, U on the N outputs.
 * n == 0 means the side is absent (no --pre_proj). */
typedef struct {
  int32_t n;
  int32_t npass;           /* 0..2 */
  QuipPass pass[2];        /* execution order */
  const int32_t* idx;      /* gather index, length n, or NULL for identity:
                              V: layout[l] = x[idx[l]] ; U: y[j] = layout[idx[j]] */
  const int32_t* inv_idx;  /* optional inverse of idx (inv_idx[idx[j]] = j), or NULL.  With it the few-token
                              forward (M <= 8) writes the last U pass straight to y (one launch fewer); the
                              result is the same without it. */
} QuipSide;

/* A packed linear layer  y = ((x * inv_scale) V^T) Q^T U + bias,
 * Q[n][k] = scales[n]*code[n][k] - zeros[n]  (Quant3Linear convention, quant.py:186-191).
 * qweight is in the native fragment-major layout (DESIGN.md, oracle/packing.py), rows
 * and columns already in the U / V layout order, scales/zeros in the same row order. */
typedef struct {
  int32_t K, N, bits;      /* bits in {2,3,4}; K % 128 == 0; N % 16 == 0 */
  int32_t flags;           /* QUIP_FLAG_* */
  const int32_t* qweight;
  const float* scales;     /* (N) */
  const float* zeros;      /* (N) */
  const void* bias;        /* fp16 (N) in output-feature order, or NULL */
  const float* inv_scale;  /* fp32 (K) = 1/scaleWH in input-feature order, or NULL */
  QuipSide V, U;
} QuipLinearDesc;

#define QUIP_FLAG_SYMMETRIC 1   /* scales*cbar == zeros for every row: the row-sum term vanishes (qfn 'b') */

/* y (M,N) fp16 = forward of x (M,K) fp16.  Replaces Quant3Linear.forward's
 * vecquant3matmul call (quant.py:222-233) for any M >= 1. */
int quip_qlinear_forward(const QuipLinearDesc* d, const void* x, void* y, int64_t M,
                         void* workspace, size_t workspace_bytes, void* stream);
int quip_qlinear_workspace_bytes(const QuipLinearDesc* d, int64_t M, size_t* out_bytes);

/* Building blocks (also exported for tests and micro-benchmarks). */
/* z (M,N) fp16 = x2 (M,K) fp16 contracted with the packed matrix + affine epilogue (+bias if given).
 * xsum (M) fp32 row sums of x2, required unless QUIP_FLAG_SYMMETRIC.  path: 0 auto, 1 few-token kernels (32-token
 * chunks; needs the workspace), 2 tcgen05 kernel. */
int quip_qgemm(const QuipLinearDesc* d, const void* x2, const float* xsum, const void* bias,
               void* z, int64_t M, int path, void* workspace, size_t workspace_bytes, void* stream);
int quip_rowsum(const void* x, float* xsum, int64_t M, int32_t K, void* stream);
/* out[m][l] = in[m][idx[l]] * scale[idx[l]] (+ bias[l]);  idx / scale / bias may be NULL. */
int quip_gather(const void* in, void* out, int64_t M, int32_t n, const int32_t* idx,
                const float* scale, const void* bias, void* stream);
/* impl: 0 auto, 1 generic CUDA-core kernel, 2 tensor-core kernels only */
int quip_rot_pass(const QuipPass* pass, const void* in, void* out, int64_t M, int32_t n, int impl,
                  void* stream);

/* Glue of a Llama decoder layer between its packed linears: what the reference's eval loop gets from the HF layer it
 * calls (llama.py:227 `layer(inps[j].unsqueeze(0), attention_mask=..., position_ids=...)`: LlamaRMSNorm, the residual
 * adds, apply_rotary_pos_emb, SiLU(gate)*up), each as one HBM pass with the HF modules' fp16 rounding points.  All
 * tensors fp16, contiguous, 16-byte aligned.
 *   quip_rmsnorm   s = x (+ residual);  y = weight * fp16(s * rsqrt(mean(s^2) + eps));  s is written to sum_out when
 *                  given (residual and sum_out may be NULL; sum_out may alias x or residual).  d % 8 == 0, d <= 32768.
 *   quip_rope      in place on q (rows, n_q_heads*head_dim) and k (rows, n_kv_heads*head_dim) with cos/sin
 *                  (rows, head_dim): out = x*cos + rotate_half(x)*sin.  head_dim % 16 == 0; k may be NULL with 0 heads.
 *   quip_silu_mul  out = silu(gate) * up over n elements (n % 8 == 0); out may alias gate or up. */
int quip_rmsnorm(const void* x, const void* residual, const void* weight, void* sum_out, void* y,
                 int64_t rows, int32_t d, float eps, void* stream);
int quip_rope(void* q, void* k, const void* cos, const void* sin, int64_t rows, int32_t n_q_heads,
              int32_t n_kv_heads, int32_t head_dim, void* stream);
int quip_silu_mul(const void* gate, const void* up, void* out, int64_t n, void* stream);
/*   quip_silu_mul_gather  the same product with the permutations of the surrounding incoherence sides folded in:
 *                  out[r][l] = silu(gate[r][idx[l] & 0xFFFF]) * up[r][idx[l] >> 16] for rows of n < 65536 features; gate / up
 *                  are the projections in their N-side layout order (quip_qlinear_forward with U.idx = NULL), out feeds a
 *                  forward with V.idx = NULL: idx[l] = u_idx_gate[v_idx_down[l]] | u_idx_up[v_idx_down[l]] << 16. */
int quip_silu_mul_gather(const void* gate, const void* up, const uint32_t* idx, void* out, int64_t rows, int32_t n,
                         void* stream);

/* One decode step of attention for `batch` sequences over a static KV cache (quip_b200/generate.py).  fp16 tensors,
 * 16-byte aligned: q (batch, n_heads*head_dim) and k_new, v_new (batch, n_kv_heads*head_dim) token-major, as the
 * projections produce them (after rotary for Llama; q already scaled for OPT); k_cache, v_cache (batch, n_kv_heads,
 * max_len, head_dim); pos (batch) int32, the position this step writes.  Sequence b stores k_new / v_new at pos[b] and
 * attends to positions 0 .. pos[b]:  out (batch, n_heads*head_dim) = softmax(scale * q K^T) V, softmax and sums in fp32,
 * the query heads h of a KV head being h / (n_heads / n_kv_heads).  Only valid cache rows are read; long contexts are
 * split along the sequence and the fp32 partials, kept in the workspace, are merged in a fixed order (deterministic).
 * head_dim 64 or 128 and 1, 2, 4 or 8 query heads per KV head, else QUIP_ERR_UNSUPPORTED.  pos[b] must lie in
 * 0 .. max_len-1 (the caller's check); a row outside it is not stored and its output is NaN. */
int quip_decode_attention(const void* q, const void* k_new, const void* v_new, void* k_cache, void* v_cache,
                          const int32_t* pos, int32_t batch, int32_t n_heads, int32_t n_kv_heads, int32_t max_len,
                          int32_t head_dim, float scale, void* out, void* workspace, size_t workspace_bytes,
                          void* stream);
int quip_decode_attention_workspace_bytes(int32_t batch, int32_t n_heads, int32_t max_len, int32_t head_dim,
                                          size_t* out_bytes);

/* Signature-compatible replacement of the reference's own native call (quant_cuda.vecquant3matmul quant.py:229-230,
 * vecquant4matmul zeroShot/models/quant.py:207-208): ONE token, fp32, on the REFERENCE's packed layout
 * (bits 3: int32 (K*3/32, N) as Quant3Linear.pack writes it; bits 4: (K/8, N); bits 2: (K/16, N)):
 *     mul[n] += sum_k (scales[n] * code[k][n] - zeros[n]) * vec[k]        (in-place accumulate, like the reference's call)
 * so a checkpoint packed by the reference runs without conversion.  K % 32 == 0.  quip_qlinear_forward on the native
 * layout is the fast path; this one is a plain HBM-streaming kernel. */
int quip_vecquant_matmul(const float* vec, const int32_t* mat, float* mul, const float* scales, const float* zeros,
                         int32_t K, int32_t N, int32_t bits, void* stream);

/* codes (N,K) uint8 row-major <-> native packed layout.  Replaces Quant3Linear.pack (quant.py:185-220). */
int quip_pack_codes(const uint8_t* codes_nk, int32_t N, int32_t K, int32_t bits, int32_t* qweight,
                    void* stream);
int quip_unpack_codes(const int32_t* qweight, int32_t N, int32_t K, int32_t bits, uint8_t* codes_nk,
                      void* stream);
/* Reference layouts -> codes (N,K): bits=3 quant.py:192-220 [(K*3/32, N) int32], bits=4
 * zeroShot/models/quant.py:193-199 [(K/8, N)], bits=2 the natural extension [(K/16, N)]. */
int quip_convert_ref(const int32_t* ref_qweight, int32_t K, int32_t N, int32_t bits,
                     uint8_t* codes_nk, void* stream);
size_t quip_packed_words(int32_t N, int32_t K, int32_t bits);

/* Quantisation-time hot loop (SURVEY section 8f rank 1): the column-sequential part of LDLQ rounding for one block of
 * <= 128 columns, all rows in one launch (reference: the Python column loops of round_ldl / round_ldl_block,
 * vector_balance.py:155-199, :218-257).  All matrices fp32, column-major over rows ("transposed": element (row r,
 * column j) at [j*ld + r]); the feedback of the finished blocks is the caller's GEMM (quip_b200/quantize.py).
 *   quip_ldlq_block    q[:, j] = clamp(floor(base[:, j] + sum_{j' > j} err[:, j'] * Lb[j'][j] + 1/2), 0, 2^bits - 1),
 *                      err[:, j] = w[:, j] - q[:, j], for j = cnt-1 .. 0.  base = w[:, blk] + err[:, done] @ L[done, blk];
 *                      Lb (cnt, cnt) row-major = L[blk, blk] - I (unit-lower LDL factor of H, strictly lower part read).
 *   quip_greedy_block  one coordinate-descent sweep over the block (vector_balance.py:267-283): for i = cnt-1 .. 0,
 *                      move = wr_i - rint(wr_i - (pre_i + sum_j s_j Hb[j][i]) / Hb[i][i]); wr_i -= move; s_i -= move.
 *                      pre = s[:, outside blk] @ Hn[outside, blk]; Hb = Hn[blk, blk]; wr, s updated in place. */
int quip_ldlq_block(const float* baseT, const float* wT, const float* Lb, float* qT, float* errT, int64_t m, int64_t ld,
                    int32_t cnt, int32_t bits, void* stream);
int quip_greedy_block(const float* preT, const float* Hb, float* wrT, float* sT, int64_t m, int64_t ld, int32_t cnt,
                      void* stream);

/* Calibration Hessian (SURVEY section 8f rank 2; reference QuantMethod.add_batch, method.py:98-120): H += X^T X for
 * X (tokens, K) fp16 row-major, H (K, K) float64 row-major.  Products on the fp16 tensor cores (exact in float32), float32
 * sums over 256 tokens, float64 carry in H.  Only the upper BLOCK triangle of 128 x 128 tiles is updated (tile row <= tile
 * column, diagonal tiles whole): mirror it once after the last batch.  K % 8 == 0. */
int quip_hessian_accumulate(const void* x, double* H, int64_t tokens, int32_t K, void* stream);

/* Optional per-launch timing of the contraction kernels with CUDA events recorded on the launch stream
 * (bench.py's roofline leg).  path: 1 = mma.sync skinny kernel, 2 = tcgen05 kernel.  quip_timing_read
 * waits for the recorded events and returns the totals since the last reset: device milliseconds,
 * launches, algorithmic flops (2*M*N*K) and algorithmic bytes (packed codes + fp16 activations in + out). */
int quip_timing_enable(int on);
int quip_timing_reset(void);
int quip_timing_read(int path, double* total_ms, int64_t* launches, double* flops, double* bytes);

/* Routing switches for ablations, tests and micro-benchmarks (defaults in parentheses); results do not depend on them.
 *   "side_fused" (1)  M > 8: a whole incoherence side in one kernel when both blocks are 32/64 wide and factors_frag is set
 *   "fewtok" (1)      M <= 8: few-token pass / gather kernels (fused input gather, output scatter + bias)
 *   "fewtok_max_m" (32) 8..32: token count up to which the few-token passes run (batched decode)
 *   "side_fewtok" (0) M <= 8: both passes of a side (+ gather / scatter, bias) in one launch: side, contraction, side
 *                     (ablation: measured slower than the two-pass route, see profiles/README.md)
 *   "pdl" (1)         programmatic dependent launch along the few-token chain
 *   "gemv" (1)        M <= 8: whole-K qgemv kernels (0: split-K mma.sync kernel)
 *   "gv_int" (1)      qgemv: int8 tensor-core path for 2-/4-bit and <= 5 tokens (0: fp16 path)
 *   "gv_tma" (1), "gv_cw" (16), "gv_rbc" (0 = auto), "gv_persist" (1)   variants of the cooperative int8 kernel
 *   "gv_stream" (32)  streaming int8 kernel when N/16 >= value * SMs (0: never)
 *   "sk_ksplit" (0)   split-K kernel (9..32 tokens): cap on the number of K splits, only ever lowering the heuristic's choice
 *                     (the workspace is sized for that); 0 = the heuristic
 *   "gather_rows", "pass_min_tiles"   tune the many-token un-projection kernels */
int quip_config(const char* key, int value);

const char* quip_last_error(void);
int quip_abi_version(void);
/* Number of kernels this library has launched on behalf of the calling process (for bench gpu_launches). */
int64_t quip_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* QUIP_B200_H_ */
