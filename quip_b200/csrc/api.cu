// C-ABI entry points (include/quip_b200.h) and the launch sequence of one packed-linear forward.
//
//   y = ((x * inv_scale)[idx_V] -> V passes) . Q^T -> U passes -> [idx_U] + bias
//
// replaces Quant3Linear.forward -> quant_cuda.vecquant3matmul (reference quant.py:222-233) and the
// un-projection the reference bakes into its dense weight (method.py:195-214).
#include <stdarg.h>
#include <string.h>

#include <map>
#include <mutex>
#include <tuple>
#include <vector>

#include "common.cuh"

namespace quip {

static thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// tuning knobs (quip_config)
static int g_side_fused = 1;     // many tokens: a whole side (gather + both passes [+ row sums]) in one kernel when the blocks allow
int g_pdl = 1;                   // few-token kernels: programmatic dependent launch (weights prefetched under the previous kernel)
static int g_use_gemv = 1;       // few-token contractions: whole-K qgemv kernel (0: the split-K kernel)
static int g_sk_ksplit = 0;      // split-K kernel: cap on the number of K splits (0: the heuristic of skinny_pick_ksplit)
static int g_side_fewtok = 0;    // <= 8 tokens: both passes of a side in ONE launch (rot_side_fewtok.cu), 3 launches per linear.
                                 // Correct on every shape but measured SLOWER than two pass launches (every CTA stages the whole
                                 // token vector): an ablation, off by default (profiles/README.md)

// ---- launch plumbing (common.cuh: launch) ----
// The attribute and the occupancy query cost more host time than a decode kernel runs: both are cached.
static std::mutex g_launch_mu;
static std::map<std::pair<const void*, int>, size_t> g_smem_limit;                   // (kernel, device) -> bytes set
static std::map<std::tuple<const void*, int, int, size_t>, int> g_occupancy;         // (kernel, device, threads, smem)
static std::map<int, int> g_sms;                                                      // device -> SM count

cudaError_t raise_smem_limit(const void* kern, size_t smem) {
  if (smem == 0) return cudaSuccess;
  int dev = 0;
  if (cudaError_t e = cudaGetDevice(&dev)) return e;
  std::lock_guard<std::mutex> lock(g_launch_mu);
  size_t& set = g_smem_limit[{kern, dev}];
  if (smem <= set) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess) set = smem;
  return e;
}

int num_sms() {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  std::lock_guard<std::mutex> lock(g_launch_mu);
  int& sms = g_sms[dev];
  if (!sms) sms = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess ? n : 148;
  return sms;
}

// 1 when the query fails: the launch that follows reports the error
int blocks_per_sm(const void* kern, int threads, size_t smem) {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || raise_smem_limit(kern, smem) != cudaSuccess) return 1;
  std::lock_guard<std::mutex> lock(g_launch_mu);
  int& occ = g_occupancy[{kern, dev, threads, smem}];
  if (!occ) occ = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, threads, smem) == cudaSuccess && n > 1 ? n : 1;
  return occ;
}

constexpr size_t WS_HEADER = 16 * 1024;     // split-K arrival counters; must be zero on first use, left zero
constexpr int SKINNY_MAX_M = 32;

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct WsPlan {
  size_t xsum, bufA, bufB, zbuf, bufC, part, total;
};

static bool side_on(const QuipSide& s) { return s.n > 0 && (s.npass > 0 || s.idx != nullptr); }

static WsPlan plan_ws(const QuipLinearDesc* d, int64_t M) {
  WsPlan p{};
  size_t off = WS_HEADER;
  p.xsum = off; off += align_up((size_t)M * sizeof(float), 256);
  const bool v_on = side_on(d->V) || d->inv_scale;
  const bool u_on = side_on(d->U);
  size_t xk = align_up((size_t)M * d->K * sizeof(__half), 256);
  size_t xn = align_up((size_t)M * d->N * sizeof(__half), 256);
  p.bufA = off; if (v_on) off += xk;
  p.bufB = off; if (v_on) off += xk;
  p.zbuf = off; if (u_on) off += xn;
  p.bufC = off; if (u_on) off += xn;
  p.part = off;
  // split-K partials of the few-token contraction: for M itself when it is small, else for one 32-token chunk (quip_qgemm
  // path 1 walks a larger M in chunks)
  const int mc = M <= SKINNY_MAX_M ? (int)M : SKINNY_MAX_M;
  off += align_up(skinny_workspace_bytes(d->N, mc, skinny_pick_ksplit(d->N, d->K, 64, mc)), 256);
  p.total = off;
  return p;
}

static int check_desc(const QuipLinearDesc* d) {
  QUIP_CHECK_ARG(d != nullptr, "null descriptor");
  QUIP_CHECK_ARG(d->bits >= 2 && d->bits <= 4, "bits must be 2, 3 or 4 (got %d)", d->bits);
  QUIP_CHECK_ARG(d->K > 0 && d->K % 128 == 0, "K=%d must be a positive multiple of 128", d->K);
  QUIP_CHECK_ARG(d->N > 0 && d->N % 16 == 0, "N=%d must be a positive multiple of 16", d->N);
  QUIP_CHECK_ARG(d->qweight && d->scales && d->zeros, "qweight / scales / zeros must be set");
  QUIP_CHECK_ARG(d->V.n == 0 || d->V.n == d->K, "V side size %d != K %d", d->V.n, d->K);
  QUIP_CHECK_ARG(d->U.n == 0 || d->U.n == d->N, "U side size %d != N %d", d->U.n, d->N);
  QUIP_CHECK_ARG(d->V.npass >= 0 && d->V.npass <= 2 && d->U.npass >= 0 && d->U.npass <= 2, "npass must be 0..2");
  return QUIP_OK;
}

// ---- optional event timing of the contraction kernels (bench.py roofline leg) ----
struct TimedLaunch {
  cudaEvent_t e0, e1;
  int path;
  double flops, bytes;
};
static bool g_timing = false;
static std::vector<TimedLaunch> g_timed;      // recorded launches since the last reset
static std::vector<TimedLaunch> g_pool;       // event pairs available for reuse
constexpr size_t TIMED_MAX = 1 << 16;

static int run_qgemm_untimed(const QuipLinearDesc* d, const __half* x2, const float* xsum, const __half* bias,
                             __half* z, int64_t M, int path, unsigned char* ws, const WsPlan& p, cudaStream_t s);

static int run_qgemm(const QuipLinearDesc* d, const __half* x2, const float* xsum, const __half* bias, __half* z,
                     int64_t M, int path, unsigned char* ws, const WsPlan& p, cudaStream_t s) {
  if (path == 0)
    path = M <= SKINNY_MAX_M ? 1 : 2;
  if (!g_timing || g_timed.size() >= TIMED_MAX) return run_qgemm_untimed(d, x2, xsum, bias, z, M, path, ws, p, s);
  TimedLaunch t;
  if (!g_pool.empty()) {
    t = g_pool.back();
    g_pool.pop_back();
  } else {
    QUIP_CUDA(cudaEventCreate(&t.e0));
    QUIP_CUDA(cudaEventCreate(&t.e1));
  }
  t.path = path;
  t.flops = 2.0 * (double)M * d->N * d->K;
  t.bytes = (double)d->N * d->K * d->bits / 8.0 + 2.0 * (double)M * (d->K + d->N);
  QUIP_CUDA(cudaEventRecord(t.e0, s));
  int e = run_qgemm_untimed(d, x2, xsum, bias, z, M, path, ws, p, s);
  QUIP_CUDA(cudaEventRecord(t.e1, s));
  g_timed.push_back(t);
  return e;
}

static int run_qgemm_untimed(const QuipLinearDesc* d, const __half* x2, const float* xsum, const __half* bias,
                             __half* z, int64_t M, int path, unsigned char* ws, const WsPlan& p, cudaStream_t s) {
  if (path == 1) {
    // the skinny kernel takes <= 32 tokens per launch and sums x itself
    for (int64_t m0 = 0; m0 < M; m0 += SKINNY_MAX_M) {
      int mc = (int)((M - m0) < SKINNY_MAX_M ? (M - m0) : SKINNY_MAX_M);
      if (g_use_gemv && qgemv_fits(d->K, mc, d->bits)) {
        if (int e = qgemv(d, x2 + m0 * d->K, bias, z + m0 * d->N, mc, s)) return e;
        continue;
      }
      int ksplit = skinny_pick_ksplit(d->N, d->K, 64, mc);
      if (g_sk_ksplit > 0 && g_sk_ksplit < ksplit) ksplit = g_sk_ksplit;   // experiments: fewer splits only (the plan sized the partials)
      if (int e = qgemm_skinny(d, x2 + m0 * d->K, bias, z + m0 * d->N, mc, ksplit,
                               reinterpret_cast<float*>(ws + p.part), reinterpret_cast<int*>(ws), s))
        return e;
    }
    return QUIP_OK;
  }
  const bool need_xsum = !(d->flags & QUIP_FLAG_SYMMETRIC);
  QUIP_CHECK_ARG(!need_xsum || xsum, "asymmetric grid needs the row sums of x");
  return qgemm_tc(d, x2, xsum, bias, z, (int)M, s);
}

}  // namespace quip

using namespace quip;

extern "C" const char* quip_last_error(void) { return g_err; }
extern "C" int quip_abi_version(void) { return QUIP_ABI_VERSION; }
extern "C" int64_t quip_launch_count(void) { return g_launches.load(); }

extern "C" int quip_config(const char* key, int value) {
  QUIP_CHECK_ARG(key != nullptr, "null key");
  if (!strcmp(key, "side_fused")) { g_side_fused = value; return QUIP_OK; }
  if (!strcmp(key, "side_fewtok")) { g_side_fewtok = value; return QUIP_OK; }
  if (!strcmp(key, "pdl")) { g_pdl = value; return QUIP_OK; }
  if (!strcmp(key, "fewtok")) { g_fewtok = value; return QUIP_OK; }
  if (!strcmp(key, "fewtok_max_m")) {
    QUIP_CHECK_ARG(value >= 8 && value <= 32, "quip_config: fewtok_max_m must be in 8..32");
    g_fewtok_max_m = value;
    return QUIP_OK;
  }
  if (!strcmp(key, "gemv")) { g_use_gemv = value; return QUIP_OK; }
  if (!strcmp(key, "gv_rbc")) { g_gv_rbc = value; return QUIP_OK; }
  if (!strcmp(key, "gv_stream")) { g_gv_stream = value; return QUIP_OK; }
  if (!strcmp(key, "gv_cw")) { g_gv_cw = value; return QUIP_OK; }
  if (!strcmp(key, "gv_tma")) { g_gv_tma = value; return QUIP_OK; }
  if (!strcmp(key, "gv_int")) { g_gv_int = value; return QUIP_OK; }
  if (!strcmp(key, "gv_persist")) { g_gv_persist = value; return QUIP_OK; }
  if (!strcmp(key, "gather_rows")) { g_gather_rows = value; return QUIP_OK; }
  if (!strcmp(key, "sk_ksplit")) { g_sk_ksplit = value; return QUIP_OK; }
  if (!strcmp(key, "pass_min_tiles")) { g_pass_min_tiles = value > 0 ? value : 1; return QUIP_OK; }
  set_error("quip_config: unknown key '%s'", key);
  return QUIP_ERR_ARG;
}

extern "C" int quip_timing_enable(int on) {
  g_timing = on != 0;
  return QUIP_OK;
}
extern "C" int quip_timing_reset(void) {
  for (auto& t : g_timed) g_pool.push_back(t);
  g_timed.clear();
  return QUIP_OK;
}
extern "C" int quip_timing_read(int path, double* total_ms, int64_t* launches, double* flops, double* bytes) {
  double ms = 0, fl = 0, by = 0;
  int64_t n = 0;
  for (auto& t : g_timed) {
    if (t.path != path) continue;
    QUIP_CUDA(cudaEventSynchronize(t.e1));
    float dt = 0.f;
    QUIP_CUDA(cudaEventElapsedTime(&dt, t.e0, t.e1));
    ms += dt; fl += t.flops; by += t.bytes; ++n;
  }
  if (total_ms) *total_ms = ms;
  if (launches) *launches = n;
  if (flops) *flops = fl;
  if (bytes) *bytes = by;
  return QUIP_OK;
}

extern "C" int quip_qlinear_workspace_bytes(const QuipLinearDesc* d, int64_t M, size_t* out) {
  if (int e = check_desc(d)) return e;
  QUIP_CHECK_ARG(out && M > 0, "bad arguments");
  *out = plan_ws(d, M).total;
  return QUIP_OK;
}

extern "C" int quip_qgemm(const QuipLinearDesc* d, const void* x2, const float* xsum, const void* bias, void* z,
                          int64_t M, int path, void* workspace, size_t workspace_bytes, void* stream) {
  if (int e = check_desc(d)) return e;
  QUIP_CHECK_ARG(x2 && z && M > 0 && M < (1ll << 31), "bad arguments");
  WsPlan p = plan_ws(d, M);
  QUIP_CHECK_ARG(path >= 0 && path <= 2, "path must be 0 (auto), 1 (few-token kernels) or 2 (tcgen05)");
  // the few-token kernels keep split-K partials + arrival counters in the workspace (path 1 loops 32-token chunks for any M)
  if (path == 1 || (path == 0 && M <= SKINNY_MAX_M)) {
    if (!workspace || workspace_bytes < p.total) {
      set_error("workspace too small: need %zu bytes, have %zu", p.total, workspace_bytes);
      return QUIP_ERR_WORKSPACE;
    }
  }
  return run_qgemm(d, (const __half*)x2, xsum, (const __half*)bias, (__half*)z, M, path, (unsigned char*)workspace, p,
                   (cudaStream_t)stream);
}

extern "C" int quip_qlinear_forward(const QuipLinearDesc* d, const void* x_, void* y_, int64_t M, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  if (int e = check_desc(d)) return e;
  QUIP_CHECK_ARG(x_ && y_ && M > 0 && M < (1ll << 31), "bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  WsPlan p = plan_ws(d, M);
  if (!workspace || workspace_bytes < p.total) {
    set_error("workspace too small: need %zu bytes, have %zu", p.total, workspace_bytes);
    return QUIP_ERR_WORKSPACE;
  }
  unsigned char* ws = (unsigned char*)workspace;
  const __half* x = (const __half*)x_;
  __half* y = (__half*)y_;
  __half* bufA = (__half*)(ws + p.bufA);
  __half* bufB = (__half*)(ws + p.bufB);
  __half* zbuf = (__half*)(ws + p.zbuf);
  __half* bufC = (__half*)(ws + p.bufC);
  float* xsum = (float*)(ws + p.xsum);
  const int K = d->K, N = d->N;

  // ---- K side: x2 = passes( (x * inv_scale)[idx] ) ----
  const __half* cur = x;
  const int vpass = d->V.n ? d->V.npass : 0;
  const bool need_xsum = !(d->flags & QUIP_FLAG_SYMMETRIC) && M > SKINNY_MAX_M;
  bool have_xsum = false;
  if (g_fewtok && g_side_fewtok && vpass == 2 && side_fewtok_ok(&d->V, K, M)) {
    // a handful of tokens: gather + 1/s + both passes in one launch, every CTA computing the first-pass rows it consumes
    if (int e = side_fewtok(&d->V, x, bufA, M, K, d->V.idx, d->inv_scale, nullptr, nullptr, s)) return e;
    cur = bufA;
  } else if (g_side_fused && M > g_fewtok_max_m && vpass == 2 && side_fused_ok(&d->V, K)) {
    // many tokens: the whole side in one kernel, 16 token rows resident in shared memory
    if (int e = side_fused(&d->V, x, bufA, M, d->V.idx, d->inv_scale, nullptr, nullptr, need_xsum ? xsum : nullptr, s)) return e;
    cur = bufA;
    have_xsum = need_xsum;
  } else {
    // few tokens: the gather (index + 1/s) rides on the first pass's operand load
    // (small blocks only: a 688-wide block is shared by 21 CTAs, which would each repeat the indexed reads)
    const bool fuse_in = g_fewtok && M <= g_fewtok_max_m && vpass > 0 && d->V.pass[0].p <= 128 && pass_fewtok_ok(&d->V.pass[0], M, K);
    if ((d->V.idx || d->inv_scale) && !fuse_in) {
      if (int e = quip_gather(cur, bufA, M, K, d->V.n ? d->V.idx : nullptr, d->inv_scale, nullptr, stream)) return e;
      cur = bufA;
    }
    for (int i = 0; i < vpass; ++i) {
      __half* dst = (cur == bufA) ? bufB : bufA;
      if (i == 0 && fuse_in) {
        if (int e = pass_fewtok(&d->V.pass[0], cur, dst, M, K, d->V.idx, d->inv_scale, nullptr, nullptr, s)) return e;
      } else if (int e = quip_rot_pass(&d->V.pass[i], cur, dst, M, K, 0, stream)) {
        return e;
      }
      cur = dst;
    }
  }
  const __half* x2 = cur;

  // ---- contraction with the packed matrix ----
  const bool u_on = side_on(d->U);
  if (need_xsum && !have_xsum)
    if (int e = quip_rowsum(x2, xsum, M, K, stream)) return e;
  __half* zdst = u_on ? zbuf : y;
  if (int e = run_qgemm(d, x2, xsum, u_on ? nullptr : (const __half*)d->bias, zdst, M, 0, ws, p, s)) return e;
  if (!u_on) return QUIP_OK;

  // ---- N side: y = passes(z)[idx] + bias ----
  if (g_fewtok && g_side_fewtok && d->U.npass == 2 && (!d->U.idx || d->U.inv_idx) && side_fewtok_ok(&d->U, N, M))
    return side_fewtok(&d->U, zbuf, y, M, N, nullptr, nullptr, d->U.inv_idx, (const __half*)d->bias, s);
  if (g_side_fused && M > g_fewtok_max_m && d->U.npass == 2 && side_fused_ok(&d->U, N))
    return side_fused(&d->U, zbuf, y, M, nullptr, nullptr, d->U.idx, (const __half*)d->bias, nullptr, s);
  const __half* zc = zbuf;
  const int np = d->U.npass;
  bool tail_gather = d->U.idx || d->bias;
  // few tokens: the last pass scatters through the inverse index and adds the bias itself
  const bool fuse_out = tail_gather && g_fewtok && M <= g_fewtok_max_m && np > 0 && (!d->U.idx || d->U.inv_idx) &&
                        pass_fewtok_ok(&d->U.pass[np - 1], M, N);
  if (fuse_out) tail_gather = false;
  for (int i = 0; i < np; ++i) {
    __half* dst = (i == np - 1 && !tail_gather) ? y : ((zc == zbuf) ? bufC : zbuf);
    if (i == np - 1 && fuse_out) {
      if (int e = pass_fewtok(&d->U.pass[i], zc, dst, M, N, nullptr, nullptr, d->U.inv_idx, (const __half*)d->bias, s)) return e;
    } else if (int e = quip_rot_pass(&d->U.pass[i], zc, dst, M, N, 0, stream)) {
      return e;
    }
    zc = dst;
  }
  if (tail_gather) return quip_gather(zc, y, M, N, d->U.idx, nullptr, d->bias, stream);
  return QUIP_OK;
}
