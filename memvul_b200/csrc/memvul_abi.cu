// C-ABI entry points of libmemvul_b200.so (declared in include/memvul_b200.h): argument checks,
// TMA tensor-map construction (cached), launch configuration.  No torch, no exceptions across the ABI.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "../../include/memvul_b200.h"
#include "attention_tcgen05.cuh"
#include "attention_tcgen05_v2.cuh"
#include "attention_tcgen05_v3.cuh"
#include "gemm_tcgen05.cuh"
#include "gemm_tcgen05_2cta.cuh"
#include "gemm_ln_tcgen05.cuh"
#include "pool_match.cuh"
#include "precise.cuh"
#include "rowwise.cuh"

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
#define CUDA_TRY(expr)                                                                      \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess)                                                                  \
      return fail(MEMVUL_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)


// ------------------------------------------------------------------ launch accounting / per-kernel timing
// Always-on launch counter (bench.py's "gpu_launches") and an opt-in mode that brackets every launch with
// CUDA events on the launching stream so bench.py can report per-kernel durations from the live run.
enum KernelClass : int {
  KC_EMBED_LN = 0, KC_GEMM_QKV, KC_ATTENTION, KC_GEMM_ATTN_OUT, KC_LAYERNORM, KC_GEMM_FFN_UP, KC_GEMM_FFN_DOWN,
  KC_POOL_MATCH, KC_OTHER, KC_ATTENTION_CLS, KC_CLS_TAIL, KC_COUNT
};
static_assert(KC_COUNT == MEMVUL_KERNEL_CLASSES, "include/memvul_b200.h lists the kernel classes");
std::atomic<long long> g_launches{0};
std::atomic<int> g_prof_on{0};
struct ProfRec { int cls; cudaEvent_t e0, e1; };
std::mutex g_prof_mu;
std::vector<ProfRec> g_prof_recs;
std::vector<cudaEvent_t> g_prof_pool;
thread_local int g_cls = KC_OTHER;

cudaEvent_t prof_event() {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (!g_prof_pool.empty()) { cudaEvent_t e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}
struct LaunchScope {
  cudaStream_t st; cudaEvent_t e0 = nullptr; int cls;
  LaunchScope(int c, cudaStream_t s) : st(s), cls(c) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (g_prof_on.load(std::memory_order_relaxed)) { e0 = prof_event(); cudaEventRecord(e0, st); }
  }
  ~LaunchScope() {
    if (e0) {
      cudaEvent_t e1 = prof_event();
      cudaEventRecord(e1, st);
      std::lock_guard<std::mutex> lk(g_prof_mu);
      g_prof_recs.push_back({cls, e0, e1});
    }
  }
};
struct ClassScope {
  int prev;
  explicit ClassScope(int c) : prev(g_cls) { g_cls = c; }
  ~ClassScope() { g_cls = prev; }
};

// ------------------------------------------------------------------ device info
struct DeviceInfo {
  int sms = 0;
  bool ok = false;
};
int device_info(DeviceInfo* out) {
  static std::mutex mu;
  static std::unordered_map<int, DeviceInfo> cache;
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(mu);
  auto it = cache.find(dev);
  if (it == cache.end()) {
    DeviceInfo d;
    int major = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&d.sms, cudaDevAttrMultiProcessorCount, dev));
    CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    if (major != 10) return fail(MEMVUL_E_CUDA, "memvul_b200 needs an sm_100a device (found compute capability %d.x)", major);
    d.ok = true;
    it = cache.emplace(dev, d).first;
  }
  *out = it->second;
  return MEMVUL_OK;
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per (device, function): cache per device, not per process
// (a second device in the same process would otherwise launch the > 48 KB kernels without the opt-in).
int ensure_dyn_smem(const void* kern, int bytes) {
  static std::mutex mu;
  static std::unordered_map<uint64_t, int> done;          // (device << 48 | function address) -> bytes set
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  const uint64_t key = (static_cast<uint64_t>(dev) << 48) ^ static_cast<uint64_t>(reinterpret_cast<uintptr_t>(kern));
  std::lock_guard<std::mutex> lk(mu);
  auto it = done.find(key);
  if (it != done.end() && it->second >= bytes) return MEMVUL_OK;
  CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  done[key] = bytes;
  return MEMVUL_OK;
}
// small per-device integer cache (occupancy results)
int* per_device_slot(int which) {
  static std::mutex mu;
  static std::unordered_map<int, int> slots;              // key = device * 16 + which; value 0 = not computed yet
  static int dummy = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return &dummy;
  std::lock_guard<std::mutex> lk(mu);
  return &slots[dev * 16 + which];                         // references into unordered_map stay valid across inserts
}

// ------------------------------------------------------------------ TMA tensor maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

struct MapKey {
  const void* base;
  uint64_t rows, cols, ld;
  uint32_t box_rows, box_cols, elem_bytes;
  bool operator==(const MapKey& o) const {
    return base == o.base && rows == o.rows && cols == o.cols && ld == o.ld && box_rows == o.box_rows &&
           box_cols == o.box_cols && elem_bytes == o.elem_bytes;
  }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.base);
    h = h * 1315423911u ^ k.rows;
    h = h * 1315423911u ^ k.cols;
    h = h * 1315423911u ^ k.ld;
    h = h * 1315423911u ^ k.box_rows;
    h = h * 1315423911u ^ (k.box_cols * 8u + k.elem_bytes);
    return h;
  }
};
// Row-major [rows, cols] matrix of fp16 (elem_bytes 2) or fp32 (4) with leading dimension ld (elements);
// box = {box_cols, box_rows} with box_cols * elem_bytes == 128 B, SWIZZLE_128B.
int make_map(const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows, uint32_t box_cols,
             uint32_t elem_bytes, CUtensorMap* out) {
  static std::mutex mu;
  static std::unordered_map<MapKey, CUtensorMap, MapKeyHash> cache;
  MapKey key{base, rows, cols, ld, box_rows, box_cols, elem_bytes};
  {
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(key);
    if (it != cache.end()) {
      *out = it->second;
      return MEMVUL_OK;
    }
  }
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(MEMVUL_E_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  if ((reinterpret_cast<uintptr_t>(base) & 15u) || ((ld * elem_bytes) & 15u) || box_cols * elem_bytes != 128)
    return fail(MEMVUL_E_INVALID, "TMA operand must be 16-byte aligned with 128-byte box rows (ptr=%p ld=%llu)", base,
                (unsigned long long)ld);
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {ld * elem_bytes};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUtensorMap m;
  CUresult r = fn(&m, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                  const_cast<void*>(base), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(MEMVUL_E_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  {
    std::lock_guard<std::mutex> lk(mu);
    if (cache.size() > 4096) cache.clear();
    cache.emplace(key, m);
  }
  *out = m;
  return MEMVUL_OK;
}
int make_map_f16(const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows, CUtensorMap* out) {
  return make_map(base, rows, cols, ld, box_rows, 64, 2, out);
}

// ------------------------------------------------------------------ launchers
template <int BN, int EPI>
int launch_gemm(const CUtensorMap& ta, const CUtensorMap& tb, int M, int N, int K, const float* bias,
                const float* resid, void* out, int sms, cudaStream_t st, const int* m_dev) {
  using Cfg = mv::GemmCfg<BN>;
  auto kern = mv::gemm_f16_tcgen05_kernel<BN, EPI>;
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(kern), Cfg::SMEM_BYTES)) return rc;
  const int tiles = ((M + Cfg::BM - 1) / Cfg::BM) * (N / BN);
  const int grid = tiles < sms ? tiles : sms;
  LaunchScope ls(g_cls, st);
  kern<<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, st>>>(ta, tb, M, N, K, bias, resid, out, N, m_dev);
  CUDA_TRY(cudaGetLastError());
  return MEMVUL_OK;
}

template <int BN>
int launch_gemm_epi(int epi, const CUtensorMap& ta, const CUtensorMap& tb, int M, int N, int K, const float* bias,
                    const float* resid, void* out, int sms, cudaStream_t st, const int* m_dev) {
  switch (epi) {
    case MEMVUL_EPI_BIAS_F16: return launch_gemm<BN, mv::EPI_BIAS_F16>(ta, tb, M, N, K, bias, resid, out, sms, st, m_dev);
    case MEMVUL_EPI_BIAS_GELU_F16: return launch_gemm<BN, mv::EPI_BIAS_GELU_F16>(ta, tb, M, N, K, bias, resid, out, sms, st, m_dev);
    case MEMVUL_EPI_BIAS_RESID_F32: return launch_gemm<BN, mv::EPI_BIAS_RESID_F32>(ta, tb, M, N, K, bias, resid, out, sms, st, m_dev);
    case MEMVUL_EPI_BIAS_F32: return launch_gemm<BN, mv::EPI_BIAS_RESID_F32>(ta, tb, M, N, K, bias, nullptr, out, sms, st, m_dev);
  }
  return fail(MEMVUL_E_INVALID, "unknown GEMM epilogue %d", epi);
}


// MEMVUL_GEMM_WAIT (default 5 = suspend-hinted TMA + MMA warps: r01n, -2..4 % on QKV / FFN-up): how the GEMM kernels' single-lane TMA / MMA warps wait (bits 0-1 TMA warp, bits 2-3 MMA warp, bits 4-5
// epilogue warps; 0 spin, 1 suspend hint, 2 hint + nanosleep -- ptx.cuh mbar_wait_idle)
static int gemm_wait_mode() {
  static const int m = [] { const char* e = getenv("MEMVUL_GEMM_WAIT"); return e ? atoi(e) & 63 : 5; }();
  return m;
}

// experiment knob: MEMVUL_GEMM_EPI_MODE = 1 (default) | 3 (math + staging, no TMA store) | 4 (TMA store only)
static int epi_mode() {
  static const int m = [] { const char* e = getenv("MEMVUL_GEMM_EPI_MODE"); return e ? atoi(e) : 1; }();
  return m;
}

template <int EPI>
int launch_gemm_2cta(const CUtensorMap& ta, const CUtensorMap& tb, int M, int N, int K, const float* bias,
                     const float* resid, void* out, int sms, cudaStream_t st, const int* m_dev) {
  using Cfg = mv::Gemm2Cfg<EPI>;
  auto kern = mv::gemm_f16_tcgen05_2cta_kernel<EPI>;
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(kern), Cfg::SMEM_BYTES)) return rc;
  static const bool nostore = getenv("MEMVUL_GEMM_NOSTORE") != nullptr;      // experiment: time the main loop alone
  static const bool direct_st = getenv("MEMVUL_GEMM_DIRECT_ST") != nullptr;   // experiment: 256-bit per-lane stores
  CUtensorMap tout, tres;
  const bool no_resid = Cfg::RESID && resid == nullptr;     // MEMVUL_EPI_BIAS_F32: fp32 output, nothing to add
  if (Cfg::RESID) {
    if (int rc = make_map(out, (uint64_t)M, (uint64_t)N, (uint64_t)N, 32, 32, 4, &tout)) return rc;
    if (no_resid) tres = tout;
    else if (int rc = make_map(resid, (uint64_t)M, (uint64_t)N, (uint64_t)N, 32, 32, 4, &tres)) return rc;
  } else {
    if (int rc = make_map(out, (uint64_t)M, (uint64_t)N, (uint64_t)N, 32, 64, 2, &tout)) return rc;
    tres = tout;
  }
  const int tiles = ((M + Cfg::BM - 1) / Cfg::BM) * (N / Cfg::BN);
  int clusters = sms / 2;
  if (tiles < clusters) clusters = tiles;
  LaunchScope ls(g_cls, st);
  kern<<<2 * clusters, Cfg::THREADS, Cfg::SMEM_BYTES, st>>>(ta, tb, tout, tres, M, N, K, bias,
                                                              (nostore ? 0 : (no_resid ? 5 : ((direct_st && !Cfg::RESID) ? 2 : epi_mode()))) | (gemm_wait_mode() << 8), out, m_dev);   // __cluster_dims__(2,1,1)
  CUDA_TRY(cudaGetLastError());
  return MEMVUL_OK;
}

int launch_gemm_2cta_epi(int epi, const CUtensorMap& ta, const CUtensorMap& tb, int M, int N, int K, const float* bias,
                         const float* resid, void* out, int sms, cudaStream_t st, const int* m_dev) {
  switch (epi) {
    case MEMVUL_EPI_BIAS_F16: return launch_gemm_2cta<mv::EPI_BIAS_F16>(ta, tb, M, N, K, bias, resid, out, sms, st, m_dev);
    case MEMVUL_EPI_BIAS_GELU_F16: return launch_gemm_2cta<mv::EPI_BIAS_GELU_F16>(ta, tb, M, N, K, bias, resid, out, sms, st, m_dev);
    case MEMVUL_EPI_BIAS_RESID_F32: return launch_gemm_2cta<mv::EPI_BIAS_RESID_F32>(ta, tb, M, N, K, bias, resid, out, sms, st, m_dev);
    case MEMVUL_EPI_BIAS_F32: return launch_gemm_2cta<mv::EPI_BIAS_RESID_F32>(ta, tb, M, N, K, bias, nullptr, out, sms, st, m_dev);
  }
  return fail(MEMVUL_E_INVALID, "unknown GEMM epilogue %d", epi);
}

// m_dev (nullable): device int holding the actual row count (<= M) of a packed batch; M is then the upper bound the
// TMA maps and the launch grid are sized for.
int gemm_impl(const void* a, const void* w, const float* bias, const float* resid, void* out, int M, int N, int K,
              int epi, cudaStream_t st, const int* m_dev = nullptr) {
  if (M <= 0 || N <= 0 || K <= 0) return fail(MEMVUL_E_INVALID, "GEMM with empty shape M=%d N=%d K=%d", M, N, K);
  if (K % 64 != 0 || N % 128 != 0)
    return fail(MEMVUL_E_INVALID, "GEMM needs K %% 64 == 0 and N %% 128 == 0 (M=%d N=%d K=%d)", M, N, K);
  if (!a || !w || !bias || !out) return fail(MEMVUL_E_INVALID, "GEMM null pointer");
  if (epi == MEMVUL_EPI_BIAS_RESID_F32 && !resid) return fail(MEMVUL_E_INVALID, "GEMM residual epilogue needs resid");
  DeviceInfo di;
  if (int rc = device_info(&di)) return rc;
  const int tiles_m = (M + 127) / 128;
  // CTA-pair kernel (256 x 256 tiles) once there is at least one tile per SM pair; MEMVUL_GEMM_MODE=1cta disables it.
  static const bool allow_2cta = [] { const char* e = getenv("MEMVUL_GEMM_MODE"); return !(e && strcmp(e, "1cta") == 0); }();
  if (allow_2cta && N % 256 == 0 && ((M + 255) / 256) * (N / 256) >= di.sms / 2) {
    CUtensorMap ta2, tb2;
    if (int rc = make_map_f16(a, (uint64_t)M, (uint64_t)K, (uint64_t)K, 128, &ta2)) return rc;
    if (int rc = make_map_f16(w, (uint64_t)N, (uint64_t)K, (uint64_t)K, 128, &tb2)) return rc;
    return launch_gemm_2cta_epi(epi, ta2, tb2, M, N, K, bias, resid, out, di.sms, st, m_dev);
  }
  const bool bn256 = (N % 256 == 0) && (tiles_m * (N / 256) >= di.sms);
  const int BN = bn256 ? 256 : 128;
  CUtensorMap ta, tb;
  if (int rc = make_map_f16(a, (uint64_t)M, (uint64_t)K, (uint64_t)K, 128, &ta)) return rc;
  if (int rc = make_map_f16(w, (uint64_t)N, (uint64_t)K, (uint64_t)K, (uint32_t)BN, &tb)) return rc;
  return bn256 ? launch_gemm_epi<256>(epi, ta, tb, M, N, K, bias, resid, out, di.sms, st, m_dev)
               : launch_gemm_epi<128>(epi, ta, tb, M, N, K, bias, resid, out, di.sms, st, m_dev);
}


// Fused residual GEMM + LayerNorm (N == 768): x32/x16 = LN(A W^T + bias + resid).  Falls back to the caller's
// two-kernel path (returns 1) when the shape does not qualify.
int gemm_ln_impl(const void* a, const void* w, const float* bias, const float* resid, const float* gamma,
                 const float* beta, float eps, float* x32, void* x16, int M, int N, int K, cudaStream_t st,
                 const int* m_dev = nullptr) {
  using Cfg = mv::GemmLnCfg;
  static const bool disabled = [] { const char* e = getenv("MEMVUL_FUSED_LN"); return e && strcmp(e, "0") == 0; }();
  if (disabled || N != Cfg::N || K % 64 != 0 || M < Cfg::BM) return 1;
  DeviceInfo di;
  if (int rc = device_info(&di)) return rc;
  auto kern = mv::gemm_ln_f16_tcgen05_kernel;
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(kern), Cfg::SMEM_BYTES)) return rc;
  int& max_clusters = *per_device_slot(0);
  if (max_clusters <= 0) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(Cfg::CLUSTER * (di.sms / Cfg::CLUSTER));
    cfg.blockDim = dim3(Cfg::THREADS);
    cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = Cfg::CLUSTER; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    int n = 0;
    CUDA_TRY(cudaOccupancyMaxActiveClusters(&n, kern, &cfg));
    if (n < 1) return fail(MEMVUL_E_CUDA, "fused GEMM+LayerNorm: no 6-CTA cluster fits on this device");
    max_clusters = n;
  }
  // TMA multicast of A across the three pairs works but measured 2-4 % slower than unicast (the main loop is not
  // L2-bound: DESIGN.md section 3), so it is opt-in: MEMVUL_LN_MULTICAST=1.
  static const bool a_mc = [] { const char* e = getenv("MEMVUL_LN_MULTICAST"); return e && strcmp(e, "1") == 0; }();
  // MEMVUL_LN_MODE: epilogue variant bits (1 direct global stores + early residual request, 2 st.async statistics
  // exchange, 4 L2 prefetch of the next tile's residual); default 2: r02c/r02d measured 83 -> 74 us at K=768 for the
  // st.async exchange alone; direct row-strided stores cost 3 k cycles per chunk against 1.4 k for the staged TMA
  // stores, and the L2 prefetch does not shorten the residual wait (the TMA queue under load, not HBM, is the
  // latency); 0 = the r01 epilogue
  static const int ln_mode = [] { const char* e = getenv("MEMVUL_LN_MODE"); return e ? atoi(e) & 7 : 2; }();
  // MEMVUL_LN_RING_SHORT: A/B ring depth (2..4) for K <= 1024 (see the kernel); longer K always uses all four stages
  static const int ring_short = [] { const char* e = getenv("MEMVUL_LN_RING_SHORT"); int v = e ? atoi(e) : 4; return v < 2 ? 2 : (v > 4 ? 4 : v); }();
  // MEMVUL_LN_XBUF (default 1): for K <= 1024 the fourth A/B stage becomes a third residual buffer per epilogue warp (kernel
  // comment); implies a ring of at most three stages
  static const int xbuf_on = [] { const char* e = getenv("MEMVUL_LN_XBUF"); return (e && atoi(e) == 0) ? 0 : 1; }();
  const int xbuf = (K <= 1024 && xbuf_on && !(ln_mode & 1)) ? 1 : 0;
  const int ring = K <= 1024 ? (xbuf && ring_short > 3 ? 3 : ring_short) : 4;
  // MEMVUL_LN_RES: how the epilogue fetches the fp32 residual boxes: "tma" (default) or "ldgsts" (per-lane cp.async
  // through the LSU path).  r02i: both wait ~3 k cycles per exposed box at K = 768 (and ~0.2 k with a 2-deep A/B ring that
  // starves the MMA): the latency is the SM's own queue of outstanding operand bytes at the L2 port, whichever unit asks.
  static const int res_ldgsts = [] { const char* e = getenv("MEMVUL_LN_RES"); return (e && strcmp(e, "ldgsts") == 0) ? 1 : 0; }();
  // MEMVUL_LN_PACE=<cycles>: minimum spacing of the producer's stage requests for K <= 1024 (see the kernel)
  static const int pace_short = [] { const char* e = getenv("MEMVUL_LN_PACE"); int v = e ? atoi(e) : 0; return v < 0 ? 0 : (v > 20000 ? 20000 : v); }();
  const int pace = K <= 1024 ? pace_short : 0;
  CUtensorMap ta, ta64, tb, tres, t32, t16;
  if (int rc = make_map_f16(a, (uint64_t)M, (uint64_t)K, (uint64_t)K, 128, &ta)) return rc;
  if (int rc = make_map_f16(a, (uint64_t)M, (uint64_t)K, (uint64_t)K, 64, &ta64)) return rc;
  if (int rc = make_map_f16(w, (uint64_t)N, (uint64_t)K, (uint64_t)K, 128, &tb)) return rc;
  if (int rc = make_map(resid, (uint64_t)M, (uint64_t)N, (uint64_t)N, 32, 32, 4, &tres)) return rc;
  if (int rc = make_map(x32, (uint64_t)M, (uint64_t)N, (uint64_t)N, 32, 32, 4, &t32)) return rc;
  if (int rc = make_map(x16, (uint64_t)M, (uint64_t)N, (uint64_t)N, 32, 64, 2, &t16)) return rc;
  const int tiles = (M + Cfg::BM - 1) / Cfg::BM;
  const int clusters = tiles < max_clusters ? tiles : max_clusters;
  // MEMVUL_LN_TRACE=<file>: debug only -- CTA 0 records clock64() per epilogue / MMA phase (tools/ln_trace.py)
  static const char* trace_path = getenv("MEMVUL_LN_TRACE");
  static unsigned long long* trace_buf = nullptr;
  if (trace_path && !trace_buf) CUDA_TRY(cudaMalloc(&trace_buf, 128 * 8));
  if (trace_buf) CUDA_TRY(cudaMemsetAsync(trace_buf, 0, 128 * 8, st));
  {
    LaunchScope ls(g_cls, st);
    kern<<<Cfg::CLUSTER * clusters, Cfg::THREADS, Cfg::SMEM_BYTES, st>>>(ta, ta64, tb, tres, t32, t16, M, K, bias, gamma, beta, eps, (a_mc ? 1 : 0) | (ln_mode << 1) | (gemm_wait_mode() << 4) | (ring << 12) | (res_ldgsts << 15) | (xbuf << 16), m_dev, trace_buf, x32, reinterpret_cast<__half*>(x16), resid, pace);
    CUDA_TRY(cudaGetLastError());
  }
  if (trace_buf) {                                  // debug: dump CTA 0's phase stamps of THIS launch
    std::vector<unsigned long long> host(128);
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaMemcpy(host.data(), trace_buf, 128 * 8, cudaMemcpyDeviceToHost));
    if (FILE* f = fopen(trace_path, "wb")) { fwrite(host.data(), 8, 128, f); fclose(f); }
  }
  return MEMVUL_OK;
}

// MEMVUL_ATT_WAIT (default 5: r01n, 118 -> 111 us): how the attention kernel's single-lane TMA / MMA warps wait (bits 0-1 TMA warp, bits 2-3 MMA warp, bits 4-5
// softmax warps; 0 spin, 1 suspend hint, 2 hint + nanosleep -- ptx.cuh mbar_wait_idle)
static int att_wait_mode() {
  static const int m = [] { const char* e = getenv("MEMVUL_ATT_WAIT"); return e ? atoi(e) & 63 : 5; }();
  // MEMVUL_ATT_STAGGER=<cycles> (bits 8..): the second CTA of every SM starts its soft-max stream that many cycles late, so
  // that the two co-resident CTAs' exponentiation phases (MUFU-bound: 2 x 64 MUFU.EX2 per thread and key block on the one
  // XU of a sub-partition) interleave instead of coinciding.  Both CTAs start together and run identical work, so without
  // the offset they stay in phase for the whole launch (r01p trace: the exp phase takes 970 cycles, twice its solo time).
  static const int stagger = [] { const char* e = getenv("MEMVUL_ATT_STAGGER"); int v = e ? atoi(e) : 0; return v < 0 ? 0 : (v > 100000 ? 100000 : v); }();
  // MEMVUL_ATT_EARLY (default 1, bit 8): the soft-max warps issue non-blocking mbarrier.test_wait for pv_done(g-1) and
  // s_full(g+1) under the exponentials instead of paying two blocking try_wait round trips per key block
  static const int early = [] { const char* e = getenv("MEMVUL_ATT_EARLY"); return (e && atoi(e) == 0) ? 0 : 1; }();
  // MEMVUL_ATT_SPEC (default 1, bit 9): speculative exponentials against the stale row maximum (attention_tcgen05.cuh)
  static const int spec = [] { const char* e = getenv("MEMVUL_ATT_SPEC"); return (e && atoi(e) == 0) ? 0 : 1; }();
  return m | (early << 8) | (spec << 9) | (stagger << 10);
}

int attention_impl(const void* qkv, const int32_t* lens, const int32_t* row_start, void* ctx, int B, int S, int H,
                   cudaStream_t st, bool first_tile_only = false) {
  if (B <= 0 || S <= 0 || S > 512) return fail(MEMVUL_E_INVALID, "attention needs 1 <= S <= 512 (B=%d S=%d)", B, S);
  if (H % 64 != 0) return fail(MEMVUL_E_INVALID, "attention needs H %% 64 == 0 (head_dim 64), H=%d", H);
  DeviceInfo di;
  if (int rc = device_info(&di)) return rc;
  CUtensorMap tq, tkv, tctx;
  if (int rc = make_map_f16(qkv, (uint64_t)B * S, (uint64_t)3 * H, (uint64_t)3 * H, 128, &tq)) return rc;
  if (int rc = make_map_f16(qkv, (uint64_t)B * S, (uint64_t)3 * H, (uint64_t)3 * H, mv::AttnCfg::BKV, &tkv)) return rc;
  if (int rc = make_map_f16(ctx, (uint64_t)B * S, (uint64_t)H, (uint64_t)H, 32, &tctx)) return rc;   // ctx write-out boxes
  // MEMVUL_ATT_V=2 selects the experimental second-generation kernel (attention_tcgen05_v2.cuh: 8 soft-max warps splitting
  // every row, separate Q K^T / P V issuers, double-buffered O).  It is parity-green but measured SLOWER (r02e: 133.7 us
  // against 116.3 us at 64 x 512): the block period is set by the MUFU phase all warps of a CTA enter together, not by
  // the per-thread chain that the split shortens.
  // Default (MEMVUL_ATT_V unset or 3): the three-streams-per-SM kernel (attention_tcgen05_v3.cuh: 3 CTAs per SM, soft-max
  // warps on 120 registers by setmaxnreg, single-buffered S / P, separate K / V rings; r02q: 106.9 against 115.8 us at
  // 64 x 512, 69.9 against 80.3 at 128 x 256, bit-identical results).  MEMVUL_ATT_V=1: the first kernel (two CTAs per SM).
  // MEMVUL_ATT_POLY=2: two of every 8 exponentials of the v3 kernel on the FMA pipe (measured slower, 111.5 us: the MUFU
  // pipe is not the limiter even with three streams).
  static const int att_v = [] { const char* e = getenv("MEMVUL_ATT_V"); int v = e ? atoi(e) : 3; return (v == 1 || v == 2) ? v : 3; }();
  static const int att_poly = [] { const char* e = getenv("MEMVUL_ATT_POLY"); return (e && atoi(e) == 2) ? 2 : 0; }();
  const bool v1 = att_v == 1;
  // MEMVUL_ATT_PTMEM=1: the v3 kernel with P handed to the tensor core through TENSOR memory (tcgen05.st + A-from-TMEM MMA:
  // no STS, no proxy fence, no 16 KB operand re-read per block).  Parity-green (r02q: 76 GPU tests + C2 / C5 config tests),
  // but not faster: 108.1 against 107.0 us at 64 x 512 and slower on short sequences (71.8 against 53.4 us at 256 x 128).
  static const int att_ptmem = [] { const char* e = getenv("MEMVUL_ATT_PTMEM"); return (e && atoi(e) == 1) ? 1 : 0; }();
  const void* v3_fn = att_ptmem ? reinterpret_cast<const void*>(mv::attention_tcgen05_v3_kernel<0, true>) : att_poly == 2 ? reinterpret_cast<const void*>(mv::attention_tcgen05_v3_kernel<2, false>)
                                    : reinterpret_cast<const void*>(mv::attention_tcgen05_v3_kernel<0, false>);
  if (v1) { if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(mv::attention_tcgen05_kernel), mv::AttnCfg::SMEM_BYTES)) return rc; }
  else if (att_v == 2) { if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(mv::attention_tcgen05_v2_kernel), mv::Attn2Cfg::SMEM_BYTES)) return rc; }
  else { if (int rc = ensure_dyn_smem(v3_fn, mv::Attn3Cfg::SMEM_BYTES)) return rc; }
  const int n_qt = first_tile_only ? 1 : (S + 127) / 128;
  const int n_items = B * (H / 64) * n_qt;
  // MEMVUL_ATT_CTAS_PER_SM=1: diagnostic (one CTA per SM: the soft-max phases without a co-resident CTA's MUFU traffic)
  static const int ctas_env = [] { const char* e = getenv("MEMVUL_ATT_CTAS_PER_SM"); return e ? atoi(e) : 0; }();
  const int ctas_max = att_v == 3 ? mv::Attn3Cfg::CTAS_PER_SM : 2;
  const int ctas_per_sm = (ctas_env >= 1 && ctas_env <= ctas_max) ? ctas_env : ctas_max;
  const int grid = n_items < ctas_per_sm * di.sms ? n_items : ctas_per_sm * di.sms;       // persistent: two CTAs per SM
  // MEMVUL_ATT_TRACE=<file>: debug only -- CTA 0 records clock64() per soft-max / MMA phase (tools/att_trace.py; the
  // MEMVUL_ATT_V=1 / 2 kernels only, like MEMVUL_ATT_{STAGGER,EARLY,SPEC})
  static const char* trace_path = getenv("MEMVUL_ATT_TRACE");
  static unsigned long long* trace_buf = nullptr;
  if (trace_path && !trace_buf) {
    CUDA_TRY(cudaMalloc(&trace_buf, 2048 * 8));
  }
  if (trace_buf) CUDA_TRY(cudaMemsetAsync(trace_buf, 0, 2048 * 8, st));
  {
    LaunchScope ls(first_tile_only ? KC_ATTENTION_CLS : KC_ATTENTION, st);
    if (v1)
      mv::attention_tcgen05_kernel<<<grid, mv::AttnCfg::THREADS, mv::AttnCfg::SMEM_BYTES, st>>>(
          tq, tkv, tctx, lens, row_start, reinterpret_cast<__half*>(ctx), B, S, H, n_qt, att_wait_mode(), trace_buf);
    else if (att_v == 2)
      mv::attention_tcgen05_v2_kernel<<<grid, mv::Attn2Cfg::THREADS, mv::Attn2Cfg::SMEM_BYTES, st>>>(
          tq, tkv, tctx, lens, row_start, reinterpret_cast<__half*>(ctx), B, S, H, n_qt, att_wait_mode(), trace_buf);
    else if (att_ptmem)
      mv::attention_tcgen05_v3_kernel<0, true><<<grid, mv::Attn3Cfg::THREADS, mv::Attn3Cfg::SMEM_BYTES, st>>>(
          tq, tkv, tctx, lens, row_start, reinterpret_cast<__half*>(ctx), B, S, H, n_qt, att_wait_mode());
    else if (att_poly == 2)
      mv::attention_tcgen05_v3_kernel<2, false><<<grid, mv::Attn3Cfg::THREADS, mv::Attn3Cfg::SMEM_BYTES, st>>>(
          tq, tkv, tctx, lens, row_start, reinterpret_cast<__half*>(ctx), B, S, H, n_qt, att_wait_mode());
    else
      mv::attention_tcgen05_v3_kernel<0, false><<<grid, mv::Attn3Cfg::THREADS, mv::Attn3Cfg::SMEM_BYTES, st>>>(
          tq, tkv, tctx, lens, row_start, reinterpret_cast<__half*>(ctx), B, S, H, n_qt, att_wait_mode());
    CUDA_TRY(cudaGetLastError());
  }
  if (trace_buf) {                                  // debug: dump CTA 0's phase stamps of THIS launch
    std::vector<unsigned long long> host(2048);
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaMemcpy(host.data(), trace_buf, 2048 * 8, cudaMemcpyDeviceToHost));
    if (FILE* f = fopen(trace_path, "wb")) { fwrite(host.data(), 8, 2048, f); fclose(f); }
  }
  return MEMVUL_OK;
}

int layernorm_impl(const float* y, const float* g, const float* b, float eps, float* x32, void* x16, int M, int H,
                   cudaStream_t st, long long x32_stride = 0) {
  if (M <= 0) return fail(MEMVUL_E_INVALID, "layernorm with M=%d", M);
  if (x32_stride == 0) x32_stride = H;
  const int blocks = (M + 7) / 8;
  LaunchScope ls(g_cls == KC_CLS_TAIL ? KC_CLS_TAIL : KC_LAYERNORM, st);
  if (H == 768)
    mv::layernorm_rows_kernel<6><<<blocks, 256, 0, st>>>(y, g, b, eps, x32, x32_stride, reinterpret_cast<__half*>(x16), M);
  else if (H == 128)
    mv::layernorm_rows_kernel<1><<<blocks, 256, 0, st>>>(y, g, b, eps, x32, x32_stride, reinterpret_cast<__half*>(x16), M);
  else
    return fail(MEMVUL_E_INVALID, "layernorm supports H in {128, 768}, got %d", H);
  CUDA_TRY(cudaGetLastError());
  return MEMVUL_OK;
}

// qkv / ctx / ffn (nullable, packed layout only): the encoder's scratch matrices whose rows past the last token the
// tail blocks zero-fill along with x32 / x16 (rowwise.cuh)
int embed_impl(const memvul_bert_weights* w, const int64_t* ids, const int64_t* tids, const int32_t* lens,
               const int32_t* row_start, int B, int S, float* x32, void* x16, int32_t* bad, cudaStream_t st,
               void* qkv = nullptr, void* ctx = nullptr, void* ffn = nullptr) {
  // 8 token rows per block, blocks never straddle sequences; packed layout: + the tail blocks that zero-fill the rows
  // past the last token
  const int blocks = B * ((S + 7) / 8) + (row_start ? mv::kEmbedTailBlocks : 0);
  auto ll = [](const int64_t* p) { return reinterpret_cast<const long long*>(p); };
  auto h = [](void* p) { return reinterpret_cast<__half*>(p); };
  LaunchScope ls(KC_EMBED_LN, st);
  if (w->hidden == 768)
    mv::embed_layernorm_kernel<6><<<blocks, 256, 0, st>>>(ll(ids), ll(tids), w->word_emb, w->pos_emb, w->type_emb,
                                                          w->emb_ln_g, w->emb_ln_b, w->ln_eps, x32, h(x16), B, S,
                                                          w->vocab, w->type_vocab, lens, row_start, bad, h(qkv), h(ctx),
                                                          h(ffn), w->intermediate);
  else if (w->hidden == 128)
    mv::embed_layernorm_kernel<1><<<blocks, 256, 0, st>>>(ll(ids), ll(tids), w->word_emb, w->pos_emb, w->type_emb,
                                                          w->emb_ln_g, w->emb_ln_b, w->ln_eps, x32, h(x16), B, S,
                                                          w->vocab, w->type_vocab, lens, row_start, bad, h(qkv), h(ctx),
                                                          h(ffn), w->intermediate);
  else
    return fail(MEMVUL_E_INVALID, "embedding supports hidden in {128, 768}, got %d", w->hidden);
  CUDA_TRY(cudaGetLastError());
  return MEMVUL_OK;
}

__global__ void mask_to_lens_kernel(const uint8_t* __restrict__ mask, int B, int S, int32_t* lens, int32_t* bad) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  int cnt = 0, last = -1;
  for (int s = lane; s < S; s += 32)
    if (mask[static_cast<size_t>(b) * S + s]) { ++cnt; last = s; }
  for (int o = 16; o > 0; o >>= 1) {
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
  }
  if (lane == 0) {
    lens[b] = cnt;
    if (cnt == 0 || last != cnt - 1) atomicOr(bad, 1);     // empty, or not a prefix mask
  }
}

// row_start[0..B] = exclusive prefix sum of lens (one block; B is a batch size, at most a few thousand)
__global__ void __launch_bounds__(1024) lens_to_row_start_kernel(const int32_t* __restrict__ lens, int B,
                                                                 int32_t* __restrict__ row_start) {
  __shared__ int warp_tot[32];
  __shared__ int carry_s;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (int base = 0; base < B; base += blockDim.x) {
    const int i = base + threadIdx.x;
    const int v = i < B ? lens[i] : 0;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_tot[wid] = x;
    __syncthreads();
    if (wid == 0) {
      int t = warp_tot[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, t, o);
        if (lane >= o) t += y;
      }
      warp_tot[lane] = t;                                   // inclusive scan of the warp totals
    }
    __syncthreads();
    const int carry = carry_s;
    const int incl = x + (wid ? warp_tot[wid - 1] : 0) + carry;
    if (i < B) row_start[i] = incl - v;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry_s = incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) row_start[B] = carry_s;
}

struct Workspace {
  __half* x16; __half* qkv; __half* ctx; __half* ffn;
  float* x32_cls; __half* x16_cls; __half* ctx_cls; __half* ffn_cls;     // [B, *] rows of the CLS-only last layer
  float* x32_packed;                                                      // packed residual stream (PACKED without CLS_ONLY)
  size_t bytes;
};
Workspace carve(const memvul_bert_weights* w, int B, int S, void* base, int flags) {
  const size_t M = static_cast<size_t>(B) * S, H = w->hidden, I = w->intermediate;
  auto up = [](size_t x) { return (x + 1023) & ~size_t(1023); };
  uint8_t* p = reinterpret_cast<uint8_t*>(base);
  size_t off = 0;
  Workspace ws;
  ws.x16 = reinterpret_cast<__half*>(p + off); off += up(M * H * 2);
  ws.qkv = reinterpret_cast<__half*>(p + off); off += up(M * 3 * H * 2);
  ws.ctx = reinterpret_cast<__half*>(p + off); off += up(M * H * 2);
  ws.ffn = reinterpret_cast<__half*>(p + off); off += up(M * I * 2);
  const size_t Bp = static_cast<size_t>(B);
  ws.x32_cls = reinterpret_cast<float*>(p + off); off += up(Bp * H * 4);
  ws.x16_cls = reinterpret_cast<__half*>(p + off); off += up(Bp * H * 2);
  ws.ctx_cls = reinterpret_cast<__half*>(p + off); off += up(Bp * H * 2);
  ws.ffn_cls = reinterpret_cast<__half*>(p + off); off += up(Bp * I * 2);
  ws.x32_packed = nullptr;
  if ((flags & MEMVUL_ENC_PACKED) && !(flags & MEMVUL_ENC_CLS_ONLY)) {
    ws.x32_packed = reinterpret_cast<float*>(p + off); off += up(M * H * 4);
  }
  ws.bytes = off;
  return ws;
}

// ------------------------------------------------------------------ accuracy mode (MEMVUL_ENC_PRECISE, precise.cuh)
int split3_impl(const float* x, void* out, int M, int K, int act, cudaStream_t st, const int* m_dev) {
  if (M <= 0 || K <= 0 || K % 4 != 0) return fail(MEMVUL_E_INVALID, "split3 needs M > 0 and K %% 4 == 0 (M=%d K=%d)", M, K);
  DeviceInfo di;
  if (int rc = device_info(&di)) return rc;
  const long long total = static_cast<long long>(M) * (K / 4);
  long long blocks = (total + 255) / 256;
  if (blocks > di.sms * 16LL) blocks = di.sms * 16LL;
  LaunchScope ls(g_cls == KC_CLS_TAIL ? KC_CLS_TAIL : KC_LAYERNORM, st);
  if (act == 1) mv::split3_rows_kernel<1><<<static_cast<int>(blocks), 256, 0, st>>>(x, reinterpret_cast<__half*>(out), M, K, m_dev);
  else mv::split3_rows_kernel<0><<<static_cast<int>(blocks), 256, 0, st>>>(x, reinterpret_cast<__half*>(out), M, K, m_dev);
  CUDA_TRY(cudaGetLastError());
  return MEMVUL_OK;
}

int attention_f32_impl(const float* qkv, const int32_t* lens, const int32_t* row_start, float* ctx, int B, int S, int H,
                       cudaStream_t st) {
  if (B <= 0 || S <= 0 || S > 512) return fail(MEMVUL_E_INVALID, "attention needs 1 <= S <= 512 (B=%d S=%d)", B, S);
  if (H % 64 != 0) return fail(MEMVUL_E_INVALID, "attention needs H %% 64 == 0 (head_dim 64), H=%d", H);
  if (B > 65535) return fail(MEMVUL_E_INVALID, "fp32 attention takes at most 65535 sequences per call (B=%d)", B);
  DeviceInfo di;
  if (int rc = device_info(&di)) return rc;
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(mv::attention_f32_kernel), mv::AttnF32Cfg::SMEM_BYTES)) return rc;
  const int n_qt = (S + mv::AttnF32Cfg::BQ - 1) / mv::AttnF32Cfg::BQ;
  LaunchScope ls(KC_ATTENTION, st);
  mv::attention_f32_kernel<<<dim3(n_qt, H / 64, B), 256, mv::AttnF32Cfg::SMEM_BYTES, st>>>(qkv, lens, row_start, ctx, B, S, H, n_qt);
  CUDA_TRY(cudaGetLastError());
  return MEMVUL_OK;
}

struct PreciseWs {
  float* x32;       // [M,H]   residual stream (token-major; the caller's hidden_out holds it in the padded layout)
  __half* xs;       // [M,3H]  split operand of the QKV / attn-out / FFN-up GEMMs
  float* qkv32;     // [M,3H]
  float* ctx32;     // [M,H]
  float* h32;       // [M,I]
  __half* hs;       // [M,3I]  split GELU output = operand of the FFN-down GEMM
  size_t bytes;
};
PreciseWs carve_precise(const memvul_bert_weights* w, int B, int S, void* base) {
  const size_t M = static_cast<size_t>(B) * S, H = w->hidden, I = w->intermediate;
  auto up = [](size_t x) { return (x + 1023) & ~size_t(1023); };
  uint8_t* p = reinterpret_cast<uint8_t*>(base);
  size_t off = 0;
  PreciseWs ws;
  ws.x32 = reinterpret_cast<float*>(p + off); off += up(M * H * 4);
  ws.xs = reinterpret_cast<__half*>(p + off); off += up(M * 3 * H * 2);
  ws.qkv32 = reinterpret_cast<float*>(p + off); off += up(M * 3 * H * 4);
  ws.ctx32 = reinterpret_cast<float*>(p + off); off += up(M * H * 4);
  ws.h32 = reinterpret_cast<float*>(p + off); off += up(M * I * 4);
  ws.hs = reinterpret_cast<__half*>(p + off); off += up(M * 3 * I * 2);
  ws.bytes = off;
  return ws;
}

// The encoder with split-fp16 operands (precise.cuh): same layer structure, every GEMM is a K' = 3K problem on the
// tcgen05 kernels with fp32 output, everything between the GEMMs is fp32.  w->layer[*].w_* are the K-concatenated
// [N, 3K] matrices [W_hi | W_hi | W_lo].
int encoder_forward_precise(const memvul_bert_weights* w, const int64_t* token_ids, const int64_t* type_ids,
                            const int32_t* lens, const int32_t* row_start, int B, int S, float* hidden_out,
                            void* workspace, size_t workspace_bytes, int flags, int32_t* bad_flag, cudaStream_t st) {
  const bool cls_only = (flags & MEMVUL_ENC_CLS_ONLY) != 0;
  const bool packed = (flags & MEMVUL_ENC_PACKED) != 0;
  PreciseWs ws = carve_precise(w, B, S, workspace);
  if (ws.bytes > workspace_bytes)
    return fail(MEMVUL_E_WORKSPACE, "workspace too small: need %zu bytes, got %zu", ws.bytes, workspace_bytes);
  const int M = B * S, H = w->hidden, I = w->intermediate;
  const int32_t* rs = packed ? row_start : nullptr;
  const int* m_dev = packed ? row_start + B : nullptr;
  float* x32 = packed ? ws.x32 : hidden_out;          // padded layout: the residual stream IS the output tensor
  // K1 (the fp16 copy it also writes is not used in this mode: it lands in the hs scratch)
  if (int rc = embed_impl(w, token_ids, type_ids, lens, rs, B, S, x32, ws.hs, bad_flag, st)) return rc;
  for (int l = 0; l < w->layers; ++l) {
    const memvul_bert_layer& L = w->layer[l];
    if (int rc = split3_impl(x32, ws.xs, M, H, 0, st, m_dev)) return rc;
    { ClassScope cs(KC_GEMM_QKV);
      if (int rc = gemm_impl(ws.xs, L.w_qkv, L.b_qkv, nullptr, ws.qkv32, M, 3 * H, 3 * H, MEMVUL_EPI_BIAS_F32, st, m_dev)) return rc; }
    if (int rc = attention_f32_impl(ws.qkv32, lens, rs, ws.ctx32, B, S, H, st)) return rc;
    if (int rc = split3_impl(ws.ctx32, ws.xs, M, H, 0, st, m_dev)) return rc;
    { ClassScope cs(KC_GEMM_ATTN_OUT);
      if (int rc = gemm_impl(ws.xs, L.w_ao, L.b_ao, x32, x32, M, H, 3 * H, MEMVUL_EPI_BIAS_RESID_F32, st, m_dev)) return rc; }
    if (int rc = layernorm_impl(x32, L.ln1_g, L.ln1_b, w->ln_eps, x32, nullptr, M, H, st)) return rc;
    if (int rc = split3_impl(x32, ws.xs, M, H, 0, st, m_dev)) return rc;
    { ClassScope cs(KC_GEMM_FFN_UP);
      if (int rc = gemm_impl(ws.xs, L.w_ff1, L.b_ff1, nullptr, ws.h32, M, I, 3 * H, MEMVUL_EPI_BIAS_F32, st, m_dev)) return rc; }
    if (int rc = split3_impl(ws.h32, ws.hs, M, I, 1, st, m_dev)) return rc;
    { ClassScope cs(KC_GEMM_FFN_DOWN);
      if (int rc = gemm_impl(ws.hs, L.w_ff2, L.b_ff2, x32, x32, M, H, 3 * I, MEMVUL_EPI_BIAS_RESID_F32, st, m_dev)) return rc; }
    if (int rc = layernorm_impl(x32, L.ln2_g, L.ln2_b, w->ln_eps, x32, nullptr, M, H, st)) return rc;
  }
  if (packed) {
    LaunchScope ls(KC_OTHER, st);
    if (cls_only) mv::scatter_cls_rows_kernel<<<B, 192, 0, st>>>(ws.x32, row_start, hidden_out, B, S, H);
    else mv::unpack_rows_kernel<<<(M + 7) / 8, 256, 0, st>>>(ws.x32, row_start, lens, hidden_out, B, S, H);
    CUDA_TRY(cudaGetLastError());
  }
  return MEMVUL_OK;
}

int check_weights(const memvul_bert_weights* w) {
  if (!w || !w->layer) return fail(MEMVUL_E_INVALID, "null weights");
  if (w->hidden != 768 && w->hidden != 128) return fail(MEMVUL_E_INVALID, "hidden must be 768 or 128, got %d", w->hidden);
  if (w->heads * 64 != w->hidden) return fail(MEMVUL_E_INVALID, "head_dim must be 64 (hidden=%d heads=%d)", w->hidden, w->heads);
  if (w->intermediate % 128 != 0) return fail(MEMVUL_E_INVALID, "intermediate must be a multiple of 128, got %d", w->intermediate);
  if (w->layers <= 0) return fail(MEMVUL_E_INVALID, "layers=%d", w->layers);
  return MEMVUL_OK;
}

}  // namespace

extern "C" {

int memvul_abi_version(void) { return MEMVUL_ABI_VERSION; }
const char* memvul_last_error(void) { return g_err; }

size_t memvul_encoder_workspace_bytes(const memvul_bert_weights* w, int B, int S, int flags) {
  if (!w || B <= 0 || S <= 0) return 0;
  if (flags & MEMVUL_ENC_PRECISE) return carve_precise(w, B, S, nullptr).bytes;
  return carve(w, B, S, nullptr, flags).bytes;
}

int memvul_gemm_f16(const void* a, const void* w, const float* bias, const float* resid, void* out, int M, int N,
                    int K, int epilogue, void* stream) {
  return gemm_impl(a, w, bias, resid, out, M, N, K, epilogue, static_cast<cudaStream_t>(stream));
}


int memvul_gemm_ln_f16(const void* a, const void* w, const float* bias, const float* resid, const float* gamma,
                       const float* beta, float eps, float* x32, void* x16, int M, int N, int K, void* stream) {
  if (!a || !w || !bias || !resid || !gamma || !beta || !x32 || !x16) return fail(MEMVUL_E_INVALID, "gemm_ln null pointer");
  int rc = gemm_ln_impl(a, w, bias, resid, gamma, beta, eps, x32, x16, M, N, K, static_cast<cudaStream_t>(stream));
  if (rc == 1) return fail(MEMVUL_E_INVALID, "gemm_ln needs N == 768, K %% 64 == 0, M >= 256 (M=%d N=%d K=%d)", M, N, K);
  return rc;
}

int memvul_attention_f16(const void* qkv, const int32_t* lens, const int32_t* row_start, void* ctx, int B, int S,
                         int H, void* stream) {
  if (!qkv || !lens || !ctx) return fail(MEMVUL_E_INVALID, "attention null pointer");
  return attention_impl(qkv, lens, row_start, ctx, B, S, H, static_cast<cudaStream_t>(stream));
}

int memvul_attention_f32(const float* qkv, const int32_t* lens, const int32_t* row_start, float* ctx, int B, int S,
                         int H, void* stream) {
  if (!qkv || !lens || !ctx) return fail(MEMVUL_E_INVALID, "attention null pointer");
  return attention_f32_impl(qkv, lens, row_start, ctx, B, S, H, static_cast<cudaStream_t>(stream));
}

int memvul_split3_f16(const float* x, void* out, int M, int K, int gelu, void* stream) {
  if (!x || !out) return fail(MEMVUL_E_INVALID, "split3 null pointer");
  return split3_impl(x, out, M, K, gelu ? 1 : 0, static_cast<cudaStream_t>(stream), nullptr);
}

int memvul_layernorm(const float* y, const float* gamma, const float* beta, float eps, float* x32, void* x16, int M,
                     int H, void* stream) {
  if (!y || !gamma || !beta) return fail(MEMVUL_E_INVALID, "layernorm null pointer");
  return layernorm_impl(y, gamma, beta, eps, x32, x16, M, H, static_cast<cudaStream_t>(stream));
}

int memvul_embed_layernorm(const memvul_bert_weights* w, const int64_t* token_ids, const int64_t* type_ids,
                           const int32_t* lens, const int32_t* row_start, int B, int S, float* x32, void* x16,
                           int32_t* bad_flag, void* stream) {
  if (!w || !token_ids || !x32 || !x16) return fail(MEMVUL_E_INVALID, "embed null pointer");
  if (B <= 0 || S <= 0 || S > w->max_pos) return fail(MEMVUL_E_INVALID, "embed needs 1 <= S <= max_pos (B=%d S=%d)", B, S);
  if (row_start && !lens) return fail(MEMVUL_E_INVALID, "embed: the packed layout needs lens as well as row_start");
  return embed_impl(w, token_ids, type_ids, lens, row_start, B, S, x32, x16, bad_flag, static_cast<cudaStream_t>(stream));
}

int memvul_mask_to_lens(const uint8_t* mask, int B, int S, int32_t* lens, int32_t* row_start, int32_t* bad_flag,
                        void* stream) {
  if (!mask || !lens || !bad_flag || B <= 0 || S <= 0) return fail(MEMVUL_E_INVALID, "mask_to_lens bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  {
    LaunchScope ls(KC_OTHER, st);
    mask_to_lens_kernel<<<(B + 7) / 8, 256, 0, st>>>(mask, B, S, lens, bad_flag);
    CUDA_TRY(cudaGetLastError());
  }
  if (row_start) {
    LaunchScope ls(KC_OTHER, st);
    lens_to_row_start_kernel<<<1, 1024, 0, st>>>(lens, B, row_start);
    CUDA_TRY(cudaGetLastError());
  }
  return MEMVUL_OK;
}

int memvul_encoder_forward(const memvul_bert_weights* w, const int64_t* token_ids, const int64_t* type_ids,
                           const int32_t* lens, const int32_t* row_start, int B, int S, float* hidden_out,
                           void* workspace, size_t workspace_bytes, int flags, int32_t* bad_flag, void* stream) {
  if (int rc = check_weights(w)) return rc;
  if (!token_ids || !lens || !hidden_out || !workspace) return fail(MEMVUL_E_INVALID, "encoder null pointer");
  if (B <= 0 || S <= 0 || S > 512 || S > w->max_pos)
    return fail(MEMVUL_E_INVALID, "encoder needs 1 <= S <= min(512, max_pos) (B=%d S=%d)", B, S);
  const bool cls_only = (flags & MEMVUL_ENC_CLS_ONLY) != 0;
  const bool packed = (flags & MEMVUL_ENC_PACKED) != 0;
  if (packed && !row_start) return fail(MEMVUL_E_INVALID, "MEMVUL_ENC_PACKED needs row_start (memvul_mask_to_lens fills it)");
  if (flags & MEMVUL_ENC_PRECISE)
    return encoder_forward_precise(w, token_ids, type_ids, lens, row_start, B, S, hidden_out, workspace, workspace_bytes,
                                   flags, bad_flag, static_cast<cudaStream_t>(stream));
  Workspace ws = carve(w, B, S, workspace, flags);
  if (ws.bytes > workspace_bytes)
    return fail(MEMVUL_E_WORKSPACE, "workspace too small: need %zu bytes, got %zu", ws.bytes, workspace_bytes);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int M = B * S, H = w->hidden, I = w->intermediate;     // M: row count (padded) or its upper bound (packed)
  const int32_t* rs = packed ? row_start : nullptr;
  const int* m_dev = packed ? row_start + B : nullptr;           // device-side row count T = sum(lens)
  // residual stream: the caller's hidden_out, except for a packed full-output run (unpacked at the end)
  float* x32 = (packed && !cls_only) ? ws.x32_packed : hidden_out;
  // packed: the embedding also zero-fills the scratch rows past the last token that tiles and key blocks read but no
  // kernel of this call writes, so the workspace's previous contents never reach a result
  if (int rc = embed_impl(w, token_ids, type_ids, lens, rs, B, S, x32, ws.x16, bad_flag, st, ws.qkv, ws.ctx, ws.ffn))
    return rc;
  for (int l = 0; l < w->layers; ++l) {
    const memvul_bert_layer& L = w->layer[l];
    if (cls_only && l == w->layers - 1) {
      // Last layer, [CLS]-only tail: keys/values need every row, but only query row 0 of each sequence is consumed
      // downstream, so attention runs on the first query tile and everything after it on B gathered rows.
      { ClassScope cs(KC_GEMM_QKV);
      if (int rc = gemm_impl(ws.x16, L.w_qkv, L.b_qkv, nullptr, ws.qkv, M, 3 * H, H, MEMVUL_EPI_BIAS_F16, st, m_dev)) return rc; }
      if (int rc = attention_impl(ws.qkv, lens, rs, ws.ctx, B, S, H, st, /*first_tile_only=*/true)) return rc;
      ClassScope tail(KC_CLS_TAIL);              // the B-row launches are accounted apart from the full-size classes
      { LaunchScope ls(KC_CLS_TAIL, st);
        mv::gather_cls_rows_kernel<<<B, 192, 0, st>>>(x32, ws.ctx, ws.x32_cls, ws.ctx_cls, rs, B, S, H);
        CUDA_TRY(cudaGetLastError()); }
      if (int rc = gemm_impl(ws.ctx_cls, L.w_ao, L.b_ao, ws.x32_cls, ws.x32_cls, B, H, H, MEMVUL_EPI_BIAS_RESID_F32, st)) return rc;
      if (int rc = layernorm_impl(ws.x32_cls, L.ln1_g, L.ln1_b, w->ln_eps, ws.x32_cls, ws.x16_cls, B, H, st)) return rc;
      if (int rc = gemm_impl(ws.x16_cls, L.w_ff1, L.b_ff1, nullptr, ws.ffn_cls, B, I, H, MEMVUL_EPI_BIAS_GELU_F16, st)) return rc;
      if (int rc = gemm_impl(ws.ffn_cls, L.w_ff2, L.b_ff2, ws.x32_cls, ws.x32_cls, B, H, I, MEMVUL_EPI_BIAS_RESID_F32, st)) return rc;
      // final LayerNorm scatters row b into hidden_out[b*S] (the [CLS] slot of the padded layout)
      if (int rc = layernorm_impl(ws.x32_cls, L.ln2_g, L.ln2_b, w->ln_eps, hidden_out, nullptr, B, H, st, (long long)S * H)) return rc;
      break;
    }
    { ClassScope cs(KC_GEMM_QKV);
    if (int rc = gemm_impl(ws.x16, L.w_qkv, L.b_qkv, nullptr, ws.qkv, M, 3 * H, H, MEMVUL_EPI_BIAS_F16, st, m_dev)) return rc; }
    if (int rc = attention_impl(ws.qkv, lens, rs, ws.ctx, B, S, H, st)) return rc;
    { ClassScope cs(KC_GEMM_ATTN_OUT);
      int rc = gemm_ln_impl(ws.ctx, L.w_ao, L.b_ao, x32, L.ln1_g, L.ln1_b, w->ln_eps, x32, ws.x16, M, H, H, st, m_dev);
      if (rc < 0) return rc;
      if (rc == 1) {      // shape not covered by the fused kernel: GEMM + stand-alone LayerNorm
        if (int rc2 = gemm_impl(ws.ctx, L.w_ao, L.b_ao, x32, x32, M, H, H, MEMVUL_EPI_BIAS_RESID_F32, st, m_dev)) return rc2;
        if (int rc2 = layernorm_impl(x32, L.ln1_g, L.ln1_b, w->ln_eps, x32, ws.x16, M, H, st)) return rc2;
      } }
    { ClassScope cs(KC_GEMM_FFN_UP);
    if (int rc = gemm_impl(ws.x16, L.w_ff1, L.b_ff1, nullptr, ws.ffn, M, I, H, MEMVUL_EPI_BIAS_GELU_F16, st, m_dev)) return rc; }
    { ClassScope cs(KC_GEMM_FFN_DOWN);
      int rc = gemm_ln_impl(ws.ffn, L.w_ff2, L.b_ff2, x32, L.ln2_g, L.ln2_b, w->ln_eps, x32, ws.x16, M, H, I, st, m_dev);
      if (rc < 0) return rc;
      if (rc == 1) {
        if (int rc2 = gemm_impl(ws.ffn, L.w_ff2, L.b_ff2, x32, x32, M, H, I, MEMVUL_EPI_BIAS_RESID_F32, st, m_dev)) return rc2;
        if (int rc2 = layernorm_impl(x32, L.ln2_g, L.ln2_b, w->ln_eps, x32, ws.x16, M, H, st)) return rc2;
      } }
  }
  if (packed && !cls_only) {          // packed residual stream -> the padded [B,S,H] tensor the interface returns
    LaunchScope ls(KC_OTHER, st);
    mv::unpack_rows_kernel<<<(M + 7) / 8, 256, 0, st>>>(ws.x32_packed, row_start, lens, hidden_out, B, S, H);
    CUDA_TRY(cudaGetLastError());
  }
  return MEMVUL_OK;
}


long long memvul_launch_count(void) { return g_launches.load(); }

int memvul_profile_enable(int on) {
  g_prof_on.store(on ? 1 : 0);
  return MEMVUL_OK;
}

int memvul_profile_read(int n_classes, double* ms_out, long long* count_out) {
  if (n_classes < KC_COUNT || !ms_out || !count_out) return fail(MEMVUL_E_INVALID, "profile_read needs %d slots", (int)KC_COUNT);
  CUDA_TRY(cudaDeviceSynchronize());
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (int i = 0; i < n_classes; ++i) { ms_out[i] = 0.0; count_out[i] = 0; }
  for (const ProfRec& r : g_prof_recs) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, r.e0, r.e1) == cudaSuccess) { ms_out[r.cls] += ms; count_out[r.cls] += 1; }
    g_prof_pool.push_back(r.e0);
    g_prof_pool.push_back(r.e1);
  }
  g_prof_recs.clear();
  return KC_COUNT;
}

int memvul_bank_prepare(const float* bank, const float* w_proj, int G, int D, float* vterm, void* stream) {
  if (!bank || !w_proj || !vterm || G <= 0 || D <= 0) return fail(MEMVUL_E_INVALID, "bank_prepare bad argument");
  LaunchScope ls(KC_OTHER, static_cast<cudaStream_t>(stream));
  mv::bank_vterm_kernel<<<(G + 7) / 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(bank, w_proj, vterm, G, D);
  CUDA_TRY(cudaGetLastError());
  return MEMVUL_OK;
}

int memvul_pool_match(const float* cls, int64_t cls_stride, const float* w_pool, const float* b_pool,
                      const float* w_head, const float* b_head, const float* w_proj, const float* bank,
                      const float* vterm, int B, int G, int H, int D, int same_idx, float* pooled, float* u,
                      float* uterm, uint64_t* best_key, float* logits, float* probs, int32_t* best_idx,
                      float* best_probs, int phase_mask, void* stream) {
  if (B <= 0 || H <= 0 || D <= 0 || H % 128 != 0 || H > 768 || D % 4 != 0 || D > 1024)
    return fail(MEMVUL_E_INVALID, "pool_match needs H %% 128 == 0, H <= 768, D %% 4 == 0, D <= 1024 (B=%d H=%d D=%d)", B, H, D);
  if (phase_mask <= 0 || phase_mask > MEMVUL_PM_ALL) return fail(MEMVUL_E_INVALID, "bad phase_mask %d", phase_mask);
  if ((phase_mask & (MEMVUL_PM_MATCH | MEMVUL_PM_FINAL)) &&
      (G <= 0 || !bank || !vterm || !logits || !probs || !best_key || !best_idx || !best_probs || !uterm))
    return fail(MEMVUL_E_INVALID, "pool_match: match phases need a non-empty bank and output buffers (G=%d)", G);
  if ((phase_mask & MEMVUL_PM_POOL) && (!cls || !w_pool || !b_pool || !pooled)) return fail(MEMVUL_E_INVALID, "pool_match: POOL needs cls/w_pool/b_pool/pooled");
  if ((phase_mask & MEMVUL_PM_HEADER) && (!w_head || !b_head || !pooled || !u)) return fail(MEMVUL_E_INVALID, "pool_match: HEADER needs w_head/b_head/pooled/u");
  if ((phase_mask & MEMVUL_PM_UTERM) && (!w_proj || !u || !uterm || !best_key)) return fail(MEMVUL_E_INVALID, "pool_match: UTERM needs w_proj/u/uterm/best_key");
  if (same_idx != 0 && same_idx != 1) return fail(MEMVUL_E_INVALID, "same_idx must be 0 or 1, got %d", same_idx);
  DeviceInfo di;
  if (int rc = device_info(&di)) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // Large problems (config-4 class) use the shared-memory tiled match: 1 block / SM with 167 KB of dynamic smem.
  static const bool tiled_ok = [] { const char* e = getenv("MEMVUL_MATCH_TILED"); return !(e && strcmp(e, "0") == 0); }();
  const bool tiled = tiled_ok && (phase_mask & MEMVUL_PM_MATCH) && D == mv::MatchTileCfg::D && B >= 32 &&
                     static_cast<long long>(B) * G >= (1LL << 18);
  const int dyn_smem = tiled ? mv::MatchTileCfg::SMEM_BYTES : 0;
  if (tiled)
    if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(mv::pool_match_kernel), dyn_smem)) return rc;
  int& bps = *per_device_slot(tiled ? 2 : 1);
  if (bps == 0) {
    int n = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, mv::pool_match_kernel, 256, dyn_smem));
    if (n < 1) return fail(MEMVUL_E_CUDA, "pool_match kernel does not fit on an SM");
    bps = n > 4 ? 4 : n;
  }
  const int grid = di.sms * bps;
  const int nwarps = grid * 8;
  mv::PoolMatchParams p;
  p.cls = cls; p.cls_stride = cls_stride;
  p.wp = w_pool; p.bp = b_pool; p.wh = w_head; p.bh = b_head; p.wproj = w_proj;
  p.bank = bank; p.vterm = vterm; p.pooled = pooled; p.u = u; p.uterm = uterm;
  p.best_key = reinterpret_cast<unsigned long long*>(best_key);
  p.logits = logits; p.probs = probs; p.best_idx = best_idx; p.best_probs = best_probs;
  p.B = B; p.G = G; p.H = H; p.D = D; p.same_idx = same_idx; p.phase_mask = phase_mask; p.tiled = tiled ? 1 : 0;
  // b_chunk: aim at ~4 work items per resident warp so the tail is short, but keep each anchor quad's
  // registers alive across as many queries as possible.
  const long long units = static_cast<long long>(B) * ((G + 3) / 4);
  long long bc = units / (4LL * nwarps);
  if (bc < 1) bc = 1;
  if (bc > B) bc = B;
  p.b_chunk = static_cast<int>(bc);
  if ((phase_mask & MEMVUL_PM_MATCH) && !(phase_mask & (MEMVUL_PM_POOL | MEMVUL_PM_UTERM)))
    CUDA_TRY(cudaMemsetAsync(best_key, 0, sizeof(uint64_t) * B, st));
  const bool multi = (phase_mask & (phase_mask - 1)) != 0;
  if (tiled) {        // Wd of both classes -> constant memory (pool_match.cuh: c_match_wd), stream-ordered
    CUDA_TRY(cudaMemcpyToSymbolAsync(mv::c_match_wd, w_proj + 2 * D, sizeof(float) * D, 0, cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaMemcpyToSymbolAsync(mv::c_match_wd, w_proj + 3 * D + 2 * D, sizeof(float) * D, sizeof(float) * D, cudaMemcpyDeviceToDevice, st));
  }
  LaunchScope ls(KC_POOL_MATCH, st);
  if (multi) {
    void* args[] = {&p};
    CUDA_TRY(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(mv::pool_match_kernel), dim3(grid), dim3(256), args, dyn_smem, st));
  } else {
    mv::pool_match_kernel<<<grid, 256, dyn_smem, st>>>(p);
    CUDA_TRY(cudaGetLastError());
  }
  return MEMVUL_OK;
}

int memvul_single_head(const float* feat, const float* w_cls, int B, int D, float* logits, float* probs, void* stream) {
  if (!feat || !w_cls || !logits || !probs || B <= 0 || D <= 0) return fail(MEMVUL_E_INVALID, "single_head bad argument");
  LaunchScope ls(KC_OTHER, static_cast<cudaStream_t>(stream));
  mv::single_head_kernel<<<(B + 7) / 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(feat, w_cls, logits, probs, B, D);
  CUDA_TRY(cudaGetLastError());
  return MEMVUL_OK;
}

}  // extern "C"
