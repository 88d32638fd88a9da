// Host side of libaf2b200.so: TMA descriptor construction, kernel launches and the per-module
// orchestration behind the C ABI declared in include/af2b200.h.
#include <cuda.h>
#include <cuda_runtime.h>
#include <cudaTypedefs.h>
#include <nvtx3/nvToolsExt.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/af2b200.h"
#include "attention_tc.cuh"
#include "chan2tok_tma.cuh"
#include "gemm_tc.cuh"
#include "ff_tc.cuh"
#include "proj_tc.cuh"
#include "simt_kernels.cuh"
#include "strict_kernels.cuh"
#include "glue_kernels.cuh"

using namespace af2;

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define CUDA_OK(expr)                                                                            \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) return fail(AF2_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)
#define AF2_TRY(expr)            \
  do {                           \
    int _r = (expr);             \
    if (_r != AF2_OK) return _r; \
  } while (0)

// Per-device state: the dynamic-shared-memory opt-in, the SM count and the cluster occupancy are properties of a
// device, and one process may drive several (ops.py keeps per-device workspaces), so every cache is indexed by ordinal.
constexpr int MAX_DEVICES = 64;
int cur_dev() {
  int dev = 0;
  cudaGetDevice(&dev);
  return (dev >= 0 && dev < MAX_DEVICES) ? dev : 0;
}
int sm_count() {
  static int n[MAX_DEVICES] = {0};
  const int dev = cur_dev();
  if (n[dev] == 0) {
    cudaDeviceGetAttribute(&n[dev], cudaDevAttrMultiProcessorCount, dev);
    if (n[dev] <= 0) n[dev] = 148;
  }
  return n[dev];
}

// AF2_X_EVICT_LAST=1: accesses to a fp32 residual stream whose size suits the L2 (48..100 MB: the pair tensor at C2) carry an
// evict_last hint, so most of it stays L2-resident from kernel to kernel (experiment, DESIGN.md)
int g_x_evict_last = 0;
inline int x_hint(long long tokens, int d) {
  const double mb = (double)tokens * d * 4 / 1e6;
  return (g_x_evict_last && mb >= 48.0 && mb <= 100.0) ? 1 : 0;
}

// Programmatic dependent launch (common.cuh): AF2_PDL=0 launches without the attribute (then wait / launch_dependents are no-ops)
int g_pdl = 1;
template <class... KArgs, class... Args>
cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = g_pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

struct NvtxRange {   // one NVTX range per C-ABI call (sub-op granularity for nsys / ncu --nvtx)
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

// ---------------------------------------------------------------------------------------------
// launch accounting + optional per-kernel-class CUDA-event profiling (bench.py roofline numbers)
// ---------------------------------------------------------------------------------------------
enum KClass { KC_GEMM_LINEAR = 0, KC_GEMM_CHANNEL = 1, KC_ATTENTION = 2, KC_LAYERNORM = 3, KC_CHAN2TOK = 4, KC_MISC = 5, KC_COUNT = 6 };
struct ProfRec { cudaEvent_t a, b; int cls; double flops, bytes; };
unsigned long long g_launches = 0;
bool g_prof = false;
std::vector<ProfRec> g_recs;
std::vector<cudaEvent_t> g_pool;

cudaEvent_t prof_event() {
  if (!g_pool.empty()) { cudaEvent_t e = g_pool.back(); g_pool.pop_back(); return e; }
  cudaEvent_t e; cudaEventCreate(&e); return e;
}
struct ProfScope {
  cudaStream_t s; bool on; ProfRec r;
  ProfScope(cudaStream_t st, int cls, double flops, double bytes) : s(st), on(g_prof) {
    ++g_launches;
    if (on) { r.a = prof_event(); r.b = prof_event(); r.cls = cls; r.flops = flops; r.bytes = bytes; cudaEventRecord(r.a, s); }
  }
  ~ProfScope() { if (on) { cudaEventRecord(r.b, s); g_recs.push_back(r); } }
};

PFN_cuTensorMapEncodeTiled_v12000 encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }
  return fn;
}

// bf16 tensor map. dims[0] is the contiguous dimension; strides_bytes[i] is the stride of dims[i+1].
int make_tmap(CUtensorMap* m, const void* base, int rank, const unsigned long long* dims,
              const unsigned long long* strides_bytes, const unsigned* box, CUtensorMapSwizzle swz,
              CUtensorMapDataType dt = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16,
              CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_256B) {
  auto fn = encode_fn();
  if (!fn) return fail(AF2_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t gdim[5];
  cuuint64_t gstr[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
  }
  for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i];
  if (reinterpret_cast<uintptr_t>(base) & 15) return fail(AF2_ERR_BAD_ARG, "TMA base pointer not 16-byte aligned");
  for (int i = 0; i + 1 < rank; ++i)
    if (gstr[i] & 15) return fail(AF2_ERR_BAD_ARG, "TMA stride %d (%llu B) not a multiple of 16", i, (unsigned long long)gstr[i]);
  CUresult r = fn(m, dt, rank, const_cast<void*>(base), gdim, gstr, bx, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swz, promo,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(AF2_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return AF2_OK;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
inline long long align_up(long long v, long long a) { return (v + a - 1) / a * a; }

// bump allocator over the caller's workspace
struct Arena {
  char* base;
  long long size, off;
  bool ok;
  Arena(void* b, long long s) : base(static_cast<char*>(b)), size(s), off(0), ok(true) {}
  template <class T>
  T* take(long long count) {
    long long bytes = align_up(count * (long long)sizeof(T), 256);
    if (off + bytes > size) {
      ok = false;
      return nullptr;
    }
    T* p = reinterpret_cast<T*>(base + off);
    off += bytes;
    return p;
  }
};

// -------------------------------------------------------------------------------------------------
// GEMM launch
// -------------------------------------------------------------------------------------------------
struct GemmCall {
  const void* A; long long lda; long long a_batch;
  const void* Bm; long long ldb; long long b_batch;
  int M, N, K, batch;
  bool mn_major;
  int bn;                 // 64 / 128 / 256
  // epilogue
  int mode, act, layout, use_rowscale;
  void* out; long long ld_out; long long out_batch;
  const float* bias; const float* rowscale; const float* resid; long long ld_resid;
  int cm_inner, cm_pitch;
  int out_cols;           // 0: N (N/2 for GATED); else explicit number of valid output columns
  // split-bf16 operands (strict precision, GemmParams::nseg): nseg = 3 (2 planes) or 6 (3 planes); a_half / b_half = element stride between planes
  int nseg; long long a_half, b_half;
  // gathered operands (GemmParams::a_pr / b_pr): rows (K-major) or columns (MN-major) per piece, element stride between pieces
  int a_pr, b_pr; long long a_piece, b_piece;
};

template <int BN, int STAGES, bool MN, int EK>
int launch_gemm_inst(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const CUtensorMap& tr,
                     const GemmParams& p, cudaStream_t s) {
  using L = GemmSmem<BN, STAGES>;
  static bool configured[MAX_DEVICES] = {false};
  auto kern = gemm_tc_kernel<BN, STAGES, MN, EK>;
  if (!configured[cur_dev()]) {
    CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL));
    configured[cur_dev()] = true;
  }
  const int m_tiles = (p.M + GEMM_BM - 1) / GEMM_BM;
  const long long total = (long long)p.batch * m_tiles * p.num_ntiles;
  if (total <= 0) return AF2_OK;
  const int grid = (int)(total < sm_count() ? total : sm_count());
  const double flops = 2.0 * p.batch * (double)p.M * p.N * p.K;    // algorithmic (a split-operand launch issues 3x this)
  const double obytes = (p.tile.mode == EPI_STORE_BF16 ? 2.0 : (p.tile.mode == EPI_GATED_BF16 ? 1.0 : (p.tile.mode == EPI_RESID_F32 ? 8.0 : 4.0)));
  const double bytes = p.batch * ((double)p.M * p.K * 2 + (p.batch > 1 ? (double)p.N * p.K * 2 : 0) + (double)p.M * p.N * obytes) +
                       (p.batch > 1 ? 0 : (double)p.N * p.K * 2);
  ProfScope ps(s, p.batch > 1 ? KC_GEMM_CHANNEL : KC_GEMM_LINEAR, flops, bytes);
  CUDA_OK(launch_pdl(kern, dim3(grid), dim3(GEMM_THREADS), L::TOTAL, s, ta, tb, tc, tr, p));
  return AF2_OK;
}

int launch_gemm(const GemmCall& c, cudaStream_t s) {
  if (c.M <= 0 || c.N <= 0 || c.K <= 0 || c.batch <= 0) return AF2_OK;
  CUtensorMap ta, tb;
  const int BN = c.bn;
  if (c.nseg > 1) {
    // rank-4 maps (k | mn, row | k, plane, batch) over split-bf16 operands: 2 planes for nseg 3, 3 planes for nseg 6
    const unsigned long long npl = c.nseg == 6 ? 3ull : 2ull;
    const unsigned long long ab = (unsigned long long)(c.batch > 1 ? c.a_batch : 0) * 2, bb_ = (unsigned long long)(c.batch > 1 ? c.b_batch : 0) * 2;
    if (!c.mn_major) {
      unsigned long long da[4] = {(unsigned long long)c.K, (unsigned long long)c.M, npl, (unsigned long long)c.batch};
      unsigned long long sa[3] = {(unsigned long long)c.lda * 2, (unsigned long long)c.a_half * 2, ab ? ab : (unsigned long long)c.a_half * 8};
      unsigned ba[4] = {64, 128, 1, 1};
      AF2_TRY(make_tmap(&ta, c.A, 4, da, sa, ba, CU_TENSOR_MAP_SWIZZLE_128B));
      unsigned long long db[4] = {(unsigned long long)c.K, (unsigned long long)c.N, npl, (unsigned long long)c.batch};
      unsigned long long sb[3] = {(unsigned long long)c.ldb * 2, (unsigned long long)c.b_half * 2, bb_ ? bb_ : (unsigned long long)c.b_half * 8};
      unsigned bx[4] = {64, (unsigned)BN, 1, 1};
      AF2_TRY(make_tmap(&tb, c.Bm, 4, db, sb, bx, CU_TENSOR_MAP_SWIZZLE_128B));
    } else {
      unsigned long long da[4] = {(unsigned long long)c.M, (unsigned long long)c.K, npl, (unsigned long long)c.batch};
      unsigned long long sa[3] = {(unsigned long long)c.lda * 2, (unsigned long long)c.a_half * 2, ab ? ab : (unsigned long long)c.a_half * 8};
      unsigned bx[4] = {64, 64, 1, 1};
      AF2_TRY(make_tmap(&ta, c.A, 4, da, sa, bx, CU_TENSOR_MAP_SWIZZLE_128B));
      unsigned long long db[4] = {(unsigned long long)c.N, (unsigned long long)c.K, npl, (unsigned long long)c.batch};
      unsigned long long sb[3] = {(unsigned long long)c.ldb * 2, (unsigned long long)c.b_half * 2, bb_ ? bb_ : (unsigned long long)c.b_half * 8};
      AF2_TRY(make_tmap(&tb, c.Bm, 4, db, sb, bx, CU_TENSOR_MAP_SWIZZLE_128B));
    }
  } else if (!c.mn_major) {
    unsigned long long da[3] = {(unsigned long long)c.K, (unsigned long long)c.M, (unsigned long long)c.batch};
    unsigned long long sa[2] = {(unsigned long long)c.lda * 2, (unsigned long long)(c.batch > 1 ? c.a_batch : c.lda * c.M) * 2};
    unsigned ba[3] = {64, 128, 1};
    AF2_TRY(make_tmap(&ta, c.A, 3, da, sa, ba, CU_TENSOR_MAP_SWIZZLE_128B));
    unsigned long long db[3] = {(unsigned long long)c.K, (unsigned long long)c.N, (unsigned long long)c.batch};
    unsigned long long sb[2] = {(unsigned long long)c.ldb * 2, (unsigned long long)(c.batch > 1 && c.b_batch ? c.b_batch : c.ldb * c.N) * 2};
    unsigned bb[3] = {64, (unsigned)BN, 1};
    AF2_TRY(make_tmap(&tb, c.Bm, 3, db, sb, bb, CU_TENSOR_MAP_SWIZZLE_128B));
  } else {
    unsigned long long da[3] = {(unsigned long long)c.M, (unsigned long long)c.K, (unsigned long long)c.batch};
    unsigned long long sa[2] = {(unsigned long long)c.lda * 2, (unsigned long long)(c.batch > 1 ? c.a_batch : c.lda * c.K) * 2};
    unsigned bx[3] = {64, 64, 1};
    AF2_TRY(make_tmap(&ta, c.A, 3, da, sa, bx, CU_TENSOR_MAP_SWIZZLE_128B));
    unsigned long long db[3] = {(unsigned long long)c.N, (unsigned long long)c.K, (unsigned long long)c.batch};
    unsigned long long sb[2] = {(unsigned long long)c.ldb * 2, (unsigned long long)(c.batch > 1 ? c.b_batch : c.ldb * c.K) * 2};
    AF2_TRY(make_tmap(&tb, c.Bm, 3, db, sb, bx, CU_TENSOR_MAP_SWIZZLE_128B));
  }
  // gathered ("pieces") operands: replace the plain map by a rank-4 map (k | mn, row | k, piece, batch)
  if (c.nseg <= 1 && (c.a_pr > 0 || c.b_pr > 0)) {
    const unsigned long long bsa = (unsigned long long)(c.batch > 1 ? c.a_batch : c.lda) * 2, bsb = (unsigned long long)(c.batch > 1 ? c.b_batch : c.ldb) * 2;
    if (!c.mn_major) {
      if (c.a_pr > 0) {
        if (c.a_pr % 128 != 0) return fail(AF2_ERR_BAD_ARG, "gemm: gathered A pieces of %d rows (need a multiple of 128)", c.a_pr);
        unsigned long long da[4] = {(unsigned long long)c.K, (unsigned long long)c.a_pr, (unsigned long long)((c.M + c.a_pr - 1) / c.a_pr), (unsigned long long)c.batch};
        unsigned long long sa[3] = {(unsigned long long)c.lda * 2, (unsigned long long)c.a_piece * 2, bsa};
        unsigned ba[4] = {64, 128, 1, 1};
        AF2_TRY(make_tmap(&ta, c.A, 4, da, sa, ba, CU_TENSOR_MAP_SWIZZLE_128B));
      }
      if (c.b_pr > 0) {
        if (!((c.b_pr % BN) == 0 || (BN % c.b_pr) == 0) || c.b_pr % 8) return fail(AF2_ERR_BAD_ARG, "gemm: gathered B pieces of %d rows do not tile BN=%d", c.b_pr, BN);
        unsigned long long db[4] = {(unsigned long long)c.K, (unsigned long long)c.b_pr, (unsigned long long)((c.N + c.b_pr - 1) / c.b_pr), (unsigned long long)c.batch};
        unsigned long long sb[3] = {(unsigned long long)c.ldb * 2, (unsigned long long)c.b_piece * 2, bsb};
        unsigned bb[4] = {64, (unsigned)(c.b_pr >= BN ? BN : c.b_pr), (unsigned)(c.b_pr >= BN ? 1 : BN / c.b_pr), 1};
        AF2_TRY(make_tmap(&tb, c.Bm, 4, db, sb, bb, CU_TENSOR_MAP_SWIZZLE_128B));
      }
    } else {
      unsigned bx[4] = {64, 64, 1, 1};
      if (c.a_pr > 0) {
        if (c.a_pr % 64) return fail(AF2_ERR_BAD_ARG, "gemm: gathered MN-major A pieces of %d columns (need a multiple of 64)", c.a_pr);
        unsigned long long da[4] = {(unsigned long long)c.a_pr, (unsigned long long)c.K, (unsigned long long)((c.M + c.a_pr - 1) / c.a_pr), (unsigned long long)c.batch};
        unsigned long long sa[3] = {(unsigned long long)c.lda * 2, (unsigned long long)c.a_piece * 2, bsa};
        AF2_TRY(make_tmap(&ta, c.A, 4, da, sa, bx, CU_TENSOR_MAP_SWIZZLE_128B));
      }
      if (c.b_pr > 0) {
        if (c.b_pr % 64) return fail(AF2_ERR_BAD_ARG, "gemm: gathered MN-major B pieces of %d columns (need a multiple of 64)", c.b_pr);
        unsigned long long db[4] = {(unsigned long long)c.b_pr, (unsigned long long)c.K, (unsigned long long)((c.N + c.b_pr - 1) / c.b_pr), (unsigned long long)c.batch};
        unsigned long long sb[3] = {(unsigned long long)c.ldb * 2, (unsigned long long)c.b_piece * 2, bsb};
        AF2_TRY(make_tmap(&tb, c.Bm, 4, db, sb, bx, CU_TENSOR_MAP_SWIZZLE_128B));
      }
    }
  }
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.M = c.M; p.N = c.N; p.K = c.K; p.batch = c.batch; p.nseg = c.nseg > 1 ? c.nseg : 1;
  if (c.nseg <= 1) { p.a_pr = c.a_pr; p.b_pr = c.b_pr; }
  p.x_evict_last = (c.mode == EPI_RESID_F32) ? x_hint(c.M, c.N) : 0;
  p.num_ntiles = (c.N + BN - 1) / BN;
  p.out_cols = c.out_cols > 0 ? c.out_cols : ((c.mode == EPI_GATED_BF16) ? c.N / 2 : c.N);
  p.rowscale = c.rowscale; p.resid = c.resid; p.ld_resid = c.ld_resid;
  p.out_batch_stride = c.out_batch;
  p.cm_inner = c.cm_inner > 0 ? c.cm_inner : 1; p.cm_pitch = c.cm_pitch > 0 ? c.cm_pitch : 1;
  p.tile.mode = c.mode; p.tile.act = c.act; p.tile.layout = c.layout; p.tile.use_rowscale = c.use_rowscale;
  p.tile.out = c.out; p.tile.bias = c.bias; p.tile.ld = c.ld_out;
  // ---- output path: TMA store through swizzled smem staging whenever the output is a legal TMA tensor ----
  const bool out_f32 = (c.mode == EPI_RESID_F32 || c.mode == EPI_STORE_F32);
  const int es = out_f32 ? 4 : 2;
  const int W = (c.mode == EPI_GATED_BF16) ? BN / 2 : BN;
  bool direct = false;
  if (!out_f32 && (W % 64) != 0) direct = true;
  if ((reinterpret_cast<uintptr_t>(c.out) & 15) != 0) direct = true;
  if (c.layout == LAYOUT_TOKEN) {
    if ((c.ld_out * es) % 16 != 0) direct = true;
    if (c.batch > 1 && (c.out_batch * es) % 16 != 0) direct = true;
  } else {
    if (c.cm_pitch != c.cm_inner || (c.ld_out * 2) % 16 != 0 || c.batch != 1 || out_f32) direct = true;
  }
  if (c.mode == EPI_RESID_F32 && ((c.ld_resid * 4) % 16 != 0 || (reinterpret_cast<uintptr_t>(c.resid) & 15) != 0)) direct = true;
  // warp-autonomous residual epilogue: one column tile, one batch, whole accumulator tile valid
  const bool resid_w = !direct && c.mode == EPI_RESID_F32 && BN == 256 && !c.mn_major && c.batch == 1 && c.N <= 256 &&
                       p.out_cols == 256;
  CUtensorMap tc = ta, tr = ta;
  if (!direct) {
    const CUtensorMapDataType dt = out_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    if (c.layout == LAYOUT_TOKEN) {
      unsigned long long dc[3] = {(unsigned long long)p.out_cols, (unsigned long long)c.M, (unsigned long long)c.batch};
      unsigned long long sc[2] = {(unsigned long long)c.ld_out * es, (unsigned long long)(c.batch > 1 ? c.out_batch : c.ld_out * c.M) * es};
      unsigned bc[3] = {(unsigned)(out_f32 ? 32 : 64), (unsigned)(resid_w ? 32 : 128), 1};
      AF2_TRY(make_tmap(&tc, c.out, 3, dc, sc, bc, CU_TENSOR_MAP_SWIZZLE_128B, dt));
      if (c.mode == EPI_RESID_F32) {
        unsigned long long sr[2] = {(unsigned long long)c.ld_resid * 4, (unsigned long long)c.ld_resid * c.M * 4};
        AF2_TRY(make_tmap(&tr, c.resid, 3, dc, sr, bc, CU_TENSOR_MAP_SWIZZLE_128B, dt));
      }
    } else {
      unsigned long long dc[3] = {(unsigned long long)c.M, (unsigned long long)p.out_cols, 1ull};
      unsigned long long sc[2] = {(unsigned long long)c.ld_out * 2, (unsigned long long)c.ld_out * p.out_cols * 2};
      unsigned bc[3] = {64, 64, 1};
      AF2_TRY(make_tmap(&tc, c.out, 3, dc, sc, bc, CU_TENSOR_MAP_SWIZZLE_128B, dt));
    }
  }
  p.direct = direct ? 1 : 0;
  // compile-time epilogue specialisation for the big-tile instantiation
  int ek = EK_GENERIC;
  if (!direct && BN == 256) {
    if (c.mode == EPI_STORE_BF16 && c.layout == LAYOUT_TOKEN && c.act == ACT_NONE && !c.use_rowscale) ek = EK_STORE_TOK;
    else if (c.mode == EPI_STORE_BF16 && c.layout == LAYOUT_TOKEN && c.act == ACT_SIGMOID && !c.use_rowscale) ek = EK_STORE_TOK_SIG;
    else if (c.mode == EPI_STORE_BF16 && c.layout == LAYOUT_CHANNEL && c.act == ACT_NONE) ek = EK_STORE_CH;
    else if (c.mode == EPI_GATED_BF16 && c.layout == LAYOUT_TOKEN && c.act == ACT_GELU && !c.use_rowscale) ek = EK_GATED_TOK_GELU;
    else if (c.mode == EPI_GATED_BF16 && c.layout == LAYOUT_CHANNEL && c.act == ACT_SIGMOID) ek = EK_GATED_CH_SIG;
    else if (c.mode == EPI_RESID_F32) ek = resid_w ? EK_RESID_F32_W : EK_RESID_F32;
    else if (c.mode == EPI_STORE_F32) ek = EK_STORE_F32;
  }
  if (c.mn_major) {
    if (BN == 256) {
      if (ek == EK_STORE_F32) return launch_gemm_inst<256, 3, true, EK_STORE_F32>(ta, tb, tc, tr, p, s);
      return launch_gemm_inst<256, 3, true, EK_GENERIC>(ta, tb, tc, tr, p, s);
    }
    if (BN == 128) return launch_gemm_inst<128, 4, true, EK_GENERIC>(ta, tb, tc, tr, p, s);
    return launch_gemm_inst<64, 6, true, EK_GENERIC>(ta, tb, tc, tr, p, s);
  }
  if (BN == 256) {
    switch (ek) {
      case EK_STORE_TOK: return launch_gemm_inst<256, 3, false, EK_STORE_TOK>(ta, tb, tc, tr, p, s);
      case EK_STORE_TOK_SIG: return launch_gemm_inst<256, 3, false, EK_STORE_TOK_SIG>(ta, tb, tc, tr, p, s);
      case EK_STORE_CH: return launch_gemm_inst<256, 3, false, EK_STORE_CH>(ta, tb, tc, tr, p, s);
      case EK_GATED_TOK_GELU: return launch_gemm_inst<256, 3, false, EK_GATED_TOK_GELU>(ta, tb, tc, tr, p, s);
      case EK_GATED_CH_SIG: return launch_gemm_inst<256, 3, false, EK_GATED_CH_SIG>(ta, tb, tc, tr, p, s);
      case EK_RESID_F32: return launch_gemm_inst<256, 3, false, EK_RESID_F32>(ta, tb, tc, tr, p, s);
      case EK_RESID_F32_W: return launch_gemm_inst<256, 3, false, EK_RESID_F32_W>(ta, tb, tc, tr, p, s);
      case EK_STORE_F32: return launch_gemm_inst<256, 3, false, EK_STORE_F32>(ta, tb, tc, tr, p, s);
      default: return launch_gemm_inst<256, 3, false, EK_GENERIC>(ta, tb, tc, tr, p, s);
    }
  }
  if (BN == 128) return launch_gemm_inst<128, 4, false, EK_GENERIC>(ta, tb, tc, tr, p, s);
  return launch_gemm_inst<64, 6, false, EK_GENERIC>(ta, tb, tc, tr, p, s);
}

int pick_bn(int n) { return n > 128 ? 256 : (n > 64 ? 128 : 64); }

GemmCall linear_call(const void* A, long long lda, const void* W, long long ldw, int M, int N, int K) {
  GemmCall c;
  memset(&c, 0, sizeof(c));
  c.A = A; c.lda = lda; c.Bm = W; c.ldb = ldw; c.M = M; c.N = N; c.K = K; c.batch = 1;
  c.mn_major = false; c.bn = pick_bn(N);
  return c;
}

// -------------------------------------------------------------------------------------------------
// LayerNorm launch
// -------------------------------------------------------------------------------------------------
int launch_layernorm(const LnParams& p, cudaStream_t s) {
  if (p.T <= 0) return AF2_OK;
  if (p.d % 4 != 0 || p.d > 1024) return fail(AF2_ERR_BAD_ARG, "LayerNorm: dim %d must be a multiple of 4 and <= 1024", p.d);
  const long long blocks_needed = (p.T + 7) / 8;
  const long long cap = (long long)sm_count() * 16;
  const int grid = (int)(blocks_needed < cap ? blocks_needed : cap);
  ProfScope ps(s, KC_LAYERNORM, 0.0, (double)p.T * p.d * (p.y ? 6.0 : 4.0) + (p.wb ? (double)p.T * p.heads * 2 : 0));
  if (p.d <= 128) layernorm_rows_kernel<1><<<grid, 256, 0, s>>>(p);
  else if (p.d <= 256) layernorm_rows_kernel<2><<<grid, 256, 0, s>>>(p);
  else if (p.d <= 512) layernorm_rows_kernel<4><<<grid, 256, 0, s>>>(p);
  else layernorm_rows_kernel<8><<<grid, 256, 0, s>>>(p);
  CUDA_OK(cudaGetLastError());
  return AF2_OK;
}

// pair bias <x_raw, w_edge> of T tokens (d % 32 == 0, d <= 256, heads <= 8), else the LayerNorm kernel's bias path
bool pair_bias_fast_ok(int d, int heads) { return d % 32 == 0 && d >= 32 && d <= 256 && heads <= 8; }
int launch_pair_bias(const float* x, long long T, int d, const float* wb, __nv_bfloat16* bias_out, int heads, long long bias_hs,
                     int n_inner, int pitch, cudaStream_t s, int transpose = 0) {
  if (T <= 0) return AF2_OK;
  PairBiasParams p;
  p.x = x; p.T = T; p.d = d; p.wb = wb; p.bias_out = bias_out; p.heads = heads; p.bias_hs = bias_hs; p.n_inner = n_inner; p.pitch = pitch;
  p.x_evict_last = x_hint(T, d);
  p.transpose = transpose;
  if (T > 0x7fffffffLL) return fail(AF2_ERR_BAD_ARG, "pair_bias: too many tokens");
  const bool mma = (d == 256 || d == 128);
  const long long need = mma ? (T + 127) / 128 : (T + 31) / 32;   // 8 warps x 16 (tensor-core kernel) / 4 tokens per block iteration
  const long long cap = (long long)sm_count() * 3;     // persistent: 3 resident blocks per SM
  const int grid = (int)(need < cap ? need : cap);
  ProfScope ps(s, KC_LAYERNORM, 0.0, (double)T * d * 4 + (double)T * heads * 2);
  if (mma && d == 256) CUDA_OK(launch_pdl(pair_bias_mma_kernel<16>, dim3(grid), dim3(256), 0, s, p));
  else if (mma) CUDA_OK(launch_pdl(pair_bias_mma_kernel<8>, dim3(grid), dim3(256), 0, s, p));
  else {
    switch (d / 32) {
      case 7: pair_bias_kernel<7><<<grid, 256, 0, s>>>(p); break;
      case 6: pair_bias_kernel<6><<<grid, 256, 0, s>>>(p); break;
      case 5: pair_bias_kernel<5><<<grid, 256, 0, s>>>(p); break;
      case 3: pair_bias_kernel<3><<<grid, 256, 0, s>>>(p); break;
      case 2: pair_bias_kernel<2><<<grid, 256, 0, s>>>(p); break;
      default: pair_bias_kernel<1><<<grid, 256, 0, s>>>(p); break;
    }
  }
  CUDA_OK(cudaGetLastError());
  return AF2_OK;
}

template <int D>
int launch_chan_to_token_tma(const ChanLnParams& p, long long T, cudaStream_t s) {
  using L = Chan2TokSmem<D>;
  static bool configured[MAX_DEVICES] = {false};
  auto kern = chan_to_token_tma_kernel<D>;
  if (!configured[cur_dev()]) {
    CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL));
    configured[cur_dev()] = true;
  }
  CUtensorMap tx, tg, ty;
  {
    unsigned long long dx[2] = {(unsigned long long)T, (unsigned long long)D};
    unsigned long long sx[1] = {(unsigned long long)p.chan_stride * 4};
    unsigned bx[2] = {C2T_TOK, (unsigned)D};
    AF2_TRY(make_tmap(&tx, p.src, 2, dx, sx, bx, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_DATA_TYPE_FLOAT32));
    unsigned long long dy[2] = {(unsigned long long)D, (unsigned long long)T};
    unsigned long long sy[1] = {(unsigned long long)D * 2};
    unsigned by[2] = {64, C2T_TOK};
    AF2_TRY(make_tmap(&ty, p.y, 2, dy, sy, by, CU_TENSOR_MAP_SWIZZLE_128B));
    if (p.mode == 0) AF2_TRY(make_tmap(&tg, p.gate, 2, dy, sy, by, CU_TENSOR_MAP_SWIZZLE_128B));
    else tg = ty;
  }
  Chan2TokParams q;
  q.T = T; q.mode = p.mode; q.gamma = p.gamma; q.beta = p.beta; q.scale = p.scale; q.scale_const = p.scale_const; q.eps = p.eps;
  const long long tiles = (T + C2T_TOK - 1) / C2T_TOK;
  const int grid = (int)(tiles < sm_count() ? tiles : sm_count());
  ProfScope ps(s, KC_CHAN2TOK, 0.0, (double)T * D * (p.mode == 0 ? 8.0 : 6.0));
  CUDA_OK(launch_pdl(kern, dim3(grid), dim3(L::THREADS), L::TOTAL, s, tx, tg, ty, q));
  return AF2_OK;
}

int g_c2t_tma = 1;   // 0: tile-per-CTA kernel (AF2_C2T_TMA=0)
int g_attn_bias_t = 0;      // 1: pair bias stored transposed ([h][key][query]) so the bias MMA's B operand is K-major (AF2_ATTN_BIAS_T)
int g_attn_ident_tmem = 1;  // 1: bias-MMA identity operand in tensor memory (AF2_ATTN_IDENT_TMEM=0: shared-memory strip)
int g_attn_skip = 0;       // DEBUG timing experiments (AF2_ATTN_SKIP bitmask, results wrong)
int g_attn_k3 = 0;         // 1: three K stages in the attention kernel's resident-bias mode (AF2_ATTN_K3)
int g_attn_headmajor = 0;  // EXPERIMENT: attention reads a head-major copy of q|k|v (AF2_ATTN_HEADMAJOR=1)
long long* g_attn_trace = nullptr;   // device buffer of 1024 stamps when AF2_ATTN_TRACE=1 (debug only)
int g_attn_l2pf = 0;      // 1: attention K producer prefetches upcoming K / V / Q / gate boxes into L2 (AF2_ATTN_L2PF)
int g_attn_group = 1;     // 1: attention CTAs grouped per (h, b') unit for 2..8 query blocks (AF2_ATTN_GROUP=0: n > 256 ungrouped)
int g_gather_fused = 1;   // 1: contractions over all-gathered operand pieces in ONE launch (AF2_GATHER_FUSED=0: one launch per piece)

int launch_chan_to_token(const ChanLnParams& p, cudaStream_t s) {
  const long long T = (long long)p.rows * p.n;
  if (g_c2t_tma && p.pitch == p.n && (p.d == 256 || p.d == 128) && (p.chan_stride % 4) == 0 && T > 0 && T < (1ll << 31) &&
      aligned16(p.src) && aligned16(p.y) && (p.mode != 0 || aligned16(p.gate))) {
    // dense token grid: persistent TMA-pipelined kernel
    return p.d == 256 ? launch_chan_to_token_tma<256>(p, T, s) : launch_chan_to_token_tma<128>(p, T, s);
  }
  if (p.pitch == p.n && p.d % 64 == 0 && p.d <= 256 && (T % 4) == 0) {
    // dense token grid: 64-token tiles, fully coalesced
    const size_t smem = (size_t)p.d * 64 * sizeof(float) + 8 * 64 * 2 * sizeof(float);
    static bool configured[MAX_DEVICES] = {false};
    if (!configured[cur_dev()]) {
      CUDA_OK(cudaFuncSetAttribute(chan_to_token_tile_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 256 * 64 * 4 + 4096));
      CUDA_OK(cudaFuncSetAttribute(chan_to_token_tile_kernel<24>, cudaFuncAttributeMaxDynamicSharedMemorySize, 192 * 64 * 4 + 4096));
      configured[cur_dev()] = true;
    }
    ProfScope ps(s, KC_CHAN2TOK, 0.0, (double)T * p.d * (p.mode == 0 ? 8.0 : 6.0));
    const unsigned grid = (unsigned)((T + 63) / 64);
    switch (p.d / 64) {
      case 4: chan_to_token_tile_kernel<32><<<grid, 512, smem, s>>>(p, T); break;
      case 3: chan_to_token_tile_kernel<24><<<grid, 512, smem, s>>>(p, T); break;
      case 2: chan_to_token_tile_kernel<16><<<grid, 512, smem, s>>>(p, T); break;
      default: chan_to_token_tile_kernel<8><<<grid, 512, smem, s>>>(p, T); break;
    }
    CUDA_OK(cudaGetLastError());
    return AF2_OK;
  }
  const size_t smem = (size_t)p.d * 33 * sizeof(float);
  static size_t configured[MAX_DEVICES] = {0};
  if (smem > 48 * 1024 && smem > configured[cur_dev()]) {
    CUDA_OK(cudaFuncSetAttribute(chan_to_token_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured[cur_dev()] = smem;
  }
  dim3 grid((p.n + 31) / 32, p.rows);
  ProfScope ps(s, KC_CHAN2TOK, 0.0, (double)p.rows * p.n * p.d * (p.mode == 0 ? 8.0 : 6.0));
  chan_to_token_kernel<<<grid, 256, smem, s>>>(p);
  CUDA_OK(cudaGetLastError());
  return AF2_OK;
}

// -------------------------------------------------------------------------------------------------
// attention launch (one folded batch group)
// -------------------------------------------------------------------------------------------------
template <int DH>
int launch_attention_inst(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const CUtensorMap& tbias,
                          const CUtensorMap& tg, const CUtensorMap& to, const AttnParams& p, cudaStream_t s) {
  using L = AttnSmem<DH>;
  static bool configured[MAX_DEVICES] = {false};
  auto kern = attention_tc_kernel<DH>;
  if (!configured[cur_dev()]) {
    CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL));
    configured[cur_dev()] = true;
  }
  const int nqb = (p.n + 127) / 128;
  const long long items = (long long)nqb * p.heads * p.nbatch;
  if (items <= 0) return AF2_OK;
  int grid = (int)(items < sm_count() ? items : sm_count());           // persistent CTAs
  if (nqb >= 2 && nqb <= 8 && g_attn_group) grid = grid / nqb * nqb;    // groups of nqb CTAs share the K/V of their (h, b') units
  const double tokens = (double)p.n * p.nbatch;
  ProfScope ps(s, KC_ATTENTION, 4.0 * tokens * p.n * p.heads * DH,
               tokens * p.heads * DH * 2.0 * 5 + (p.has_bias ? (double)p.heads * p.n * p.n * 2 : 0));
  CUDA_OK(launch_pdl(kern, dim3(grid), dim3(ATTN_THREADS), L::TOTAL, s, tq, tk, tv, tbias, tg, to, p));
  return AF2_OK;
}

// qkv: bf16 [tokens, 3I] (q | k | v), token(b', i) = b' * tok_sb + i * tok_si
int launch_attention(const __nv_bfloat16* qkv, int heads, int dh, int n, int nbatch, long long tok_sb, long long tok_si,
                     const __nv_bfloat16* bias, int npad, const uint8_t* mask, const __nv_bfloat16* gate,
                     __nv_bfloat16* out, cudaStream_t s, const __nv_bfloat16* qkv_hm = nullptr, long long hm_tokens = 0, int bias_t = 0) {
  const long long I = (long long)heads * dh;
  const long long ld = 3 * I;
  CUtensorMap tq, tk, tv, tb, tg, to;
  unsigned long long dims[4] = {(unsigned long long)dh, (unsigned long long)n, (unsigned long long)heads, (unsigned long long)nbatch};
  unsigned long long str[3] = {(unsigned long long)(tok_si * ld * 2), (unsigned long long)(dh * 2), (unsigned long long)(tok_sb * ld * 2)};
  if (qkv_hm) {   // head-major q|k|v [3H][hm_tokens][dh] (experiment AF2_ATTN_HEADMAJOR)
    str[0] = (unsigned long long)(tok_si * dh * 2); str[1] = (unsigned long long)(hm_tokens * dh * 2); str[2] = (unsigned long long)(tok_sb * dh * 2);
  }
  unsigned box[4] = {(unsigned)dh, 128, 1, 1};
  const CUtensorMapSwizzle swz = (dh == 64) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  // A box row is ONE head's slice of a token (dh * 2 bytes); the bytes next to it belong to other heads, which other CTAs
  // read at other times, so the L2 fill granularity must not exceed the row (256B promotion doubled the DRAM reads).
  const CUtensorMapL2promotion promo = (dh == 64) ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B : CU_TENSOR_MAP_L2_PROMOTION_L2_64B;
  const CUtensorMapDataType bf = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  if (qkv_hm) {
    const long long part = (long long)heads * hm_tokens * dh;
    AF2_TRY(make_tmap(&tq, qkv_hm, 4, dims, str, box, swz, bf, CU_TENSOR_MAP_L2_PROMOTION_L2_256B));
    AF2_TRY(make_tmap(&tk, qkv_hm + part, 4, dims, str, box, swz, bf, CU_TENSOR_MAP_L2_PROMOTION_L2_256B));
    AF2_TRY(make_tmap(&tv, qkv_hm + 2 * part, 4, dims, str, box, swz, bf, CU_TENSOR_MAP_L2_PROMOTION_L2_256B));
  } else {
    AF2_TRY(make_tmap(&tq, qkv, 4, dims, str, box, swz, bf, promo));
    AF2_TRY(make_tmap(&tk, qkv + I, 4, dims, str, box, swz, bf, promo));
    AF2_TRY(make_tmap(&tv, qkv + 2 * I, 4, dims, str, box, swz, bf, promo));
  }
  unsigned long long gstr[3] = {(unsigned long long)(tok_si * I * 2), (unsigned long long)(dh * 2), (unsigned long long)(tok_sb * I * 2)};
  AF2_TRY(make_tmap(&tg, gate, 4, dims, gstr, box, swz, bf, promo));
  unsigned obox[4] = {(unsigned)dh, 32, 1, 1};            // the output leaves per 32-row quarter of a query block
  AF2_TRY(make_tmap(&to, out, 4, dims, gstr, obox, swz));
  if (bias) {
    unsigned long long bd[3] = {(unsigned long long)npad, (unsigned long long)n, (unsigned long long)heads};
    unsigned long long bs[2] = {(unsigned long long)npad * 2, (unsigned long long)n * npad * 2};
    unsigned bb[3] = {64, 128, 1};
    AF2_TRY(make_tmap(&tb, bias, 3, bd, bs, bb, CU_TENSOR_MAP_SWIZZLE_128B));
  } else {
    tb = tq;
  }
  AttnParams p;
  memset(&p, 0, sizeof(p));
  p.n = n; p.heads = heads; p.nbatch = nbatch; p.has_bias = bias != nullptr;
  p.mask = mask; p.mask_sb = tok_sb; p.mask_si = tok_si;
  p.gate = gate; p.out = out; p.tok_sb = tok_sb; p.tok_si = tok_si; p.ld_gate = I; p.ld_out = I;
  p.l2_prefetch = g_attn_l2pf;
  p.k_stages3 = g_attn_k3;
  p.dbg_skip = g_attn_skip;
  p.ident_tmem = g_attn_ident_tmem;
  p.bias_t = bias_t;
  p.trace = g_attn_trace;
  if (dh == 64) return launch_attention_inst<64>(tq, tk, tv, tb, tg, to, p, s);
  if (dh == 32) return launch_attention_inst<32>(tq, tk, tv, tb, tg, to, p, s);
  return fail(AF2_ERR_BAD_ARG, "attention: dim_head %d unsupported (32 or 64)", dh);
}

#include "proj_launch.inl"

// 1 (default): FeedForward blocks that ff_tc_kernel takes run as that one fused launch; 0: LN->W1->GEGLU (proj_tc) + residual
// GEMM, two launches (af2_set_ff_fused, AF2_FF_FUSED)
int g_ff_fused = 1;

// shapes the fused transition kernel takes: d = 128 / 256 (pair-MMA N = d, K = d in pairs of 64-wide k-blocks), whole 64-unit
// hidden chunks, the per-256-row-tile W1 packing of the fused projection path
bool ff_fused_ok(const af2_ff_weights* w, int d, int hidden) {
  return g_ff_fused && g_proj_ctas == 2 && w->w_cat && w->w_ext && w->bn == 256 && (d == 128 || d == 256) &&
         hidden % FF_CHUNK == 0 && aligned16(w->w2) && aligned16(w->b2);
}

int launch_ff_fused(const af2_ff_weights* w, float* x, long long T, int d, int hidden, cudaStream_t s) {
  if (T <= 0) return AF2_OK;
  if (!aligned16(x)) return fail(AF2_ERR_BAD_ARG, "feed_forward: x not 16-byte aligned");
  using L = FfSmem;
  static bool configured_dev[MAX_DEVICES] = {false};
  static int max_clusters_dev[MAX_DEVICES] = {0};
  int& max_clusters = max_clusters_dev[cur_dev()];
  if (!configured_dev[cur_dev()]) {
    CUDA_OK(cudaFuncSetAttribute(ff_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL));
    cudaLaunchConfig_t qc;
    memset(&qc, 0, sizeof(qc));
    qc.gridDim = dim3(sm_count(), 1, 1); qc.blockDim = dim3(FF_THREADS, 1, 1); qc.dynamicSmemBytes = L::TOTAL;
    cudaLaunchAttribute qa[1];
    qa[0].id = cudaLaunchAttributeClusterDimension; qa[0].val.clusterDim.x = 2; qa[0].val.clusterDim.y = 1; qa[0].val.clusterDim.z = 1;
    qc.attrs = qa; qc.numAttrs = 1;
    int nc = 0;
    if (cudaOccupancyMaxActiveClusters(&nc, ff_tc_kernel, &qc) != cudaSuccess || nc <= 0) { cudaGetLastError(); nc = sm_count() / 2; }
    max_clusters = nc < sm_count() / 2 ? nc : sm_count() / 2;
    configured_dev[cur_dev()] = true;
  }
  const int n1p = (hidden + 127) / 128 * 256;          // packed W1 rows (w_cat)
  CUtensorMap tw1, tb1, tw2, tx;
  {
    unsigned long long dw[2] = {(unsigned long long)d, (unsigned long long)n1p};
    unsigned long long sw[1] = {(unsigned long long)d * 2};
    unsigned bw[2] = {64, 64};
    AF2_TRY(make_tmap(&tw1, w->w_cat, 2, dw, sw, bw, CU_TENSOR_MAP_SWIZZLE_128B));
    unsigned long long dx[2] = {16ull, (unsigned long long)n1p};
    unsigned long long sx[1] = {32ull};
    unsigned bx[2] = {16, 64};
    AF2_TRY(make_tmap(&tb1, w->w_ext, 2, dx, sx, bx, CU_TENSOR_MAP_SWIZZLE_32B));
    unsigned long long d2[2] = {(unsigned long long)hidden, (unsigned long long)d};
    unsigned long long s2[1] = {(unsigned long long)hidden * 2};
    unsigned b2[2] = {64, (unsigned)(d / 2)};
    AF2_TRY(make_tmap(&tw2, w->w2, 2, d2, s2, b2, CU_TENSOR_MAP_SWIZZLE_128B));
    unsigned long long dxr[2] = {(unsigned long long)d, (unsigned long long)T};
    unsigned long long sxr[1] = {(unsigned long long)d * 4};
    unsigned bxr[2] = {32, 32};
    AF2_TRY(make_tmap(&tx, x, 2, dxr, sxr, bxr, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_DATA_TYPE_FLOAT32));
  }
  FfParams p;
  memset(&p, 0, sizeof(p));
  p.x = x; p.b2 = w->b2; p.T = T; p.d = d; p.hidden = hidden; p.inv_d = 1.0f / (float)d; p.eps = 1e-5f;
  p.m_units = (int)((T + 255) / 256);
  const int clusters = p.m_units < max_clusters ? p.m_units : max_clusters;
  // algorithmic FLOPs of both Linear layers; bytes: x read + written once, both weight matrices once
  const double flops = 2.0 * T * (double)d * hidden * 3;
  const double bytes = (double)T * d * 8 + (double)n1p * d * 2 + (double)d * hidden * 2;
  ProfScope ps(s, KC_GEMM_LINEAR, flops, bytes);
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(clusters * 2, 1, 1); cfg.blockDim = dim3(FF_THREADS, 1, 1); cfg.dynamicSmemBytes = L::TOTAL; cfg.stream = s;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = g_pdl ? 2 : 1;
  CUDA_OK(cudaLaunchKernelEx(&cfg, ff_tc_kernel, tw1, tb1, tw2, tx, p));
  return AF2_OK;
}

// OuterMean normaliser of pair rows [row0, row0 + rows) of one batch element (quirk Q3): bit-packed kernel when the packed
// mask fits in shared memory, else the byte-loop kernel
int launch_outer_scale(const uint8_t* mask, float* scale, uint32_t* words, int row0, int rows, int S, int N, float eps, cudaStream_t s);

int ew_grid(long long n) {
  long long b = (n + 255) / 256;
  long long cap = (long long)sm_count() * 8;
  return (int)(b < cap ? (b > 0 ? b : 1) : cap);
}

int launch_outer_scale(const uint8_t* mask, float* scale, uint32_t* words, int row0, int rows, int S, int N, float eps, cudaStream_t s) {
  const long long T = (long long)rows * N;
  if (T <= 0) return AF2_OK;
  const int nw = (S + 31) / 32;
  const size_t smem = (size_t)nw * N * 4;
  ProfScope ps(s, KC_MISC, 0.0, 0.0);
  if (words && smem <= 160 * 1024) {
    static size_t configured[MAX_DEVICES] = {0};
    if (smem > 48 * 1024 && smem > configured[cur_dev()]) {
      CUDA_OK(cudaFuncSetAttribute(outer_scale_bits_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      configured[cur_dev()] = smem;
    }
    mask_pack_bits_kernel<<<ew_grid((long long)nw * N), 256, 0, s>>>(mask, words, S, N);
    CUDA_OK(cudaGetLastError());
    const long long need = (T + 255) / 256;
    const int grid = (int)(need < sm_count() ? need : sm_count());
    outer_scale_bits_kernel<<<grid, 256, smem, s>>>(words, scale, row0, rows, S, N, eps);
  } else {
    outer_scale_rows_kernel<<<ew_grid(T), 256, 0, s>>>(mask, scale, row0, rows, S, N, eps);
  }
  CUDA_OK(cudaGetLastError());
  return AF2_OK;
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

const char* af2_last_error(void) { return g_err; }
int af2_abi_version(void) { return 2; }

unsigned long long af2_launch_count(void) { return g_launches; }

void af2_profile_enable(int on) {
  g_prof = on != 0;
  if (g_prof) {
    for (auto& r : g_recs) { g_pool.push_back(r.a); g_pool.push_back(r.b); }
    g_recs.clear();
  }
}

// Sums the recorded launches of kernel class `cls` (synchronises the device). Returns the launch count.
long long af2_profile_read(int cls, double* ms, double* flops, double* bytes) {
  cudaDeviceSynchronize();
  double t = 0, f = 0, b = 0;
  long long n = 0;
  for (auto& r : g_recs) {
    if (r.cls != cls) continue;
    float e = 0.f;
    if (cudaEventElapsedTime(&e, r.a, r.b) == cudaSuccess) t += e;
    f += r.flops; b += r.bytes; ++n;
  }
  if (ms) *ms = t;
  if (flops) *flops = f;
  if (bytes) *bytes = b;
  return n;
}

// debug: copies the clock64 stamps of the last fused-projection launch (AF2_PROJ_TRACE=1) to `out` (2048 entries)
int af2_debug_proj_trace(long long* out) {
  if (!g_proj_trace) return fail(AF2_ERR_BAD_ARG, "projection trace not enabled (AF2_PROJ_TRACE=1)");
  CUDA_OK(cudaDeviceSynchronize());
  CUDA_OK(cudaMemcpy(out, g_proj_trace, 2048 * sizeof(long long), cudaMemcpyDeviceToHost));
  return AF2_OK;
}

// debug: copies the clock64 stamps of CTA 0 of the last attention launch (AF2_ATTN_TRACE=1) to `out` (1024 entries) and clears them
int af2_debug_attn_trace(long long* out) {
  if (!g_attn_trace) return fail(AF2_ERR_BAD_ARG, "attention trace not enabled (AF2_ATTN_TRACE=1)");
  CUDA_OK(cudaDeviceSynchronize());
  CUDA_OK(cudaMemcpy(out, g_attn_trace, 1024 * sizeof(long long), cudaMemcpyDeviceToHost));
  CUDA_OK(cudaMemset(g_attn_trace, 0, 1024 * sizeof(long long)));
  return AF2_OK;
}

void af2_set_proj_mode(int ctas) { g_proj_ctas = ctas < 0 ? 2 : (ctas > 2 ? 2 : ctas); }
void af2_set_ff_fused(int on) { g_ff_fused = on != 0; }

int af2_check_device(void) {
  if (const char* e = getenv("AF2_PROJ_CTAS")) af2_set_proj_mode(atoi(e));
  if (const char* e = getenv("AF2_FF_FUSED")) af2_set_ff_fused(atoi(e));
  if (const char* e = getenv("AF2_C2T_TMA")) g_c2t_tma = atoi(e) != 0;
  if (const char* e = getenv("AF2_PROJ_PRODTILES")) g_proj_prod_tiles = atof(e);
  if (const char* e = getenv("AF2_PROJ_BALANCE")) g_proj_balance = atoi(e) != 0;
  if (const char* e = getenv("AF2_PROJ_WIDE")) g_proj_wide = atoi(e) != 0;
  if (const char* e = getenv("AF2_PROJ_L2PF")) g_proj_l2pf = atoi(e) != 0;
  if (const char* e = getenv("AF2_GATHER_FUSED")) g_gather_fused = atoi(e) != 0;
  if (const char* e = getenv("AF2_ATTN_GROUP")) g_attn_group = atoi(e) != 0;
  if (const char* e = getenv("AF2_ATTN_L2PF")) g_attn_l2pf = atoi(e) != 0;
  if (const char* e = getenv("AF2_ATTN_HEADMAJOR")) g_attn_headmajor = atoi(e) != 0;
  if (const char* e = getenv("AF2_ATTN_K3")) g_attn_k3 = atoi(e) != 0;
  if (const char* e = getenv("AF2_ATTN_SKIP")) g_attn_skip = atoi(e);
  if (const char* e = getenv("AF2_ATTN_IDENT_TMEM")) g_attn_ident_tmem = atoi(e) != 0;
  if (const char* e = getenv("AF2_ATTN_BIAS_T")) g_attn_bias_t = atoi(e) != 0;
  if (const char* e = getenv("AF2_ATTN_TRACE")) {
    if (atoi(e) != 0 && !g_attn_trace) {
      if (cudaMalloc(&g_attn_trace, 1024 * sizeof(long long)) != cudaSuccess) g_attn_trace = nullptr;
      else cudaMemset(g_attn_trace, 0, 1024 * sizeof(long long));
    }
  }
  if (const char* e = getenv("AF2_X_EVICT_LAST")) g_x_evict_last = atoi(e) != 0;
  if (const char* e = getenv("AF2_PDL")) g_pdl = atoi(e) != 0;
  if (const char* e = getenv("AF2_PROJ_TRACE")) {
    if (atoi(e) != 0 && !g_proj_trace) {
      if (cudaMalloc(&g_proj_trace, 2048 * sizeof(long long)) != cudaSuccess) g_proj_trace = nullptr;
      else cudaMemset(g_proj_trace, 0, 2048 * sizeof(long long));
    }
  }
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return fail(AF2_ERR_CUDA, "no CUDA device");
  int major = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (major != 10) return fail(AF2_ERR_UNSUPPORTED_DEVICE, "libaf2b200 is built for sm_100a only; device has compute capability %d.x", major);
  return AF2_OK;
}

// ------------------------------------------------------------------------------------------------
long long af2_feed_forward_workspace(long long tokens, int d, int hidden) {
  return align_up(tokens * d * 2, 256) + align_up(tokens * hidden * 2, 256) + 1024;
}

int af2_feed_forward(const af2_ff_weights* w, float* x, long long tokens, int d, int hidden, void* workspace,
                     long long workspace_bytes, af2_stream_t stream) {
  NvtxRange nvtx_("af2_feed_forward");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (!w || !x) return fail(AF2_ERR_BAD_ARG, "feed_forward: null argument");
  if (d % 8 || hidden % 8) return fail(AF2_ERR_BAD_ARG, "feed_forward: d=%d and hidden=%d must be multiples of 8", d, hidden);
  if (tokens > 0x7fffffffLL) return fail(AF2_ERR_BAD_ARG, "feed_forward: too many tokens");
  if (ff_fused_ok(w, d, hidden)) return launch_ff_fused(w, x, tokens, d, hidden, s);   // LN -> W1 -> GEGLU -> W2 -> residual, h on chip
  Arena ar(workspace, workspace_bytes);
  __nv_bfloat16* xn = ar.take<__nv_bfloat16>(tokens * d);
  __nv_bfloat16* hbuf = ar.take<__nv_bfloat16>(tokens * hidden);
  if (!ar.ok) return fail(AF2_ERR_WORKSPACE, "feed_forward: workspace too small");
  // h = a * gelu(g)
  const int half = w->bn / 2;
  const int n1p = (hidden + half - 1) / half * w->bn;   // packed accumulator columns
  if (g_proj_ctas > 0 && w->w_cat && w->bn == 256 && proj_dim_ok(d)) {
    // fused LayerNorm -> Linear -> GEGLU (A-stationary CTA-pair kernel)
    ProjCall pc;
    memset(&pc, 0, sizeof(pc));
    pc.x = x; pc.T = tokens; pc.d = d;
    pc.w_cat = w->w_cat; pc.w_ext = w->w_ext; pc.nseg = 1;
    pc.seg[0] = ProjOut{n1p / 256, EK_GATED_TOK_GELU, hidden, hbuf, hidden};
    AF2_TRY(launch_proj(pc, s));
  } else {
    LnParams lp;
    memset(&lp, 0, sizeof(lp));
    lp.x = x; lp.gamma = w->ln_gamma; lp.beta = w->ln_beta; lp.y = xn; lp.T = tokens; lp.d = d; lp.eps = 1e-5f;
    AF2_TRY(launch_layernorm(lp, s));
    GemmCall c1 = linear_call(xn, d, w->w1, d, (int)tokens, n1p, d);
    c1.bn = w->bn; c1.mode = EPI_GATED_BF16; c1.act = ACT_GELU; c1.layout = LAYOUT_TOKEN;
    c1.out = hbuf; c1.ld_out = hidden; c1.bias = w->b1; c1.out_cols = hidden;
    AF2_TRY(launch_gemm(c1, s));
  }
  GemmCall c2 = linear_call(hbuf, hidden, w->w2, hidden, (int)tokens, d, hidden);
  c2.mode = EPI_RESID_F32; c2.out = x; c2.ld_out = d; c2.bias = w->b2; c2.resid = x; c2.ld_resid = d;
  AF2_TRY(launch_gemm(c2, s));
  return AF2_OK;
}

// ------------------------------------------------------------------------------------------------
long long af2_axial_attention_workspace(int B, int h, int wdim, int d, int heads, int dim_head, int row_attn) {
  const long long T = (long long)B * h * wdim, I = (long long)heads * dim_head;
  const int n = row_attn ? wdim : h;
  const long long npad = align_up(n, 8);
  return align_up(T * d * 2, 256) + 2 * align_up(T * 3 * I * 2, 256) + 2 * align_up(T * I * 2, 256) +
         align_up((long long)B * heads * n * npad * 2, 256) + 1024;
}

static int axial_attention_impl(const af2_attn_weights* w, float* x, const float* edges, const void* pre_bias,
                                const unsigned char* mask, int B, int h, int wdim, int d, int heads, int dim_head,
                                int row_attn, void* workspace, long long workspace_bytes, af2_stream_t stream, int tied = 0) {
  NvtxRange nvtx_(row_attn ? "af2_axial_attention(row)" : "af2_axial_attention(col)");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (!w || !x) return fail(AF2_ERR_BAD_ARG, "axial_attention: null argument");
  if (dim_head != 32 && dim_head != 64) return fail(AF2_ERR_BAD_ARG, "axial_attention: dim_head %d unsupported (32 or 64)", dim_head);
  if (d % 8) return fail(AF2_ERR_BAD_ARG, "axial_attention: dim %d must be a multiple of 8", d);
  const long long T = (long long)B * h * wdim, I = (long long)heads * dim_head;
  if (T > 0x7fffffffLL) return fail(AF2_ERR_BAD_ARG, "axial_attention: too many tokens");
  const int n = row_attn ? wdim : h;
  const int nb = row_attn ? h : wdim;
  const int npad = (int)align_up(n, 8);
  const bool has_bias = pre_bias != nullptr || (edges != nullptr && w->w_edge != nullptr);
  Arena ar(workspace, workspace_bytes);
  __nv_bfloat16* xn = ar.take<__nv_bfloat16>(T * d);
  __nv_bfloat16* qkv = ar.take<__nv_bfloat16>(T * 3 * I);
  __nv_bfloat16* gate = ar.take<__nv_bfloat16>(T * I);
  __nv_bfloat16* og = ar.take<__nv_bfloat16>(T * I);
  __nv_bfloat16* bias = ar.take<__nv_bfloat16>((long long)B * heads * n * npad);
  __nv_bfloat16* qkv_hm = ar.take<__nv_bfloat16>(T * 3 * I);
  if (!ar.ok) return fail(AF2_ERR_WORKSPACE, "axial_attention: workspace too small");
  if (pre_bias) bias = const_cast<__nv_bfloat16*>(static_cast<const __nv_bfloat16*>(pre_bias));   // [B][H][n][npad], zero padded

  // 1. LayerNorm (+ pair bias from the RAW edges; fused when the edges are x itself)
  const bool fused_proj = g_proj_ctas > 0 && w->w_cat && proj_dim_ok(d) && (I % 8) == 0;
  LnParams lp;
  memset(&lp, 0, sizeof(lp));
  lp.x = x; lp.gamma = w->ln_gamma; lp.beta = w->ln_beta; lp.y = xn; lp.T = T; lp.d = d; lp.eps = 1e-5f;
  const bool fuse_bias = has_bias && !pre_bias && edges == x && B == 1;
  // transposed bias [h][key][query] (K-major operand of the bias MMA) whenever the dedicated pair-bias kernel produces it
  const bool bias_t = g_attn_bias_t && has_bias && !pre_bias && pair_bias_fast_ok(d, heads) && !(fuse_bias && !fused_proj);
  // pad key columns are loaded by TMA next to valid ones: keep them finite (zero)
  if (has_bias && !pre_bias && npad != n) CUDA_OK(cudaMemsetAsync(bias, 0, (size_t)B * heads * n * npad * 2, s));
  if (fuse_bias) {
    lp.wb = w->w_edge; lp.bias_out = bias; lp.heads = heads; lp.bias_hs = (long long)n * npad; lp.n_inner = n; lp.pitch = npad;
  }
  if (!fused_proj) {
    AF2_TRY(launch_layernorm(lp, s));
  } else if (fuse_bias) {
    // pair bias only (raw x . w_edge); the LayerNorm itself is fused into the projection
    if (pair_bias_fast_ok(d, heads)) {
      AF2_TRY(launch_pair_bias(x, T, d, w->w_edge, bias, heads, (long long)n * npad, n, npad, s, bias_t ? 1 : 0));
    } else {
      lp.y = nullptr;
      AF2_TRY(launch_layernorm(lp, s));
    }
  }
  if (has_bias && !fuse_bias && !pre_bias && pair_bias_fast_ok(d, heads)) {
    for (int b = 0; b < B; ++b)
      AF2_TRY(launch_pair_bias(edges + (long long)b * n * n * d, (long long)n * n, d, w->w_edge, bias + (long long)b * heads * n * npad,
                               heads, (long long)n * npad, n, npad, s, bias_t ? 1 : 0));
  } else if (has_bias && !fuse_bias && !pre_bias) {
    for (int b = 0; b < B; ++b) {
      LnParams bp;
      memset(&bp, 0, sizeof(bp));
      bp.x = edges + (long long)b * n * n * d; bp.T = (long long)n * n; bp.d = d; bp.eps = 1e-5f;
      bp.wb = w->w_edge; bp.bias_out = bias + (long long)b * heads * n * npad; bp.heads = heads;
      bp.bias_hs = (long long)n * npad; bp.n_inner = n; bp.pitch = npad;
      AF2_TRY(launch_layernorm(bp, s));
    }
  }
  // 2. projections
  if (fused_proj) {
    // one launch: LayerNorm (+ pair bias) -> [q | k | v] and sigmoid(gating)
    ProjCall pc;
    memset(&pc, 0, sizeof(pc));
    pc.x = x; pc.T = T; pc.d = d;
    pc.w_cat = w->w_cat; pc.w_ext = w->w_ext; pc.nseg = 2;
    pc.seg[0] = ProjOut{(int)((3 * I + 255) / 256), EK_STORE_TOK, (int)(3 * I), qkv, 3 * I};
    pc.seg[1] = ProjOut{(int)((I + 255) / 256), EK_STORE_TOK_SIG, (int)I, gate, I};
    AF2_TRY(launch_proj(pc, s));
  } else {
    GemmCall cq = linear_call(xn, d, w->w_qkv, d, (int)T, (int)(3 * I), d);
    cq.mode = EPI_STORE_BF16; cq.layout = LAYOUT_TOKEN; cq.out = qkv; cq.ld_out = 3 * I;
    AF2_TRY(launch_gemm(cq, s));
    GemmCall cg = linear_call(xn, d, w->w_gate, d, (int)T, (int)I, d);
    cg.mode = EPI_STORE_BF16; cg.act = ACT_SIGMOID; cg.layout = LAYOUT_TOKEN; cg.out = gate; cg.ld_out = I; cg.bias = w->b_gate;
    AF2_TRY(launch_gemm(cg, s));
  }
  // 3. attention per batch element
  const long long tok_sb = row_attn ? wdim : 1, tok_si = row_attn ? 1 : wdim;
  for (int b = 0; b < B; ++b) {
    const long long t0 = (long long)b * h * wdim;
    if (tied) {   // MSAColumnGlobalAttention-style tied queries (alphafold2.py:142-151): q <- mean over the folded batch
      ProfScope ps(s, KC_MISC, 0.0, 0.0);
      tie_queries_kernel<__nv_bfloat16><<<ew_grid((long long)n * I), 256, 0, s>>>(qkv + t0 * 3 * I, 3 * I, (int)I, n, nb, tok_sb, tok_si);
      CUDA_OK(cudaGetLastError());
    }
    const long long Tb = (long long)h * wdim;
    if (g_attn_headmajor && dim_head % 8 == 0) {
      ProfScope ps(s, KC_MISC, 0.0, 0.0);
      qkv_to_headmajor_kernel<<<ew_grid(Tb * 3 * I / 8), 256, 0, s>>>(reinterpret_cast<const uint4*>(qkv + t0 * 3 * I),
                                                                        reinterpret_cast<uint4*>(qkv_hm + t0 * 3 * I), Tb, (int)(3 * I), dim_head);
      CUDA_OK(cudaGetLastError());
    }
    AF2_TRY(launch_attention(qkv + t0 * 3 * I, heads, dim_head, n, nb, tok_sb, tok_si,
                             has_bias ? bias + (long long)b * heads * n * npad : nullptr, npad,
                             mask ? mask + t0 : nullptr, gate + t0 * I, og + t0 * I, s,
                             (g_attn_headmajor && dim_head % 8 == 0) ? qkv_hm + t0 * 3 * I : nullptr, Tb, bias_t ? 1 : 0));
  }
  // 4. to_out + bias + residual
  GemmCall co = linear_call(og, I, w->w_out, I, (int)T, d, (int)I);
  co.mode = EPI_RESID_F32; co.out = x; co.ld_out = d; co.bias = w->b_out; co.resid = x; co.ld_resid = d;
  AF2_TRY(launch_gemm(co, s));
  return AF2_OK;
}

// ------------------------------------------------------------------------------------------------
long long af2_triangle_multiply_workspace(int B, int N, int d) {
  const long long T = (long long)B * N * N;
  const long long np8 = align_up(N, 8), np4 = align_up(N, 4);
  return 3 * align_up(T * d * 2, 256)                               // xn, gate, tn
         + 2 * align_up((long long)d * B * N * np8 * 2, 256)          // Lc, Rc
         + align_up((long long)d * B * N * np4 * 4, 256)              // Oc
         + align_up(T * 4, 256) + 1024;                               // mask as float
}

int af2_triangle_multiply(const af2_trimul_weights* w, float* x, const unsigned char* mask, int B, int N, int d,
                          int ingoing, void* workspace, long long workspace_bytes, af2_stream_t stream) {
  NvtxRange nvtx_("af2_triangle_multiply");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (!w || !x) return fail(AF2_ERR_BAD_ARG, "triangle_multiply: null argument");
  if (d % 32) return fail(AF2_ERR_BAD_ARG, "triangle_multiply: dim %d must be a multiple of 32", d);
  const long long T = (long long)B * N * N;
  if (T > 0x7fffffffLL) return fail(AF2_ERR_BAD_ARG, "triangle_multiply: too many tokens");
  const int np8 = (int)align_up(N, 8), np4 = (int)align_up(N, 4);
  const long long cs_lr = (long long)B * N * np8;   // channel stride of Lc / Rc
  const long long cs_o = (long long)B * N * np4;    // channel stride of Oc
  Arena ar(workspace, workspace_bytes);
  __nv_bfloat16* xn = ar.take<__nv_bfloat16>(T * d);
  __nv_bfloat16* gate = ar.take<__nv_bfloat16>(T * d);
  __nv_bfloat16* tn = ar.take<__nv_bfloat16>(T * d);
  __nv_bfloat16* Lc = ar.take<__nv_bfloat16>(d * cs_lr);
  __nv_bfloat16* Rc = ar.take<__nv_bfloat16>(d * cs_lr);
  float* Oc = ar.take<float>(d * cs_o);
  float* maskf = ar.take<float>(T);
  if (!ar.ok) return fail(AF2_ERR_WORKSPACE, "triangle_multiply: workspace too small");

  const bool fused_front = g_proj_ctas > 0 && w->w_cat && w->bn == 256 && proj_dim_ok(d) && np8 == N;
  if (fused_front) {
    ProjCall pc;
    memset(&pc, 0, sizeof(pc));
    pc.x = x; pc.T = T; pc.d = d;
    pc.w_cat = w->w_cat; pc.w_ext = w->w_ext; pc.rowmask = mask; pc.nseg = 3;
    const int tl = (d + 127) / 128;
    pc.seg[0] = ProjOut{tl, EK_GATED_CH_SIG, d, Lc, cs_lr};
    pc.seg[1] = ProjOut{tl, EK_GATED_CH_SIG, d, Rc, cs_lr};
    pc.seg[2] = ProjOut{(d + 255) / 256, EK_STORE_TOK_SIG, d, gate, (long long)d};
    AF2_TRY(launch_proj(pc, s));
  }
  LnParams lp;
  memset(&lp, 0, sizeof(lp));
  lp.x = x; lp.gamma = w->ln_gamma; lp.beta = w->ln_beta; lp.y = xn; lp.T = T; lp.d = d; lp.eps = 1e-5f;
  if (!fused_front) AF2_TRY(launch_layernorm(lp, s));
  if (mask && !fused_front) {
    { ProfScope ps(s, KC_MISC, 0.0, 0.0); mask_to_float_kernel<<<ew_grid(T), 256, 0, s>>>(mask, maskf, T); }
    CUDA_OK(cudaGetLastError());
  }
  if (np8 != N) {   // pad columns of the channel-major operands are read by TMA as K / MN padding: keep them zero
    CUDA_OK(cudaMemsetAsync(Lc, 0, (size_t)d * cs_lr * 2, s));
    CUDA_OK(cudaMemsetAsync(Rc, 0, (size_t)d * cs_lr * 2, s));
  }
  // left / right: (proj + b) * mask * sigmoid(gate + b)  -> channel-major [c][b*N + i][k]
  const int half = w->bn / 2;
  const int npk = (d + half - 1) / half * w->bn;
  for (int side = 0; side < 2 && !fused_front; ++side) {
    GemmCall c = linear_call(xn, d, side ? w->w_right : w->w_left, d, (int)T, npk, d);
    c.bn = w->bn; c.mode = EPI_GATED_BF16; c.act = ACT_SIGMOID; c.layout = LAYOUT_CHANNEL;
    c.out = side ? Rc : Lc; c.ld_out = cs_lr; c.bias = side ? w->b_right : w->b_left;
    c.use_rowscale = mask != nullptr; c.rowscale = maskf; c.cm_inner = N; c.cm_pitch = np8; c.out_cols = d;
    AF2_TRY(launch_gemm(c, s));
  }
  GemmCall cg = linear_call(xn, d, w->w_ogate, d, (int)T, d, d);
  cg.mode = EPI_STORE_BF16; cg.act = ACT_SIGMOID; cg.layout = LAYOUT_TOKEN; cg.out = gate; cg.ld_out = d; cg.bias = w->b_ogate;
  if (!fused_front) AF2_TRY(launch_gemm(cg, s));
  // per-channel contraction, batch = channels
  for (int b = 0; b < B; ++b) {
    GemmCall c;
    memset(&c, 0, sizeof(c));
    const long long boff = (long long)b * N * np8;
    if (!ingoing) {   // O_c = L_c R_c^T : both K-major (k contiguous)
      c.A = Lc + boff; c.Bm = Rc + boff; c.mn_major = false;
    } else {          // O_c[i][j] = sum_k R_c[k][i] L_c[k][j] : both MN-major
      c.A = Rc + boff; c.Bm = Lc + boff; c.mn_major = true;
    }
    c.lda = np8; c.ldb = np8; c.a_batch = cs_lr; c.b_batch = cs_lr;
    c.M = N; c.N = N; c.K = N; c.batch = d; c.bn = pick_bn(N);
    c.mode = EPI_STORE_F32; c.layout = LAYOUT_TOKEN; c.out = Oc + (long long)b * N * np4; c.ld_out = np4; c.out_batch = cs_o;
    AF2_TRY(launch_gemm(c, s));
  }
  // LN over channels * out_gate -> token-major bf16
  ChanLnParams cp;
  memset(&cp, 0, sizeof(cp));
  cp.src = Oc; cp.chan_stride = cs_o; cp.pitch = np4; cp.rows = B * N; cp.n = N; cp.d = d; cp.mode = 0;
  cp.gamma = w->on_gamma; cp.beta = w->on_beta; cp.gate = gate; cp.eps = 1e-5f; cp.y = tn;
  AF2_TRY(launch_chan_to_token(cp, s));
  GemmCall co = linear_call(tn, d, w->w_out, d, (int)T, d, d);
  co.mode = EPI_RESID_F32; co.out = x; co.ld_out = d; co.bias = w->b_out; co.resid = x; co.ld_resid = d;
  AF2_TRY(launch_gemm(co, s));
  return AF2_OK;
}

// ------------------------------------------------------------------------------------------------
long long af2_outer_mean_workspace(int B, int S, int N, int d) {
  const long long Tm = (long long)B * S * N, Tx = (long long)B * N * N;
  const long long np8 = align_up(N, 8), np4 = align_up(N, 4);
  return align_up(Tm * d * 2, 256) + align_up((long long)2 * d * B * S * np8 * 2, 256) +
         align_up((long long)d * B * N * np4 * 4, 256) + align_up(Tx * d * 2, 256) + align_up(Tm * 4, 256) +
         align_up(Tx * 4, 256) + align_up((long long)((S + 31) / 32) * N * 4, 256) + 1024;
}

int af2_outer_mean(const af2_outer_weights* w, float* x, const float* m, const unsigned char* msa_mask, int B, int S,
                   int N, int d, float eps, void* workspace, long long workspace_bytes, af2_stream_t stream) {
  NvtxRange nvtx_("af2_outer_mean");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (!w || !x || !m) return fail(AF2_ERR_BAD_ARG, "outer_mean: null argument");
  if (d % 32) return fail(AF2_ERR_BAD_ARG, "outer_mean: dim %d must be a multiple of 32", d);
  const long long Tm = (long long)B * S * N, Tx = (long long)B * N * N;
  if (Tm > 0x7fffffffLL || Tx > 0x7fffffffLL) return fail(AF2_ERR_BAD_ARG, "outer_mean: too many tokens");
  const int np8 = (int)align_up(N, 8), np4 = (int)align_up(N, 4);
  const long long cs_lr = (long long)B * S * np8, cs_o = (long long)B * N * np4;
  Arena ar(workspace, workspace_bytes);
  __nv_bfloat16* mn = ar.take<__nv_bfloat16>(Tm * d);
  __nv_bfloat16* LRc = ar.take<__nv_bfloat16>(2LL * d * cs_lr);
  float* Oc = ar.take<float>(d * cs_o);
  __nv_bfloat16* tn = ar.take<__nv_bfloat16>(Tx * d);
  float* maskf = ar.take<float>(Tm);
  float* scale = ar.take<float>(Tx);
  uint32_t* mwords = ar.take<uint32_t>((long long)((S + 31) / 32) * N);
  if (!ar.ok) return fail(AF2_ERR_WORKSPACE, "outer_mean: workspace too small");

  const bool fused_front = g_proj_ctas > 0 && w->w_cat && proj_dim_ok(d) && np8 == N;
  LnParams lp;
  memset(&lp, 0, sizeof(lp));
  lp.x = m; lp.gamma = w->ln_gamma; lp.beta = w->ln_beta; lp.y = mn; lp.T = Tm; lp.d = d; lp.eps = 1e-5f;
  if (!fused_front) AF2_TRY(launch_layernorm(lp, s));
  if (msa_mask) {
    if (!fused_front) { ProfScope ps(s, KC_MISC, 0.0, 0.0); mask_to_float_kernel<<<ew_grid(Tm), 256, 0, s>>>(msa_mask, maskf, Tm); }
    CUDA_OK(cudaGetLastError());
    for (int b = 0; b < B; ++b)
      AF2_TRY(launch_outer_scale(msa_mask + (long long)b * S * N, scale + (long long)b * N * N, mwords, 0, N, S, N, eps, s));
  }
  if (np8 != N) CUDA_OK(cudaMemsetAsync(LRc, 0, (size_t)2 * d * cs_lr * 2, s));
  // [left | right] = (LN(m) W^T + b) * mask  -> channel-major [c][b*S + s][i]
  if (fused_front) {
    ProjCall pc;
    memset(&pc, 0, sizeof(pc));
    pc.x = m; pc.T = Tm; pc.d = d;
    pc.w_cat = w->w_cat; pc.w_ext = w->w_ext; pc.rowmask = msa_mask; pc.nseg = 1;
    pc.seg[0] = ProjOut{(2 * d + 255) / 256, EK_STORE_CH, 2 * d, LRc, cs_lr};
    AF2_TRY(launch_proj(pc, s));
  } else {
    GemmCall c = linear_call(mn, d, w->w_lr, d, (int)Tm, 2 * d, d);
    c.mode = EPI_STORE_BF16; c.layout = LAYOUT_CHANNEL; c.out = LRc; c.ld_out = cs_lr; c.bias = w->b_lr;
    c.use_rowscale = msa_mask != nullptr; c.rowscale = maskf; c.cm_inner = N; c.cm_pitch = np8;
    AF2_TRY(launch_gemm(c, s));
  }
  // O_c[i][j] = sum_s L_c[s][i] R_c[s][j]  (MN-major operands, K = S)
  for (int b = 0; b < B; ++b) {
    GemmCall g;
    memset(&g, 0, sizeof(g));
    g.A = LRc + (long long)b * S * np8; g.Bm = LRc + (long long)d * cs_lr + (long long)b * S * np8;
    g.mn_major = true; g.lda = np8; g.ldb = np8; g.a_batch = cs_lr; g.b_batch = cs_lr;
    g.M = N; g.N = N; g.K = S; g.batch = d; g.bn = pick_bn(N);
    g.mode = EPI_STORE_F32; g.layout = LAYOUT_TOKEN; g.out = Oc + (long long)b * N * np4; g.ld_out = np4; g.out_batch = cs_o;
    AF2_TRY(launch_gemm(g, s));
  }
  ChanLnParams cp;
  memset(&cp, 0, sizeof(cp));
  cp.src = Oc; cp.chan_stride = cs_o; cp.pitch = np4; cp.rows = B * N; cp.n = N; cp.d = d; cp.mode = 1;
  cp.scale = msa_mask ? scale : nullptr; cp.scale_const = 1.0f / (float)S; cp.y = tn;
  AF2_TRY(launch_chan_to_token(cp, s));
  GemmCall co = linear_call(tn, d, w->w_out, d, (int)Tx, d, d);
  co.mode = EPI_RESID_F32; co.out = x; co.ld_out = d; co.bias = w->b_out; co.resid = x; co.ld_resid = d;
  AF2_TRY(launch_gemm(co, s));
  return AF2_OK;
}


int af2_axial_attention(const af2_attn_weights* w, float* x, const float* edges, const unsigned char* mask, int B,
                        int h, int wdim, int d, int heads, int dim_head, int row_attn, void* workspace,
                        long long workspace_bytes, af2_stream_t stream) {
  return axial_attention_impl(w, x, edges, nullptr, mask, B, h, wdim, d, heads, dim_head, row_attn, workspace,
                              workspace_bytes, stream);
}

// same with flags: bit 0 = tied queries (global_query_attn of the extra-MSA stack, alphafold2.py:142-151, 250)
int af2_axial_attention_ex(const af2_attn_weights* w, float* x, const float* edges, const unsigned char* mask, int B,
                           int h, int wdim, int d, int heads, int dim_head, int row_attn, int flags, void* workspace,
                           long long workspace_bytes, af2_stream_t stream) {
  return axial_attention_impl(w, x, edges, nullptr, mask, B, h, wdim, d, heads, dim_head, row_attn, workspace,
                              workspace_bytes, stream, flags & 1);
}

int af2_axial_attention_prebias(const af2_attn_weights* w, float* x, const void* bias_bf16, const unsigned char* mask,
                                int B, int h, int wdim, int d, int heads, int dim_head, int row_attn, void* workspace,
                                long long workspace_bytes, af2_stream_t stream) {
  return axial_attention_impl(w, x, nullptr, bias_bf16, mask, B, h, wdim, d, heads, dim_head, row_attn, workspace,
                              workspace_bytes, stream);
}

// bias rows of a shard of the pair tensor: out[h][r][j] (pitch npad, caller zero-fills the pad) = <x[r, j, :], w_edge[h, :]>
int af2_pair_bias(const float* x_rows, const float* w_edge, void* bias_out, int rows, int n, int d, int heads,
                  af2_stream_t stream) {
  NvtxRange nvtx_("af2_pair_bias");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (!x_rows || !w_edge || !bias_out) return fail(AF2_ERR_BAD_ARG, "pair_bias: null argument");
  const int npad = (int)align_up(n, 8);
  if (pair_bias_fast_ok(d, heads))
    return launch_pair_bias(x_rows, (long long)rows * n, d, w_edge, static_cast<__nv_bfloat16*>(bias_out), heads, (long long)rows * npad,
                            n, npad, s);
  LnParams bp;
  memset(&bp, 0, sizeof(bp));
  bp.x = x_rows; bp.T = (long long)rows * n; bp.d = d; bp.eps = 1e-5f;
  bp.wb = w_edge; bp.bias_out = static_cast<__nv_bfloat16*>(bias_out); bp.heads = heads;
  bp.bias_hs = (long long)rows * npad; bp.n_inner = n; bp.pitch = npad;
  return launch_layernorm(bp, s);
}

// ------------------------------------------------------------------------------------------------
// stage-level triangle multiply (used by the sharded path; pieces = number of gathered operand shards)
// ------------------------------------------------------------------------------------------------
long long af2_triangle_project_workspace(long long tokens, int d) {
  return align_up(tokens * d * 2, 256) + align_up(tokens * 4, 256) + 1024;
}

int af2_triangle_project(const af2_trimul_weights* w, const float* x, const unsigned char* mask, long long tokens,
                         int inner, int d, void* Lc, void* Rc, long long chan_stride, void* gate, void* workspace,
                         long long workspace_bytes, af2_stream_t stream) {
  NvtxRange nvtx_("af2_triangle_project");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (!w || !x || !Lc || !Rc || !gate) return fail(AF2_ERR_BAD_ARG, "triangle_project: null argument");
  if (d % 32) return fail(AF2_ERR_BAD_ARG, "triangle_project: dim %d must be a multiple of 32", d);
  if (tokens % inner) return fail(AF2_ERR_BAD_ARG, "triangle_project: tokens must be a multiple of inner");
  const int pitch = (int)align_up(inner, 8);
  Arena ar(workspace, workspace_bytes);
  __nv_bfloat16* xn = ar.take<__nv_bfloat16>(tokens * d);
  float* maskf = ar.take<float>(tokens);
  if (!ar.ok) return fail(AF2_ERR_WORKSPACE, "triangle_project: workspace too small");
  if (g_proj_ctas > 0 && w->w_cat && w->bn == 256 && proj_dim_ok(d) && pitch == inner) {
    ProjCall pc;
    memset(&pc, 0, sizeof(pc));
    pc.x = x; pc.T = tokens; pc.d = d;
    pc.w_cat = w->w_cat; pc.w_ext = w->w_ext; pc.rowmask = mask; pc.nseg = 3;
    const int tl = (d + 127) / 128;
    pc.seg[0] = ProjOut{tl, EK_GATED_CH_SIG, d, Lc, chan_stride};
    pc.seg[1] = ProjOut{tl, EK_GATED_CH_SIG, d, Rc, chan_stride};
    pc.seg[2] = ProjOut{(d + 255) / 256, EK_STORE_TOK_SIG, d, gate, (long long)d};
    return launch_proj(pc, s);
  }
  LnParams lp;
  memset(&lp, 0, sizeof(lp));
  lp.x = x; lp.gamma = w->ln_gamma; lp.beta = w->ln_beta; lp.y = xn; lp.T = tokens; lp.d = d; lp.eps = 1e-5f;
  AF2_TRY(launch_layernorm(lp, s));
  if (mask) {
    { ProfScope ps(s, KC_MISC, 0.0, 0.0); mask_to_float_kernel<<<ew_grid(tokens), 256, 0, s>>>(mask, maskf, tokens); }
    CUDA_OK(cudaGetLastError());
  }
  if (pitch != inner) {
    CUDA_OK(cudaMemsetAsync(Lc, 0, (size_t)d * chan_stride * 2, s));
    CUDA_OK(cudaMemsetAsync(Rc, 0, (size_t)d * chan_stride * 2, s));
  }
  const int half = w->bn / 2;
  const int npk = (d + half - 1) / half * w->bn;
  for (int side = 0; side < 2; ++side) {
    GemmCall c = linear_call(xn, d, side ? w->w_right : w->w_left, d, (int)tokens, npk, d);
    c.bn = w->bn; c.mode = EPI_GATED_BF16; c.act = ACT_SIGMOID; c.layout = LAYOUT_CHANNEL;
    c.out = side ? Rc : Lc; c.ld_out = chan_stride; c.bias = side ? w->b_right : w->b_left;
    c.use_rowscale = mask != nullptr; c.rowscale = maskf; c.cm_inner = inner; c.cm_pitch = pitch; c.out_cols = d;
    AF2_TRY(launch_gemm(c, s));
  }
  GemmCall cg = linear_call(xn, d, w->w_ogate, d, (int)tokens, d, d);
  cg.mode = EPI_STORE_BF16; cg.act = ACT_SIGMOID; cg.layout = LAYOUT_TOKEN; cg.out = gate; cg.ld_out = d; cg.bias = w->b_ogate;
  AF2_TRY(launch_gemm(cg, s));
  return AF2_OK;
}

long long af2_triangle_contract_workspace(int rows, int cols, int d) {
  return align_up((long long)d * rows * align_up(cols, 4) * 4, 256) + align_up((long long)rows * cols * d * 2, 256) + 1024;
}

// x [rows, cols, d] (local shard, updated in place) += to_out(LN_c(O) * gate) with
//   outgoing: O[i][j] = sum_k L[i][k] R[j][k]; L = Lc [c][rows][pitch(K)], piece p of Rg = [c][cols/pieces][pitch(K)]
//   ingoing : O[i][j] = sum_k R[k][i] L[k][j]; L = Lc [c][K][pitch(cols)],  piece p of Rg = [c][K][pitch(rows/pieces)]
int af2_triangle_contract(const af2_trimul_weights* w, float* x, const void* Lc, long long cs_l, const void* Rg,
                          long long cs_r, long long piece_stride, int pieces, const void* gate, int rows, int cols,
                          int K, int d, int ingoing, void* workspace, long long workspace_bytes, af2_stream_t stream) {
  NvtxRange nvtx_("af2_triangle_contract");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (!w || !x || !Lc || !Rg || !gate || pieces < 1) return fail(AF2_ERR_BAD_ARG, "triangle_contract: bad argument");
  if ((!ingoing && cols % pieces) || (ingoing && rows % pieces)) return fail(AF2_ERR_BAD_ARG, "triangle_contract: pieces must divide the gathered axis");
  const long long T = (long long)rows * cols;
  const int cp4 = (int)align_up(cols, 4);
  const long long cs_o = (long long)rows * cp4;
  Arena ar(workspace, workspace_bytes);
  float* Oc = ar.take<float>(d * cs_o);
  __nv_bfloat16* tn = ar.take<__nv_bfloat16>(T * d);
  if (!ar.ok) return fail(AF2_ERR_WORKSPACE, "triangle_contract: workspace too small");
  const __nv_bfloat16* L = static_cast<const __nv_bfloat16*>(Lc);
  const __nv_bfloat16* R = static_cast<const __nv_bfloat16*>(Rg);
  // one launch over all gathered pieces when their size tiles the kernel's boxes (rank-4 tensor maps), else one per piece
  bool fused_pieces = false;
  if (pieces > 1 && g_gather_fused) {
    GemmCall c;
    memset(&c, 0, sizeof(c));
    c.batch = d; c.K = K; c.mode = EPI_STORE_F32; c.layout = LAYOUT_TOKEN; c.ld_out = cp4; c.out_batch = cs_o; c.out = Oc;
    if (!ingoing) {
      const int pc = cols / pieces, bn = pick_bn(cols);
      if (pc % 8 == 0 && (pc % bn == 0 || bn % pc == 0)) {
        c.A = L; c.lda = align_up(K, 8); c.a_batch = cs_l;
        c.Bm = R; c.ldb = align_up(K, 8); c.b_batch = cs_r; c.b_pr = pc; c.b_piece = piece_stride;
        c.mn_major = false; c.M = rows; c.N = cols; c.bn = bn;
        fused_pieces = true;
      }
    } else {
      const int pr = rows / pieces;
      if (pr % 64 == 0) {
        c.A = R; c.lda = align_up(pr, 8); c.a_batch = cs_r; c.a_pr = pr; c.a_piece = piece_stride;
        c.Bm = L; c.ldb = align_up(cols, 8); c.b_batch = cs_l;
        c.mn_major = true; c.M = rows; c.N = cols; c.bn = pick_bn(cols);
        fused_pieces = true;
      }
    }
    if (fused_pieces) AF2_TRY(launch_gemm(c, s));
  }
  for (int p = 0; p < pieces && !fused_pieces; ++p) {
    GemmCall c;
    memset(&c, 0, sizeof(c));
    c.batch = d; c.K = K; c.mode = EPI_STORE_F32; c.layout = LAYOUT_TOKEN; c.ld_out = cp4; c.out_batch = cs_o;
    if (!ingoing) {
      const int pc = cols / pieces;
      c.A = L; c.lda = align_up(K, 8); c.a_batch = cs_l;
      c.Bm = R + p * piece_stride; c.ldb = align_up(K, 8); c.b_batch = cs_r;
      c.mn_major = false; c.M = rows; c.N = pc; c.bn = pick_bn(pc);
      c.out = Oc + (long long)p * pc;
    } else {
      const int pr = rows / pieces;
      c.A = R + p * piece_stride; c.lda = align_up(pr, 8); c.a_batch = cs_r;
      c.Bm = L; c.ldb = align_up(cols, 8); c.b_batch = cs_l;
      c.mn_major = true; c.M = pr; c.N = cols; c.bn = pick_bn(cols);
      c.out = Oc + (long long)p * pr * cp4;
    }
    AF2_TRY(launch_gemm(c, s));
  }
  ChanLnParams cp;
  memset(&cp, 0, sizeof(cp));
  cp.src = Oc; cp.chan_stride = cs_o; cp.pitch = cp4; cp.rows = rows; cp.n = cols; cp.d = d; cp.mode = 0;
  cp.gamma = w->on_gamma; cp.beta = w->on_beta; cp.gate = static_cast<const __nv_bfloat16*>(gate); cp.eps = 1e-5f; cp.y = tn;
  AF2_TRY(launch_chan_to_token(cp, s));
  GemmCall co = linear_call(tn, d, w->w_out, d, (int)T, d, d);
  co.mode = EPI_RESID_F32; co.out = x; co.ld_out = d; co.bias = w->b_out; co.resid = x; co.ld_resid = d;
  AF2_TRY(launch_gemm(co, s));
  return AF2_OK;
}

// ------------------------------------------------------------------------------------------------
// stage-level outer mean
// ------------------------------------------------------------------------------------------------
long long af2_outer_project_workspace(long long tokens, int d) {
  return align_up(tokens * d * 2, 256) + align_up(tokens * 4, 256) + 1024;
}

// m [S, inner, d] local columns -> LRc bf16 [2d][S*pitch(inner)]: channels [0,d) = left, [d,2d) = right
int af2_outer_project(const af2_outer_weights* w, const float* m, const unsigned char* msa_mask, long long tokens,
                      int inner, int d, void* LRc, long long chan_stride, void* workspace, long long workspace_bytes,
                      af2_stream_t stream) {
  NvtxRange nvtx_("af2_outer_project");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (!w || !m || !LRc) return fail(AF2_ERR_BAD_ARG, "outer_project: null argument");
  if (d % 32) return fail(AF2_ERR_BAD_ARG, "outer_project: dim %d must be a multiple of 32", d);
  const int pitch = (int)align_up(inner, 8);
  Arena ar(workspace, workspace_bytes);
  __nv_bfloat16* mn = ar.take<__nv_bfloat16>(tokens * d);
  float* maskf = ar.take<float>(tokens);
  if (!ar.ok) return fail(AF2_ERR_WORKSPACE, "outer_project: workspace too small");
  if (g_proj_ctas > 0 && w->w_cat && proj_dim_ok(d) && pitch == inner) {
    ProjCall pc;
    memset(&pc, 0, sizeof(pc));
    pc.x = m; pc.T = tokens; pc.d = d;
    pc.w_cat = w->w_cat; pc.w_ext = w->w_ext; pc.rowmask = msa_mask; pc.nseg = 1;
    pc.seg[0] = ProjOut{(2 * d + 255) / 256, EK_STORE_CH, 2 * d, LRc, chan_stride};
    return launch_proj(pc, s);
  }
  LnParams lp;
  memset(&lp, 0, sizeof(lp));
  lp.x = m; lp.gamma = w->ln_gamma; lp.beta = w->ln_beta; lp.y = mn; lp.T = tokens; lp.d = d; lp.eps = 1e-5f;
  AF2_TRY(launch_layernorm(lp, s));
  if (msa_mask) {
    { ProfScope ps(s, KC_MISC, 0.0, 0.0); mask_to_float_kernel<<<ew_grid(tokens), 256, 0, s>>>(msa_mask, maskf, tokens); }
    CUDA_OK(cudaGetLastError());
  }
  if (pitch != inner) CUDA_OK(cudaMemsetAsync(LRc, 0, (size_t)2 * d * chan_stride * 2, s));
  GemmCall c = linear_call(mn, d, w->w_lr, d, (int)tokens, 2 * d, d);
  c.mode = EPI_STORE_BF16; c.layout = LAYOUT_CHANNEL; c.out = LRc; c.ld_out = chan_stride; c.bias = w->b_lr;
  c.use_rowscale = msa_mask != nullptr; c.rowscale = maskf; c.cm_inner = inner; c.cm_pitch = pitch;
  AF2_TRY(launch_gemm(c, s));
  return AF2_OK;
}

long long af2_outer_contract_workspace(int rows, int N, int d) {
  return align_up((long long)d * rows * align_up(N, 4) * 4, 256) + align_up((long long)rows * N * d * 2, 256) +
         align_up((long long)rows * N * 4, 256) + align_up((long long)N * 4096 / 8, 256) + 1024;    // + packed mask bits (S <= 4096)
}

// x [rows, N, d] (pair rows row0..row0+rows, updated in place) += proj_out( sum_s L[s][i] R[s][j] * scale[i][j] )
//   L = Lc [c][S][pitch(rows)] (local columns), piece p of Rg = [c][S][pitch(N/pieces)]
int af2_outer_contract(const af2_outer_weights* w, float* x, const void* Lc, long long cs_l, const void* Rg,
                       long long cs_r, long long piece_stride, int pieces, const unsigned char* msa_mask_full,
                       int row0, int rows, int N, int S, int d, float eps, void* workspace, long long workspace_bytes,
                       af2_stream_t stream) {
  NvtxRange nvtx_("af2_outer_contract");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (!w || !x || !Lc || !Rg || pieces < 1 || N % pieces) return fail(AF2_ERR_BAD_ARG, "outer_contract: bad argument");
  const long long T = (long long)rows * N;
  const int np4 = (int)align_up(N, 4);
  const long long cs_o = (long long)rows * np4;
  Arena ar(workspace, workspace_bytes);
  float* Oc = ar.take<float>(d * cs_o);
  __nv_bfloat16* tn = ar.take<__nv_bfloat16>(T * d);
  float* scale = ar.take<float>(T);
  uint32_t* mwords = (S <= 4096) ? ar.take<uint32_t>((long long)((S + 31) / 32) * N) : nullptr;
  if (!ar.ok) return fail(AF2_ERR_WORKSPACE, "outer_contract: workspace too small");
  if (msa_mask_full) AF2_TRY(launch_outer_scale(msa_mask_full, scale, mwords, row0, rows, S, N, eps, s));
  const __nv_bfloat16* L = static_cast<const __nv_bfloat16*>(Lc);
  const __nv_bfloat16* R = static_cast<const __nv_bfloat16*>(Rg);
  const int pc = N / pieces;
  const bool fused_pieces = pieces > 1 && g_gather_fused && pc % 64 == 0;
  if (fused_pieces) {   // one launch: B columns j = p * pc + jj addressed through a rank-4 map over the gathered pieces
    GemmCall g;
    memset(&g, 0, sizeof(g));
    g.A = L; g.lda = align_up(rows, 8); g.a_batch = cs_l;
    g.Bm = R; g.ldb = align_up(pc, 8); g.b_batch = cs_r; g.b_pr = pc; g.b_piece = piece_stride;
    g.mn_major = true; g.M = rows; g.N = N; g.K = S; g.batch = d; g.bn = pick_bn(N);
    g.mode = EPI_STORE_F32; g.layout = LAYOUT_TOKEN; g.out = Oc; g.ld_out = np4; g.out_batch = cs_o;
    AF2_TRY(launch_gemm(g, s));
  }
  for (int p = 0; p < pieces && !fused_pieces; ++p) {
    GemmCall g;
    memset(&g, 0, sizeof(g));
    g.A = L; g.lda = align_up(rows, 8); g.a_batch = cs_l;
    g.Bm = R + p * piece_stride; g.ldb = align_up(pc, 8); g.b_batch = cs_r;
    g.mn_major = true; g.M = rows; g.N = pc; g.K = S; g.batch = d; g.bn = pick_bn(pc);
    g.mode = EPI_STORE_F32; g.layout = LAYOUT_TOKEN; g.out = Oc + (long long)p * pc; g.ld_out = np4; g.out_batch = cs_o;
    AF2_TRY(launch_gemm(g, s));
  }
  ChanLnParams cp;
  memset(&cp, 0, sizeof(cp));
  cp.src = Oc; cp.chan_stride = cs_o; cp.pitch = np4; cp.rows = rows; cp.n = N; cp.d = d; cp.mode = 1;
  cp.scale = msa_mask_full ? scale : nullptr; cp.scale_const = 1.0f / (float)S; cp.y = tn;
  AF2_TRY(launch_chan_to_token(cp, s));
  GemmCall co = linear_call(tn, d, w->w_out, d, (int)T, d, d);
  co.mode = EPI_RESID_F32; co.out = x; co.ld_out = d; co.bias = w->b_out; co.resid = x; co.ld_resid = d;
  AF2_TRY(launch_gemm(co, s));
  return AF2_OK;
}

// ------------------------------------------------------------------------------------------------
int af2_rotary(const float* x, const float* sin_, const float* cos_, float* y, int b, int h, int n, int dh, int rot,
               int sincos_batch, af2_stream_t stream) {
  NvtxRange nvtx_("af2_rotary");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (dh % 2 || rot % 2 || rot > dh) return fail(AF2_ERR_BAD_ARG, "rotary: dh=%d rot=%d must be even, rot <= dh", dh, rot);
  const long long pairs = (long long)b * h * n * (dh / 2);
  if (pairs == 0) return AF2_OK;
  { ProfScope ps(s, KC_MISC, 0.0, 0.0); rotary_kernel<<<ew_grid(pairs), 256, 0, s>>>(x, sin_, cos_, y, b, h, n, dh, rot, sincos_batch); }
  CUDA_OK(cudaGetLastError());
  return AF2_OK;
}

int af2_layernorm_bf16(const float* x, const float* gamma, const float* beta, void* y_bf16, long long T, int d,
                       float eps, af2_stream_t stream) {
  LnParams lp;
  memset(&lp, 0, sizeof(lp));
  lp.x = x; lp.gamma = gamma; lp.beta = beta; lp.y = static_cast<__nv_bfloat16*>(y_bf16); lp.T = T; lp.d = d; lp.eps = eps;
  return launch_layernorm(lp, static_cast<cudaStream_t>(stream));
}

int af2_gemm_bf16_f32(const void* A, long long lda, long long a_batch, const void* Bm, long long ldb, long long b_batch,
                      float* C, long long ldc, long long c_batch, int M, int N, int K, int batch, int mn_major,
                      af2_stream_t stream) {
  GemmCall c;
  memset(&c, 0, sizeof(c));
  c.A = A; c.lda = lda; c.a_batch = a_batch; c.Bm = Bm; c.ldb = ldb; c.b_batch = b_batch;
  c.M = M; c.N = N; c.K = K; c.batch = batch; c.mn_major = mn_major != 0; c.bn = pick_bn(N);
  c.mode = EPI_STORE_F32; c.layout = LAYOUT_TOKEN; c.out = C; c.ld_out = ldc; c.out_batch = c_batch;
  return launch_gemm(c, static_cast<cudaStream_t>(stream));
}

}  // extern "C"

#include "strict_api.inl"
#include "peer_api.inl"
