// Runtime plumbing of the C ABI: status/last-error, architecture gate, TMA descriptor encoding, and the
// runtime-dispatched GEMM entry (llb_gemm_bf16).
#include <stdarg.h>
#include <stdlib.h>

#include <mutex>
#include <unordered_map>
#include <vector>

#include "llb_gemm.cuh"

namespace llb {

static thread_local std::string g_last_error;

void set_error(const std::string& msg) { g_last_error = msg; }

int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

static int64_t g_kernel_launches[LLB_KERN_FAMILIES];
void note_kernel(int family, int64_t n) {
  if (family >= 0 && family < LLB_KERN_FAMILIES) __atomic_add_fetch(&g_kernel_launches[family], n, __ATOMIC_RELAXED);
}

// ---- live profiling -------------------------------------------------------------------------------
namespace {
struct ProfRec {
  int slot;
  cudaEvent_t a, b;
};
bool g_prof_on = false;
std::vector<ProfRec> g_prof_recs;
std::vector<cudaEvent_t> g_prof_pool;
double g_prof_ms[LLB_PROF_SLOTS];
int64_t g_prof_n[LLB_PROF_SLOTS];
cudaEvent_t prof_event() {
  if (!g_prof_pool.empty()) {
    cudaEvent_t e = g_prof_pool.back();
    g_prof_pool.pop_back();
    return e;
  }
  cudaEvent_t e;
  cudaEventCreate(&e);
  return e;
}
void prof_drain() {
  for (auto& r : g_prof_recs) {
    float ms = 0.f;
    if (cudaEventSynchronize(r.b) == cudaSuccess && cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
      g_prof_ms[r.slot] += ms;
      g_prof_n[r.slot] += 1;
    }
    g_prof_pool.push_back(r.a);
    g_prof_pool.push_back(r.b);
  }
  g_prof_recs.clear();
}
}  // namespace

bool profile_on() { return g_prof_on; }
void profile_begin(int slot, cudaStream_t s) {
  ProfRec r{slot, prof_event(), prof_event()};
  cudaEventRecord(r.a, s);
  g_prof_recs.push_back(r);
}
void profile_end(cudaStream_t s) { cudaEventRecord(g_prof_recs.back().b, s); }

int launch_failed(const void* kern, cudaError_t e) {
  (void)cudaGetLastError();   // the launch's error is reported here, not by a later status check
  const char* name = nullptr;
  if (cudaFuncGetName(&name, kern) != cudaSuccess || !name) {
    (void)cudaGetLastError();
    name = "?";
  }
  return fail(LLB_ERR_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(e));
}

int reserve_dynamic_smem(const void* kern, size_t smem) {
  static std::mutex mu;
  static std::unordered_map<const void*, size_t> reserved;
  std::lock_guard<std::mutex> lock(mu);
  size_t& have = reserved[kern];
  if (smem <= have) return LLB_OK;
  const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return launch_failed(kern, e);
  have = smem;
  return LLB_OK;
}

bool pdl_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("LLB_PDL");
    on = (e && e[0] == '0') ? 0 : 1;
  }
  return on == 1;
}

int num_sms() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 1;
  }
  return sms;
}

int require_sm100() {
  static int status = 1;  // 1 = unknown
  if (status == 1) {
    int dev = 0, major = 0, minor = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
    if (e != cudaSuccess) return fail(LLB_ERR_CUDA, "no usable CUDA device: %s", cudaGetErrorString(e));
    if (major != 10)
      return fail(LLB_ERR_ARCH, "llamole_b200 is sm_100a-only (tcgen05/TMEM/TMA); device %d is sm_%d%d and there is no fallback path",
                  dev, major, minor);
    status = LLB_OK;
  }
  return status;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// Descriptor cache: a sampling step re-issues the same ~130 GEMMs on the same buffers every step, and
// cuTensorMapEncodeTiled costs 1-2 us a call (three to five calls per GEMM) -- at small batch that was most of the step.
// Direct-mapped, per host thread, keyed on everything that defines the map.
namespace {
struct TmapKey {
  const void* ptr;
  int elem_bytes, rows, cols, ld, box_cols, box_rows, swizzle;
  bool operator==(const TmapKey& o) const {
    return ptr == o.ptr && elem_bytes == o.elem_bytes && rows == o.rows && cols == o.cols && ld == o.ld && box_cols == o.box_cols &&
           box_rows == o.box_rows && swizzle == o.swizzle;
  }
};
struct TmapSlot {
  TmapKey key{};
  bool valid = false;
  CUtensorMap map;
};
constexpr int TMAP_CACHE_SLOTS = 2048;
}  // namespace

int make_tensor_map_2d(CUtensorMap* out, const void* ptr, int elem_bytes, int rows, int cols, int ld_elems, int box_cols,
                       int box_rows, int swizzle_bytes) {
  static thread_local std::vector<TmapSlot> cache(TMAP_CACHE_SLOTS);
  const TmapKey key{ptr, elem_bytes, rows, cols, ld_elems, box_cols, box_rows, swizzle_bytes};
  uint64_t hsh = reinterpret_cast<uintptr_t>(ptr) * 0x9E3779B97F4A7C15ull;
  hsh ^= ((uint64_t)(uint32_t)rows << 32 | (uint32_t)cols) * 0xC2B2AE3D27D4EB4Full;
  hsh ^= ((uint64_t)(uint32_t)ld_elems << 24 | (uint32_t)box_cols << 12 | (uint32_t)box_rows << 4 | (uint32_t)(elem_bytes ^ swizzle_bytes)) * 0x165667B19E3779F9ull;
  TmapSlot& slot = cache[(hsh >> 40) % TMAP_CACHE_SLOTS];
  if (slot.valid && slot.key == key) {
    *out = slot.map;
    return LLB_OK;
  }
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(LLB_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld_elems * elem_bytes};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType dt = elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                : (swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE);
  CUresult r = fn(out, dt, 2, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(LLB_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for rows=%d cols=%d ld=%d elem=%d box=%dx%d ptr=%p", (int)r, rows,
                cols, ld_elems, elem_bytes, box_cols, box_rows, ptr);
  slot.key = key, slot.map = *out, slot.valid = true;
  return LLB_OK;
}

// Pick the N tile of the single-CTA kernel by a small time model (clocks per CTA, measured in the latency regime,
// profiles/r2_latency_timeline.txt): a tile's k-loop issues K/16 MMAs, each taking max(95, BN/2) clocks -- one tcgen05.mma of
// M = 128 is accepted every ~95 clocks however narrow it is, so halving the tile does NOT halve its time --, its epilogue and
// hand-over cost ~600 + 6 BN, and the tiles run in ceil(tiles / SMs) rounds.
static int pick_bn(int M, int N, int K, int group_n = 0) {
  const int sms = num_sms();
  const int mt = ceil_div(M, GEMM_BM);
  int best = 256;
  double best_cost = 1e30;
  const int cand[3] = {256, 128, 64};
  for (int i = 0; i < 3; ++i) {
    if (group_n > 0 && group_n % cand[i] != 0) continue;   // a tile must not straddle two groups
    const int tiles = mt * ceil_div(N, cand[i]);
    const double per_mma = cand[i] / 2 > 95 ? cand[i] / 2 : 95;
    const double cost = (double)ceil_div(tiles, sms) * (ceil_div(K, 16) * per_mma + 600.0 + 6.0 * cand[i]);
    if (cost < best_cost) {
      best_cost = cost;
      best = cand[i];
    }
  }
  return best;
}

template <int ACT, bool F32>
static int gemm_dispatch_bn(const void* A, int lda, const void* W, int ldw, const float* bias, void* C, int ldc, int M,
                            int N, int K, cudaStream_t stream, LaunchCounter* ctr, GemmGroups grp) {
  LLB_CHECK_ARG(bias == nullptr || (reinterpret_cast<uintptr_t>(bias) & 15) == 0, "gemm: bias must be 16-byte aligned");
  EpiBiasAct<ACT, F32> epi{C, ldc, bias};
  switch (pick_bn(M, N, K, grp.group_n)) {
    case 256: return launch_gemm<256>(A, lda, W, ldw, M, N, K, epi, stream, ctr, grp);
    case 128: return launch_gemm<128>(A, lda, W, ldw, M, N, K, epi, stream, ctr, grp);
    default: return launch_gemm<64>(A, lda, W, ldw, M, N, K, epi, stream, ctr, grp);
  }
}

template <bool F32>
static int gemm_dispatch_act(const void* A, int lda, const void* W, int ldw, const float* bias, void* C, int ldc, int M,
                             int N, int K, int act, cudaStream_t stream, LaunchCounter* ctr, GemmGroups grp) {
  switch (act) {
    case LLB_ACT_NONE: return gemm_dispatch_bn<LLB_ACT_NONE, F32>(A, lda, W, ldw, bias, C, ldc, M, N, K, stream, ctr, grp);
    case LLB_ACT_GELU: return gemm_dispatch_bn<LLB_ACT_GELU, F32>(A, lda, W, ldw, bias, C, ldc, M, N, K, stream, ctr, grp);
    case LLB_ACT_SILU: return gemm_dispatch_bn<LLB_ACT_SILU, F32>(A, lda, W, ldw, bias, C, ldc, M, N, K, stream, ctr, grp);
    case LLB_ACT_SOFTSIGN:
      return gemm_dispatch_bn<LLB_ACT_SOFTSIGN, F32>(A, lda, W, ldw, bias, C, ldc, M, N, K, stream, ctr, grp);
  }
  return fail(LLB_ERR_INVALID, "gemm: unknown activation %d", act);
}

int gemm_bias_act(const void* A, int lda, const void* W, int ldw, const float* bias, void* C, int ldc, int M, int N,
                  int K, int act, bool out_f32, cudaStream_t stream, LaunchCounter* ctr, GemmGroups grp) {
  return out_f32 ? gemm_dispatch_act<true>(A, lda, W, ldw, bias, C, ldc, M, N, K, act, stream, ctr, grp)
                 : gemm_dispatch_act<false>(A, lda, W, ldw, bias, C, ldc, M, N, K, act, stream, ctr, grp);
}

}  // namespace llb

extern "C" {

const char* llb_last_error(void) { return llb::g_last_error.c_str(); }

int llb_version(void) { return 100; }

int llb_profile_enable(int on) {
  llb::prof_drain();
  llb::g_prof_on = on != 0;
  for (int i = 0; i < LLB_PROF_SLOTS; ++i) llb::g_prof_ms[i] = 0.0, llb::g_prof_n[i] = 0;
  return LLB_OK;
}

int llb_profile_read(int slot, double* total_ms, int64_t* launches) {
  LLB_CHECK_ARG(slot >= 0 && slot < LLB_PROF_SLOTS && total_ms && launches, "llb_profile_read: bad argument");
  llb::prof_drain();
  *total_ms = llb::g_prof_ms[slot];
  *launches = llb::g_prof_n[slot];
  llb::g_prof_ms[slot] = 0.0;
  llb::g_prof_n[slot] = 0;
  return LLB_OK;
}

const char* llb_profile_slot_name(int slot) {
  static const char* names[LLB_PROF_SLOTS] = {
      "gemm_qkv", "gemm_proj", "gemm_fc1", "gemm_fc2", "gemm_adaln", "gemm_other", "attention", "ln_mod_res", "dit_step",
      "dit_misc", "gin_aggregate", "gin_pool", "gin_gemm_mlp0", "gin_gemm_mlp4", "gin_rowln", "gin_misc", "gin_gemm_head",
      "gin_topk", "gin_gemm_stats"};
  return (slot >= 0 && slot < LLB_PROF_SLOTS) ? names[slot] : "?";
}

int64_t llb_kernel_launches(int family) {
  return (family >= 0 && family < LLB_KERN_FAMILIES) ? __atomic_load_n(&llb::g_kernel_launches[family], __ATOMIC_RELAXED) : -1;
}

int llb_arch_check(int device) {
  int major = 0, minor = 0;
  cudaError_t e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device);
  if (e != cudaSuccess) return llb::fail(LLB_ERR_CUDA, "device %d: %s", device, cudaGetErrorString(e));
  if (major != 10)
    return llb::fail(LLB_ERR_ARCH, "device %d is sm_%d%d; llamole_b200 runs on sm_100 (B200) only and has no fallback", device,
                     major, minor);
  return LLB_OK;
}

int llb_gemm_bf16(const void* A, int lda, const void* W, int ldw, const float* bias, void* C, int ldc, int M, int N,
                  int K, int act, int out_fp32, llb_stream_t stream) {
  LLB_TRY(llb::require_sm100());
  LLB_CHECK_ARG(A && W && C, "llb_gemm_bf16: null operand");
  return llb::gemm_bias_act(A, lda, W, ldw, bias, C, ldc, M, N, K, act, out_fp32 != 0, (cudaStream_t)stream, nullptr);
}

}  // extern "C"

LLB_STEP_TRACE_INSTALL(llb_trace_install_runtime)
