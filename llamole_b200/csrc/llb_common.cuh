// Shared device/host helpers for the llamole_b200 kernels (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "../../include/llamole_b200.h"

namespace llb {

// ------------------------------------------------------------------------------------------------
// Host-side status handling.  Every C-ABI entry returns an int status; the message of the last failure
// on the calling thread is kept for llb_last_error().
// ------------------------------------------------------------------------------------------------
void set_error(const std::string& msg);
int fail(int code, const char* fmt, ...);

#define LLB_CUDA_OK(expr)                                                                           \
  do {                                                                                              \
    cudaError_t _e = (expr);                                                                        \
    if (_e != cudaSuccess)                                                                          \
      return ::llb::fail(LLB_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),     \
                         __FILE__, __LINE__);                                                       \
  } while (0)

#define LLB_CHECK_ARG(cond, ...)                                                                    \
  do {                                                                                              \
    if (!(cond)) return ::llb::fail(LLB_ERR_INVALID, __VA_ARGS__);                                  \
  } while (0)

#define LLB_TRY(expr)                                                                               \
  do {                                                                                              \
    int _s = (expr);                                                                                \
    if (_s != LLB_OK) return _s;                                                                    \
  } while (0)

int num_sms();
int require_sm100();  // LLB_OK or LLB_ERR_ARCH (no fallback by design)

// Event bracket around one kernel launch (no-op unless llb_profile_enable(1)).
bool profile_on();
void profile_begin(int slot, cudaStream_t s);
void profile_end(cudaStream_t s);
struct ProfScope {
  cudaStream_t s;
  bool on;
  ProfScope(int slot, cudaStream_t stream) : s(stream), on(profile_on()) {
    if (on) profile_begin(slot, s);
  }
  ~ProfScope() {
    if (on) profile_end(s);
  }
};

void note_kernel(int family, int64_t n = 1);   // llb_kernel_launches counters (n < 0: a stream capture issued nothing)

// Programmatic dependent launch: the kernel may start while its predecessor in the stream still runs; whatever it does before
// pdl_wait() (barrier init, TMEM allocation, descriptor prefetch, loads of WEIGHTS) overlaps the predecessor's tail.  Every access
// to data a predecessor produced (or still reads) comes after pdl_wait(), which returns once all prerequisite grids have completed
// and flushed.  Kernels launched the ordinary way execute both instructions as no-ops.
bool pdl_enabled();   // LLB_PDL=0 launches everything the ordinary way (A-B comparison)
template <class T>
struct pdl_ident {
  using type = T;
};
// Set to make the NEXT launch_pdl of this thread an ordinary launch (a full dependency on everything before it in the stream):
// what some later kernel reads AHEAD of its own dependency wait must have been produced before such a launch.
inline bool& pdl_full_barrier_next() {
  static thread_local bool flag = false;
  return flag;
}
template <class... KArgs>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, typename pdl_ident<KArgs>::type... args) {
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = s;
  cfg.attrs = attr, cfg.numAttrs = (pdl_enabled() && !pdl_full_barrier_next()) ? 1 : 0;
  pdl_full_barrier_next() = false;
  return cudaLaunchKernelEx(&cfg, kern, args...);
}

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// Bump allocator over a caller-provided workspace.
struct Arena {
  uint8_t* base;
  size_t cap, off;
  Arena(void* p, size_t bytes) : base((uint8_t*)p), cap(bytes), off(0) {}
  template <class T>
  T* take(size_t n) {
    off = align_up(off, 256);
    T* p = (T*)(base ? base + off : nullptr);
    off += n * sizeof(T);
    return p;
  }
  bool ok() const { return off <= cap; }
};

// ------------------------------------------------------------------------------------------------
// Device math
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }
// d gelu_erf / dx = Phi(x) + x phi(x) (backward passes)
__device__ __forceinline__ float gelu_erf_grad(float x) {
  return 0.5f * (1.0f + erff(x * 0.70710678118654752f)) + x * 0.39894228040143268f * expf(-0.5f * x * x);
}
// Exact-erf GELU restated as gelu(x) = max(x, 0) - |x| * Phi(-|x|) with Phi(-a) = 2^P(a), P a degree-5 minimax fit
// of log2(Phi(-a)) on [0, 6] (leading coefficient negative, so P -> -inf and the correction -> 0 beyond the fit range).
// Max |error| against the fp64 erf form is 6.4e-7 over [-8, 8] (tools/fit_gelu.py), i.e. fp32 round-off of the
// surrounding arithmetic, for 6 FFMA + 1 FMNMX + 1 MUFU.EX2 per element -- erff costs ~35 instructions, the previous
// Abramowitz-Stegun form 16 + 2 MUFU, and both made the fc1 epilogue slow the tensor pipe down.
__device__ __forceinline__ float ex2_approx(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float gelu_fast(float x) {
  const float a = fabsf(x);
  float p = -0.0004733077904837858f;
  p = fmaf(p, a, 0.007084582472665392f);
  p = fmaf(p, a, -0.05182752433176751f);
  p = fmaf(p, a, -0.45999221096226367f);
  p = fmaf(p, a, -1.150787981711536f);
  p = fmaf(p, a, -1.0000376025053335f);
  return fmaf(-a, ex2_approx(p), fmaxf(x, 0.0f));
}
// The same form with a degree-3 exponent polynomial (tools/fit_gelu3.py): max |error| 5.5e-5 against the fp64 erf form, 1/35 of a
// bf16 half-ulp at 1 -- for results that are rounded to bf16 right away (GEMM epilogues with bf16 output, GIN messages), where
// two FFMAs per element are worth more than digits the rounding discards: 4 FFMA + 1 FMNMX + 1 MUFU.EX2.
__device__ __forceinline__ float gelu_bf16(float x) {
  const float a = fabsf(x);
  float p = -0.024885521646689234f;
  p = fmaf(p, a, -0.49882014726711105f);
  p = fmaf(p, a, -1.129246088530717f);
  p = fmaf(p, a, -1.0035316221396362f);
  return fmaf(-a, ex2_approx(p), fmaxf(x, 0.0f));
}
// Same function with 2^p evaluated on the FMA pipe (round-to-nearest split p = i + f, degree-4 polynomial for 2^f,
// exponent add), i.e. no MUFU instruction at all: 16 FP32/INT instructions instead of 8 + 1 MUFU.  Max |error| vs the
// fp64 erf form 1.1e-6.  Used where the MUFU / MIO queue is the scarcer resource (see the fc1 epilogue notes in DESIGN.md).
__device__ __forceinline__ float gelu_fma_only(float x) {
  const float a = fabsf(x);
  float p = -0.0004733077904837858f;
  p = fmaf(p, a, 0.007084582472665392f);
  p = fmaf(p, a, -0.05182752433176751f);
  p = fmaf(p, a, -0.45999221096226367f);
  p = fmaf(p, a, -1.150787981711536f);
  p = fmaf(p, a, -1.0000376025053335f);
  p = fmaxf(p, -125.0f);
  const float t = p + 12582912.0f;                  // 1.5 * 2^23: the integer part of p lands in the low mantissa bits
  const float f = p - (t - 12582912.0f);            // in [-0.5, 0.5]
  float e = 0.009570098074450925f;
  e = fmaf(e, f, 0.05591786664763956f);
  e = fmaf(e, f, 0.24024744980255675f);
  e = fmaf(e, f, 0.6931218139887697f);
  e = fmaf(e, f, 0.9999992613818445f);
  const float h = __int_as_float(__float_as_int(e) + (__float_as_int(t) << 23));   // e * 2^i (the magic constant's bits shift out)
  return fmaf(-a, h, fmaxf(x, 0.0f));
}
__device__ __forceinline__ float silu(float x) { return x / (1.0f + __expf(-x)); }
__device__ __forceinline__ float softsign(float x) { return x / (1.0f + fabsf(x)); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }

// ------------------------------------------------------------------------------------------------
// Philox-4x32-10 counter RNG (same function restated on the host in oracle/llamole_oracle.py).
// counter = (pos, mol, stream, group), key = (seed lo, seed hi); one call serves 4 consecutive classes.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}
// Exp(1) variate from 32 bits: u = (bits + 0.5) 2^-32 (exact in fp64, rounded once to fp32), q = -log(u).
__device__ __forceinline__ float exp1_from_bits(uint32_t bits) {
  float u = (float)(((double)bits + 0.5) * (1.0 / 4294967296.0));
  return -logf(u);
}

// ------------------------------------------------------------------------------------------------
// sm_100a PTX wrappers: mbarrier, TMA, tcgen05 / TMEM
// ------------------------------------------------------------------------------------------------
// Warp index as a value the compiler KNOWS to be warp-uniform (a shuffle result), so that the role branches are uniform
// branches and everything a role derives from kernel arguments, loop counters and shared-memory bases stays in uniform
// registers.  Without it every tcgen05.mma / tcgen05.commit / TMA issue is wrapped in an ELECT + R2UR waterfall loop
// (~20 extra instructions each), which made the single MMA-issuing thread nearly as slow as the tensor pipe itself.
__device__ __forceinline__ int uniform_warp_idx() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }
// One elected lane of a converged warp (deterministic: the same lane every time, as tcgen05.commit requires).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

#ifdef LLB_STEP_TRACE
// Debug-only timeline of the latency regime (tools/step_trace.py builds the library with -DLLB_STEP_TRACE; never in the product
// build): CTA 0 of every kernel appends {tag, info, globaltimer} records; one buffer pointer per translation unit.
static __device__ unsigned long long* g_step_trace;
__device__ __forceinline__ void step_stamp(unsigned long long tag, unsigned long long info) {
  unsigned long long* t = g_step_trace;
  if (t) {
    const unsigned long long i = atomicAdd(t, 1ull);
    if (i < 20000) {
      unsigned long long now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      t[1 + 3 * i] = tag, t[2 + 3 * i] = info, t[3 + 3 * i] = now;
    }
  }
}
#define LLB_STAMP(tag, info, cond) do { if (blockIdx.x == 0 && (cond)) step_stamp((tag), (info)); } while (0)
#define LLB_STEP_TRACE_INSTALL(name) extern "C" int name(void* p) { return cudaMemcpyToSymbol(llb::g_step_trace, &p, sizeof(p)) == cudaSuccess ? 0 : 1; }
#else
#define LLB_STAMP(tag, info, cond) do { } while (0)
#define LLB_STEP_TRACE_INSTALL(name)
#endif
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// explicit shared-space accesses by 32-bit address (a generic pointer into shared memory compiles to the slow generic LD / ST)
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a pipeline bug must surface as a launch failure, never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  long long start = clock64();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3ffu) == 0 && clock64() - start > 8000000000ll) {
      printf("llamole_b200: mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
      __trap();
    }
  }
}

// generic-proxy shared-memory writes -> visible to the async proxy (TMA stores, tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void l2_prefetch_tile(const CUtensorMap* map, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T, both operands K-major bf16, fp32 accumulate.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
// mbarrier arrives once all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread = lane of the warp's TMEM quarter).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 16 consecutive 32-bit columns <- 16 registers per thread (thread = lane of the warp's TMEM quarter).
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// D[tmem] (+)= A[tmem] * B[smem]: A is read from tensor memory (lane = row, 32-bit column = two consecutive K elements).
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// UMMA shared-memory descriptor, K-major operand, 128-byte swizzle, rows of 64 bf16 (128 B):
//   start address >> 4 | LBO (ignored for swizzled K-major, 1) | SBO = 1024 B (8 rows x 128 B) | version 1 | SWIZZLE_128B (2)
// (bit layout: cute/arch/mma_sm100_desc.hpp, union SmemDescriptor)
__device__ __forceinline__ uint64_t umma_desc_k128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor for kind::f16: D fp32, A/B bf16, both K-major, M x N tile.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// The same with both operands in IEEE fp16 (a_format = b_format = 0) when `ab_f16` is set: where an operand is an activation of
// order one (GELU(LayerNorm(.)) of the GIN node MLP) fp16 carries three more mantissa bits than bf16 at the same cost.
__host__ __device__ constexpr uint32_t umma_idesc_ab(int M, int N, bool ab_f16) {
  return umma_idesc_bf16(M, N) & ~(ab_f16 ? ((1u << 7) | (1u << 10)) : 0u);
}
// Degree-3 GELU (gelu_bf16) on a pair of fp16 values: 3 HFMA2 + ex2.approx.f16x2 + HMNMX2 + HFMA2 for TWO elements.  Error of the
// fp16 evaluation ~3e-4 absolute (about one fp16 ulp at 0.5), an eighth of a bf16 ulp; for epilogues that store fp16.
__device__ __forceinline__ __half2 gelu_h2(__half2 x) {
  const __half2 a = __habs2(x);
  __half2 p = __float2half2_rn(-0.024885521646689234f);
  p = __hfma2(p, a, __float2half2_rn(-0.49882014726711105f));
  p = __hfma2(p, a, __float2half2_rn(-1.129246088530717f));
  p = __hfma2(p, a, __float2half2_rn(-1.0035316221396362f));
  return __hfma2(__hneg2(a), h2exp2(p), __hmax2(x, __float2half2_rn(0.0f)));
}

}  // namespace llb
