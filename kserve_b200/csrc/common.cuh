// Common device helpers for the sm_100a kernels: error handling, bf16 helpers and thin
// wrappers over the Blackwell PTX used by the hot path (mbarrier, TMA, tcgen05/TMEM).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <string>

namespace b200 {

typedef __nv_bfloat16 bf16;

// ---------------------------------------------------------------------------------------------
// host-side error plumbing: every C-ABI entry returns an int status; the text is kept per thread.
// ---------------------------------------------------------------------------------------------
void set_last_error(const std::string& msg);

#define B200_CUDA_OK(expr)                                                                       \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) {                                                                     \
      ::b200::set_last_error(std::string(#expr) + " failed: " + cudaGetErrorString(_e) + " at " + \
                             __FILE__ + ":" + std::to_string(__LINE__));                         \
      return -1;                                                                                 \
    }                                                                                            \
  } while (0)

#define B200_REQUIRE(cond, msg)                                                          \
  do {                                                                                   \
    if (!(cond)) {                                                                       \
      ::b200::set_last_error(std::string("requirement failed: ") + #cond + ": " + (msg)); \
      return -2;                                                                         \
    }                                                                                    \
  } while (0)

// ---------------------------------------------------------------------------------------------
// small device utilities
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

__device__ __forceinline__ float2 unpack_bf16x2(uint32_t u) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(v);
}

// 128-bit streaming load that does not allocate in L1 (weights / KV pages are read once per step).
__device__ __forceinline__ uint4 ld_nc_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

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

// ---------------------------------------------------------------------------------------------
// Optional per-CTA timeline (debug): when enabled through b200_debug_trace(), thread 0 of every CTA appends
// {kind, block, globaltimer at entry, at exit}; off by default (one predictable branch per CTA).
// ---------------------------------------------------------------------------------------------
struct TraceRec { unsigned long long t0, t1, tmid; int kind, block; };
__device__ TraceRec* g_trace_buf = nullptr;
__device__ unsigned int g_trace_cap = 0;
__device__ unsigned int g_trace_cnt = 0;
enum TraceKind : int { TK_GEMM = 1, TK_RMSNORM = 2, TK_ROPE = 3, TK_ATTN_DECODE = 4, TK_ARGMAX = 6,
                       TK_STEP = 7, TK_EMBED = 8, TK_ATTN_PREFILL = 9, TK_OTHER = 10 };
__device__ __forceinline__ unsigned long long global_timer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
struct TraceScope {
  unsigned long long t0 = 0, tmid = 0;
  int kind;
  __device__ __forceinline__ void mark() { if (threadIdx.x == 0 && t0 != 0) tmid = global_timer(); }
  __device__ __forceinline__ explicit TraceScope(int k) : kind(k) {
    if (threadIdx.x == 0 && g_trace_buf != nullptr) t0 = global_timer();
  }
  __device__ __forceinline__ ~TraceScope() {
    if (threadIdx.x == 0 && t0 != 0) {
      const unsigned int i = atomicAdd(&g_trace_cnt, 1u);
      if (i < g_trace_cap) {
        TraceRec r; r.t0 = t0; r.t1 = global_timer(); r.tmid = tmid; r.kind = kind; r.block = blockIdx.x;
        g_trace_buf[i] = r;
      }
    }
  }
};

// ---------------------------------------------------------------------------------------------
// Recoverable faults of the cross-GPU / cross-CTA waits.  A tensor-parallel peer that died, or was never launched, must
// not take this rank's CUDA context with it: a wait that times out records a code here and the kernel carries on with
// whatever data it has (every later wait then gives up at once), instead of __trap()ing — which would poison the context
// of every rank for good.  The host reads the code at its next synchronisation point (b200_engine_fault), fails the call,
// marks the engine unusable, and the model server reports the model as not ready.  Codes: 1 peer flag, 2 all-reduce
// packet, 3 candidate exchange, 4 stream-K piece.
// ---------------------------------------------------------------------------------------------
__device__ int g_fault_code = 0;
__device__ __forceinline__ bool fault_raised() { return *reinterpret_cast<volatile int*>(&g_fault_code) != 0; }
__device__ __forceinline__ void fault_raise(int code) { atomicCAS(&g_fault_code, 0, code); }
// One step of a bounded spin: false = keep waiting, true = give up (time-out reached, or another wait already failed).
// The bound is wall time (%globaltimer, looked at every 1024 polls): g_wait_timeout_ns, default 5 s — far beyond any
// legitimate wait of a decode step, short enough that a lost peer fails the request instead of hanging the server.
__device__ unsigned long long g_wait_timeout_ns = 5000000000ull;
struct SpinGuard { uint32_t polls = 0; unsigned long long t0 = 0; };
__device__ __forceinline__ bool spin_give_up(SpinGuard& g, int code) {
  if ((++g.polls & 0x3ff) != 0) return false;
  if (fault_raised()) return true;
  const unsigned long long now = global_timer();
  if (g.t0 == 0) { g.t0 = now; return false; }
  if (now - g.t0 > *reinterpret_cast<volatile unsigned long long*>(&g_wait_timeout_ns)) { fault_raise(code); return true; }
  return false;
}

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch: a kernel lets its successor start (prologue, weight prefetch) while it is
// still running, and blocks only where it first touches data the predecessor produced.  Both are no-ops when
// the kernel was launched without the programmatic-stream-serialization attribute.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------
// mbarrier
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a pipeline bug traps (-> a CUDA error the host reports) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) {
      printf("b200: mbarrier wait timeout (block %d thread %d parity %u)\n", blockIdx.x, threadIdx.x, parity);
      __trap();
    }
  }
}

// ---------------------------------------------------------------------------------------------
// TMA (cp.async.bulk.tensor) — 2D tile load, completion on an mbarrier, with an L2 cache hint
// ---------------------------------------------------------------------------------------------
constexpr uint64_t kEvictNormal = 0x1000000000000000ull;
constexpr uint64_t kEvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kEvictLast = 0x14F0000000000000ull;

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c_inner,
                                            int c_outer, uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c_inner), "r"(c_outer), "l"(hint)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

// ---------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]; issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives when all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread i of the warp gets row (lane base + i).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,"
      "%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// UMMA shared-memory descriptor for a K-major bf16 tile whose rows are 128 B (64 elements) wide and
// stored with the 128-byte swizzle TMA writes (CU_TENSOR_MAP_SWIZZLE_128B): 8-row groups are 1024 B
// apart (SBO), LBO is unused for swizzled K-major layouts (encoded 1), version=1 (sm_100), layout=2.
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, M x N tile.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---------------------------------------------------------------------------------------------
// legacy warp-level MMA (m16n8k16 bf16) + ldmatrix + cp.async: used by the attention kernels
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mma_m16n8k16_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void cp_async_16(uint32_t smem_dst, const void* gsrc, bool valid) {
  int sz = valid ? 16 : 0;  // src-size 0 => zero fill
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_dst), "l"(gsrc), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

}  // namespace b200
