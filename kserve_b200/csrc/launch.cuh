// Host-side launchers: TMA tensor-map cache, GEMM dispatch, op launch helpers.
#pragma once
#include <cstring>
#include <map>
#include <mutex>
#include <tuple>

#include "attention.cuh"
#include "attention_tc.cuh"
#include "common.cuh"
#include "gemm_tcgen05.cuh"
#include "gemm_2cta.cuh"
#include "ops.cuh"
#include "p2p.cuh"
#include "moe.cuh"
#include "cb.cuh"
#include "sampling.cuh"

namespace b200 {

// ---------------------------------------------------------------------------------------------
// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time libcuda dependency,
// so the library also loads on a GPU-less box for the symbol-export test).
// ---------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  });
  return fn;
}

// 2D bf16 row-major [rows][cols] (cols contiguous), box = [box_rows][64], 128B swizzle, OOB -> zeros.
inline int make_tmap_2d(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld_elems,
                        uint32_t box_rows) {
  PFN_encodeTiled fn = get_encode_fn();
  B200_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled entry point not available (no CUDA driver?)");
  B200_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "TMA base must be 16-byte aligned");
  B200_REQUIRE((ld_elems * 2) % 16 == 0, "TMA row pitch must be a multiple of 16 bytes");
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld_elems * 2};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  B200_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
  return 0;
}

struct TmapCache {
  std::map<std::tuple<const void*, uint64_t, uint64_t, uint32_t>, CUtensorMap> maps;
  int get(const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows, const CUtensorMap** out) {
    auto key = std::make_tuple(ptr, rows, cols, box_rows);
    auto it = maps.find(key);
    if (it == maps.end()) {
      CUtensorMap m;
      int rc = make_tmap_2d(&m, ptr, rows, cols, cols, box_rows);
      if (rc) return rc;
      it = maps.emplace(key, m).first;
    }
    *out = &it->second;
    return 0;
  }
  // called between forward passes (no descriptor pointer outstanding): micro-batch views of ragged prompts key new
  // maps by their row offset, so the table is bounded here
  void trim(size_t max_entries = 2048) {
    if (maps.size() > max_entries) maps.clear();
  }
};

// Every kernel of the forward path is launched with programmatic stream serialization so that its prologue
// (and, for the weight-streaming GEMMs, its first weight tiles) overlaps the tail of its predecessor.
// B200_NO_PDL=1 disables it (A/B measurement).
inline bool pdl_enabled() {
  static const bool v = getenv("B200_NO_PDL") == nullptr;
  return v;
}
// set by the engine per phase: decode kernels are 5-50 us and benefit; the ms-scale prefill kernels do not
// (early-launched successors only take SM slots away), measured r01: TTFT 410 -> 449 ms with PDL on.
inline bool& pdl_phase() {
  static bool v = false;
  return v;
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (pdl_enabled() && pdl_phase()) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

template <int BLOCK_N, int EPI>
int launch_gemm_inst(const CUtensorMap* ta, const CUtensorMap* tb, const GemmParams& p, int grid, cudaStream_t s) {
  auto kern = gemm_tn_kernel<BLOCK_N, EPI>;
  static bool configured = false;  // per instantiation
  if (!configured) {
    B200_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, GemmCfg<BLOCK_N>::kSmemBytes));
    configured = true;
  }
  B200_CUDA_OK(launch_k(kern, dim3(grid), dim3(kGemmThreads), GemmCfg<BLOCK_N>::kSmemBytes, s, *ta, *tb, p));
  return 0;
}

template <int EPI>
int launch_gemm_2cta_inst(const CUtensorMap* ta, const CUtensorMap* tb, const GemmParams& p, int num_sms, cudaStream_t s) {
  auto kern = gemm_tn_2cta_kernel<EPI>;
  static bool configured = false;
  if (!configured) {
    B200_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, k2SmemBytes));
    configured = true;
  }
  const int units = ((p.m_tiles + 1) / 2) * p.n_tiles;
  const int clusters = std::min(units, num_sms / 2);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2 * clusters); cfg.blockDim = dim3(kGemmThreads); cfg.dynamicSmemBytes = k2SmemBytes; cfg.stream = s;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (pdl_enabled() && pdl_phase()) ? 2 : 1;
  B200_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, *ta, *tb, p));
  return 0;
}

struct GemmArgs {
  const bf16* A; int a_rows;        // rows of the A buffer as declared to TMA (>= M)
  const bf16* B; int b_rows;        // rows of the B buffer as declared to TMA (>= N)
  int M, N, K;
  int epi, block_n, splits;
  void* out; const bf16* residual; long long ldo; long long split_stride; int out_cols;
  bool stream_a;                    // true: A is the weight (decode) -> evict-first on A, keep B
  float* sk_ws = nullptr;           // stream-K workspace / flags (optional): enables balanced scheduling for
  int* sk_flags = nullptr;          // single-split swap-AB GEMMs whose tile count is not a multiple of the SM count
  size_t sk_ws_floats = 0;          // capacity of the workspace
  int sk_tiles = 0;                 // capacity of the flag array
  const int* m_rt = nullptr;        // device-side runtime bounds (MoE expert token counts)
  const int* n_rt = nullptr;
  const int* row_off = nullptr;
  int groups = 0;                   // > 0: grouped swap-AB problem (see GemmParams::group_m_tiles); A rows = groups * M,
  long long group_out_stride = 0;   // n_rt / row_off are arrays of `groups` entries
  const RopeKvParams* rope = nullptr;   // EPI_ROPE_KV: where RoPE(k) / v go and the tables (q is rotated in place in `out`)
};

inline int launch_gemm(TmapCache& cache, const GemmArgs& a, int num_sms, cudaStream_t s) {
  B200_REQUIRE(a.K % 8 == 0, "K must be a multiple of 8");
  const CUtensorMap *ta, *tb;
  int rc = cache.get(a.A, a.a_rows, a.K, kGemmBlockM, &ta);
  if (rc) return rc;
  rc = cache.get(a.B, a.b_rows, a.K, a.block_n, &tb);
  if (rc) return rc;
  GemmParams p;
  p.M = a.M; p.N = a.N; p.K = a.K;
  p.m_tiles = (a.M + kGemmBlockM - 1) / kGemmBlockM;
  p.n_tiles = (a.N + a.block_n - 1) / a.block_n;
  p.kb_total = (a.K + kGemmBlockK - 1) / kGemmBlockK;
  p.splits = a.splits < 1 ? 1 : (a.splits > p.kb_total ? p.kb_total : a.splits);
  p.kb_per_split = (p.kb_total + p.splits - 1) / p.splits;
  p.splits = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;  // no empty splits
  B200_REQUIRE(p.splits == a.splits || a.epi != EPI_T_PARTIAL, "caller must use effective_splits() for partials");
  p.out = a.out; p.residual = a.residual; p.ldo = a.ldo; p.split_stride = a.split_stride; p.out_cols = a.out_cols;
  p.hint_a = a.stream_a ? kEvictFirst : kEvictLast;
  p.hint_b = a.stream_a ? kEvictLast : kEvictNormal;
  p.m_rt = a.m_rt; p.n_rt = a.n_rt; p.row_off = a.row_off;
  p.group_m_tiles = 0; p.group_out_stride = a.group_out_stride;
  if (a.groups > 0) {
    B200_REQUIRE(a.stream_a && a.n_rt && a.row_off && !a.m_rt && a.N <= a.block_n, "grouped GEMM: swap-AB with per-group n_rt / row_off");
    p.group_m_tiles = p.m_tiles;
    p.m_tiles *= a.groups;
  }
  p.prefetch_a = (a.stream_a && !a.n_rt && !a.m_rt) ? 1 : 0;
  const int units = p.m_tiles * p.n_tiles * p.splits;
  int grid = units < num_sms ? units : num_sms;
  p.sched = 0; p.sk_slots = 0; p.sk_ws = a.sk_ws; p.sk_flags = a.sk_flags;
  // only when every tile is cut into at most two pieces (m_tiles >= SMs): finishing many-piece tiles inside the
  // kernel serialises the reduction on the tile owner and measured slower than split-K + a reducing consumer
  const bool sk_any = getenv("B200_STREAMK_ANY") != nullptr;
  if (a.groups == 0 && a.sk_ws && a.sk_flags && a.stream_a && p.splits == 1 && p.n_tiles == 1 && p.m_tiles <= a.sk_tiles &&
      (p.m_tiles >= num_sms || sk_any) && (p.m_tiles % num_sms) != 0 && (a.epi == EPI_T_STORE || a.epi == EPI_T_SWIGLU)) {
    const long long W = (long long)p.m_tiles * p.kb_total;
    const int g2 = (int)std::min<long long>(num_sms, W);
    const long long per_min = W / g2;                                   // >= 1
    const int slots = (int)((p.kb_total + per_min - 1) / per_min) + 1;    // pieces a tile can be cut into, minus the owner
    if ((size_t)p.m_tiles * slots * a.block_n * kGemmBlockM <= a.sk_ws_floats) {
      p.sched = 1; p.sk_slots = slots; grid = g2;
    }
  }
  B200_REQUIRE(p.splits == 1 || a.epi == EPI_T_PARTIAL, "split-K only with the fp32 partial epilogue");
  p.rope_tok_seq = nullptr; p.rope_tok_pos = nullptr; p.rope_page_table = nullptr; p.rope_max_pages = 0;
  p.rope_kcache = nullptr; p.rope_vcache = nullptr; p.rope_cos = nullptr; p.rope_sin = nullptr; p.rope_nh = 0; p.rope_nkv = 0;
  if (a.epi == EPI_ROPE_KV) {
    B200_REQUIRE(a.block_n == 256 && a.rope && a.N == (a.rope->nh + 2 * a.rope->nkv) * kHeadDim,
                 "EPI_ROPE_KV is the 2-CTA prefill QKV projection");
    p.rope_tok_seq = a.rope->tok_seq; p.rope_tok_pos = a.rope->tok_pos; p.rope_page_table = a.rope->page_table;
    p.rope_max_pages = a.rope->max_pages; p.rope_kcache = a.rope->kcache; p.rope_vcache = a.rope->vcache;
    p.rope_cos = a.rope->cos_tab; p.rope_sin = a.rope->sin_tab; p.rope_nh = a.rope->nh; p.rope_nkv = a.rope->nkv;
    const CUtensorMap* tb2;
    int rc2 = cache.get(a.B, a.b_rows, a.K, 128, &tb2);
    if (rc2) return rc2;
    return launch_gemm_2cta_inst<EPI_ROPE_KV>(ta, tb2, p, num_sms, s);
  }
  if (a.block_n == 256 && a.epi <= EPI_SWIGLU) {
    const CUtensorMap* tb2;
    int rc2 = cache.get(a.B, a.b_rows, a.K, 128, &tb2);   // each CTA of the pair stages half of the 256 weight rows
    if (rc2) return rc2;
    if (a.epi == EPI_STORE) return launch_gemm_2cta_inst<EPI_STORE>(ta, tb2, p, num_sms, s);
    if (a.epi == EPI_STORE_RES) return launch_gemm_2cta_inst<EPI_STORE_RES>(ta, tb2, p, num_sms, s);
    return launch_gemm_2cta_inst<EPI_SWIGLU>(ta, tb2, p, num_sms, s);
  }
#define B200_GEMM_CASE(BN, E) \
  if (a.block_n == BN && a.epi == E) return launch_gemm_inst<BN, E>(ta, tb, p, grid, s);
  B200_GEMM_CASE(16, EPI_T_STORE)
  B200_GEMM_CASE(16, EPI_T_SWIGLU)
  B200_GEMM_CASE(16, EPI_T_PARTIAL)
  B200_GEMM_CASE(32, EPI_T_STORE)
  B200_GEMM_CASE(32, EPI_T_SWIGLU)
  B200_GEMM_CASE(32, EPI_T_PARTIAL)
  B200_GEMM_CASE(64, EPI_T_STORE)
  B200_GEMM_CASE(64, EPI_T_SWIGLU)
  B200_GEMM_CASE(64, EPI_T_PARTIAL)
#undef B200_GEMM_CASE
  set_last_error("unsupported GEMM variant block_n=" + std::to_string(a.block_n) + " epi=" + std::to_string(a.epi));
  return -3;
}

// number of split-K slices launch_gemm will really use for a request of `want`
inline int effective_splits(int K, int want) {
  const int kb = (K + kGemmBlockK - 1) / kGemmBlockK;
  int s = want < 1 ? 1 : (want > kb ? kb : want);
  const int per = (kb + s - 1) / s;
  return (kb + per - 1) / per;
}

inline int launch_rmsnorm(int mode, bf16* x, const bf16* w, bf16* xn, int rows, int H, float eps,
                          const float* partial, int splits, long long split_stride, long long ld_partial,
                          const bf16* y, cudaStream_t s) {
  B200_REQUIRE(H % 8 == 0, "hidden size must be a multiple of 8");
  const size_t smem = (size_t)(H + 32) * sizeof(float);
  static bool configured = false;
  if (!configured) {
    B200_CUDA_OK(cudaFuncSetAttribute(rmsnorm_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    B200_CUDA_OK(cudaFuncSetAttribute(rmsnorm_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    B200_CUDA_OK(cudaFuncSetAttribute(rmsnorm_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    configured = true;
  }
  B200_REQUIRE(smem <= 96 * 1024, "hidden size too large for the rmsnorm kernel");
  if (rows == 0) return 0;
  const float* np = nullptr;
  const bf16* ny = nullptr;
  // prefill-sized launches of the plain / post-all-reduce norm: the warp-per-row kernel
  if (mode != 1 && rows >= 256) {
#define B200_NORM_ROWS(NVV)                                                                                                       \
    if (H == NVV * 256) {                                                                                                          \
      if (mode == 0) B200_CUDA_OK(launch_k(rmsnorm_rows_kernel<0, NVV>, dim3((rows + 7) / 8), dim3(256), 0, s, x, w, xn, rows, eps, ny)); \
      else B200_CUDA_OK(launch_k(rmsnorm_rows_kernel<2, NVV>, dim3((rows + 7) / 8), dim3(256), 0, s, x, w, xn, rows, eps, y));           \
      return 0;                                                                                                                    \
    }
    B200_NORM_ROWS(2) B200_NORM_ROWS(4) B200_NORM_ROWS(8) B200_NORM_ROWS(16) B200_NORM_ROWS(32)
#undef B200_NORM_ROWS
  }
  if (mode == 0) B200_CUDA_OK(launch_k(rmsnorm_kernel<0>, dim3(rows), dim3(kNormThreads), smem, s, x, w, xn, H, eps, np, 0, 0LL, 0LL, ny));
  else if (mode == 1) B200_CUDA_OK(launch_k(rmsnorm_kernel<1>, dim3(rows), dim3(kNormThreads), smem, s, x, w, xn, H, eps, partial, splits, split_stride, ld_partial, ny));
  else B200_CUDA_OK(launch_k(rmsnorm_kernel<2>, dim3(rows), dim3(kNormThreads), smem, s, x, w, xn, H, eps, np, 0, 0LL, 0LL, y));
  return 0;
}

constexpr int kDecodeSmem = 4096 + 2 * kDecStages * kTileBytes + 10 * kHeadDim * 4 + 2 * kHeadDim * 2;

// tcgen05 prefill attention: q rows [q_rows][ldq] (head h at column h*128), paged caches [num_pages][nkv][64][128]
inline int launch_attn_prefill_tc(TmapCache& cache, const bf16* q, int q_rows, long long ldq, const bf16* kcache,
                                  const bf16* vcache, int num_pages, const AttnTcParams& p, int B, int max_len, cudaStream_t s) {
  static bool configured = false;
  if (!configured) {
    B200_CUDA_OK(cudaFuncSetAttribute(attn_prefill_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmem));
    configured = true;
  }
  const CUtensorMap *tq, *tk, *tv;
  int rc = cache.get(q, (uint64_t)q_rows, (uint64_t)ldq, 128, &tq);
  if (rc) return rc;
  const uint64_t kv_rows = (uint64_t)num_pages * p.nkv * kPageTokens;
  if ((rc = cache.get(kcache, kv_rows, kHeadDim, 64, &tk))) return rc;
  if ((rc = cache.get(vcache, kv_rows, kHeadDim, 64, &tv))) return rc;
  dim3 grid((max_len + kTcQ - 1) / kTcQ, p.nh, B);
  B200_CUDA_OK(launch_k(attn_prefill_tc_kernel, grid, dim3(kTcThreads), kTcSmem, s, *tq, *tk, *tv, p));
  return 0;
}

inline int launch_attn_decode(const AttnDecodeParams& p, int B, cudaStream_t s) {
  static bool configured = false;
  if (!configured) {
    B200_CUDA_OK(cudaFuncSetAttribute(attn_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kDecodeSmem));
    configured = true;
  }
  B200_REQUIRE(p.G >= 1 && p.G <= 8, "GQA group size must be in [1, 8]");
  B200_REQUIRE(p.splits == 1 || p.split_counter, "split decode attention needs the arrival counters of its merge");
  dim3 grid(B * p.nkv, p.splits);
  B200_CUDA_OK(launch_k(attn_decode_kernel, grid, dim3(kAttnThreads), kDecodeSmem, s, p));
  return 0;
}

}  // namespace b200
