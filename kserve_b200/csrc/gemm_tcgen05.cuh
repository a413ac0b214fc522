// Persistent, warp-specialised bf16 GEMM for sm_100a:  D[M,N] = A[M,K] * B[N,K]^T  (both K-major).
//
//   warp 0   : TMA producer  (cp.async.bulk.tensor -> 128B-swizzled smem ring, mbarrier complete_tx)
//   warp 1   : MMA issuer    (one thread, tcgen05.mma cta_group::1 kind::f16, fp32 accumulators in TMEM)
//   warps 2-5: epilogue      (tcgen05.ld -> registers -> fused epilogue -> global), double-buffered TMEM
//
// This kernel is the decode GEMM (SURVEY.md §8a rows 13-17); prefill runs on the 2-CTA kernel (gemm_2cta.cuh).
// A = weight [N_out,K] (M = N_out), B = activations [batch,K] ("swap-AB": the 128-row MMA M dimension is filled
// by weight rows, the small batch rides in the MMA N dimension, so no tensor-core work is wasted on padding and
// each CTA streams a contiguous weight slab) -> transposed epilogues, optional split-K with fp32 partials.
#pragma once
#include "common.cuh"

namespace b200 {

enum GemmEpi : int {
  // row-major epilogues of the 2-CTA prefill kernel
  EPI_STORE = 0,      // out[m][n] = bf16(acc)
  EPI_STORE_RES = 1,  // out[m][n] = bf16(bf16(acc) + residual[m][n])           (o_proj / down_proj + residual)
  EPI_SWIGLU = 2,     // B rows interleaved {16 gate,16 up}: out[m][n/2] = bf16(bf16(silu(g)) * u)
  // transposed epilogues of the swap-AB decode kernel
  EPI_T_STORE = 3,    // out[n][m] = bf16(acc)                                    (swap-AB)
  EPI_T_SWIGLU = 4,   // A rows interleaved {16 gate,16 up}: out[n][m/2] = ...    (swap-AB)
  EPI_T_PARTIAL = 5,  // ws[split][n][m] = acc (fp32)                             (swap-AB split-K)
  EPI_ROPE_KV = 6,    // prefill QKV projection (2-CTA kernel only): columns are [q heads | k heads | v heads] x 128;
                      // q <- RoPE(q) in place in `out`, RoPE(k) and v go straight to the paged KV cache
};

struct GemmParams {
  int M, N, K;
  int m_tiles, n_tiles, splits;
  int kb_total;       // ceil(K / 64)
  int kb_per_split;   // ceil(kb_total / splits)
  void* out;
  const bf16* residual;
  long long ldo;           // leading dimension of out (elements)
  long long split_stride;  // EPI_T_PARTIAL: elements between split slices
  int out_cols;            // logical number of output columns (bounds for SWIGLU modes = N/2 resp. M/2)
  unsigned long long hint_a, hint_b;
  int prefetch_a;          // A (weights) does not depend on the previous kernel: stream it before griddepcontrol.wait
  // sched == 1: "stream-K" — the m_tiles * kb_total k-block iterations are cut into gridDim.x equal contiguous
  // ranges, so every SM streams the same number of weight bytes whatever the tile count (few tiles under tensor
  // parallelism, 224 tiles on 148 SMs, ...).  A tile covered by several CTAs is finished by the CTA that owns
  // its last k-block: the others park fp32 partials in sk_ws[tile][piece] and bump sk_flags[tile]; the owner
  // waits for the count, adds the pieces in piece order (deterministic) and runs the normal epilogue.
  // Each CTA processes its non-final piece first and its tile-finishing piece last, so nobody waits on a CTA
  // that is itself waiting.  Requires n_tiles == 1 and splits == 1.
  // runtime extents (device counters, e.g. tokens routed to one MoE expert): when set they replace M (row-major
  // kernels) / N (swap-AB kernels) and the kernel first waits for its predecessor to read them; 0 => nothing to do
  const int* m_rt;
  const int* n_rt;
  const int* row_off;      // device row offset of the activation / output rows inside a grouped (per-expert) buffer
                           // (2-CTA kernel: rows of A and of the output; swap-AB kernel: rows of B and output rows n)
  // grouped (per-expert) swap-AB problem in ONE launch: A = [groups][M][K] stacked weights, m_tiles = groups * group_m_tiles;
  // tile m_t belongs to group g = m_t / group_m_tiles whose activation rows are row_off[g] .. + n_rt[g] (tiles of
  // empty groups are skipped: their weights are never streamed) and whose outputs start at out + g * group_out_stride
  int group_m_tiles;
  long long group_out_stride;
  // EPI_ROPE_KV: one output row = one prompt token (HF bf16 rounding points of apply_rotary_pos_emb; bit-identical to rope_kv_kernel)
  const int32_t* rope_tok_seq; const int32_t* rope_tok_pos;   // [M] page-table row / position of each token
  const int32_t* rope_page_table; int rope_max_pages;
  bf16* rope_kcache; bf16* rope_vcache;                      // this layer's [page][kv_head][64][128]
  const bf16* rope_cos; const bf16* rope_sin;                // [max_pos][64]
  int rope_nh, rope_nkv;
  int sched;
  int sk_slots;            // partial slots per tile
  float* sk_ws;            // [m_tiles][sk_slots][BLOCK_N][128] fp32
  int* sk_flags;           // [m_tiles] arrival counters, 0 between launches
};

constexpr int kGemmBlockM = 128;
constexpr int kGemmBlockK = 64;
constexpr int kGemmThreads = 192;
constexpr int kGemmGroupM = 16;

template <int BLOCK_N>
struct GemmCfg {
  static constexpr int kABytes = kGemmBlockM * kGemmBlockK * 2;  // 16 KB
  static constexpr int kBBytes = BLOCK_N * kGemmBlockK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = BLOCK_N >= 128 ? 6 : 8;
  static constexpr int kTmemCols = (2 * BLOCK_N < 32) ? 32 : 2 * BLOCK_N;  // power of two for 16..64
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/;
};

// SiLU on an already bf16-rounded input whose result is rounded to bf16 again: the fast exp / divide intrinsics
// (rel. error ~1e-6) cannot change the bf16 result except on exact rounding ties, and keep the epilogue short.
__device__ __forceinline__ float silu_f(float x) { return __fdividef(x, 1.0f + __expf(-x)); }


struct GemmSeg { int m_t, n_t, kb0, kb1, split, type, slot; };  // type: 0 full tile, 1 partial piece -> workspace slot, 2 tile-finishing piece (adds `slot` parked pieces)

__device__ __forceinline__ int sk_owner(long long it, long long W, int P) {   // CTA whose range contains iteration `it`
  int c = (int)((it * P) / W);
  while (W * (c + 1) / P <= it) ++c;
  while (W * c / P > it) --c;
  return c;
}

// The work list of this CTA: its idx-th segment
__device__ __forceinline__ bool gemm_get_seg(const GemmParams& p, int idx, GemmSeg& g, int m_tiles_rt) {
  g.slot = 0;
  if (m_tiles_rt <= 0) return false;
  if (p.sched == 0) {
    const int u = (int)blockIdx.x + idx * (int)gridDim.x;
    if (u >= m_tiles_rt * p.n_tiles * p.splits) return false;
    const int tile = u / p.splits;
    g.split = u - tile * p.splits;
    const int per_group = kGemmGroupM * p.n_tiles;
    const int grp = tile / per_group;
    const int first_m = grp * kGemmGroupM;
    const int gsize = min(m_tiles_rt - first_m, kGemmGroupM);
    const int r = tile - grp * per_group;
    g.m_t = first_m + r % gsize;
    g.n_t = r / gsize;
    g.kb0 = g.split * p.kb_per_split;
    g.kb1 = min(g.kb0 + p.kb_per_split, p.kb_total);
    g.type = 0;
    return true;
  }
  const int P = (int)gridDim.x, c = (int)blockIdx.x, KB = p.kb_total;
  const long long W = (long long)p.m_tiles * KB;
  const long long lo = W * c / P, hi = W * (c + 1) / P;
  if (lo >= hi) return false;
  const int t0 = (int)(lo / KB), k_lo = (int)(lo % KB);
  const int t1 = (int)((hi - 1) / KB), k_hi = (int)((hi - 1) % KB) + 1;
  const int has_piece = (k_hi < KB) ? 1 : 0;                                   // last tile of the range is finished by a later CTA
  const int has_tail = (k_lo > 0 && !(t0 == t1 && has_piece)) ? 1 : 0;          // first tile was started by an earlier CTA, we finish it
  const int f0 = t0 + ((k_lo > 0) ? 1 : 0), f1 = t1 - has_piece;
  const int n_full = max(0, f1 - f0 + 1);
  g.n_t = 0; g.split = 0;
  if (idx < has_piece) {
    g.m_t = t1; g.kb0 = (t0 == t1) ? k_lo : 0; g.kb1 = k_hi; g.type = 1;
    g.slot = c - sk_owner((long long)t1 * KB, W, P);
    return true;
  }
  idx -= has_piece;
  if (idx < n_full) { g.m_t = f0 + idx; g.kb0 = 0; g.kb1 = KB; g.type = 0; return true; }
  idx -= n_full;
  if (idx < has_tail) {
    g.m_t = t0; g.kb0 = k_lo; g.kb1 = KB; g.type = 2;
    g.slot = c - sk_owner((long long)t0 * KB, W, P);   // number of parked pieces to wait for
    return true;
  }
  return false;
}

template <int BLOCK_N, int EPI>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tn_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
               const GemmParams p) {
  TraceScope _ts(TK_GEMM + 100 * EPI + 1000 * (p.M >> 7));
  using Cfg = GemmCfg<BLOCK_N>;
  constexpr int STAGES = Cfg::kStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::kStageBytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + STAGES;
  uint64_t* tmem_full = bars + 2 * STAGES;
  uint64_t* tmem_empty = bars + 2 * STAGES + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  pdl_launch_dependents();

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 128);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, Cfg::kTmemCols);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  int M_rt = p.M, N_rt = p.N;
  const int gmt = p.group_m_tiles;
  if (p.m_rt != nullptr || p.n_rt != nullptr) {   // extents produced by the previous kernel
    pdl_wait();
    if (p.m_rt) M_rt = min(p.M, *p.m_rt);
    if (p.n_rt && !gmt) N_rt = min(p.N, *p.n_rt);
  }
  const int m_tiles_rt = gmt ? p.m_tiles : ((M_rt <= 0 || N_rt <= 0) ? 0 : (M_rt + kGemmBlockM - 1) / kGemmBlockM);
  int roff_b = (p.row_off && !gmt) ? *p.row_off : 0;   // (read after the wait above: set together with m_rt / n_rt)

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      bool first = true;
      GemmSeg sg;
      for (int idx = 0; gemm_get_seg(p, idx, sg, m_tiles_rt); ++idx) {
        const int m_t = sg.m_t, n_t = sg.n_t, kb0 = sg.kb0, kb1 = sg.kb1;
        int a_row = m_t * kGemmBlockM, b_off = roff_b;
        if (gmt) {
          const int g = m_t / gmt;
          if (p.n_rt[g] <= 0) continue;
          a_row = g * p.M + (m_t - g * gmt) * kGemmBlockM;
          b_off = p.row_off[g];
        }
        int kb = kb0;
        if (first) {
          first = false;
          if (p.prefetch_a) {
            // Weight tiles of the first k-blocks are requested before the previous kernel has finished; only the
            // activation tiles wait for it.  (All stages are free at this point: no empty-barrier wait needed.)
            const int npre = min(STAGES, kb1 - kb0);
            for (int i = 0; i < npre; ++i) {
              mbar_arrive_expect_tx(&full_bar[i], Cfg::kStageBytes);
              tma_load_2d(smem + i * Cfg::kStageBytes, &tmap_a, &full_bar[i], (kb0 + i) * kGemmBlockK, a_row, p.hint_a);
            }
            pdl_wait();
            _ts.mark();
            for (int i = 0; i < npre; ++i)
              tma_load_2d(smem + i * Cfg::kStageBytes + Cfg::kABytes, &tmap_b, &full_bar[i], (kb0 + i) * kGemmBlockK, n_t * BLOCK_N + b_off, p.hint_b);
            kb = kb0 + npre;
            if (npre == STAGES) { stage = 0; phase = 1; } else { stage = npre; }
          } else {
            pdl_wait();
          }
        }
        for (; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * Cfg::kStageBytes;
          uint8_t* sb = sa + Cfg::kABytes;
          mbar_arrive_expect_tx(&full_bar[stage], Cfg::kStageBytes);
          tma_load_2d(sa, &tmap_a, &full_bar[stage], kb * kGemmBlockK, a_row, p.hint_a);
          tma_load_2d(sb, &tmap_b, &full_bar[stage], kb * kGemmBlockK, n_t * BLOCK_N + b_off, p.hint_b);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(kGemmBlockM, BLOCK_N);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      GemmSeg sg;
      for (int idx = 0; gemm_get_seg(p, idx, sg, m_tiles_rt); ++idx) {
        const int kb0 = sg.kb0, kb1 = sg.kb1;
        if (gmt && p.n_rt[sg.m_t / gmt] <= 0) continue;
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tcgen05_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BLOCK_N;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tcgen05_fence_after();
          const uint32_t sa = smem_u32(smem + stage * Cfg::kStageBytes);
          const uint64_t adesc = make_smem_desc_sw128(sa);
          const uint64_t bdesc = make_smem_desc_sw128(sa + Cfg::kABytes);
#pragma unroll
          for (int k = 0; k < kGemmBlockK / 16; ++k) {
            // advance 16 elements (32 B) along K inside the 128 B swizzle atom: +2 in the (addr>>4) field
            umma_bf16(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);  // smem slot reusable once these MMAs retire
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tmem_full[acc]);  // accumulator complete -> epilogue
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------------ epilogue (4 warps = 128 TMEM lanes)
    const int q = warp & 3;  // TMEM lane quadrant this warp may access
    pdl_wait();              // outputs / residual must not be touched before the previous kernel is complete
    int acc = 0;
    uint32_t acc_phase = 0;
    GemmSeg sg;
    for (int idx = 0; gemm_get_seg(p, idx, sg, m_tiles_rt); ++idx) {
      const int n_t = sg.n_t, s = sg.split;
      int m_t = sg.m_t;
      long long out_off = 0;   // elements
      if (gmt) {
        const int g = m_t / gmt;
        N_rt = min(p.N, p.n_rt[g]);
        if (N_rt <= 0) continue;
        roff_b = p.row_off[g];
        m_t -= g * gmt;         // tile index inside the group: output features are per expert
        out_off = (long long)g * p.group_out_stride;
      }
      const int m = m_t * kGemmBlockM + q * 32 + lane;  // accumulator row of this thread
      const int n0 = n_t * BLOCK_N;
      mbar_wait(&tmem_full[acc], acc_phase);
      tcgen05_fence_after();
      const long long sk_piece = (long long)BLOCK_N * kGemmBlockM;
      float* skw = (sg.type != 0) ? p.sk_ws + ((long long)sg.m_t * p.sk_slots) * sk_piece + q * 32 + lane : nullptr;
      if (sg.type == 2) {   // wait until every other piece of this tile has been parked
        if (threadIdx.x == 64) {
          SpinGuard spins;
          while (*reinterpret_cast<volatile int*>(p.sk_flags + sg.m_t) != sg.slot)
            if (spin_give_up(spins, 4)) break;
          __threadfence();
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
      }
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * BLOCK_N;
      constexpr int CH = (BLOCK_N >= 32) ? 32 : 16;
#pragma unroll 1
      for (int c0 = 0; c0 < BLOCK_N; c0 += CH) {
        if (n0 + c0 >= N_rt) break;  // warp-uniform: nothing valid in this chunk
        float v[CH];
        {
          uint32_t r[CH];
          if constexpr (CH == 32) tmem_ld_32x32(taddr + c0, r); else tmem_ld_32x16(taddr + c0, r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < CH; ++j) v[j] = __uint_as_float(r[j]);
        }
        const int nvalid = min(CH, N_rt - (n0 + c0));
        if (sg.type == 1) {          // park the fp32 accumulators of this piece, the tile's owner finishes it
          float* w = skw + (long long)sg.slot * sk_piece;
#pragma unroll
          for (int j = 0; j < CH; ++j) w[(long long)(c0 + j) * kGemmBlockM] = v[j];
          continue;
        }
        if (sg.type == 2) {          // pieces are added in piece (= k) order, then this CTA's own tail
          float acc[CH];
#pragma unroll
          for (int j = 0; j < CH; ++j) acc[j] = 0.f;
          for (int sl = 0; sl < sg.slot; ++sl) {
            const float* w = skw + (long long)sl * sk_piece;
#pragma unroll
            for (int j = 0; j < CH; ++j) acc[j] += __ldcg(w + (long long)(c0 + j) * kGemmBlockM);
          }
#pragma unroll
          for (int j = 0; j < CH; ++j) v[j] += acc[j];
        }
        if constexpr (EPI == EPI_T_STORE) {
          if (m < M_rt) {
            bf16* o = reinterpret_cast<bf16*>(p.out) + out_off + (long long)(n0 + c0 + roff_b) * p.ldo + m;
#pragma unroll
            for (int j = 0; j < CH; ++j)
              if (j < nvalid) o[(long long)j * p.ldo] = __float2bfloat16_rn(v[j]);
          }
        } else if constexpr (EPI == EPI_T_SWIGLU) {
          // rows of a 32-row warp slab: lanes 0-15 gate, lanes 16-31 up, for output feature (slab/2 + lane)
          const int f = ((m_t * kGemmBlockM + q * 32) >> 1) + (lane & 15);
          bf16* o = reinterpret_cast<bf16*>(p.out) + out_off + (long long)(n0 + c0 + roff_b) * p.ldo + f;
#pragma unroll
          for (int j = 0; j < CH; j += 2) {
            // lanes 16-31 hold `up`: hand two bf16 columns per shuffle to the gate lane 16 below
            const uint32_t mine = pack_bf16x2(v[j], v[j + 1]);
            const uint32_t other = __shfl_down_sync(0xffffffffu, mine, 16);
            if (lane < 16 && f < p.out_cols) {
              const float2 g2 = unpack_bf16x2(mine), u2 = unpack_bf16x2(other);
              if (j < nvalid) o[(long long)j * p.ldo] = __float2bfloat16_rn(bf16_round(silu_f(g2.x)) * u2.x);
              if (j + 1 < nvalid) o[(long long)(j + 1) * p.ldo] = __float2bfloat16_rn(bf16_round(silu_f(g2.y)) * u2.y);
            }
          }
        } else {  // EPI_T_PARTIAL
          if (m < M_rt) {
            float* o = reinterpret_cast<float*>(p.out) + out_off + (long long)s * p.split_stride +
                       (long long)(n0 + c0) * p.ldo + m;
#pragma unroll
            for (int j = 0; j < CH; ++j)
              if (j < nvalid) o[(long long)j * p.ldo] = v[j];
          }
        }
      }
      tcgen05_fence_before();
      mbar_arrive(&tmem_empty[acc]);
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      if (sg.type == 1) {          // publish the partial
        __threadfence();
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (threadIdx.x == 64) atomicAdd(p.sk_flags + sg.m_t, 1);
      } else if (sg.type == 2) {   // consumed: leave the flag clean for the next launch / graph replay
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (threadIdx.x == 64) atomicExch(p.sk_flags + sg.m_t, 0);
      }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

}  // namespace b200
