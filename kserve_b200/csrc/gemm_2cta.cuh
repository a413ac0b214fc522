// 2-CTA (cta_group::2) variant of the prefill GEMM: a CTA pair on one TPC computes a 256 x 256 tile with one
// tcgen05.mma.cta_group::2 (M = 256) per K step.  Each CTA stages its own 128 rows of A and HALF of the B tile
// (128 of the 256 weight rows); the tensor cores of both SMs read both halves, so shared-memory traffic per SM
// drops by a third versus the 1-CTA kernel, which ncu shows pinned at ~75 % L1/shared throughput
// (profiles/r01_ncu_full_summary.json).
//
//   leader (cluster rank 0): arms the full barriers (tx bytes of BOTH CTAs), issues every MMA, multicasts the
//                            commits (smem-slot free / accumulator ready) to both CTAs
//   both CTAs              : TMA producer for their halves (complete_tx on the LEADER's barrier), own epilogue of
//                            their 128 accumulator rows, arrive on the leader's tmem_empty barrier
#pragma once
#include "common.cuh"
#include "gemm_tcgen05.cuh"

namespace b200 {

constexpr int k2StageBytes = 2 * kGemmBlockM * kGemmBlockK * 2;  // A 16 KB + B-half 16 KB
constexpr int k2Stages = 6;
constexpr int k2SmemBytes = k2Stages * k2StageBytes + 1024 + 256;
constexpr int k2BlockN = 256;

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;  // clears the CTA-rank bit of a shared::cluster address -> leader CTA

__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* map, uint64_t* leader_bar, int c_inner,
                                                int c_outer, uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(leader_bar) & kPeerBitMask), "r"(c_inner), "r"(c_outer), "l"(hint)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar) {  // arrives on `bar`'s offset in BOTH CTAs
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {  // arrive on the same barrier in cluster rank 0
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(0));
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}

// output tiles are written once and read by a LATER kernel: they go out as cache-streaming stores so that the (up to
// 940 MB per GEMM) output stream does not push the A / B tiles the other CTAs are about to re-read out of L2
__device__ __forceinline__ void st_out_v4(bf16* p, const uint4& o) {
  asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(o.x), "r"(o.y), "r"(o.z), "r"(o.w) : "memory");
}

// m-pairs (256 rows each) per raster group.  r02 (tools/prefill_gemm.py, T = 32768): groups of 12 m-pairs + cache-streaming
// output stores: gate/up 5.47 -> 4.76 ms, down 3.34 -> 2.57 ms, qkv 1.126 -> 1.108 ms
constexpr int k2GroupPairs = 12;

struct Gemm2Unit { int m_pair, n_t; };
__device__ __forceinline__ bool gemm2_get_unit(const GemmParams& p, int idx, int cluster_id, int num_clusters, Gemm2Unit& u, int m_tiles_rt) {
  const int m_pairs = (m_tiles_rt + 1) >> 1;
  const int t = cluster_id + idx * num_clusters;
  if (t >= m_pairs * p.n_tiles) return false;
  constexpr int G = k2GroupPairs;
  const int per_group = G * p.n_tiles;
  const int grp = t / per_group;
  const int first = grp * G;
  const int gsize = min(m_pairs - first, G);
  const int r = t - grp * per_group;
  u.m_pair = first + r % gsize;
  u.n_t = r / gsize;
  return true;
}

template <int EPI>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tn_2cta_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, const GemmParams p) {
  TraceScope _ts(TK_GEMM + 100 * EPI + 50);
  constexpr int STAGES = k2Stages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * k2StageBytes);
  uint64_t* full_bar = bars;                 // used in the leader CTA only
  uint64_t* empty_bar = bars + STAGES;       // per CTA
  uint64_t* tmem_full = bars + 2 * STAGES;   // per CTA
  uint64_t* tmem_empty = bars + 2 * STAGES + 2;  // used in the leader CTA only (256 arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
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
      mbar_init(&tmem_empty[i], 256);
    }
    fence_barrier_init();
  }
  cluster_sync_all();   // barriers of both CTAs initialised before any cross-CTA signal
  if (warp == 1) tmem_alloc_2sm(tmem_slot, 512);
  tcgen05_fence_before();
  cluster_sync_all();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  int M_rt = p.M;
  if (p.m_rt != nullptr) {   // rows produced by the previous kernel (tokens routed to this MoE expert)
    pdl_wait();
    M_rt = min(p.M, *p.m_rt);
  }
  const int m_tiles_rt = M_rt <= 0 ? 0 : (M_rt + kGemmBlockM - 1) / kGemmBlockM;
  const int roff = p.row_off ? *p.row_off : 0;

  if (warp == 0) {
    // ---------------------------------------------------------------- TMA producer (both CTAs)
    if (lane == 0) {
      pdl_wait();
      int stage = 0;
      uint32_t phase = 0;
      Gemm2Unit u;
      for (int idx = 0; gemm2_get_unit(p, idx, cluster_id, num_clusters, u, m_tiles_rt); ++idx) {
        const int m0 = u.m_pair * 256 + (int)rank * kGemmBlockM;
        const int n0 = u.n_t * k2BlockN + (int)rank * 128;
        for (int kb = 0; kb < p.kb_total; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * k2StageBytes;
          if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * k2StageBytes);
          tma_load_2d_2sm(sa, &tmap_a, &full_bar[stage], kb * kGemmBlockK, m0 + roff, p.hint_a);
          tma_load_2d_2sm(sa + kGemmBlockM * kGemmBlockK * 2, &tmap_b, &full_bar[stage], kb * kGemmBlockK, n0, p.hint_b);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ---------------------------------------------------------------- MMA issuer (leader CTA only)
    if (leader && lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(256, k2BlockN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      Gemm2Unit u;
      for (int idx = 0; gemm2_get_unit(p, idx, cluster_id, num_clusters, u, m_tiles_rt); ++idx) {
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tcgen05_fence_after();
        const uint32_t tmem_d = tmem_base + acc * k2BlockN;
        for (int kb = 0; kb < p.kb_total; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tcgen05_fence_after();
          const uint32_t sa = smem_u32(smem + stage * k2StageBytes);
          const uint64_t adesc = make_smem_desc_sw128(sa);
          const uint64_t bdesc = make_smem_desc_sw128(sa + kGemmBlockM * kGemmBlockK * 2);
#pragma unroll
          for (int k = 0; k < kGemmBlockK / 16; ++k)
            umma_bf16_2sm(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          umma_commit_2sm(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit_2sm(&tmem_full[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
    __syncwarp();
  } else {
    // ---------------------------------------------------------------- epilogue (both CTAs, own 128 rows)
    const int q = warp & 3;
    pdl_wait();
    int acc = 0;
    uint32_t acc_phase = 0;
    Gemm2Unit u;
    for (int idx = 0; gemm2_get_unit(p, idx, cluster_id, num_clusters, u, m_tiles_rt); ++idx) {
      const int m = u.m_pair * 256 + (int)rank * kGemmBlockM + q * 32 + lane;
      const int n0 = u.n_t * k2BlockN;
      mbar_wait(&tmem_full[acc], acc_phase);
      tcgen05_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * k2BlockN;
      constexpr int CH = 32;
      if constexpr (EPI == EPI_ROPE_KV) {
        // the tile's 256 columns are two whole heads; this thread owns token row m
        const bool row_ok = m < M_rt;
        int pos = 0;
        long long page_row = 0;     // (page * nkv) * 64 + slot: row of kv head 0 of this token inside the [.. ][64][128] cache
        if (row_ok) {
          pos = p.rope_tok_pos[m + roff];
          const int page = p.rope_page_table[(long long)p.rope_tok_seq[m + roff] * p.rope_max_pages + (pos >> 6)];
          page_row = (long long)page * p.rope_nkv * 64 + (pos & 63);
        }
#pragma unroll 1
        for (int hh = 0; hh < 2; ++hh) {
          const int col0 = n0 + hh * 128;
          if (col0 >= p.N) break;
          const int head = col0 >> 7;
          if (head >= p.rope_nh + p.rope_nkv) {           // ---- V head: copy to the cache
            const int kvh = head - p.rope_nh - p.rope_nkv;
            bf16* vrow = p.rope_vcache + (page_row + (long long)kvh * 64) * 128;
#pragma unroll 1
            for (int c0 = 0; c0 < 128; c0 += CH) {
              uint32_t r[CH];
              tmem_ld_32x32(taddr + hh * 128 + c0, r);
              tmem_ld_wait();
              if (row_ok) {
#pragma unroll
                for (int j = 0; j < CH; j += 8) {
                  uint4 o;
                  o.x = pack_bf16x2(__uint_as_float(r[j + 0]), __uint_as_float(r[j + 1]));
                  o.y = pack_bf16x2(__uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
                  o.z = pack_bf16x2(__uint_as_float(r[j + 4]), __uint_as_float(r[j + 5]));
                  o.w = pack_bf16x2(__uint_as_float(r[j + 6]), __uint_as_float(r[j + 7]));
                  *reinterpret_cast<uint4*>(vrow + c0 + j) = o;
                }
              }
            }
            continue;
          }
          // ---- q or k head: rotate-half RoPE on the pairs (d, d + 64)
          bf16* dst = head < p.rope_nh ? reinterpret_cast<bf16*>(p.out) + (long long)(m + roff) * p.ldo + col0
                                       : p.rope_kcache + (page_row + (long long)(head - p.rope_nh) * 64) * 128;
#pragma unroll 1
          for (int c = 0; c < 64; c += CH) {
            uint32_t r1[CH], r2[CH];
            tmem_ld_32x32(taddr + hh * 128 + c, r1);
            tmem_ld_32x32(taddr + hh * 128 + 64 + c, r2);
            tmem_ld_wait();
            if (row_ok) {
#pragma unroll
              for (int j = 0; j < CH; j += 8) {
                const uint4 cu = *reinterpret_cast<const uint4*>(p.rope_cos + (long long)pos * 64 + c + j);
                const uint4 su = *reinterpret_cast<const uint4*>(p.rope_sin + (long long)pos * 64 + c + j);
                const uint32_t cw[4] = {cu.x, cu.y, cu.z, cu.w}, sw[4] = {su.x, su.y, su.z, su.w};
                float o1[8], o2[8];
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                  const float2 cs = unpack_bf16x2(cw[t]), sn = unpack_bf16x2(sw[t]);
                  const float a0 = bf16_round(__uint_as_float(r1[j + 2 * t])), a1 = bf16_round(__uint_as_float(r1[j + 2 * t + 1]));
                  const float b0 = bf16_round(__uint_as_float(r2[j + 2 * t])), b1 = bf16_round(__uint_as_float(r2[j + 2 * t + 1]));
                  o1[2 * t] = bf16_round(a0 * cs.x) + bf16_round(-b0 * sn.x);
                  o1[2 * t + 1] = bf16_round(a1 * cs.y) + bf16_round(-b1 * sn.y);
                  o2[2 * t] = bf16_round(b0 * cs.x) + bf16_round(a0 * sn.x);
                  o2[2 * t + 1] = bf16_round(b1 * cs.y) + bf16_round(a1 * sn.y);
                }
                uint4 w1, w2;
                w1.x = pack_bf16x2(o1[0], o1[1]); w1.y = pack_bf16x2(o1[2], o1[3]); w1.z = pack_bf16x2(o1[4], o1[5]); w1.w = pack_bf16x2(o1[6], o1[7]);
                w2.x = pack_bf16x2(o2[0], o2[1]); w2.y = pack_bf16x2(o2[2], o2[3]); w2.z = pack_bf16x2(o2[4], o2[5]); w2.w = pack_bf16x2(o2[6], o2[7]);
                *reinterpret_cast<uint4*>(dst + c + j) = w1;
                *reinterpret_cast<uint4*>(dst + 64 + c + j) = w2;
              }
            }
          }
        }
      } else {
#pragma unroll 1
      for (int c0 = 0; c0 < k2BlockN; c0 += CH) {
        if (n0 + c0 >= p.N) break;
        float v[CH];
        {
          uint32_t r[CH];
          tmem_ld_32x32(taddr + c0, r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < CH; ++j) v[j] = __uint_as_float(r[j]);
        }
        const int nvalid = min(CH, p.N - (n0 + c0));
        if (m >= M_rt) continue;
        if constexpr (EPI == EPI_STORE || EPI == EPI_STORE_RES) {
          bf16* orow = reinterpret_cast<bf16*>(p.out) + (long long)(m + roff) * p.ldo + n0 + c0;
          const bf16* rrow = (EPI == EPI_STORE_RES) ? p.residual + (long long)(m + roff) * p.ldo + n0 + c0 : nullptr;
          const bool vec = (nvalid == CH) && ((p.ldo & 7) == 0) && ((reinterpret_cast<uintptr_t>(p.out) & 15) == 0);
          if (vec) {
#pragma unroll
            for (int j = 0; j < CH; j += 8) {
              float f[8];
#pragma unroll
              for (int t = 0; t < 8; ++t) f[t] = v[j + t];
              if constexpr (EPI == EPI_STORE_RES) {
                uint4 rr = *reinterpret_cast<const uint4*>(rrow + j);
                const uint32_t rw[4] = {rr.x, rr.y, rr.z, rr.w};
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                  float2 r2 = unpack_bf16x2(rw[t]);
                  f[2 * t] = bf16_round(f[2 * t]) + r2.x;
                  f[2 * t + 1] = bf16_round(f[2 * t + 1]) + r2.y;
                }
              }
              uint4 o;
              o.x = pack_bf16x2(f[0], f[1]); o.y = pack_bf16x2(f[2], f[3]);
              o.z = pack_bf16x2(f[4], f[5]); o.w = pack_bf16x2(f[6], f[7]);
              st_out_v4(orow + j, o);
            }
          } else {
            for (int j = 0; j < nvalid; ++j) {
              float f = v[j];
              if constexpr (EPI == EPI_STORE_RES) f = bf16_round(f) + __bfloat162float(rrow[j]);
              orow[j] = __float2bfloat16_rn(f);
            }
          }
        } else {  // EPI_SWIGLU: columns [c0,c0+16) gate, [c0+16,c0+32) up
          const int oc = (n0 + c0) >> 1;
          bf16* orow = reinterpret_cast<bf16*>(p.out) + (long long)(m + roff) * p.ldo + oc;
          float h[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) h[j] = bf16_round(silu_f(bf16_round(v[j]))) * bf16_round(v[16 + j]);
          if (oc + 16 <= p.out_cols && (p.ldo & 7) == 0) {
            uint4 o0, o1;
            o0.x = pack_bf16x2(h[0], h[1]);   o0.y = pack_bf16x2(h[2], h[3]);
            o0.z = pack_bf16x2(h[4], h[5]);   o0.w = pack_bf16x2(h[6], h[7]);
            o1.x = pack_bf16x2(h[8], h[9]);   o1.y = pack_bf16x2(h[10], h[11]);
            o1.z = pack_bf16x2(h[12], h[13]); o1.w = pack_bf16x2(h[14], h[15]);
            st_out_v4(orow, o0);
            st_out_v4(orow + 8, o1);
          } else {
            for (int j = 0; j < 16 && oc + j < p.out_cols; ++j) orow[j] = __float2bfloat16_rn(h[j]);
          }
        }
      }
      }   // EPI != EPI_ROPE_KV
      tcgen05_fence_before();
      mbar_arrive_leader(&tmem_empty[acc]);
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }

  tcgen05_fence_before();
  cluster_sync_all();   // nobody touches the peer's barriers / TMEM after this point
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc_2sm(tmem_base, 512);
  }
}

}  // namespace b200
