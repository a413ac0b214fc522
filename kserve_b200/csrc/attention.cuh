// Decode attention over the paged KV cache (SURVEY.md §8a row 15: LlamaAttention.forward + SDPA with GQA); the
// prefill attention is the tcgen05 kernel in attention_tc.cuh.
//
//   attn_decode_kernel : one query token per sequence, split over the KV length (flash-decoding),
//                        the G query heads that share a KV head are packed into the MMA M dimension;
//                        the last split CTA to arrive merges the per-split partials.
//
// KV pages are [page][kv_head][64 tokens][128 dims] bf16, so one (page, kv_head) tile is a contiguous
// 16 KB block that is staged with 128-bit cp.async into XOR-swizzled shared memory and consumed with
// ldmatrix + mma.sync.m16n8k16 (fp32 softmax / accumulation).  The warp-level MMA path suffices here: the
// kernel is HBM-bound (the KV read).
#pragma once
#include "common.cuh"
#include "ops.cuh"

namespace b200 {

constexpr int kAttnThreads = 128;
constexpr int kDecStages = 3;   // cp.async ring of the decode kernel: two KV tiles (64 KB) in flight per CTA
constexpr int kTileBytes = kPageTokens * kHeadDim * 2;  // 16 KB

// byte offset of 16-byte chunk `c` (0..15) of row `r` in a [rows][128] bf16 tile with XOR swizzle
__device__ __forceinline__ uint32_t swz(int r, int c) { return (uint32_t)(r * 256 + ((c ^ (r & 7)) << 4)); }

// stage one 64x128 bf16 tile (contiguous in global memory) into swizzled smem; 128 threads
__device__ __forceinline__ void load_kv_tile(uint32_t sdst, const bf16* gsrc) {
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    const int idx = threadIdx.x + it * kAttnThreads;
    const int r = idx >> 4, c = idx & 15;
    cp_async_16(sdst + swz(r, c), gsrc + r * kHeadDim + c * 8, true);
  }
}

struct AttnDecodeParams {
  const bf16* q; long long ldq;        // [B][ldq] roped queries of the current token
  bf16* out; long long ldo;            // [B][ldo]
  const bf16* kcache; const bf16* vcache;
  const int32_t* page_table; int max_pages;
  const int32_t* seq_slot;             // [B]
  const int32_t* tok_pos;              // [B] position of the current token; context = pos + 1
  int nh, nkv, G, splits;
  float* part_o;                       // [B*nkv][splits][G][128]
  float* part_ml;                      // [B*nkv][splits][G][2]
  float scale_log2;
  // Fused RoPE + KV append: when fuse_rope != 0 the kernel reads the raw QKV projection of the current token
  // (bf16 [B][ld_qkv], or fp32 split-K partials), applies rotate-half RoPE with the same rounding points as
  // rope_kv_kernel, uses the roped q / new k,v directly and appends k,v to the paged cache — one kernel
  // boundary less on the decode critical path.
  int fuse_rope;
  const bf16* qkv; long long ld_qkv;
  const float* qkv_partial; int qkv_splits; long long qkv_split_stride; long long ld_qkv_partial;
  const bf16* cos_tab; const bf16* sin_tab;
  bf16* kcache_w; bf16* vcache_w;
  // splits > 1: per-(sequence, kv head) arrival counters (zero between launches; required).  The LAST split CTA to
  // arrive merges the partials itself (in split order: deterministic) — no separate combine kernel on the
  // tensor-parallel decode path, where few (sequence, kv head) pairs per GPU force the split.
  int* split_counter;
};

// called by every CTA of a split launch after its partial (or its "empty" marker) is in global memory
__device__ __forceinline__ void attn_decode_arrive_and_merge(const AttnDecodeParams& p, int bh, int b, int kvh) {
  __shared__ int s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(p.split_counter + bh, 1) == p.splits - 1) ? 1 : 0;
  __syncthreads();
  if (!s_last) return;
  if (threadIdx.x == 0) p.split_counter[bh] = 0;
  __threadfence();
  const int G = p.G, d = threadIdx.x;
  const long long base = (long long)bh * p.splits * G;
  for (int r = 0; r < G; ++r) {
    float M = -INFINITY;
    for (int s = 0; s < p.splits; ++s) M = fmaxf(M, __ldcg(p.part_ml + (base + (long long)s * G + r) * 2));
    float L = 0.f, acc = 0.f;
    for (int s = 0; s < p.splits; ++s) {
      const long long row = base + (long long)s * G + r;
      const float ms = __ldcg(p.part_ml + row * 2);
      const float f = (ms == -INFINITY) ? 0.f : exp2f(ms - M);
      L += __ldcg(p.part_ml + row * 2 + 1) * f;
      acc += __ldcg(p.part_o + row * kHeadDim + d) * f;
    }
    p.out[(long long)b * p.ldo + (kvh * G + r) * kHeadDim + d] = __float2bfloat16_rn(acc / L);
  }
}

__global__ void __launch_bounds__(kAttnThreads) attn_decode_kernel(const AttnDecodeParams p) {
  TraceScope _ts(TK_ATTN_DECODE);
  pdl_launch_dependents();
  pdl_wait();
  _ts.mark();
  extern __shared__ __align__(1024) uint8_t smem[];
  const int bh = blockIdx.x, split = blockIdx.y;
  const int b = bh / p.nkv, kvh = bh - b * p.nkv;
  const int ctx = p.tok_pos[b] + 1;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int G = p.G;
  const int ntiles = (ctx + 63) >> 6;
  const int per = (ntiles + p.splits - 1) / p.splits;
  const int t0 = split * per, t1 = min(ntiles, t0 + per);
  float* po = p.part_o + ((long long)bh * p.splits + split) * G * kHeadDim;
  float* pml = p.part_ml + ((long long)bh * p.splits + split) * G * 2;
  if (t0 >= t1) {  // empty split (uniform for the CTA)
    if (p.splits > 1 && threadIdx.x < G) { pml[threadIdx.x * 2] = -INFINITY; pml[threadIdx.x * 2 + 1] = 0.f; }
    if (p.splits > 1 && p.split_counter) attn_decode_arrive_and_merge(p, bh, b, kvh);
    return;
  }
  const uint32_t sQ = smem_u32(smem);       // 16 rows x 256 B = 4 KB
  const uint32_t sK = sQ + 4096;                      // kDecStages x 16 KB
  const uint32_t sV = sK + kDecStages * kTileBytes;   // kDecStages x 16 KB
  const int32_t* pages = p.page_table + (long long)p.seq_slot[b] * p.max_pages;
  const long long tile_stride = (long long)p.nkv * kPageTokens * kHeadDim;
  const long long head_off = (long long)kvh * kPageTokens * kHeadDim;

  const int pos = ctx - 1;
  const int jt = pos >> 6;  // KV tile that receives the current token
  float* s_raw = reinterpret_cast<float*>(smem + 4096 + 2 * kDecStages * kTileBytes);   // [(G+2)][128] fp32
  bf16* s_newk = reinterpret_cast<bf16*>(s_raw + 10 * kHeadDim);           // [128]
  bf16* s_newv = s_newk + kHeadDim;                                          // [128]
  // fill the ring: kDecStages-1 tiles in flight before any compute (one commit group per ring slot, empty or not)
#pragma unroll
  for (int st = 0; st < kDecStages - 1; ++st) {
    if (t0 + st < t1) {
      const long long pg = pages[t0 + st];
      load_kv_tile(sK + st * kTileBytes, p.kcache + pg * tile_stride + head_off);
      load_kv_tile(sV + st * kTileBytes, p.vcache + pg * tile_stride + head_off);
    }
    cp_async_commit();
  }
  if (p.fuse_rope) {
    const int ngroups = (G + 2) * 16;
    for (int gi = threadIdx.x; gi < ngroups; gi += kAttnThreads) {
      const int hl = gi >> 4, c = (gi & 15) * 8;
      const int col = (hl < G ? (kvh * G + hl) : (hl == G ? p.nh + kvh : p.nh + p.nkv + kvh)) * kHeadDim + c;
      float f[8];
      if (p.qkv_partial) {
        float a[8];
        sum_partials8(p.qkv_partial + (long long)b * p.ld_qkv_partial + col, p.qkv_splits, p.qkv_split_stride, a);
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] = bf16_round(a[i]);
      } else {
        uint4 u = *reinterpret_cast<const uint4*>(p.qkv + (long long)b * p.ld_qkv + col);
        const uint32_t uw[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float2 v2 = unpack_bf16x2(uw[i]);
          f[2 * i] = v2.x;
          f[2 * i + 1] = v2.y;
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) s_raw[hl * kHeadDim + c + i] = f[i];
    }
    __syncthreads();
    const int items = (G + 1) * 8 + 16;   // roped heads (q heads + k) x 8 threads, then 16 threads copy v
    for (int it = threadIdx.x; it < items; it += kAttnThreads) {
      if (it < (G + 1) * 8) {
        const int hl = it >> 3, c = (it & 7) * 8;
        float cs[8], sn[8], o1[8], o2[8];
        {
          uint4 cu = *reinterpret_cast<const uint4*>(p.cos_tab + (long long)pos * 64 + c);
          uint4 su = *reinterpret_cast<const uint4*>(p.sin_tab + (long long)pos * 64 + c);
          const uint32_t cw[4] = {cu.x, cu.y, cu.z, cu.w}, sw[4] = {su.x, su.y, su.z, su.w};
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            float2 a2 = unpack_bf16x2(cw[i]), b2 = unpack_bf16x2(sw[i]);
            cs[2 * i] = a2.x; cs[2 * i + 1] = a2.y;
            sn[2 * i] = b2.x; sn[2 * i + 1] = b2.y;
          }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float x1 = s_raw[hl * kHeadDim + c + i], x2 = s_raw[hl * kHeadDim + c + 64 + i];
          o1[i] = bf16_round(x1 * cs[i]) + bf16_round(-x2 * sn[i]);
          o2[i] = bf16_round(x2 * cs[i]) + bf16_round(x1 * sn[i]);
        }
        if (hl < G) {
          *reinterpret_cast<uint4*>(smem + swz(hl, c >> 3)) = pack8(o1);
          *reinterpret_cast<uint4*>(smem + swz(hl, (c >> 3) + 8)) = pack8(o2);
        } else {
          *reinterpret_cast<uint4*>(s_newk + c) = pack8(o1);
          *reinterpret_cast<uint4*>(s_newk + c + 64) = pack8(o2);
        }
      } else {
        const int c = (it - (G + 1) * 8) * 8;
        float f[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] = s_raw[(G + 1) * kHeadDim + c + i];
        *reinterpret_cast<uint4*>(s_newv + c) = pack8(f);
      }
    }
    // padding rows of the 16-row Q tile
    for (int idx = threadIdx.x; idx < (16 - G) * 16; idx += kAttnThreads)
      *reinterpret_cast<uint4*>(smem + swz(G + (idx >> 4), idx & 15)) = make_uint4(0, 0, 0, 0);
    __syncthreads();
    if (jt >= t0 && jt < t1 && threadIdx.x < 32) {   // the split that owns the current token appends it to the cache
      const int c = (threadIdx.x & 15) * 8, slot = pos & 63;
      const long long off = (long long)pages[jt] * tile_stride + head_off + slot * kHeadDim + c;
      if (threadIdx.x < 16) *reinterpret_cast<uint4*>(p.kcache_w + off) = *reinterpret_cast<const uint4*>(s_newk + c);
      else *reinterpret_cast<uint4*>(p.vcache_w + off) = *reinterpret_cast<const uint4*>(s_newv + c);
    }
  } else {
    // Q: G rows valid, the rest zero
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int idx = threadIdx.x + it * kAttnThreads;
      const int r = idx >> 4, c = idx & 15;
      const bool valid = r < G;
      const bf16* src = p.q + (long long)b * p.ldq + (kvh * G + (valid ? r : 0)) * kHeadDim + c * 8;
      cp_async_16(sQ + swz(r, c), src, valid);
    }
    cp_async_commit();
    cp_async_wait<0>();   // (test path) keep the group accounting of the ring simple
  }

  uint32_t qf[8][4];
  float o[16][4];
#pragma unroll
  for (int i = 0; i < 16; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
  float m0 = -INFINITY, l0 = 0.f;  // only row g (< 8) matters: rows >= G are padding

  for (int j = t0; j < t1; ++j) {
    const int buf = (j - t0) % kDecStages;
    cp_async_wait<kDecStages - 2>();   // tile j has landed
    __syncthreads();                   // ... for every thread, and everyone is done with tile j-1's slot
    {
      const int jn = j + kDecStages - 1;   // refill the slot tile j-1 used
      if (jn < t1) {
        const int nb = (jn - t0) % kDecStages;
        const long long pg = pages[jn];
        load_kv_tile(sK + nb * kTileBytes, p.kcache + pg * tile_stride + head_off);
        load_kv_tile(sV + nb * kTileBytes, p.vcache + pg * tile_stride + head_off);
      }
      cp_async_commit();
    }
    if (j == t0) {
#pragma unroll
      for (int ks = 0; ks < 8; ++ks)
        ldmatrix_x4(qf[ks], sQ + swz((lane & 7) + 8 * ((lane >> 3) & 1), 2 * ks + (lane >> 4)));
    }
    const uint32_t sKb = sK + buf * kTileBytes, sVb = sV + buf * kTileBytes;
    if (p.fuse_rope && j == jt) {   // the row of the current token is not in the cache copy that was just staged
      if (threadIdx.x < 32) {
        const int c = threadIdx.x & 15, slot = pos & 63;
        uint8_t* base = smem + 4096 + (threadIdx.x < 16 ? 0 : kDecStages * kTileBytes) + buf * kTileBytes;
        *reinterpret_cast<uint4*>(base + swz(slot, c)) =
            *reinterpret_cast<const uint4*>((threadIdx.x < 16 ? s_newk : s_newv) + c * 8);
      }
      __syncthreads();
    }
    float s[2][4];
    s[0][0] = s[0][1] = s[0][2] = s[0][3] = 0.f;
    s[1][0] = s[1][1] = s[1][2] = s[1][3] = 0.f;
    const int trow = warp * 16;  // this warp's 16 tokens of the tile
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      uint32_t bfr[4];
      ldmatrix_x4(bfr, sKb + swz(trow + (lane & 7) + 8 * (lane >> 4), 2 * ks + ((lane >> 3) & 1)));
      mma_m16n8k16_bf16(s[0], qf[ks], bfr[0], bfr[1]);
      mma_m16n8k16_bf16(s[1], qf[ks], bfr[2], bfr[3]);
    }
    float mx = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int kp = j * 64 + trow + nt * 8 + 2 * t + e;
        float v = s[nt][e] * p.scale_log2;
        if (kp >= ctx) v = -INFINITY;
        s[nt][e] = v;
        mx = fmaxf(mx, v);
      }
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
    const float mn = fmaxf(m0, mx);
    const float msafe = (mn == -INFINITY) ? 0.f : mn;  // whole 16-token slice masked and nothing seen yet
    const float c0 = exp2f(m0 - msafe);
    m0 = mn;
    l0 *= c0;
#pragma unroll
    for (int i = 0; i < 16; ++i) { o[i][0] *= c0; o[i][1] *= c0; }
    float pr[2][2];
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) {
      pr[nt][0] = exp2f(s[nt][0] - msafe);
      pr[nt][1] = exp2f(s[nt][1] - msafe);
      l0 += pr[nt][0] + pr[nt][1];
    }
    uint32_t a[4];
    a[0] = pack_bf16x2(pr[0][0], pr[0][1]);
    a[1] = 0u;  // rows 8..15 are padding
    a[2] = pack_bf16x2(pr[1][0], pr[1][1]);
    a[3] = 0u;
#pragma unroll
    for (int dp = 0; dp < 8; ++dp) {
      uint32_t bfr[4];
      ldmatrix_x4_trans(bfr, sVb + swz(trow + (lane & 7) + 8 * ((lane >> 3) & 1), 2 * dp + (lane >> 4)));
      mma_m16n8k16_bf16(o[2 * dp], a, bfr[0], bfr[1]);
      mma_m16n8k16_bf16(o[2 * dp + 1], a, bfr[2], bfr[3]);
    }
  }
  cp_async_wait<0>();
  __syncthreads();   // all warps done with the ring before it is reused for the merge
  // ---- merge the 4 warps (each saw a disjoint quarter of every tile) through shared memory
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
  l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  float* sm_m = reinterpret_cast<float*>(smem + 4096);  // [4][8]
  float* sm_l = sm_m + 32;                               // [4][8]
  float* sm_o = sm_l + 32;                               // [4][8][128]
  if (t == 0) { sm_m[warp * 8 + g] = m0; sm_l[warp * 8 + g] = l0; }
#pragma unroll
  for (int nt = 0; nt < 16; ++nt) {
    sm_o[(warp * 8 + g) * kHeadDim + nt * 8 + 2 * t] = o[nt][0];
    sm_o[(warp * 8 + g) * kHeadDim + nt * 8 + 2 * t + 1] = o[nt][1];
  }
  __syncthreads();
  const int d = threadIdx.x;  // 128 threads <-> 128 dims
  for (int r = 0; r < G; ++r) {
    float M = -INFINITY;
#pragma unroll
    for (int w = 0; w < 4; ++w) M = fmaxf(M, sm_m[w * 8 + r]);
    float L = 0.f, acc = 0.f;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      const float mw = sm_m[w * 8 + r];
      const float f = (mw == -INFINITY) ? 0.f : exp2f(mw - M);
      L += sm_l[w * 8 + r] * f;
      acc += sm_o[(w * 8 + r) * kHeadDim + d] * f;
    }
    if (p.splits == 1) {
      p.out[(long long)b * p.ldo + (kvh * G + r) * kHeadDim + d] = __float2bfloat16_rn(acc / L);
    } else {
      po[r * kHeadDim + d] = acc;
      if (d == 0) { pml[r * 2] = M; pml[r * 2 + 1] = L; }
    }
  }
  if (p.splits > 1 && p.split_counter) attn_decode_arrive_and_merge(p, bh, b, kvh);
}

}  // namespace b200
