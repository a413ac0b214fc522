// HBM-bound element-wise / reduction kernels of the LLM path (embedding gather, RMSNorm with fused
// residual / split-K reduce, RoPE + paged-KV append, greedy argmax, per-step sequence bookkeeping).
// All are coalesced 128-bit accesses; the arithmetic reproduces the rounding points of the HF bf16
// modules the reference executes (modeling_llama.py:62-67 RMSNorm, :146-168 RoPE).
#pragma once
#include "common.cuh"
#include "p2p_base.cuh"

namespace b200 {

constexpr int kPageTokens = 64;   // tokens per KV page == KV tile of the attention kernels
constexpr int kHeadDim = 128;

// -------------------------------------------------------------------------------------------------
// embedding gather: x[t][:] = table[tok[t]][:]
// -------------------------------------------------------------------------------------------------
__global__ void embed_gather_kernel(const int32_t* __restrict__ tokens, const bf16* __restrict__ table,
                                    bf16* __restrict__ x, int H, int vocab_rows) {
  TraceScope _ts(TK_EMBED);
  pdl_launch_dependents();
  pdl_wait();
  _ts.mark();
  const int t = blockIdx.x;
  int tok = tokens[t];
  tok = max(0, min(tok, vocab_rows - 1));
  const uint4* src = reinterpret_cast<const uint4*>(table + (long long)tok * H);
  uint4* dst = reinterpret_cast<uint4*>(x + (long long)t * H);
  for (int i = threadIdx.x; i < H / 8; i += blockDim.x) dst[i] = ld_nc_v4(src + i);
}

__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) red[w] = v;
  __syncthreads();
  const int nw = blockDim.x >> 5;
  float t = (l < nw) ? red[l] : 0.f;
  t = warp_sum(t);
  __syncthreads();
  return t;
}

// -------------------------------------------------------------------------------------------------
// RMSNorm (LlamaRMSNorm.forward): xn = w * bf16( x * rsqrt(mean(x^2) + eps) ), fp32 internally.
// MODE 0: plain.                         x read-only.
// MODE 1: x += bf16(sum_s partial[s])    (split-K fp32 partials of the preceding row-parallel GEMM)
// MODE 2: x += y (bf16)                  (already reduced, e.g. after the TP all-reduce)
// In modes 1/2 the updated residual stream x is written back (bf16), then normalised.
// One CTA per row; the row lives in shared memory as fp32 between the two passes.
// -------------------------------------------------------------------------------------------------
// sum of split-K partials for 8 consecutive elements; all loads of up to 4 splits are issued before the first
// add (memory-level parallelism: this sits on the decode critical path), accumulation order is s = 0,1,2,...
__device__ __forceinline__ void sum_partials8(const float* __restrict__ base, int splits, long long split_stride, float (&a)[8]) {
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = 0.f;
  for (int s0 = 0; s0 < splits; s0 += 4) {
    float4 v[4][2];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (s0 + j < splits) {
        const float4* pp = reinterpret_cast<const float4*>(base + (long long)(s0 + j) * split_stride);
        v[j][0] = pp[0];
        v[j][1] = pp[1];
      } else {
        v[j][0] = make_float4(0.f, 0.f, 0.f, 0.f);
        v[j][1] = v[j][0];
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (s0 + j < splits) {
        a[0] += v[j][0].x; a[1] += v[j][0].y; a[2] += v[j][0].z; a[3] += v[j][0].w;
        a[4] += v[j][1].x; a[5] += v[j][1].y; a[6] += v[j][1].z; a[7] += v[j][1].w;
      }
    }
  }
}

constexpr int kNormThreads = 512;
__device__ int g_trace_split = 0;
__device__ __forceinline__ bool getenv_trace_split() { return g_trace_split != 0; }

template <int MODE>
__global__ void __launch_bounds__(kNormThreads)
rmsnorm_kernel(bf16* __restrict__ x, const bf16* __restrict__ w, bf16* __restrict__ xn, int H, float eps,
               const float* __restrict__ partial, int splits, long long split_stride, long long ld_partial,
               const bf16* __restrict__ y) {
  TraceScope _ts(TK_RMSNORM);
  pdl_launch_dependents();
  extern __shared__ float row[];  // H floats + 32
  float* red = row + H;
  const int r = blockIdx.x;
  bf16* xr = x + (long long)r * H;
  // the norm weight does not depend on the previous kernel: fetch it before the dependency wait
  const bool single = H <= (int)blockDim.x * 8;
  uint4 wpre = make_uint4(0, 0, 0, 0);
  if (single && (int)threadIdx.x * 8 < H) wpre = *reinterpret_cast<const uint4*>(w + threadIdx.x * 8);
  pdl_wait();
  _ts.mark();
  float ss = 0.f;
  for (int i = threadIdx.x * 8; i < H; i += blockDim.x * 8) {
    uint4 u = *reinterpret_cast<const uint4*>(xr + i);
    float f[8];
    if constexpr (MODE == 1) {
      float a[8];
      sum_partials8(partial + (long long)r * ld_partial + i, splits, split_stride, a);
      const uint32_t uw[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        float2 p2 = unpack_bf16x2(uw[t]);
        f[2 * t] = bf16_round(p2.x + bf16_round(a[2 * t]));
        f[2 * t + 1] = bf16_round(p2.y + bf16_round(a[2 * t + 1]));
      }
    } else if constexpr (MODE == 2) {
      uint4 yu = *reinterpret_cast<const uint4*>(y + (long long)r * H + i);
      const uint32_t uw[4] = {u.x, u.y, u.z, u.w}, yw[4] = {yu.x, yu.y, yu.z, yu.w};
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        float2 p2 = unpack_bf16x2(uw[t]), q2 = unpack_bf16x2(yw[t]);
        f[2 * t] = bf16_round(p2.x + q2.x);
        f[2 * t + 1] = bf16_round(p2.y + q2.y);
      }
    } else {
      const uint32_t uw[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        float2 p2 = unpack_bf16x2(uw[t]);
        f[2 * t] = p2.x;
        f[2 * t + 1] = p2.y;
      }
    }
    if constexpr (MODE != 0) {
      uint4 o;
      o.x = pack_bf16x2(f[0], f[1]); o.y = pack_bf16x2(f[2], f[3]);
      o.z = pack_bf16x2(f[4], f[5]); o.w = pack_bf16x2(f[6], f[7]);
      *reinterpret_cast<uint4*>(xr + i) = o;
    }
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      row[i + t] = f[t];
      ss += f[t] * f[t];
    }
  }
  if (getenv_trace_split()) _ts.mark();
  const float tot = block_sum(ss, red);
  const float rs = 1.0f / sqrtf(tot / (float)H + eps);  // IEEE sqrt + div, as torch.rsqrt on CPU
  bf16* o = xn + (long long)r * H;
  for (int i = threadIdx.x * 8; i < H; i += blockDim.x * 8) {
    uint4 wu = single ? wpre : *reinterpret_cast<const uint4*>(w + i);
    const uint32_t ww[4] = {wu.x, wu.y, wu.z, wu.w};
    float g[8];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      float2 w2 = unpack_bf16x2(ww[t]);
      g[2 * t] = w2.x * bf16_round(row[i + 2 * t] * rs);          // cast to bf16 BEFORE the weight multiply
      g[2 * t + 1] = w2.y * bf16_round(row[i + 2 * t + 1] * rs);
    }
    uint4 ov;
    ov.x = pack_bf16x2(g[0], g[1]); ov.y = pack_bf16x2(g[2], g[3]);
    ov.z = pack_bf16x2(g[4], g[5]); ov.w = pack_bf16x2(g[6], g[7]);
    *reinterpret_cast<uint4*>(o + i) = ov;
  }
}

// Many-row variant for the prefill (thousands of rows): one WARP per row, the whole row in registers (NV 16-byte
// vectors per lane, all loads issued before the first use), warp-shuffle reduction, no shared memory, no block
// barriers; 8 rows per CTA.  The one-CTA-per-row kernel above spends most of its time launching 32768 CTAs and in two
// block-wide barriers per row (r01 ncu: 0.47 of the HBM peak).  MODE 0: xn = norm(x) * w;  MODE 2: x += y first.
// Same rounding points; the sum of squares is accumulated lane-wise then across lanes (fp32) instead of thread-wise
// then across warps.
template <int MODE, int NV>
__global__ void __launch_bounds__(256)
rmsnorm_rows_kernel(bf16* __restrict__ x, const bf16* __restrict__ w, bf16* __restrict__ xn, int rows, float eps,
                    const bf16* __restrict__ y) {
  TraceScope _ts(TK_RMSNORM);
  pdl_launch_dependents();
  pdl_wait();
  _ts.mark();
  constexpr int H = NV * 256;
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= rows) return;
  bf16* xr = x + (long long)r * H;
  uint4 u[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) u[v] = *reinterpret_cast<const uint4*>(xr + (v * 32 + lane) * 8);
  if constexpr (MODE == 2) {
    uint4 yu[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) yu[v] = ld_nc_v4(y + (long long)r * H + (v * 32 + lane) * 8);
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const uint32_t uw[4] = {u[v].x, u[v].y, u[v].z, u[v].w}, yw[4] = {yu[v].x, yu[v].y, yu[v].z, yu[v].w};
      uint32_t o[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        float2 p2 = unpack_bf16x2(uw[t]), q2 = unpack_bf16x2(yw[t]);
        o[t] = pack_bf16x2(p2.x + q2.x, p2.y + q2.y);
      }
      u[v] = make_uint4(o[0], o[1], o[2], o[3]);
      *reinterpret_cast<uint4*>(xr + (v * 32 + lane) * 8) = u[v];
    }
  }
  float ss = 0.f;
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const uint32_t uw[4] = {u[v].x, u[v].y, u[v].z, u[v].w};
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      float2 p2 = unpack_bf16x2(uw[t]);
      ss += p2.x * p2.x;
      ss += p2.y * p2.y;
    }
  }
  const float tot = warp_sum(ss);
  const float rs = 1.0f / sqrtf(tot / (float)H + eps);
  bf16* o = xn + (long long)r * H;
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const uint4 wu = *reinterpret_cast<const uint4*>(w + (v * 32 + lane) * 8);
    const uint32_t uw[4] = {u[v].x, u[v].y, u[v].z, u[v].w}, ww[4] = {wu.x, wu.y, wu.z, wu.w};
    uint32_t ov[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      float2 p2 = unpack_bf16x2(uw[t]), w2 = unpack_bf16x2(ww[t]);
      ov[t] = pack_bf16x2(w2.x * bf16_round(p2.x * rs), w2.y * bf16_round(p2.y * rs));   // cast to bf16 BEFORE the weight multiply
    }
    *reinterpret_cast<uint4*>(o + (v * 32 + lane) * 8) = make_uint4(ov[0], ov[1], ov[2], ov[3]);
  }
}

// sum split-K partials into a bf16 matrix (used before the TP all-reduce): y[r][i] = bf16(sum_s p[s][r][i])
__global__ void reduce_partials_kernel(const float* __restrict__ partial, int splits, long long split_stride,
                                       long long ld_partial, bf16* __restrict__ y, int H) {
  TraceScope _ts(TK_OTHER);
  pdl_launch_dependents();
  pdl_wait();
  _ts.mark();
  const int r = blockIdx.x;
  for (int i = threadIdx.x; i < H; i += blockDim.x) {
    float a = 0.f;
    for (int s = 0; s < splits; ++s) a += partial[s * split_stride + (long long)r * ld_partial + i];
    y[(long long)r * H + i] = __float2bfloat16_rn(a);
  }
}

// -------------------------------------------------------------------------------------------------
// RoPE (apply_rotary_pos_emb, rotate-half form, every product/sum rounded to bf16 as the bf16 HF
// module does) fused with the paged KV-cache append.  One CTA per token.
//   qkv      : bf16 [T][ld] (q heads | k heads | v heads)   or, when `partial` != null,
//              fp32 split-K partials [splits][T][ld_partial] of the same matrix.
//   q_out    : bf16 [T][ldq]  (may alias qkv for the in-place prefill case)
//   K/V cache: [page][kv_head][64][128] per layer; page = page_table[seq][pos / 64]
// -------------------------------------------------------------------------------------------------
struct RopeKvParams {
  const bf16* qkv; long long ld;
  const float* partial; int splits; long long split_stride; long long ld_partial;
  bf16* q_out; long long ldq;
  bf16* kcache; bf16* vcache;            // this layer's base
  const int32_t* page_table; int max_pages;  // [seq][max_pages]
  const int32_t* tok_seq;                // [T] sequence slot of each token
  const int32_t* tok_pos;                // [T] position within the sequence
  const bf16* cos_tab; const bf16* sin_tab;  // [max_pos][64]
  int nh, nkv;
  int T;                                 // tokens in this launch (one CTA each)
};

__device__ __forceinline__ void load8(const RopeKvParams& p, int t, int col, float (&f)[8]) {
  if (p.partial) {
    float a[8];
    sum_partials8(p.partial + (long long)t * p.ld_partial + col, p.splits, p.split_stride, a);
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] = bf16_round(a[i]);
  } else {
    uint4 u = *reinterpret_cast<const uint4*>(p.qkv + (long long)t * p.ld + col);
    const uint32_t uw[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float2 v = unpack_bf16x2(uw[i]);
      f[2 * i] = v.x;
      f[2 * i + 1] = v.y;
    }
  }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 o;
  o.x = pack_bf16x2(f[0], f[1]); o.y = pack_bf16x2(f[2], f[3]);
  o.z = pack_bf16x2(f[4], f[5]); o.w = pack_bf16x2(f[6], f[7]);
  return o;
}

__global__ void __launch_bounds__(512) rope_kv_kernel(const RopeKvParams p) {
  TraceScope _ts(TK_ROPE);
  pdl_launch_dependents();
  pdl_wait();
  _ts.mark();
  const int rope_items = (p.nh + p.nkv) * 8;   // 8 threads per roped head (each 8 dims of both halves)
  const int copy_items = p.nkv * 16;           // 16 threads per V head
  for (int t = blockIdx.x; t < p.T; t += gridDim.x) {   // launched with one CTA per token
  const int pos = p.tok_pos[t];
  const int seq = p.tok_seq[t];
  const int page = p.page_table[(long long)seq * p.max_pages + pos / kPageTokens];
  const int slot = pos % kPageTokens;
  for (int it = threadIdx.x; it < rope_items + copy_items; it += blockDim.x) {
    if (it < rope_items) {
      const int head = it >> 3, c = (it & 7) * 8;  // dims [c, c+8) and [c+64, c+72)
      const int col = head * kHeadDim;
      float x1[8], x2[8], cs[8], sn[8];
      load8(p, t, col + c, x1);
      load8(p, t, col + c + 64, x2);
      {
        uint4 cu = *reinterpret_cast<const uint4*>(p.cos_tab + (long long)pos * 64 + c);
        uint4 su = *reinterpret_cast<const uint4*>(p.sin_tab + (long long)pos * 64 + c);
        const uint32_t cw[4] = {cu.x, cu.y, cu.z, cu.w}, sw[4] = {su.x, su.y, su.z, su.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float2 a = unpack_bf16x2(cw[i]), b = unpack_bf16x2(sw[i]);
          cs[2 * i] = a.x; cs[2 * i + 1] = a.y;
          sn[2 * i] = b.x; sn[2 * i + 1] = b.y;
        }
      }
      float o1[8], o2[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        o1[i] = bf16_round(x1[i] * cs[i]) + bf16_round(-x2[i] * sn[i]);
        o2[i] = bf16_round(x2[i] * cs[i]) + bf16_round(x1[i] * sn[i]);
      }
      if (head < p.nh) {
        bf16* q = p.q_out + (long long)t * p.ldq + head * kHeadDim;
        *reinterpret_cast<uint4*>(q + c) = pack8(o1);
        *reinterpret_cast<uint4*>(q + c + 64) = pack8(o2);
      } else {
        const int kvh = head - p.nh;
        bf16* k = p.kcache + ((long long)page * p.nkv + kvh) * (kPageTokens * kHeadDim) + slot * kHeadDim;
        *reinterpret_cast<uint4*>(k + c) = pack8(o1);
        *reinterpret_cast<uint4*>(k + c + 64) = pack8(o2);
      }
    } else {
      const int j = it - rope_items;
      const int kvh = j >> 4, c = (j & 15) * 8;
      float f[8];
      load8(p, t, (p.nh + p.nkv + kvh) * kHeadDim + c, f);
      bf16* v = p.vcache + ((long long)page * p.nkv + kvh) * (kPageTokens * kHeadDim) + slot * kHeadDim;
      *reinterpret_cast<uint4*>(v + c) = pack8(f);
    }
  }
  }
}

// SwiGLU over split-K partials of the interleaved gate/up projection (used when the per-GPU weight has too few
// 128-row tiles to fill the SMs without split-K, i.e. under tensor parallelism):
//   h[r][f] = bf16( bf16(silu(bf16(sum_s gate_s))) * bf16(sum_s up_s) ),  partial columns interleaved {16 gate,16 up}
__global__ void __launch_bounds__(512)
swiglu_reduce_kernel(const float* __restrict__ partial, int splits, long long split_stride, long long ld_partial,
                     bf16* __restrict__ h, int I) {
  TraceScope _ts(TK_OTHER);
  pdl_launch_dependents();
  pdl_wait();
  _ts.mark();
  const int r = blockIdx.x;
  for (int f = threadIdx.x * 8; f < I; f += blockDim.x * 8) {
    const int gcol = ((f >> 4) << 5) + (f & 15);
    float g[8], u[8], o[8];
    sum_partials8(partial + (long long)r * ld_partial + gcol, splits, split_stride, g);
    sum_partials8(partial + (long long)r * ld_partial + gcol + 16, splits, split_stride, u);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float gg = bf16_round(g[i]);
      o[i] = bf16_round(__fdividef(gg, 1.0f + __expf(-gg))) * bf16_round(u[i]);
    }
    *reinterpret_cast<uint4*>(h + (long long)r * I + f) = pack8(o);
  }
}

// -------------------------------------------------------------------------------------------------
// greedy argmax over bf16 logits (== argmax of logits.float(), transformers generation/utils.py:2762,
// 2793); ties -> lowest index like torch.argmax on CPU.  Also emits (max, idx) for the vocab-parallel case.
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
argmax_kernel(const bf16* __restrict__ logits, long long ld, int V, int idx_offset, float* __restrict__ out_val,
              int32_t* __restrict__ out_idx, const P2P pp, int use_p2p) {
  TraceScope _ts(TK_ARGMAX);
  pdl_launch_dependents();
  pdl_wait();
  _ts.mark();
  // grid = (B, chunks): chunk c scans [c*per, (c+1)*per) of the row and writes candidate slot [c][b]; the step
  // kernel merges the slots exactly like the per-rank candidates of the vocabulary-parallel case
  const int b = blockIdx.x, B = gridDim.x;
  const int per = (V + gridDim.y - 1) / gridDim.y;
  const int v0 = blockIdx.y * per, v1 = min(V, v0 + per);
  const bf16* row = logits + (long long)b * ld;
  float best = -INFINITY;
  int bi = 0x7fffffff;
  for (int i = v0 + threadIdx.x; i < v1; i += blockDim.x) {
    const float v = __bfloat162float(row[i]);
    if (v > best || (v == best && i < bi)) { best = v; bi = i; }
  }
  __shared__ float sv[32];
  __shared__ int si[32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
  }
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { sv[w] = best; si[w] = bi; }
  __syncthreads();
  if (w == 0) {
    const int nw = blockDim.x >> 5;
    best = (l < nw) ? sv[l] : -INFINITY;
    bi = (l < nw) ? si[l] : 0x7fffffff;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
    }
    if (l == 0) {
      const int gi = (bi == 0x7fffffff) ? bi : bi + idx_offset;
      out_val[blockIdx.y * B + b] = best;
      out_idx[blockIdx.y * B + b] = gi;
      if (use_p2p) push_candidate(pp, b, best, gi);   // vocab-parallel (single chunk): hand the candidate to every rank
    }
  }
}

// -------------------------------------------------------------------------------------------------
// Per-step sequence bookkeeping, entirely on device so the host never synchronises per token
// (the reference syncs every step: generation/utils.py:2804-2805).  One CTA.
//   * merges vocab-parallel (val, idx) candidates [ranks][B] (ranks == 1 without TP)
//   * forced tokens (teacher forcing in tests), EOS -> finished rows emit pad (utils.py:2796-2797)
//   * appends the token to out_tokens[b][step], feeds it back as next input, cur_len[b] += 1
//   * batch-wide stop sequences (stop_sequence_stopping_criteria.py:36-48) and max_new_tokens
// -------------------------------------------------------------------------------------------------
struct StepState {
  int32_t step;           // number of tokens generated so far (per row; all rows advance together)
  int32_t done;           // 1 once generation ended
  int32_t stop_triggered; // 1 iff a stop sequence matched (finish_reason == "stop")
  int32_t max_new;
};

struct StepParams {
  const float* cand_val; const int32_t* cand_idx; int ranks; int B;
  const int32_t* forced; int forced_ld;   // optional [B][max_new]
  int32_t* out_tokens; int out_ld;        // [B][max_new]
  int32_t* next_tok;                      // [B] input of the next decode step
  int32_t* cur_len;                       // [B] tokens in the KV cache of each row
  int32_t* tok_pos;                       // [B] position of the next input token (== cur_len before increment)
  int32_t* finished;                      // [B]
  const int32_t* eos; int num_eos; int32_t pad_token;
  const int32_t* stop_tok; const int32_t* stop_off; int num_stop;  // flattened stop sequences
  StepState* st;
  P2P pp; int use_p2p;                    // vocab-parallel candidates arrive through peer memory
  uint32_t* seen; int seen_words; int V;  // repetition-penalty bitmap [B][seen_words] (null when the penalty is off)
};

__global__ void __launch_bounds__(128) step_update_kernel(const StepParams p) {
  TraceScope _ts(TK_STEP);
  pdl_launch_dependents();
  pdl_wait();
  _ts.mark();
  __shared__ int s_stop, s_unfinished;
  StepState* st = p.st;
  if (p.use_p2p && threadIdx.x == 0) p.pp.row_epoch[0] += 1;   // epoch base of the next step's peer all-reduces
  if (st->done) return;
  const int step = st->step;
  if (threadIdx.x == 0) { s_stop = 0; s_unfinished = 0; }
  __syncthreads();
  for (int b = threadIdx.x; b < p.B; b += blockDim.x) {
    float best = p.cand_val[b];
    int tok = p.cand_idx[b];
    if (p.use_p2p) merge_candidates(p.pp, b, best, tok);
    for (int r = 1; r < p.ranks && !p.use_p2p; ++r) {
      const float v = p.cand_val[r * p.B + b];
      const int i = p.cand_idx[r * p.B + b];
      if (v > best || (v == best && i < tok)) { best = v; tok = i; }
    }
    if (p.forced) tok = p.forced[b * p.forced_ld + step];
    int fin = p.finished[b];
    if (fin) tok = p.pad_token;
    p.out_tokens[b * p.out_ld + step] = tok;
    if (p.seen && tok >= 0 && tok < p.V) atomicOr(p.seen + (long long)b * p.seen_words + (tok >> 5), 1u << (tok & 31));
    for (int e = 0; e < p.num_eos; ++e)
      if (!fin && tok == p.eos[e]) fin = 1;
    p.finished[b] = fin;
    if (!fin) atomicAdd(&s_unfinished, 1);
    p.next_tok[b] = tok;
    const int len = p.cur_len[b];   // tokens already in the KV cache == position of the token just chosen
    p.tok_pos[b] = len;
    p.cur_len[b] = len + 1;
    // stop sequences: compare the generated suffix (only generated tokens count)
    const int gen = step + 1;
    for (int s = 0; s < p.num_stop; ++s) {
      const int o = p.stop_off[s], n = p.stop_off[s + 1] - o;
      if (n == 0 || n > gen) continue;
      bool eq = true;
      for (int i = 0; i < n && eq; ++i) eq = p.out_tokens[b * p.out_ld + gen - n + i] == p.stop_tok[o + i];
      if (eq) atomicExch(&s_stop, 1);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    st->step = step + 1;
    if (s_stop) { st->stop_triggered = 1; st->done = 1; }
    if (s_unfinished == 0) st->done = 1;
    if (step + 1 >= st->max_new) st->done = 1;
  }
}

// xl[b][:] = x[row_idx[b]][:]   (last prompt token of each sequence before the LM head)
__global__ void gather_rows_kernel(const bf16* __restrict__ x, const int32_t* __restrict__ row_idx,
                                   bf16* __restrict__ out, int H) {
  TraceScope _ts(TK_OTHER);
  pdl_launch_dependents();
  pdl_wait();
  _ts.mark();
  const uint4* src = reinterpret_cast<const uint4*>(x + (long long)row_idx[blockIdx.x] * H);
  uint4* dst = reinterpret_cast<uint4*>(out + (long long)blockIdx.x * H);
  for (int i = threadIdx.x; i < H / 8; i += blockDim.x) dst[i] = src[i];
}

}  // namespace b200
