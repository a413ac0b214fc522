// Sparse mixture-of-experts block (Mixtral: SURVEY.md §8a row 18, transformers modeling_mixtral.py:62-135):
//   router  : logits = xn * Wr^T (bf16 result), softmax in fp32, top-k (k = 2), renormalised fp32 weights
//   dispatch: tokens are grouped per expert into one compact row buffer (deterministic order: token index)
//   experts : the same tcgen05 GEMM kernels as the dense MLP, one launch per expert, bounded at run time by the
//             device-side token count of that expert (GemmParams::m_rt / n_rt / row_off)
//   combine : out[t] = bf16(bf16(y_e1[t] * w1) + bf16(y_e2[t] * w2)) in ascending expert order, exactly the
//             bf16 index_add_ sequence of MixtralExperts.forward, then residual add + next RMSNorm (fused)
#pragma once
#include "common.cuh"
#include "ops.cuh"

namespace b200 {

constexpr int kMaxExperts = 16;
constexpr int kTopK = 2;

// one warp per token
__global__ void __launch_bounds__(128)
moe_router_kernel(const bf16* __restrict__ xn, const bf16* __restrict__ wr, int T, int H, int E,
                  int32_t* __restrict__ tok_expert, float* __restrict__ tok_weight) {
  TraceScope _ts(TK_OTHER);
  pdl_launch_dependents();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t = blockIdx.x * 4 + warp;
  if (t >= T) return;
  float logit[kMaxExperts];
  const bf16* xr = xn + (long long)t * H;
  for (int e = 0; e < E; ++e) {
    const bf16* w = wr + (long long)e * H;
    float acc = 0.f;
    for (int i = lane * 8; i < H; i += 256) {
      const uint4 xu = *reinterpret_cast<const uint4*>(xr + i), wu = *reinterpret_cast<const uint4*>(w + i);
      const uint32_t xw[4] = {xu.x, xu.y, xu.z, xu.w}, ww[4] = {wu.x, wu.y, wu.z, wu.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 a = unpack_bf16x2(xw[j]), b = unpack_bf16x2(ww[j]);
        acc += a.x * b.x + a.y * b.y;
      }
    }
    logit[e] = bf16_round(warp_sum(acc));   // F.linear output is bf16
  }
  if (lane == 0) {
    float mx = -INFINITY;
    for (int e = 0; e < E; ++e) mx = fmaxf(mx, logit[e]);
    float p[kMaxExperts], sum = 0.f;
    for (int e = 0; e < E; ++e) { p[e] = expf(logit[e] - mx); sum += p[e]; }
    for (int e = 0; e < E; ++e) p[e] /= sum;
    int i0 = 0;
    for (int e = 1; e < E; ++e) if (p[e] > p[i0]) i0 = e;           // lowest index wins ties
    int i1 = (i0 == 0) ? 1 : 0;
    for (int e = 0; e < E; ++e) if (e != i0 && p[e] > p[i1]) i1 = e;
    const float s2 = p[i0] + p[i1];
    tok_expert[t * 2] = i0; tok_expert[t * 2 + 1] = i1;
    tok_weight[t * 2] = p[i0] / s2; tok_weight[t * 2 + 1] = p[i1] / s2;
  }
}

// Single CTA: per-expert counts, compact segment offsets (8-row aligned) and the row of every (token, k)
// assignment inside its expert's segment, in token order (deterministic).
//   count[e], off[e] (row offset of expert e in the grouped buffers), tok_row[t*2+k] = off[e] + position
__global__ void __launch_bounds__(1024)
moe_offsets_kernel(const int32_t* __restrict__ tok_expert, int T, int E, int32_t* __restrict__ count,
                   int32_t* __restrict__ off, int32_t* __restrict__ tok_row) {
  TraceScope _ts(TK_OTHER);
  pdl_launch_dependents();
  pdl_wait();
  __shared__ int s_cnt[kMaxExperts][32];   // per warp
  __shared__ int s_base[kMaxExperts][32];
  __shared__ int s_off[kMaxExperts + 1];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int per = (T + 1023) / 1024;
  const int t0 = min(T, tid * per), t1 = min(T, t0 + per);
  int local[kMaxExperts];
  for (int e = 0; e < E; ++e) local[e] = 0;
  for (int t = t0; t < t1; ++t) { local[tok_expert[t * 2]]++; local[tok_expert[t * 2 + 1]]++; }
  // exclusive scan over threads per expert: warp scan + warp totals
  int excl[kMaxExperts];
  for (int e = 0; e < E; ++e) {
    int v = local[e], inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += n;
    }
    excl[e] = inc - v;
    if (lane == 31) s_cnt[e][warp] = inc;
  }
  __syncthreads();
  if (tid < E) {
    int run = 0;
    for (int w = 0; w < 32; ++w) { s_base[tid][w] = run; run += s_cnt[tid][w]; }
    count[tid] = run;
  }
  __syncthreads();
  if (tid == 0) {
    int o = 0;
    for (int e = 0; e < E; ++e) {
      s_off[e] = o; off[e] = o;
      int c = 0;
      for (int w = 0; w < 32; ++w) c += s_cnt[e][w];
      o += (c + 7) & ~7;
    }
    s_off[E] = o; off[E] = o;
  }
  __syncthreads();
  int pos[kMaxExperts];
  for (int e = 0; e < E; ++e) pos[e] = s_off[e] + s_base[e][warp] + excl[e];
  for (int t = t0; t < t1; ++t) {
    const int e0 = tok_expert[t * 2], e1 = tok_expert[t * 2 + 1];
    tok_row[t * 2] = pos[e0]++;
    tok_row[t * 2 + 1] = pos[e1]++;
  }
}

// xg[tok_row[t*2+k]][:] = xn[t][:]
__global__ void __launch_bounds__(128)
moe_gather_kernel(const bf16* __restrict__ xn, const int32_t* __restrict__ tok_row, bf16* __restrict__ xg, int H) {
  TraceScope _ts(TK_OTHER);
  pdl_launch_dependents();
  pdl_wait();
  const int t = blockIdx.x;
  const uint4* src = reinterpret_cast<const uint4*>(xn + (long long)t * H);
  uint4* d0 = reinterpret_cast<uint4*>(xg + (long long)tok_row[t * 2] * H);
  uint4* d1 = reinterpret_cast<uint4*>(xg + (long long)tok_row[t * 2 + 1] * H);
  for (int i = threadIdx.x; i < H / 8; i += blockDim.x) {
    const uint4 v = src[i];
    d0[i] = v;
    d1[i] = v;
  }
}

// Decode (T <= 64 rows).  r01 timeline: the one-warp-per-token router walked E dependent dot products (47 us per
// layer at T = 32), and a variant in which every CTA recomputed all T * E logits pulled 4 MB per CTA through L2
// (58 us).  Here: one CTA per token with one warp per expert (8 KB of x + 8 KB of router row per warp, loads
// batched 8 deep), then one kernel that rebuilds the (tiny) placement tables in every CTA and copies its token.
// Same arithmetic and the same deterministic token-order placement as the prefill kernels above.
constexpr int kMoeDecodeMaxT = 64;
__global__ void __launch_bounds__(32 * kMaxExperts)
moe_router_decode_kernel(const bf16* __restrict__ xn, const bf16* __restrict__ wr, int H, int E,
                         int32_t* __restrict__ tok_expert, float* __restrict__ tok_weight) {
  TraceScope _ts(TK_OTHER);
  pdl_launch_dependents();
  __shared__ float s_logit[kMaxExperts];
  const int e = threadIdx.x >> 5, lane = threadIdx.x & 31, t = blockIdx.x;
  pdl_wait();
  _ts.mark();
  {
    const bf16* xr = xn + (long long)t * H;
    const bf16* w = wr + (long long)e * H;
    float acc = 0.f;
#pragma unroll 8
    for (int i = lane * 8; i < H; i += 256) {
      const uint4 xu = *reinterpret_cast<const uint4*>(xr + i), wu = *reinterpret_cast<const uint4*>(w + i);
      const uint32_t xw[4] = {xu.x, xu.y, xu.z, xu.w}, ww[4] = {wu.x, wu.y, wu.z, wu.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 a = unpack_bf16x2(xw[j]), b = unpack_bf16x2(ww[j]);
        acc += a.x * b.x + a.y * b.y;
      }
    }
    acc = bf16_round(warp_sum(acc));   // F.linear output is bf16
    if (lane == 0) s_logit[e] = acc;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float mx = -INFINITY;
    for (int x = 0; x < E; ++x) mx = fmaxf(mx, s_logit[x]);
    float p[kMaxExperts], sum = 0.f;
    for (int x = 0; x < E; ++x) { p[x] = expf(s_logit[x] - mx); sum += p[x]; }
    for (int x = 0; x < E; ++x) p[x] /= sum;
    int i0 = 0;
    for (int x = 1; x < E; ++x) if (p[x] > p[i0]) i0 = x;           // lowest index wins ties
    int i1 = (i0 == 0) ? 1 : 0;
    for (int x = 0; x < E; ++x) if (x != i0 && p[x] > p[i1]) i1 = x;
    const float s2 = p[i0] + p[i1];
    tok_expert[t * 2] = i0; tok_expert[t * 2 + 1] = i1;
    tok_weight[t * 2] = p[i0] / s2; tok_weight[t * 2 + 1] = p[i1] / s2;
  }
}

// grid T: every CTA rebuilds count / off / tok_row from the 2T expert picks (ballot prefix per expert), CTA t
// copies token t into its two expert segments, CTA 0 publishes the tables.
__global__ void __launch_bounds__(256)
moe_place_gather_kernel(const bf16* __restrict__ xn, const int32_t* __restrict__ tok_expert, int T, int H, int E,
                        int32_t* __restrict__ count, int32_t* __restrict__ off, int32_t* __restrict__ tok_row,
                        bf16* __restrict__ xg) {
  TraceScope _ts(TK_OTHER);
  pdl_launch_dependents();
  __shared__ int s_e[kMoeDecodeMaxT * 2], s_rel[kMoeDecodeMaxT * 2];
  __shared__ int s_cnt[kMaxExperts], s_off[kMaxExperts + 1];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int A = T * 2;
  pdl_wait();
  _ts.mark();
  for (int a = threadIdx.x; a < kMoeDecodeMaxT * 2; a += blockDim.x) s_e[a] = a < A ? tok_expert[a] : -1;
  __syncthreads();
  for (int e = warp; e < E; e += 8) {
    int base = 0;
    for (int c = 0; c < kMoeDecodeMaxT * 2; c += 32) {
      const bool hit = s_e[c + lane] == e;
      const unsigned m = __ballot_sync(0xffffffffu, hit);
      if (hit) s_rel[c + lane] = base + __popc(m & ((1u << lane) - 1u));
      base += __popc(m);
    }
    if (lane == 0) s_cnt[e] = base;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int o = 0;
    for (int e = 0; e < E; ++e) { s_off[e] = o; o += (s_cnt[e] + 7) & ~7; }
    s_off[E] = o;
  }
  __syncthreads();
  if (blockIdx.x == 0) {
    for (int a = threadIdx.x; a < A; a += blockDim.x) tok_row[a] = s_off[s_e[a]] + s_rel[a];
    if ((int)threadIdx.x < E) count[threadIdx.x] = s_cnt[threadIdx.x];
    if ((int)threadIdx.x <= E) off[threadIdx.x] = s_off[threadIdx.x];
  }
  const int t = blockIdx.x;
  const uint4* src = reinterpret_cast<const uint4*>(xn + (long long)t * H);
  uint4* d0 = reinterpret_cast<uint4*>(xg + (long long)(s_off[s_e[t * 2]] + s_rel[t * 2]) * H);
  uint4* d1 = reinterpret_cast<uint4*>(xg + (long long)(s_off[s_e[t * 2 + 1]] + s_rel[t * 2 + 1]) * H);
  for (int i = threadIdx.x; i < H / 8; i += blockDim.x) {
    const uint4 v = src[i];
    d0[i] = v;
    d1[i] = v;
  }
}

// Combine + residual + next RMSNorm over the bf16 expert output rows yg[row][H].  TP: writes the per-rank partial
// sum to `ysum` instead (the caller all-reduces it and applies the residual / norm afterwards).
struct MoeCombineParams {
  bf16* x; const bf16* w; bf16* xn; int H; float eps;
  const int32_t* tok_expert; const float* tok_weight; const int32_t* tok_row;
  const bf16* yg;
  bf16* ysum;   // non-null under tensor parallelism
};

__global__ void __launch_bounds__(kNormThreads) moe_combine_norm_kernel(const MoeCombineParams p) {
  TraceScope _ts(TK_RMSNORM);
  pdl_launch_dependents();
  extern __shared__ float row[];
  const int H = p.H;
  float* red = row + H;
  const int r = blockIdx.x;
  pdl_wait();
  _ts.mark();
  int ea = p.tok_expert[r * 2], eb = p.tok_expert[r * 2 + 1];
  float wa = p.tok_weight[r * 2], wb = p.tok_weight[r * 2 + 1];
  int ra = p.tok_row[r * 2], rb = p.tok_row[r * 2 + 1];
  if (eb < ea) {   // MixtralExperts.forward walks the experts in ascending index
    int ti = ea; ea = eb; eb = ti;
    float tf = wa; wa = wb; wb = tf;
    ti = ra; ra = rb; rb = ti;
  }
  bf16* xr = p.x + (long long)r * H;
  float ss = 0.f;
  for (int i = threadIdx.x * 8; i < H; i += blockDim.x * 8) {
    float ya[8], yb[8];
    const uint4 ua = *reinterpret_cast<const uint4*>(p.yg + (long long)ra * H + i);
    const uint4 ub = *reinterpret_cast<const uint4*>(p.yg + (long long)rb * H + i);
    const uint32_t aw[4] = {ua.x, ua.y, ua.z, ua.w}, bw[4] = {ub.x, ub.y, ub.z, ub.w};
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const float2 a2 = unpack_bf16x2(aw[t]), b2 = unpack_bf16x2(bw[t]);
      ya[2 * t] = a2.x; ya[2 * t + 1] = a2.y;
      yb[2 * t] = b2.x; yb[2 * t + 1] = b2.y;
    }
    float f[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) f[t] = bf16_round(bf16_round(ya[t] * wa) + bf16_round(yb[t] * wb));
    if (p.ysum) {
      *reinterpret_cast<uint4*>(p.ysum + (long long)r * H + i) = pack8(f);
      continue;
    }
    const uint4 xu = *reinterpret_cast<const uint4*>(xr + i);
    const uint32_t xw[4] = {xu.x, xu.y, xu.z, xu.w};
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const float2 x2 = unpack_bf16x2(xw[t]);
      f[2 * t] = bf16_round(x2.x + f[2 * t]);
      f[2 * t + 1] = bf16_round(x2.y + f[2 * t + 1]);
    }
    *reinterpret_cast<uint4*>(xr + i) = pack8(f);
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      row[i + t] = f[t];
      ss += f[t] * f[t];
    }
  }
  if (p.ysum) return;
  const float tot = block_sum(ss, red);
  const float rs = 1.0f / sqrtf(tot / (float)H + p.eps);
  bf16* o = p.xn + (long long)r * H;
  for (int i = threadIdx.x * 8; i < H; i += blockDim.x * 8) {
    const uint4 wu = *reinterpret_cast<const uint4*>(p.w + i);
    const uint32_t ww[4] = {wu.x, wu.y, wu.z, wu.w};
    float g[8];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const float2 w2 = unpack_bf16x2(ww[t]);
      g[2 * t] = w2.x * bf16_round(row[i + 2 * t] * rs);
      g[2 * t + 1] = w2.y * bf16_round(row[i + 2 * t + 1] * rs);
    }
    *reinterpret_cast<uint4*>(o + i) = pack8(g);
  }
}

}  // namespace b200
