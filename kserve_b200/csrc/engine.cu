// The generation engine behind the C ABI in include/kserve_b200.h.
//
// Replaces what the reference delegates to `transformers` at
// python/huggingfaceserver/huggingfaceserver/generative_model.py:328 (`self._model.generate(**kwargs)`):
// prefill over the packed (un-padded) prompt tokens, then a CUDA-graph-captured decode step per token,
// with sampling (greedy), EOS / stop-sequence / max-length checks kept on the device.
#include <dlfcn.h>
#include <math.h>

#include <algorithm>
#include <deque>
#include <climits>
#include <memory>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/kserve_b200.h"
#include "batcher.cuh"
#include "launch.cuh"

namespace b200 {

static thread_local std::string g_last_error;
void set_last_error(const std::string& msg) { g_last_error = msg; }

// ---------------------------------------------------------------------------------------------------
// NCCL, resolved at run time (only needed when tp_size > 1)
// ---------------------------------------------------------------------------------------------------
struct Nccl {
  typedef struct { char internal[128]; } UniqueId;
  typedef void* Comm;
  int (*GetUniqueId)(UniqueId*) = nullptr;
  int (*CommInitRank)(Comm*, int, UniqueId, int) = nullptr;
  int (*CommDestroy)(Comm) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, Comm, cudaStream_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, Comm, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool ok = false;
  static constexpr int kBf16 = 9, kFloat = 7, kInt32 = 2, kSum = 0;
  static Nccl& get() {
    static Nccl n;
    static std::once_flag once;
    std::call_once(once, [] {
      void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
      if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
      if (!h) return;
      n.GetUniqueId = (decltype(n.GetUniqueId))dlsym(h, "ncclGetUniqueId");
      n.CommInitRank = (decltype(n.CommInitRank))dlsym(h, "ncclCommInitRank");
      n.CommDestroy = (decltype(n.CommDestroy))dlsym(h, "ncclCommDestroy");
      n.AllReduce = (decltype(n.AllReduce))dlsym(h, "ncclAllReduce");
      n.AllGather = (decltype(n.AllGather))dlsym(h, "ncclAllGather");
      n.GetErrorString = (decltype(n.GetErrorString))dlsym(h, "ncclGetErrorString");
      n.ok = n.GetUniqueId && n.CommInitRank && n.AllReduce && n.AllGather;
    });
    return n;
  }
};

#define B200_NCCL_OK(expr)                                                                  \
  do {                                                                                      \
    int _r = (expr);                                                                        \
    if (_r != 0) {                                                                          \
      Nccl& _n = Nccl::get();                                                               \
      set_last_error(std::string(#expr) + " failed: " +                                     \
                     (_n.GetErrorString ? _n.GetErrorString(_r) : std::to_string(_r)));     \
      return -4;                                                                            \
    }                                                                                       \
  } while (0)

template <class T>
static int dmalloc(T** p, size_t n) {
  B200_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(p), n * sizeof(T)));
  return 0;
}

struct LayerW {
  bf16 *wqkv = nullptr, *wo = nullptr, *wgu = nullptr, *wdown = nullptr, *ln1 = nullptr, *ln2 = nullptr;
  bf16 *wr = nullptr, *wgu_e = nullptr, *wdown_e = nullptr;   // MoE: router [E][H], experts [E][2I][H] / [E][H][I]
};

}  // namespace b200

using namespace b200;

struct b200_engine {
  b200_model_config_t cfg;
  int num_sms = 148;
  cudaStream_t stream = nullptr;
  cudaStream_t stream2 = nullptr;            // second micro-batch of a tensor-parallel prefill
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;
  // per-rank dims
  int H, nh, nkv, G, I, V, Vl, v0, qkv_cols, L;
  int E = 0;   // experts (0 = dense)
  // MoE dispatch state / grouped buffers
  int32_t *tok_expert = nullptr, *tok_row = nullptr, *e_count = nullptr, *e_off = nullptr;
  float* tok_weight = nullptr;
  bf16 *xg = nullptr, *hg = nullptr, *yg = nullptr;
  int g_rows = 0;
  // weights
  bf16 *embed = nullptr, *lm_head = nullptr, *final_norm = nullptr;
  std::vector<LayerW> layers;
  std::unordered_map<std::string, int> seen;
  bool finalized = false;
  bf16 *cos_tab = nullptr, *sin_tab = nullptr;
  // KV cache
  bf16 *kcache = nullptr, *vcache = nullptr;
  long long layer_stride = 0;  // elements per layer in each cache
  int num_pages = 0, max_pages = 0;
  int32_t* d_page_table = nullptr;
  std::vector<int32_t> h_page_table;
  // activations
  int cap_T = 0;  // rows of the token-major buffers
  int rows_cap = 0;   // min(max_batch, kMaxRows): rows of the per-step buffers (logits, xl, partials, candidates)
  bf16 *x = nullptr, *xn = nullptr, *qkv = nullptr, *attn = nullptr, *hbuf = nullptr, *ybuf = nullptr, *xl = nullptr,
       *qdec = nullptr, *logits = nullptr;
  float* ws = nullptr;
  size_t ws_elems = 0;
  float* sk_ws = nullptr;   // stream-K partials / flags
  int* sk_flags = nullptr;
  int sk_tiles = 0;
  size_t sk_ws_floats = 0;
  float *part_o = nullptr, *part_ml = nullptr;
  int* attn_split_cnt = nullptr;   // [max_batch * nkv] arrival counters of the split decode attention
  float* cand_val = nullptr;
  int32_t* cand_idx = nullptr;
  float* cand_val_all = nullptr;
  int32_t* cand_idx_all = nullptr;
  // token bookkeeping (device)
  int32_t *d_tok = nullptr, *d_tok_seq = nullptr, *d_tok_pos = nullptr, *d_cu = nullptr, *d_seq_slot = nullptr,
          *d_last_rows = nullptr, *d_cur_len = nullptr, *d_next_tok = nullptr, *d_dec_pos = nullptr,
          *d_finished = nullptr, *d_out_tokens = nullptr, *d_forced = nullptr, *d_eos = nullptr,
          *d_stop_tok = nullptr, *d_stop_off = nullptr;
  StepState* d_state = nullptr;
  int out_ld = 0;
  // raw request staging (device-side concat/pad)
  long long *d_raw_ids = nullptr, *d_raw_mask = nullptr, *d_pred = nullptr;
  int32_t *d_flat = nullptr, *d_offs = nullptr;
  long long *h_raw = nullptr, *h_pred = nullptr;
  // pinned staging
  int32_t* h_stage = nullptr;
  size_t h_stage_elems = 0;
  StepState* h_state = nullptr;
  int32_t* h_out_tokens = nullptr;
  // staged request
  struct Staged {
    int B = 0, S = 0, T = 0, max_len = 0, max_new = 0;
    std::vector<int> lens;
    std::vector<int64_t> input;  // [B][S] copy of the prompt (with pads) for output assembly
    int32_t pad = 0;
    int num_eos = 0, num_stop = 0;
    bool forced = false;
    bool prefilled = false;
    bool sample_on = false, rep_on = false;   // processed-score path (sampling.cuh) / repetition-penalty bitmap in use
    int per_seq_pages = 0;
  } st;
  // host-DRAM KV tier: pinned copies of the pages of swapped-out sequences (slot -> buffer)
  std::unordered_map<int, bf16*> host_kv;
  std::unordered_map<int, size_t> host_kv_bytes;
  bool staged_mask = false;
  // graphs per batch size
  std::unordered_map<int, cudaGraphExec_t> graphs;
  std::unordered_map<int, int> graph_nodes;
  TmapCache tmaps;
  // comm
  Nccl::Comm comm = nullptr;
  // peer-memory exchange (decode): IPC-shared block of this rank + mapped blocks of the peers
  unsigned char* ar_local = nullptr;
  void* ar_peer_map[kMaxTp] = {nullptr};
  int *row_epoch = nullptr, *cand_epoch = nullptr;
  int ar_index = 0;   // index of the next peer all-reduce inside the forward pass being recorded
  int big_epoch[2] = {0, 0};   // prefill all-reduce epochs, one per micro-batch stream (identical on every rank)
  int* big_cnt = nullptr;      // [2] CTA arrival counters of allreduce_big_kernel
  bool ybuf_in_block = false;  // ybuf lives inside the IPC-shared exchange block (tp > 1)
  bool p2p_ready = false;
  P2P p2p{};
  b200_timing_t timing{};
  int launches = 0;
  // continuous batching (cb.cuh): per-slot sequence state + the compact list of running slots
  SampleCfg* d_sample_cfg = nullptr;
  uint32_t* d_seen = nullptr;        // [max_batch][seen_words] token-presence bitmap (allocated on first use)
  int seen_words = 0;
  bool cb_on = false;
  CbState cb{};
  std::vector<int> cb_active;        // running slots, in row order of the decode step
  std::vector<char> cb_used;         // slot occupied (running or finished-but-not-released)
  int32_t* d_cb_row_slot = nullptr;  // [max_batch]
  int32_t* d_cb_rec = nullptr;       // [max_batch][kCbInitInts]
  int32_t* h_cb = nullptr;           // pinned: init records / poll results / token reads
  bool cb_rows_dirty = false;
  int32_t* h_cb_rows = nullptr;      // pinned ring [8][kMaxRows]: the row -> slot list of the next decode pass
  unsigned long long cb_ring_pos = 0, cb_window = 0;
  int cb_num_eos = 0;
  // KV page pool of the continuous-batching mode: pages are reference counted so that 128-token blocks of a prompt
  // can be shared between requests (prefix reuse); a slot's page-table row is filled at admit
  struct CbPending {                     // a prompt whose tokens are not all in the cache yet (chunked prefill)
    int slot;
    std::vector<int32_t> toks;
    int done;                            // tokens already in the cache (shared prefix + prefilled chunks), multiple of 128
    std::vector<unsigned long long> block_hash;   // chain hash of every full 128-token block of the prompt
  };
  struct PrefixEntry { int p0, p1; unsigned long long parent, tick; std::vector<int32_t> toks; };
  std::deque<CbPending> cb_pending;
  std::vector<std::vector<int>> cb_slot_pages;
  std::vector<int> cb_free_pages, cb_page_ref;
  std::unordered_map<unsigned long long, PrefixEntry> cb_prefix;
  unsigned long long cb_tick = 0;
  int cb_chunk_tokens = 0;               // 0: a prompt is prefilled completely inside b200_cb_admit
  bool cb_prefix_on = false;
  long long cb_stat[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // prompt tokens admitted / served from shared pages / prefilled, evictions, prefill passes
  std::vector<char> cb_swapped;          // slot's KV pages live in host DRAM (b200_cb_swap_out)
  std::vector<int> cb_swap_pages;        // number of pages parked per swapped slot
  SampleCfg* d_cb_cfg = nullptr;         // [max_batch] per-slot logits-processor / sampling configuration
  std::vector<char> cb_slot_sampling;    // slot uses the processed-score path
  int cb_sampling_slots = 0;
  int32_t* d_kv_off = nullptr;           // [80] tokens of each prefill row's sequence that are already cached
  bool faulted = false;                  // a cross-GPU / cross-CTA wait timed out (common.cuh: g_fault_code)
};

namespace b200 {

constexpr int kMaxRows = 64;   // rows of one decode / LM-head pass (swap-AB GEMM block_n, peer-exchange rows)
static int pick_block_n(int B) { return B <= 16 ? 16 : (B <= 32 ? 32 : 64); }

// peer-memory all-reduce + residual + RMSNorm of the decode step: one-shot LL up to 4 ranks, two-shot (reduce-scatter +
// all-gather, 4x less NVLink traffic) at 8 ranks.  Measured r02: TP = 8 decode 2.64 -> 2.20 ms/step with two-shot; at TP = 4
// two-shot is slower (2.57 vs 2.46 ms/step: one more NVLink hop for only 2x less traffic).
typedef void (*ArKernel)(const P2P, bf16*, const bf16*, bf16*, float, const float*, int, long long, long long, const bf16*, int, int);
static ArKernel ar_kernel(const b200_engine* e) {
  constexpr int kTwoShotMinTp = 8;
  return (e->cfg.tp_size >= kTwoShotMinTp && (e->H / e->cfg.tp_size) % 8 == 0) ? allreduce2_norm_kernel : allreduce_norm_kernel;
}

static int pick_splits(const b200_engine* e, int n_out, int K) {
  const int m_tiles = (n_out + kGemmBlockM - 1) / kGemmBlockM;
  int s = e->num_sms / m_tiles;
  s = std::max(1, std::min(s, 16));
  return effective_splits(K, s);
}

// prefill: all-reduce of a micro-batch's row-parallel GEMM output (bandwidth regime): ncclAllReduce by default.  The
// engine's own peer-memory kernel (p2p.cuh: allreduce_big_kernel, B200_PREFILL_OWN_AR=1) is correct (tests/test_tp_gpu.py
// run it too) but measured slower — TTFT 228.9 vs 220.6 ms at TP = 2, 108.5 vs 99.7 ms at TP = 8 (r02): its pull-based
// reduce-scatter reaches ~300 GB/s per direction over NVLink, short of NCCL's NVLS path.
static int allreduce_bf16(b200_engine* e, bf16* buf, size_t count, cudaStream_t s) {
  if (e->cfg.tp_size == 1) return 0;
  static const bool force_nccl = getenv("B200_PREFILL_OWN_AR") == nullptr;
  constexpr int kArCtas = 64;
  if (e->p2p_ready && !force_nccl && buf >= e->ybuf && buf + count <= e->ybuf + (size_t)e->cap_T * e->H && count % 8 == 0) {
    const int lane = (s == e->stream2) ? 1 : 0;
    const int epoch = ++e->big_epoch[lane];
    allreduce_big_kernel<<<kArCtas, 256, 0, s>>>(e->p2p, (long long)e->p2p.lay.total, (long long)(buf - e->ybuf), (long long)count,
                                                 epoch, lane, e->big_cnt + lane);
    B200_CUDA_OK(cudaGetLastError());
    e->launches++;
    return 0;
  }
  Nccl& n = Nccl::get();
  B200_NCCL_OK(n.AllReduce(buf, buf, count, Nccl::kBf16, Nccl::kSum, e->comm, s));
  return 0;
}

// ---- one transformer stack pass over T token rows --------------------------------------------------
// decode == true : T == B rows, swap-AB GEMMs (+ split-K), flash-decoding attention
// decode == false: packed prompt tokens, row-major GEMMs, causal flash attention
static int forward_layers(b200_engine* e, int T_all, int B_all, int max_len, bool decode, const int32_t* kv_off = nullptr) {
  const int H = e->H, bn = pick_block_n(B_all);
  const float eps = e->cfg.rms_eps;
  const float scale_log2 = (1.0f / sqrtf((float)kHeadDim)) * 1.4426950408889634f;
  const bool tp = e->cfg.tp_size > 1;
  int rc;
  pdl_phase() = decode;
  e->ar_index = 0;
  if (!decode) e->tmaps.trim();
  // Tensor-parallel prefill runs as two micro-batches (halves of the sequences = two row ranges of the packed
  // buffers) on two streams, issued layer by layer: while one half's 256 MiB all-reduce is on the wire the other
  // half's GEMMs / attention own the SMs (SURVEY.md §8e "prefill ... overlap by token-chunking").
  struct View { long long r0; int T, b0, B; cudaStream_t s; };
  View views[2] = {{0, T_all, 0, B_all, e->stream}, {0, 0, 0, 0, e->stream2}};
  int nv = 1;
  static const int mb_min_t = getenv("B200_PREFILL_OVERLAP_MIN_T") ? atoi(getenv("B200_PREFILL_OVERLAP_MIN_T")) : 2048;
  if (!decode && tp && e->E == 0 && B_all >= 2 && T_all >= mb_min_t) {
    const int b0 = B_all / 2;
    long long r0 = 0;
    for (int b = 0; b < b0; ++b) r0 += e->st.lens[b];
    views[0] = View{0, (int)r0, 0, b0, e->stream};
    views[1] = View{r0, (int)(T_all - r0), b0, B_all - b0, e->stream2};
    nv = 2;
    B200_CUDA_OK(cudaEventRecord(e->ev_fork, e->stream));
    B200_CUDA_OK(cudaStreamWaitEvent(e->stream2, e->ev_fork, 0));
  }
  for (int v = 0; v < nv; ++v) {
    const View& vw = views[v];
    B200_CUDA_OK(launch_k(embed_gather_kernel, dim3(vw.T), dim3(128), 0, vw.s, (const int32_t*)(decode ? e->d_next_tok : e->d_tok + vw.r0),
                          (const bf16*)e->embed, e->x + vw.r0 * H, H, e->V));
    e->launches++;
    if ((rc = launch_rmsnorm(0, e->x + vw.r0 * H, e->layers[0].ln1, e->xn + vw.r0 * H, vw.T, H, eps, nullptr, 0, 0, 0, nullptr, vw.s))) return rc;
    e->launches++;
  }
  for (int l = 0; l < e->L; ++l)
  for (int v = 0; v < nv; ++v) {
    const View& vw = views[v];
    const int T = vw.T, B = vw.B;
    const long long r0 = vw.r0;        // first row of this micro-batch in the packed activation buffers (0 in decode)
    cudaStream_t s = vw.s;
    const LayerW& w = e->layers[l];
    bf16* kc = e->kcache + (long long)l * e->layer_stride;
    bf16* vc = e->vcache + (long long)l * e->layer_stride;
    // ---- QKV projection
    RopeKvParams rp{};
    rp.ld = e->qkv_cols;
    if (decode) {
      // uniform split-K with fp32 partials: the consumer kernel (attention prologue / rmsnorm) reduces them in
      // parallel, which measured faster than finishing multi-piece tiles inside the GEMM (r01: 4.30 vs 4.62 ms/step)
      const int sp = pick_splits(e, e->qkv_cols, H);
      GemmArgs a{w.wqkv, e->qkv_cols, e->xn, e->cap_T, e->qkv_cols, B, H, sp > 1 ? EPI_T_PARTIAL : EPI_T_STORE, bn, sp,
                 sp > 1 ? (void*)e->ws : (void*)e->qkv, nullptr, e->qkv_cols, (long long)B * e->qkv_cols, 0, true};
      a.sk_ws = e->sk_ws; a.sk_flags = e->sk_flags; a.sk_tiles = e->sk_tiles; a.sk_ws_floats = e->sk_ws_floats;
      if ((rc = launch_gemm(e->tmaps, a, e->num_sms, s))) return rc;
      if (sp > 1) { rp.partial = e->ws; rp.splits = sp; rp.split_stride = (long long)B * e->qkv_cols; rp.ld_partial = e->qkv_cols; }
      rp.qkv = e->qkv;
      rp.q_out = e->qdec; rp.ldq = e->nh * kHeadDim;
      rp.tok_seq = e->d_seq_slot; rp.tok_pos = e->d_dec_pos;
    } else {
      rp.qkv = e->qkv + r0 * e->qkv_cols;
      rp.q_out = e->qkv + r0 * e->qkv_cols; rp.ldq = e->qkv_cols;  // in place
      rp.tok_seq = e->d_tok_seq + r0; rp.tok_pos = e->d_tok_pos + r0;
      rp.kcache = kc; rp.vcache = vc; rp.page_table = e->d_page_table; rp.max_pages = e->max_pages;
      rp.cos_tab = e->cos_tab; rp.sin_tab = e->sin_tab; rp.nh = e->nh; rp.nkv = e->nkv;
      // RoPE + KV append in the QKV GEMM's epilogue (a separate rope_kv_kernel pass re-read and re-wrote 750 MB per layer
      // at 0.37 of the HBM peak); decode fuses them into attn_decode_kernel instead
      GemmArgs a{e->xn + r0 * H, e->cap_T - (int)r0, w.wqkv, e->qkv_cols, T, e->qkv_cols, H, EPI_ROPE_KV, 256, 1,
                 e->qkv + r0 * e->qkv_cols, nullptr, e->qkv_cols, 0, 0, false};
      a.rope = &rp;
      if ((rc = launch_gemm(e->tmaps, a, e->num_sms, s))) return rc;
    }
    e->launches++;
    // ---- attention
    if (decode) {
      AttnDecodeParams ap{};
      ap.q = e->qdec; ap.ldq = e->nh * kHeadDim; ap.out = e->attn; ap.ldo = e->nh * kHeadDim;
      ap.kcache = kc; ap.vcache = vc; ap.page_table = e->d_page_table; ap.max_pages = e->max_pages;
      ap.seq_slot = e->d_seq_slot; ap.tok_pos = e->d_dec_pos; ap.nh = e->nh; ap.nkv = e->nkv; ap.G = e->G;
      // one CTA per (sequence, kv head) already fills the machine at large batch; split the KV range only
      // when there are fewer CTAs than SMs
      const int ctas = B * e->nkv;
      ap.splits = ctas >= e->num_sms ? 1 : std::max(1, std::min((e->num_sms + ctas - 1) / ctas, 8));
      ap.part_o = e->part_o; ap.part_ml = e->part_ml; ap.scale_log2 = scale_log2;
      ap.fuse_rope = 1; ap.qkv = rp.qkv; ap.ld_qkv = rp.ld; ap.qkv_partial = rp.partial; ap.qkv_splits = rp.splits;
      ap.qkv_split_stride = rp.split_stride; ap.ld_qkv_partial = rp.ld_partial; ap.cos_tab = e->cos_tab; ap.sin_tab = e->sin_tab;
      ap.kcache_w = kc; ap.vcache_w = vc;
      ap.split_counter = e->attn_split_cnt;
      if ((rc = launch_attn_decode(ap, B, s))) return rc;
      e->launches++;
    } else {
      AttnTcParams tp_{};
      tp_.out = e->attn; tp_.ldo = e->nh * kHeadDim; tp_.page_table = e->d_page_table; tp_.max_pages = e->max_pages;
      tp_.cu_seqlens = e->d_cu + vw.b0; tp_.seq_slot = e->d_seq_slot + vw.b0; tp_.nh = e->nh; tp_.nkv = e->nkv; tp_.scale_log2 = scale_log2;
      tp_.kv_off = kv_off ? kv_off + vw.b0 : nullptr;
      if ((rc = launch_attn_prefill_tc(e->tmaps, e->qkv, e->cap_T, e->qkv_cols, kc, vc, e->num_pages, tp_, B, max_len, s))) return rc;
      e->launches++;
    }
    // ---- row-parallel projections (o_proj, down_proj) followed by residual add + next RMSNorm
    auto row_parallel = [&](const bf16* act, int K, const bf16* wmat, const bf16* next_norm) -> int {
      int rc2;
      if (decode) {
        const int sp = pick_splits(e, H, K);
        if (sp > 1) {
          GemmArgs a{wmat, H, act, e->cap_T, H, B, K, EPI_T_PARTIAL, bn, sp, e->ws, nullptr, H, (long long)B * H, 0, true};
          if ((rc2 = launch_gemm(e->tmaps, a, e->num_sms, s))) return rc2;
          e->launches++;
          if (!tp) {
            if ((rc2 = launch_rmsnorm(1, e->x, next_norm, e->xn, T, H, eps, e->ws, sp, (long long)B * H, H, nullptr, s))) return rc2;
            e->launches++;
            return 0;
          }
          if (e->p2p_ready) {   // split-K reduce + all-reduce over peer memory + residual + RMSNorm in one kernel
            B200_CUDA_OK(launch_k(ar_kernel(e), dim3(T), dim3(kNormThreads), (size_t)(H + 32) * sizeof(float), s, e->p2p,
                                  e->x, next_norm, e->xn, eps, (const float*)e->ws, sp, (long long)B * H, (long long)H, (const bf16*)nullptr,
                                  e->ar_index++, 2 * e->L));
            e->launches++;
            return 0;
          }
          B200_CUDA_OK(launch_k(reduce_partials_kernel, dim3(T), dim3(256), 0, s, (const float*)e->ws, sp, (long long)B * H, (long long)H, e->ybuf, H));
          e->launches++;
        } else {
          GemmArgs a{wmat, H, act, e->cap_T, H, B, K, EPI_T_STORE, bn, 1, e->ybuf, nullptr, H, 0, 0, true};
          a.sk_ws = e->sk_ws; a.sk_flags = e->sk_flags; a.sk_tiles = e->sk_tiles; a.sk_ws_floats = e->sk_ws_floats;
          if ((rc2 = launch_gemm(e->tmaps, a, e->num_sms, s))) return rc2;
          e->launches++;
          if (tp && e->p2p_ready) {
            B200_CUDA_OK(launch_k(ar_kernel(e), dim3(T), dim3(kNormThreads), (size_t)(H + 32) * sizeof(float), s, e->p2p,
                                  e->x, next_norm, e->xn, eps, (const float*)nullptr, 0, 0LL, 0LL, (const bf16*)e->ybuf,
                                  e->ar_index++, 2 * e->L));
            e->launches++;
            return 0;
          }
        }
      } else {
        if (!tp) {
          GemmArgs a{act, e->cap_T, wmat, H, T, H, K, EPI_STORE_RES, 256, 1, e->x, e->x, H, 0, 0, false};   // (r0 == 0: one GPU)
          if ((rc2 = launch_gemm(e->tmaps, a, e->num_sms, s))) return rc2;
          if ((rc2 = launch_rmsnorm(0, e->x, next_norm, e->xn, T, H, eps, nullptr, 0, 0, 0, nullptr, s))) return rc2;
          e->launches += 2;
          return 0;
        }
        GemmArgs a{act + r0 * K, e->cap_T - (int)r0, wmat, H, T, H, K, EPI_STORE, 256, 1, e->ybuf + r0 * H, nullptr, H, 0, 0, false};
        if ((rc2 = launch_gemm(e->tmaps, a, e->num_sms, s))) return rc2;
        e->launches++;
      }
      if ((rc2 = allreduce_bf16(e, e->ybuf + r0 * H, (size_t)T * H, s))) return rc2;
      if ((rc2 = launch_rmsnorm(2, e->x + r0 * H, next_norm, e->xn + r0 * H, T, H, eps, nullptr, 0, 0, 0, e->ybuf + r0 * H, s))) return rc2;
      e->launches++;
      return 0;
    };
    if ((rc = row_parallel(e->attn, e->nh * kHeadDim, w.wo, w.ln2))) return rc;
    const bf16* next_norm = (l + 1 < e->L) ? e->layers[l + 1].ln1 : e->final_norm;
    if (e->E > 0) {
      // ---- sparse MoE: route, group rows per expert, run the expert GEMMs bounded by the device-side counts, combine
      if (decode && T <= kMoeDecodeMaxT) {
        B200_CUDA_OK(launch_k(moe_router_decode_kernel, dim3(T), dim3(32 * e->E), 0, s, (const bf16*)e->xn, (const bf16*)w.wr, H, e->E,
                              e->tok_expert, e->tok_weight));
        B200_CUDA_OK(launch_k(moe_place_gather_kernel, dim3(T), dim3(256), 0, s, (const bf16*)e->xn, (const int32_t*)e->tok_expert, T, H, e->E,
                              e->e_count, e->e_off, e->tok_row, e->xg));
        e->launches += 2;
      } else {
        B200_CUDA_OK(launch_k(moe_router_kernel, dim3((T + 3) / 4), dim3(128), 0, s, (const bf16*)e->xn, (const bf16*)w.wr, T, H, e->E,
                              e->tok_expert, e->tok_weight));
        B200_CUDA_OK(launch_k(moe_offsets_kernel, dim3(1), dim3(1024), 0, s, (const int32_t*)e->tok_expert, T, e->E, e->e_count, e->e_off, e->tok_row));
        B200_CUDA_OK(launch_k(moe_gather_kernel, dim3(T), dim3(128), 0, s, (const bf16*)e->xn, (const int32_t*)e->tok_row, e->xg, H));
        e->launches += 3;
      }
      // decode: ONE grouped launch per projection over all experts (E * tiles fill the SMs; the weights of experts
      // without tokens are skipped); prefill: one 2-CTA launch per expert, bounded by the expert's token count
      if (decode) {
        GemmArgs a{w.wgu_e, e->E * 2 * e->I, e->xg, e->g_rows, 2 * e->I, B, H, EPI_T_SWIGLU, bn, 1, e->hg, nullptr, e->I, 0, e->I, true};
        a.n_rt = e->e_count; a.row_off = e->e_off; a.groups = e->E;
        if ((rc = launch_gemm(e->tmaps, a, e->num_sms, s))) return rc;
        GemmArgs d{w.wdown_e, e->E * H, e->hg, e->g_rows, H, B, e->I, EPI_T_STORE, bn, 1, e->yg, nullptr, H, 0, 0, true};
        d.n_rt = e->e_count; d.row_off = e->e_off; d.groups = e->E;
        if ((rc = launch_gemm(e->tmaps, d, e->num_sms, s))) return rc;
        e->launches += 2;
      }
      for (int x = 0; x < e->E && !decode; ++x) {
        const bf16* wgu = w.wgu_e + (long long)x * 2 * e->I * H;
        const bf16* wdn = w.wdown_e + (long long)x * H * e->I;
        GemmArgs a{e->xg, e->g_rows, wgu, 2 * e->I, T, 2 * e->I, H, EPI_SWIGLU, 256, 1, e->hg, nullptr, e->I, 0, e->I, false};
        a.m_rt = e->e_count + x; a.row_off = e->e_off + x;
        if ((rc = launch_gemm(e->tmaps, a, e->num_sms, s))) return rc;
        GemmArgs d{e->hg, e->g_rows, wdn, H, T, H, e->I, EPI_STORE, 256, 1, e->yg, nullptr, H, 0, 0, false};
        d.m_rt = e->e_count + x; d.row_off = e->e_off + x;
        if ((rc = launch_gemm(e->tmaps, d, e->num_sms, s))) return rc;
        e->launches += 2;
      }
      MoeCombineParams cp{};
      cp.x = e->x; cp.w = next_norm; cp.xn = e->xn; cp.H = H; cp.eps = eps;
      cp.tok_expert = e->tok_expert; cp.tok_weight = e->tok_weight; cp.tok_row = e->tok_row;
      cp.yg = e->yg;
      cp.ysum = tp ? e->ybuf : nullptr;
      B200_CUDA_OK(launch_k(moe_combine_norm_kernel, dim3(T), dim3(kNormThreads), (size_t)(H + 32) * sizeof(float), s, cp));
      e->launches++;
      if (tp && decode && e->p2p_ready) {   // all-reduce of the combined expert outputs + residual + next norm, over peer memory
        B200_CUDA_OK(launch_k(ar_kernel(e), dim3(T), dim3(kNormThreads), (size_t)(H + 32) * sizeof(float), s, e->p2p,
                              e->x, next_norm, e->xn, eps, (const float*)nullptr, 0, 0LL, 0LL, (const bf16*)e->ybuf,
                              e->ar_index++, 2 * e->L));
        e->launches++;
      } else if (tp) {
        if ((rc = allreduce_bf16(e, e->ybuf, (size_t)T * H, s))) return rc;
        if ((rc = launch_rmsnorm(2, e->x, next_norm, e->xn, T, H, eps, nullptr, 0, 0, 0, e->ybuf, s))) return rc;
        e->launches++;
      }
      continue;
    }
    // ---- gate/up projection with the SwiGLU fused into the epilogue
    if (decode) {
      const int gu_tiles = (2 * e->I + kGemmBlockM - 1) / kGemmBlockM;
      const int gsp = gu_tiles * 4 >= e->num_sms * 3 ? 1 : pick_splits(e, 2 * e->I, H);
      if (gsp > 1) {   // few tiles per GPU (tensor parallel): split-K partials + a reducing SwiGLU kernel
        GemmArgs a{w.wgu, 2 * e->I, e->xn, e->cap_T, 2 * e->I, B, H, EPI_T_PARTIAL, bn, gsp, e->ws, nullptr, 2 * e->I,
                   (long long)B * 2 * e->I, 0, true};
        if ((rc = launch_gemm(e->tmaps, a, e->num_sms, s))) return rc;
        B200_CUDA_OK(launch_k(swiglu_reduce_kernel, dim3(B), dim3(512), 0, s, (const float*)e->ws, gsp, (long long)B * 2 * e->I,
                              (long long)2 * e->I, e->hbuf, e->I));
        e->launches++;
      } else {
        GemmArgs a{w.wgu, 2 * e->I, e->xn, e->cap_T, 2 * e->I, B, H, EPI_T_SWIGLU, bn, 1, e->hbuf, nullptr, e->I, 0, e->I, true};
        a.sk_ws = e->sk_ws; a.sk_flags = e->sk_flags; a.sk_tiles = e->sk_tiles; a.sk_ws_floats = e->sk_ws_floats;
        if ((rc = launch_gemm(e->tmaps, a, e->num_sms, s))) return rc;
      }
    } else {
      GemmArgs a{e->xn + r0 * H, e->cap_T - (int)r0, w.wgu, 2 * e->I, T, 2 * e->I, H, EPI_SWIGLU, 256, 1, e->hbuf + r0 * e->I, nullptr, e->I, 0, e->I, false};
      if ((rc = launch_gemm(e->tmaps, a, e->num_sms, s))) return rc;
    }
    e->launches++;
    if ((rc = row_parallel(e->hbuf, e->I, w.wdown, next_norm))) return rc;
  }
  B200_REQUIRE(e->ar_index == 0 || e->ar_index == 2 * e->L, "peer all-reduce count per step must be 2 per layer");
  if (nv == 2) {
    B200_CUDA_OK(cudaEventRecord(e->ev_join, e->stream2));
    B200_CUDA_OK(cudaStreamWaitEvent(e->stream, e->ev_join, 0));
  }
  return 0;
}

// LM head on `rows` (B x H, already final-normed) -> logits -> per-rank argmax candidates -> step update
static int head_and_step(b200_engine* e, const bf16* rows_xn, int rows_cap, int B, const int32_t* cb_row_slot = nullptr) {
  cudaStream_t s = e->stream;
  int rc;
  GemmArgs a{e->lm_head, e->Vl, rows_xn, rows_cap, e->Vl, B, e->H, EPI_T_STORE, pick_block_n(B), 1,
             e->logits, nullptr, e->Vl, 0, 0, true};
  a.sk_ws = e->sk_ws; a.sk_flags = e->sk_flags; a.sk_tiles = e->sk_tiles; a.sk_ws_floats = e->sk_ws_floats;
  if ((rc = launch_gemm(e->tmaps, a, e->num_sms, s))) return rc;
  const int use_p2p = (e->cfg.tp_size > 1 && e->p2p_ready) ? 1 : 0;
  // one GPU: 16 CTAs per row scan slices of the 128k-entry row (a single CTA per row took 65 us of the 4.3 ms step)
  const int chunks = (e->cfg.tp_size == 1 && e->Vl >= 16384) ? 16 : 1;
  const bool processed = cb_row_slot ? e->cb_sampling_slots > 0 : e->st.sample_on;   // repetition penalty / sampling: sampling.cuh
  if (processed) {
    SampleParams sp{};
    sp.logits = e->logits; sp.ld = e->Vl; sp.V = e->Vl; sp.words = e->seen_words;
    sp.out_val = e->cand_val; sp.out_idx = e->cand_idx;
    if (cb_row_slot) { sp.seen = e->d_seen; sp.cfg = e->d_cb_cfg; sp.row_slot = cb_row_slot; sp.n_gen = e->cb.n_gen; }
    else { sp.seen = e->st.rep_on ? e->d_seen : nullptr; sp.cfg = e->d_sample_cfg; sp.st = e->d_state; }
    B200_CUDA_OK(launch_k(sample_kernel, dim3(B), dim3(1024), 0, s, sp));
  } else {
    B200_CUDA_OK(launch_k(argmax_kernel, dim3(B, chunks), dim3(1024), 0, s, (const bf16*)e->logits, (long long)e->Vl, e->Vl, e->v0, e->cand_val, e->cand_idx, e->p2p, use_p2p));
  }
  e->launches += 2;
  const float* cv = e->cand_val;
  const int32_t* ci = e->cand_idx;
  int ranks = processed ? 1 : chunks;
  if (e->cfg.tp_size > 1 && !use_p2p) {
    Nccl& n = Nccl::get();
    B200_NCCL_OK(n.AllGather(e->cand_val, e->cand_val_all, B, Nccl::kFloat, e->comm, s));
    B200_NCCL_OK(n.AllGather(e->cand_idx, e->cand_idx_all, B, Nccl::kInt32, e->comm, s));
    cv = e->cand_val_all; ci = e->cand_idx_all; ranks = e->cfg.tp_size;
  }
  if (cb_row_slot) {   // continuous batching: per-slot bookkeeping
    B200_CUDA_OK(launch_k(cb_step_kernel, dim3(1), dim3(128), 0, s, cv, ci, ranks, B, cb_row_slot, e->cb, (const int32_t*)e->d_eos, e->cb_num_eos,
                          e->p2p, use_p2p, processed ? e->d_seen : (uint32_t*)nullptr, e->seen_words, e->Vl));
    e->launches++;
    return 0;
  }
  StepParams sp{};
  sp.cand_val = cv; sp.cand_idx = ci; sp.ranks = ranks; sp.B = B;
  sp.forced = e->st.forced ? e->d_forced : nullptr; sp.forced_ld = e->out_ld;
  sp.out_tokens = e->d_out_tokens; sp.out_ld = e->out_ld;
  sp.next_tok = e->d_next_tok; sp.cur_len = e->d_cur_len; sp.tok_pos = e->d_dec_pos; sp.finished = e->d_finished;
  sp.eos = e->d_eos; sp.num_eos = e->st.num_eos; sp.pad_token = e->st.pad;
  sp.stop_tok = e->d_stop_tok; sp.stop_off = e->d_stop_off; sp.num_stop = e->st.num_stop;
  sp.st = e->d_state;
  sp.pp = e->p2p; sp.use_p2p = use_p2p;
  sp.seen = e->st.rep_on ? e->d_seen : nullptr; sp.seen_words = e->seen_words; sp.V = e->Vl;
  B200_CUDA_OK(launch_k(step_update_kernel, dim3(1), dim3(128), 0, s, sp));
  e->launches++;
  return 0;
}

static int prefill(b200_engine* e) {
  auto& st = e->st;
  int rc;
  if (st.rep_on) {   // input_ids of the reference = the prompt (pads included): the tokens the penalty applies to
    B200_CUDA_OK(cudaMemsetAsync(e->d_seen, 0, (size_t)st.B * e->seen_words * 4, e->stream));
    seen_set_kernel<<<32, 256, 0, e->stream>>>(e->d_seen, e->seen_words, e->d_tok, e->d_tok_seq, st.T, e->d_cur_len, st.B, st.S, st.pad, e->Vl);
    B200_CUDA_OK(cudaGetLastError());
    e->launches++;
  }
  if ((rc = forward_layers(e, st.T, st.B, st.max_len, false))) return rc;
  B200_CUDA_OK(launch_k(gather_rows_kernel, dim3(st.B), dim3(128), 0, e->stream, (const bf16*)e->xn, (const int32_t*)e->d_last_rows, e->xl, e->H));
  e->launches++;
  return head_and_step(e, e->xl, e->rows_cap, st.B);
}

static int decode_step_enqueue(b200_engine* e) {
  int rc;
  if ((rc = forward_layers(e, e->st.B, e->st.B, 0, true))) return rc;
  return head_and_step(e, e->xn, e->cap_T, e->st.B);
}

// One decode step through a CUDA graph captured once per key.  The first call for a key runs the step eagerly (tensor
// maps / function attributes are created outside of capture), the second captures it: one chain of programmatic
// dependent launches.
template <class Enqueue>
static int graph_step(b200_engine* e, int key, Enqueue&& enqueue) {
  auto it = e->graphs.find(key);
  if (it == e->graphs.end()) {
    const int before = e->launches;
    int rc = enqueue();
    if (rc) return rc;
    const int per_step = e->launches - before;
    B200_CUDA_OK(cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal));
    rc = enqueue();
    cudaGraph_t g = nullptr;
    cudaError_t ce = cudaStreamEndCapture(e->stream, &g);
    e->launches -= per_step;  // the captured enqueue did not execute
    if (rc) { if (g) cudaGraphDestroy(g); return rc; }
    B200_CUDA_OK(ce);
    cudaGraphExec_t ge = nullptr;
    B200_CUDA_OK(cudaGraphInstantiate(&ge, g, 0));
    cudaGraphDestroy(g);
    e->graphs[key] = ge;
    e->graph_nodes[key] = per_step;
    return 0;  // the eager step above already advanced the sequences by one token
  }
  B200_CUDA_OK(cudaGraphLaunch(it->second, e->stream));
  e->launches += e->graph_nodes[key];
  return 0;
}

static int decode_step(b200_engine* e, bool use_graph) {
  if (!use_graph) return decode_step_enqueue(e);
  const int key = e->st.B | (e->st.forced ? 1 << 8 : 0) | (e->st.num_eos << 9) | (e->st.num_stop << 14) |
                  (e->st.sample_on ? 1 << 21 : 0) | (e->st.rep_on ? 1 << 22 : 0);
  return graph_step(e, key, [&] { return decode_step_enqueue(e); });
}

// Validates the request, sizes the KV pages and resets the per-request device state.  `lens` are the real
// (un-padded) sequence lengths; S is the padded prompt width (0 for ragged batcher input).
static int stage_common(b200_engine* e, int B, int S, const std::vector<int>& lens, const b200_gen_params_t* gp) {
  B200_REQUIRE(e->finalized, "weights not finalized");
  B200_REQUIRE(!e->faulted, "engine fault: an earlier device-side wait timed out; re-create the engine");
  B200_REQUIRE(!e->cb_on, "engine is in continuous-batching mode (b200_cb_end first)");
  B200_REQUIRE(B >= 1 && B <= e->rows_cap, "batch size out of range (one generate call covers at most 64 rows)");
  B200_REQUIRE(gp->max_new_tokens >= 1, "max_new_tokens must be >= 1");
  B200_REQUIRE(gp->num_eos <= 16 && gp->num_stop <= 16, "too many eos / stop sequences");
  auto& st = e->st;
  st.B = B; st.S = S; st.max_new = gp->max_new_tokens; st.lens = lens;
  st.pad = (int32_t)gp->pad_token_id; st.num_eos = gp->num_eos; st.num_stop = gp->num_stop;
  st.forced = gp->forced_tokens != nullptr; st.prefilled = false;
  int T = 0, max_len = 0;
  for (int b = 0; b < B; ++b) {
    B200_REQUIRE(lens[b] >= 1, "empty sequence");
    T += lens[b];
    max_len = std::max(max_len, lens[b]);
  }
  const int width = std::max(S, max_len);
  B200_REQUIRE(width + gp->max_new_tokens <= e->cfg.max_seq_len, "prompt + max_new_tokens exceeds max_seq_len");
  B200_REQUIRE(width + gp->max_new_tokens <= e->cfg.max_position, "exceeds rope table");
  B200_REQUIRE(T <= e->cap_T, "packed prompt tokens exceed max_prefill_tokens");
  st.T = T; st.max_len = max_len;
  // page allocation: sequence b owns a contiguous run of pages (fresh allocator per call)
  const int per_seq = (width + gp->max_new_tokens + kPageTokens - 1) / kPageTokens;
  B200_REQUIRE(per_seq <= e->max_pages && (long long)per_seq * B <= e->num_pages, "KV page pool too small");
  st.per_seq_pages = per_seq;
  std::fill(e->h_page_table.begin(), e->h_page_table.end(), 0);
  for (int b = 0; b < B; ++b)
    for (int i = 0; i < per_seq; ++i) e->h_page_table[(size_t)b * e->max_pages + i] = b * per_seq + i;
  cudaStream_t s = e->stream;
  B200_CUDA_OK(cudaMemcpyAsync(e->d_page_table, e->h_page_table.data(), e->h_page_table.size() * 4, cudaMemcpyHostToDevice, s));
  // eos / stop / forced
  std::vector<int32_t> tmp;
  if (gp->num_eos) {
    tmp.assign(gp->num_eos, 0);
    for (int i = 0; i < gp->num_eos; ++i) tmp[i] = (int32_t)gp->eos_token_ids[i];
    B200_CUDA_OK(cudaMemcpy(e->d_eos, tmp.data(), tmp.size() * 4, cudaMemcpyHostToDevice));
  }
  if (gp->num_stop) {
    const int total = gp->stop_offsets[gp->num_stop];
    B200_REQUIRE(total <= 1024, "stop sequences too long");
    tmp.assign(total, 0);
    for (int i = 0; i < total; ++i) tmp[i] = (int32_t)gp->stop_tokens[i];
    B200_CUDA_OK(cudaMemcpy(e->d_stop_tok, tmp.data(), tmp.size() * 4, cudaMemcpyHostToDevice));
    B200_CUDA_OK(cudaMemcpy(e->d_stop_off, gp->stop_offsets, (gp->num_stop + 1) * 4, cudaMemcpyHostToDevice));
  }
  if (gp->forced_tokens) {
    tmp.assign((size_t)B * e->out_ld, 0);
    for (int b = 0; b < B; ++b)
      for (int i = 0; i < gp->max_new_tokens; ++i) tmp[(size_t)b * e->out_ld + i] = (int32_t)gp->forced_tokens[(size_t)b * gp->max_new_tokens + i];
    B200_CUDA_OK(cudaMemcpy(e->d_forced, tmp.data(), tmp.size() * 4, cudaMemcpyHostToDevice));
  }
  StepState init{0, 0, 0, gp->max_new_tokens};
  *e->h_state = init;
  B200_CUDA_OK(cudaMemcpyAsync(e->d_state, e->h_state, sizeof(StepState), cudaMemcpyHostToDevice, s));
  // logits processors / sampling (build_generation_config, generative_model.py:388-402)
  SampleCfg sc{};
  sc.rep_penalty = (gp->repetition_penalty > 0.f) ? gp->repetition_penalty : 1.0f;
  sc.temperature = (gp->temperature > 0.f) ? gp->temperature : 1.0f;
  sc.do_sample = gp->do_sample ? 1 : 0;
  sc.top_p = (gp->top_p > 0.f && gp->top_p < 1.f) ? gp->top_p : 1.0f;
  sc.top_k = gp->top_k > 0 ? std::min(gp->top_k, kSampleMaxCand) : 50;
  sc.seed = gp->seed;
  st.rep_on = sc.rep_penalty != 1.0f;
  st.sample_on = st.rep_on || sc.do_sample;
  if (st.sample_on) {
    B200_REQUIRE(e->cfg.tp_size == 1, "logits processors / sampling run on one GPU per engine (tp_size == 1)");
    if (!e->d_sample_cfg) B200_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&e->d_sample_cfg), sizeof(SampleCfg)));
    B200_CUDA_OK(cudaMemcpy(e->d_sample_cfg, &sc, sizeof(sc), cudaMemcpyHostToDevice));
    if (st.rep_on && !e->d_seen) {
      e->seen_words = (e->Vl + 31) / 32;
      B200_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&e->d_seen), (size_t)e->cfg.max_batch * e->seen_words * 4));
    }
  }
  return 0;
}

static PackOut pack_out(b200_engine* e) {
  return PackOut{e->d_tok, e->d_tok_seq, e->d_tok_pos, e->d_cu, e->d_seq_slot, e->d_last_rows, e->d_cur_len, e->d_dec_pos, e->d_finished};
}

// Padded [B][S] ids (+ left-padding mask) as they arrive on the OpenAI / V2 legs: the raw rows are copied to
// the device once and concatenated into the packed layout by pack_padded_kernel.
static int stage_prompt(b200_engine* e, const int64_t* ids, const int64_t* mask, int B, int S,
                        const b200_gen_params_t* gp) {
  B200_REQUIRE(B >= 1 && B <= e->rows_cap && S >= 1 && S <= e->cfg.max_seq_len, "bad batch shape");
  std::vector<int> lens(B, S);
  if (mask) {
    for (int b = 0; b < B; ++b) {
      int first = 0;
      while (first < S && mask[(size_t)b * S + first] == 0) ++first;
      for (int i = first; i < S; ++i)
        B200_REQUIRE(mask[(size_t)b * S + i] != 0, "attention_mask must be left padding only");
      lens[b] = S - first;
    }
  }
  int rc = stage_common(e, B, S, lens, gp);
  if (rc) return rc;
  e->staged_mask = mask != nullptr;
  e->st.input.assign(ids, ids + (size_t)B * S);
  cudaStream_t s = e->stream;
  const size_t n = (size_t)B * S;
  memcpy(e->h_raw, ids, n * 8);
  B200_CUDA_OK(cudaMemcpyAsync(e->d_raw_ids, e->h_raw, n * 8, cudaMemcpyHostToDevice, s));
  if (mask) {
    memcpy(e->h_raw + n, mask, n * 8);
    B200_CUDA_OK(cudaMemcpyAsync(e->d_raw_mask, e->h_raw + n, n * 8, cudaMemcpyHostToDevice, s));
  }
  pack_padded_kernel<<<1, 1024, 0, s>>>(e->d_raw_ids, mask ? e->d_raw_mask : nullptr, B, S, pack_out(e));
  B200_CUDA_OK(cudaGetLastError());
  e->launches++;
  return 0;
}

// Ragged rows as the batcher hands them over (one row per instance of every waiting request).
static int stage_ragged(b200_engine* e, const int64_t* const* rows, const int32_t* row_lens, int B,
                        const b200_gen_params_t* gp) {
  B200_REQUIRE(B >= 1 && B <= e->rows_cap, "batch size out of range");
  std::vector<int> lens(row_lens, row_lens + B);
  int rc = stage_common(e, B, 0, lens, gp);
  if (rc) return rc;
  e->st.input.clear();
  int32_t* flat = reinterpret_cast<int32_t*>(e->h_raw);
  int32_t* offs = flat + e->cap_T;
  int t = 0;
  for (int b = 0; b < B; ++b) {
    offs[b] = t;
    for (int i = 0; i < lens[b]; ++i) flat[t++] = (int32_t)rows[b][i];
  }
  offs[B] = t;
  cudaStream_t s = e->stream;
  B200_CUDA_OK(cudaMemcpyAsync(e->d_flat, flat, (size_t)t * 4, cudaMemcpyHostToDevice, s));
  B200_CUDA_OK(cudaMemcpyAsync(e->d_offs, offs, (size_t)(B + 1) * 4, cudaMemcpyHostToDevice, s));
  pack_ragged_kernel<<<1, 1024, 0, s>>>(e->d_flat, e->d_offs, B, pack_out(e));
  B200_CUDA_OK(cudaGetLastError());
  e->launches++;
  return 0;
}

// called right after a stream synchronisation: did any wait of the kernels just run give up?
static int check_fault(b200_engine* e) {
  int code = 0;
  B200_CUDA_OK(cudaMemcpyFromSymbol(&code, g_fault_code, sizeof(int)));
  if (code == 0) return 0;
  e->faulted = true;
  static const char* what[] = {"", "peer flag", "peer all-reduce packet", "peer candidate exchange", "stream-K piece"};
  set_last_error(std::string("engine fault: a device-side wait timed out (") + (code >= 1 && code <= 4 ? what[code] : "?") +
                 ") — a tensor-parallel peer is gone or out of step; this engine is unusable until it is re-created");
  return -8;
}

static int fetch_result(b200_engine* e, int64_t* out_ids, int32_t* out_len, int32_t* stop_triggered) {
  auto& st = e->st;
  cudaStream_t s = e->stream;
  B200_CUDA_OK(cudaMemcpyAsync(e->h_state, e->d_state, sizeof(StepState), cudaMemcpyDeviceToHost, s));
  B200_CUDA_OK(cudaMemcpyAsync(e->h_out_tokens, e->d_out_tokens, (size_t)st.B * e->out_ld * 4, cudaMemcpyDeviceToHost, s));
  B200_CUDA_OK(cudaStreamSynchronize(s));
  { int frc = check_fault(e); if (frc) return frc; }
  const int Tn = e->h_state->step;
  const int W = st.S + st.max_new;
  for (int b = 0; b < st.B; ++b) {
    for (int i = 0; i < st.S; ++i) out_ids[(size_t)b * W + i] = st.input[(size_t)b * st.S + i];
    for (int i = 0; i < st.max_new; ++i)
      out_ids[(size_t)b * W + st.S + i] = i < Tn ? (int64_t)e->h_out_tokens[(size_t)b * e->out_ld + i] : (int64_t)st.pad;
  }
  *out_len = st.S + Tn;
  if (stop_triggered) *stop_triggered = e->h_state->stop_triggered;
  return 0;
}


// ---- continuous batching ---------------------------------------------------------------------------
static int cb_alloc(b200_engine* e) {
  if (e->cb.len) return 0;
  const size_t nb = (size_t)e->cfg.max_batch;
  int rc;
  if ((rc = dmalloc(&e->cb.len, nb))) return rc;
  if ((rc = dmalloc(&e->cb.n_gen, nb))) return rc;
  if ((rc = dmalloc(&e->cb.max_new, nb))) return rc;
  if ((rc = dmalloc(&e->cb.finished, nb))) return rc;
  if ((rc = dmalloc(&e->cb.stop_hit, nb))) return rc;
  if ((rc = dmalloc(&e->cb.next_tok, nb))) return rc;
  if ((rc = dmalloc(&e->cb.stop_len, nb * kCbMaxStop))) return rc;
  if ((rc = dmalloc(&e->cb.stop_tok, nb * kCbMaxStop * kCbMaxStopLen))) return rc;
  if ((rc = dmalloc(&e->d_cb_row_slot, nb))) return rc;
  if ((rc = dmalloc(&e->d_cb_rec, nb * kCbInitInts))) return rc;
  if ((rc = dmalloc(&e->d_cb_cfg, nb))) return rc;
  if ((rc = dmalloc(&e->d_kv_off, (size_t)80))) return rc;
  e->cb.out = e->d_out_tokens; e->cb.out_ld = e->out_ld;
  const size_t host_ints = std::max(nb * kCbInitInts, std::max((size_t)e->out_ld, 4 * nb));
  B200_CUDA_OK(cudaMallocHost(reinterpret_cast<void**>(&e->h_cb), host_ints * 4));
  B200_CUDA_OK(cudaMallocHost(reinterpret_cast<void**>(&e->h_cb_rows), (size_t)8 * kMaxRows * 4));
  return 0;
}

static int cb_decode_enqueue(b200_engine* e, int R) {
  int rc;
  B200_CUDA_OK(launch_k(cb_gather_kernel, dim3(1), dim3(64), 0, e->stream, (const int32_t*)e->d_cb_row_slot, R, e->cb, e->d_next_tok,
                        e->d_seq_slot, e->d_dec_pos));
  e->launches++;
  if ((rc = forward_layers(e, R, R, 0, true))) return rc;
  return head_and_step(e, e->xn, e->cap_T, R, e->d_cb_row_slot);
}

// one decode iteration through a CUDA graph keyed by the row count.  At most kMaxRows sequences ride in one pass: with
// more than that running, a window rotates over them (round robin), so every admitted sequence keeps advancing — the
// pass streams the weights once whatever the row count, so aggregate tokens/s is that of a full 64-row batch while new
// requests do not queue for a slot (config 5: 512 concurrent clients).
static int cb_decode_step(b200_engine* e) {
  const int Rt = (int)e->cb_active.size();
  if (Rt == 0) return 0;
  const int R = std::min(Rt, kMaxRows);
  if (e->cb_rows_dirty || Rt > kMaxRows) {
    int32_t* ring = e->h_cb_rows + (size_t)(e->cb_ring_pos % 8) * kMaxRows;
    if (e->cb_ring_pos && (e->cb_ring_pos % 8) == 0) B200_CUDA_OK(cudaStreamSynchronize(e->stream));   // the ring slot's last copy is long done
    ++e->cb_ring_pos;
    const int start = Rt > kMaxRows ? (int)(e->cb_window % Rt) : 0;
    for (int r = 0; r < R; ++r) ring[r] = e->cb_active[(start + r) % Rt];
    if (Rt > kMaxRows) e->cb_window += R;
    B200_CUDA_OK(cudaMemcpyAsync(e->d_cb_row_slot, ring, (size_t)R * 4, cudaMemcpyHostToDevice, e->stream));
    e->cb_rows_dirty = false;
  }
  static const bool eager = getenv("B200_NO_GRAPH") != nullptr;
  if (eager) return cb_decode_enqueue(e, R);
  const int key = R | (1 << 20) | (e->cb_num_eos << 9) | (e->cb_sampling_slots > 0 ? 1 << 21 : 0);
  return graph_step(e, key, [&] { return cb_decode_enqueue(e, R); });
}

// ---- KV page pool + prefix cache ---------------------------------------------------------------------
static unsigned long long cb_block_hash(unsigned long long parent, const int32_t* toks) {   // FNV-1a over 128 tokens, chained
  unsigned long long h = parent ^ 0xcbf29ce484222325ull;
  for (int i = 0; i < 128; ++i) { h ^= (unsigned long long)(uint32_t)toks[i]; h *= 0x100000001b3ull; }
  return h ? h : 1ull;
}

static void cb_unref_page(b200_engine* e, int pg) {
  if (--e->cb_page_ref[pg] == 0) e->cb_free_pages.push_back(pg);
}

// frees the least recently used cached block nobody else references; false when nothing can be evicted
static bool cb_evict_one(b200_engine* e) {
  unsigned long long best_key = 0, best_tick = ~0ull;
  for (auto& kv : e->cb_prefix) {
    const auto& en = kv.second;
    if (e->cb_page_ref[en.p0] == 1 && e->cb_page_ref[en.p1] == 1 && en.tick < best_tick) { best_tick = en.tick; best_key = kv.first; }
  }
  if (best_tick == ~0ull) return false;
  auto it = e->cb_prefix.find(best_key);
  cb_unref_page(e, it->second.p0);
  cb_unref_page(e, it->second.p1);
  e->cb_prefix.erase(it);
  e->cb_stat[3]++;
  return true;
}

static int cb_take_page(b200_engine* e) {
  while (e->cb_free_pages.empty())
    if (!cb_evict_one(e)) return -1;
  const int pg = e->cb_free_pages.back();
  e->cb_free_pages.pop_back();
  e->cb_page_ref[pg] = 1;
  return pg;
}

// One prefill pass over (chunks of) the pending prompts, at most `budget` packed tokens: sequences whose last chunk is
// in this pass get their first token and join the decode batch.  Chunks end on multiples of 128 tokens (the attention
// kernel's query tiles stay aligned with its KV tiles); a prompt's cached prefix (shared pages) is never recomputed.
static int cb_prefill_pending(b200_engine* e, long long budget) {
  if (e->cb_pending.empty()) return 0;
  budget = std::min<long long>(budget, e->cap_T);
  struct Part { size_t idx; int start, count; bool fin; };
  std::vector<Part> parts;
  long long left = budget;
  for (size_t i = 0; i < e->cb_pending.size() && (int)parts.size() < e->rows_cap; ++i) {
    const auto& pd = e->cb_pending[i];
    const int rem = (int)pd.toks.size() - pd.done;
    int c = rem <= left ? rem : (int)((left / 128) * 128);
    if (c <= 0) break;
    parts.push_back(Part{i, pd.done, c, c == rem});
    left -= c;
    if (c < rem) break;       // budget exhausted inside this prompt: FIFO, later prompts wait
  }
  if (parts.empty()) return 0;
  const int n = (int)parts.size();
  int T = 0, max_len = 0, nfin = 0;
  for (auto& pt : parts) { T += pt.count; max_len = std::max(max_len, pt.count); nfin += pt.fin ? 1 : 0; }
  cudaStream_t s = e->stream;
  int32_t* flat = e->h_stage;   // tok | tok_seq | tok_pos | cu | seq_slot | kv_off | last_rows | fin_slot
  B200_REQUIRE((size_t)(3 * T + 5 * n + 1) <= e->h_stage_elems, "prompt staging buffer too small");
  int32_t *h_tok = flat, *h_seq = flat + T, *h_pos = flat + 2 * T, *h_cu = flat + 3 * T, *h_slot = h_cu + n + 1, *h_off = h_slot + n,
          *h_last = h_off + n, *h_fin = h_last + n;
  int t = 0, f = 0;
  std::vector<int> lens(n);
  for (int i = 0; i < n; ++i) {
    const auto& pd = e->cb_pending[parts[i].idx];
    h_cu[i] = t;
    for (int k = 0; k < parts[i].count; ++k, ++t) { h_tok[t] = pd.toks[parts[i].start + k]; h_seq[t] = pd.slot; h_pos[t] = parts[i].start + k; }
    h_slot[i] = pd.slot; h_off[i] = parts[i].start; lens[i] = parts[i].count;
    if (parts[i].fin) { h_last[f] = t - 1; h_fin[f] = pd.slot; ++f; }
  }
  h_cu[n] = t;
  B200_CUDA_OK(cudaMemcpyAsync(e->d_tok, h_tok, (size_t)T * 4, cudaMemcpyHostToDevice, s));
  B200_CUDA_OK(cudaMemcpyAsync(e->d_tok_seq, h_seq, (size_t)T * 4, cudaMemcpyHostToDevice, s));
  B200_CUDA_OK(cudaMemcpyAsync(e->d_tok_pos, h_pos, (size_t)T * 4, cudaMemcpyHostToDevice, s));
  B200_CUDA_OK(cudaMemcpyAsync(e->d_cu, h_cu, (size_t)(n + 1) * 4, cudaMemcpyHostToDevice, s));
  B200_CUDA_OK(cudaMemcpyAsync(e->d_seq_slot, h_slot, (size_t)n * 4, cudaMemcpyHostToDevice, s));
  B200_CUDA_OK(cudaMemcpyAsync(e->d_kv_off, h_off, (size_t)n * 4, cudaMemcpyHostToDevice, s));
  if (nfin) {
    B200_CUDA_OK(cudaMemcpyAsync(e->d_last_rows, h_last, (size_t)nfin * 4, cudaMemcpyHostToDevice, s));
    B200_CUDA_OK(cudaMemcpyAsync(e->d_cb_rec, h_fin, (size_t)nfin * 4, cudaMemcpyHostToDevice, s));   // row -> slot of the finishing rows
  }
  int rc;
  e->st.lens = lens;
  if ((rc = forward_layers(e, T, n, max_len, false, e->d_kv_off))) return rc;
  if (nfin) {
    B200_CUDA_OK(launch_k(gather_rows_kernel, dim3(nfin), dim3(128), 0, s, (const bf16*)e->xn, (const int32_t*)e->d_last_rows, e->xl, e->H));
    e->launches++;
    if ((rc = head_and_step(e, e->xl, e->rows_cap, nfin, e->d_cb_rec))) return rc;
  }
  B200_CUDA_OK(cudaStreamSynchronize(s));   // h_stage is reused by the next pass
  e->cb_stat[2] += T; e->cb_stat[4]++;
  // bookkeeping (front to back so that erasing does not disturb the indices still to be visited)
  for (int i = n - 1; i >= 0; --i) {
    auto& pd = e->cb_pending[parts[i].idx];
    pd.done += parts[i].count;
    if (!parts[i].fin) continue;
    if (e->cb_prefix_on) {   // every full 128-token block of the prompt can now be shared with later requests
      const auto& pages = e->cb_slot_pages[pd.slot];
      unsigned long long parent = 0;
      for (size_t k = 0; k < pd.block_hash.size(); ++k) {
        const unsigned long long key = pd.block_hash[k];
        if (!e->cb_prefix.count(key)) {
          b200_engine::PrefixEntry en{pages[2 * k], pages[2 * k + 1], parent, ++e->cb_tick,
                                      std::vector<int32_t>(pd.toks.begin() + 128 * k, pd.toks.begin() + 128 * (k + 1))};
          e->cb_page_ref[en.p0]++; e->cb_page_ref[en.p1]++;
          e->cb_prefix.emplace(key, std::move(en));
        }
        parent = key;
      }
    }
    e->cb_active.push_back(pd.slot);
    e->cb_rows_dirty = true;
    e->cb_pending.erase(e->cb_pending.begin() + parts[i].idx);
  }
  return 0;
}

// admit `n` new sequences: slots, KV pages (shared with cached prefixes where possible), per-sequence state; their
// prompts are prefilled here (cb_chunk_tokens == 0) or chunk by chunk between the following decode steps
static int cb_admit(b200_engine* e, int n, const int64_t* const* rows, const int32_t* lens, const int32_t* max_new,
                    const int32_t* stop_count, const int32_t* stop_offsets, const int64_t* stop_tokens,
                    const b200_gen_params_t* sampling, int32_t* slots_out) {
  B200_REQUIRE(e->cb_on, "b200_cb_begin was not called");
  B200_REQUIRE(n >= 1 && n <= e->cfg.max_batch, "nothing to admit / more prompts than slots");
  int free_slots = 0;
  for (char u : e->cb_used) free_slots += u ? 0 : 1;
  B200_REQUIRE(n <= free_slots, "not enough free slots");
  long long T = 0;
  for (int i = 0; i < n; ++i) {
    B200_REQUIRE(lens[i] >= 1 && max_new[i] >= 1, "empty sequence / max_new < 1");
    B200_REQUIRE(lens[i] + max_new[i] <= e->cfg.max_seq_len && lens[i] + max_new[i] <= e->cfg.max_position, "prompt + max_new exceeds max_seq_len");
    T += lens[i];
  }
  B200_REQUIRE(e->cb_chunk_tokens > 0 || T <= e->cap_T, "packed prompt tokens exceed max_prefill_tokens (enable chunked prefill: b200_cb_config)");
  cudaStream_t s = e->stream;
  std::vector<int> slots;
  for (int sl = 0; sl < (int)e->cb_used.size() && (int)slots.size() < n; ++sl)
    if (!e->cb_used[sl]) slots.push_back(sl);
  // ---- pages: plan every prompt first; on exhaustion everything taken so far is handed back
  std::vector<b200_engine::CbPending> plans(n);
  long long stat_prompt = 0, stat_hit = 0;      // counted only when the whole admit goes through
  auto rollback = [&](int upto) {
    for (int i = 0; i < upto; ++i) {
      for (int pg : e->cb_slot_pages[slots[i]]) cb_unref_page(e, pg);
      e->cb_slot_pages[slots[i]].clear();
    }
  };
  for (int i = 0; i < n; ++i) {
    auto& pd = plans[i];
    pd.slot = slots[i];
    pd.toks.resize(lens[i]);
    for (int k = 0; k < lens[i]; ++k) pd.toks[k] = (int32_t)rows[i][k];
    const int need = (lens[i] + max_new[i] + kPageTokens - 1) / kPageTokens;
    std::vector<int>& pages = e->cb_slot_pages[slots[i]];
    pages.clear();
    int hit_blocks = 0;
    const int full_blocks = lens[i] / 128;
    if (e->cb_prefix_on) {
      unsigned long long parent = 0;
      bool chain = true;
      for (int k = 0; k < full_blocks; ++k) {
        const unsigned long long key = cb_block_hash(parent, pd.toks.data() + 128 * k);
        pd.block_hash.push_back(key);
        // at least one token must be left to compute (its logits select the first generated token)
        if (chain && 128 * (k + 1) < lens[i]) {
          auto it = e->cb_prefix.find(key);
          if (it != e->cb_prefix.end() && it->second.parent == parent &&
              memcmp(it->second.toks.data(), pd.toks.data() + 128 * k, 128 * sizeof(int32_t)) == 0) {
            it->second.tick = ++e->cb_tick;
            e->cb_page_ref[it->second.p0]++; e->cb_page_ref[it->second.p1]++;
            pages.push_back(it->second.p0); pages.push_back(it->second.p1);
            hit_blocks = k + 1;
          } else {
            chain = false;
          }
        } else {
          chain = false;
        }
        parent = key;
      }
    }
    pd.done = hit_blocks * 128;
    while ((int)pages.size() < need) {
      const int pg = cb_take_page(e);
      if (pg < 0) {
        rollback(i + 1);
        set_last_error("KV page pool exhausted: release finished sequences first");
        return -7;
      }
      pages.push_back(pg);
    }
    stat_prompt += lens[i]; stat_hit += pd.done;
  }
  for (int i = 0; i < n; ++i) {
    const std::vector<int>& pages = e->cb_slot_pages[slots[i]];
    int32_t* row = e->h_page_table.data() + (size_t)slots[i] * e->max_pages;
    for (int k = 0; k < e->max_pages; ++k) row[k] = k < (int)pages.size() ? pages[k] : pages.back();
    B200_CUDA_OK(cudaMemcpyAsync(e->d_page_table + (size_t)slots[i] * e->max_pages, row, (size_t)e->max_pages * 4, cudaMemcpyHostToDevice, s));
  }
  // ---- per-sequence device state
  int so = 0;   // running index into stop_offsets
  for (int i = 0; i < n; ++i) {
    int32_t* r = e->h_cb + (size_t)i * kCbInitInts;
    for (int j = 0; j < kCbInitInts; ++j) r[j] = 0;
    r[0] = slots[i]; r[1] = lens[i]; r[2] = max_new[i];
    const int ns = stop_count ? stop_count[i] : 0;
    if (ns > kCbMaxStop) { rollback(n); set_last_error("too many stop sequences for one sequence"); return -2; }
    r[3] = ns;
    for (int j = 0; j < ns; ++j, ++so) {
      const int o = stop_offsets[so], len = stop_offsets[so + 1] - o;
      if (len < 0 || len > kCbMaxStopLen) { rollback(n); set_last_error("stop sequence too long"); return -2; }
      r[4 + j] = len;
      for (int k = 0; k < len; ++k) r[4 + kCbMaxStop + j * kCbMaxStopLen + k] = (int32_t)stop_tokens[o + k];
    }
  }
  B200_CUDA_OK(cudaMemcpyAsync(e->d_cb_rec, e->h_cb, (size_t)n * kCbInitInts * 4, cudaMemcpyHostToDevice, s));
  cb_init_kernel<<<n, 64, 0, s>>>(e->d_cb_rec, n, e->cb);
  B200_CUDA_OK(cudaGetLastError());
  // ---- logits processors / sampling per sequence (build_generation_config, generative_model.py:388-402)
  for (int i = 0; i < n; ++i) {
    SampleCfg sc{};
    sc.rep_penalty = 1.0f; sc.temperature = 1.0f; sc.top_p = 1.0f; sc.top_k = 50;
    bool on = false;
    if (sampling) {
      const b200_gen_params_t& gp = sampling[i];
      sc.rep_penalty = (gp.repetition_penalty > 0.f) ? gp.repetition_penalty : 1.0f;
      sc.temperature = (gp.temperature > 0.f) ? gp.temperature : 1.0f;
      sc.do_sample = gp.do_sample ? 1 : 0;
      sc.top_p = (gp.top_p > 0.f && gp.top_p < 1.f) ? gp.top_p : 1.0f;
      sc.top_k = gp.top_k > 0 ? std::min(gp.top_k, kSampleMaxCand) : 50;
      sc.seed = gp.seed;
      on = sc.rep_penalty != 1.0f || sc.do_sample;
    }
    if (on && e->cfg.tp_size != 1) { rollback(n); set_last_error("logits processors / sampling run on one GPU per engine (tp_size == 1)"); return -2; }
    B200_CUDA_OK(cudaMemcpyAsync(e->d_cb_cfg + slots[i], &sc, sizeof(sc), cudaMemcpyHostToDevice, s));   // (pageable source: staged before return)
    if (on && sc.rep_penalty != 1.0f) {
      if (!e->d_seen) {
        e->seen_words = (e->Vl + 31) / 32;
        B200_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&e->d_seen), (size_t)e->cfg.max_batch * e->seen_words * 4));
      }
      std::vector<uint32_t> bits(e->seen_words, 0u);      // the reference's input_ids = the prompt tokens
      for (int32_t tk : plans[i].toks)
        if (tk >= 0 && tk < e->Vl) bits[tk >> 5] |= 1u << (tk & 31);
      B200_CUDA_OK(cudaMemcpy(e->d_seen + (size_t)slots[i] * e->seen_words, bits.data(), bits.size() * 4, cudaMemcpyHostToDevice));
    } else if (e->d_seen && on) {
      B200_CUDA_OK(cudaMemsetAsync(e->d_seen + (size_t)slots[i] * e->seen_words, 0, (size_t)e->seen_words * 4, s));
    }
    if (on) { e->cb_slot_sampling[slots[i]] = 1; e->cb_sampling_slots++; }
  }
  if (e->cb_sampling_slots > 0 && !e->d_seen) {   // the step kernel updates the bitmaps whenever the processed path is on
    e->seen_words = (e->Vl + 31) / 32;
    B200_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&e->d_seen), (size_t)e->cfg.max_batch * e->seen_words * 4));
    B200_CUDA_OK(cudaMemset(e->d_seen, 0, (size_t)e->cfg.max_batch * e->seen_words * 4));
  }
  B200_CUDA_OK(cudaStreamSynchronize(s));   // h_cb / sc are reused
  e->cb_stat[0] += stat_prompt; e->cb_stat[1] += stat_hit;
  for (int i = 0; i < n; ++i) {
    e->cb_used[slots[i]] = 1;
    slots_out[i] = slots[i];
    e->cb_pending.push_back(std::move(plans[i]));
  }
  if (e->cb_chunk_tokens == 0) {
    while (!e->cb_pending.empty()) {
      int rc = cb_prefill_pending(e, LLONG_MAX);
      if (rc) return rc;
    }
  }
  return 0;
}

// shard copy helpers -------------------------------------------------------------------------------
static int copy_rows(bf16* dst, const bf16* src, long long row0, long long rows, long long cols, bool on_device) {
  B200_CUDA_OK(cudaMemcpy(dst, src + row0 * cols, (size_t)rows * cols * 2, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
  return 0;
}
static int copy_cols(bf16* dst, const bf16* src, long long rows, long long src_cols, long long col0, long long cols, bool on_device) {
  B200_CUDA_OK(cudaMemcpy2D(dst, cols * 2, src + col0, src_cols * 2, cols * 2, rows, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
  return 0;
}

}  // namespace b200

// =====================================================================================================
// C ABI
// =====================================================================================================
extern "C" {

const char* b200_last_error(void) { return g_last_error.c_str(); }
const char* b200_version(void) { return "kserve_b200 0.2 (sm_100a)"; }

int b200_nccl_unique_id(void* out128) {
  Nccl& n = Nccl::get();
  B200_REQUIRE(n.ok, "libnccl.so.2 could not be loaded");
  Nccl::UniqueId id;
  B200_NCCL_OK(n.GetUniqueId(&id));
  memcpy(out128, &id, 128);
  return 0;
}

int b200_engine_create(const b200_model_config_t* c, const void* nccl_id, b200_engine_t** out) {
  B200_REQUIRE(c && out, "null argument");
  B200_REQUIRE(c->head_dim == kHeadDim, "head_dim must be 128");
  B200_REQUIRE(c->tp_size >= 1 && c->tp_rank >= 0 && c->tp_rank < c->tp_size, "bad tp rank/size");
  B200_REQUIRE(c->num_heads % c->tp_size == 0 && c->num_kv_heads % c->tp_size == 0, "heads must divide tp_size");
  B200_REQUIRE(c->intermediate_size % (16 * c->tp_size) == 0, "intermediate_size must be a multiple of 16*tp_size");
  B200_REQUIRE(c->hidden_size % 64 == 0, "hidden_size must be a multiple of 64");
  // max_batch = sequences the engine can hold at once (KV pages, per-sequence state).  One forward pass still covers at most
  // kMaxRows = 64 of them: a static generate call is limited to 64 rows, the continuous batcher rotates a 64-row window
  // over the running sequences when more than 64 are live.
  B200_REQUIRE(c->max_batch >= 1 && c->max_batch <= 512, "max_batch must be in [1, 512]");
  B200_REQUIRE(c->num_heads % c->num_kv_heads == 0 && c->num_heads / c->num_kv_heads <= 8, "GQA group must be <= 8");
  int ndev = 0;
  B200_CUDA_OK(cudaGetDeviceCount(&ndev));
  B200_REQUIRE(c->device >= 0 && c->device < ndev, "no such CUDA device (this library has no CPU fallback)");
  B200_CUDA_OK(cudaSetDevice(c->device));
  cudaDeviceProp prop;
  B200_CUDA_OK(cudaGetDeviceProperties(&prop, c->device));
  B200_REQUIRE(prop.major == 10, std::string("kserve_b200 kernels are built for sm_100a only; device is sm_") +
                                     std::to_string(prop.major) + std::to_string(prop.minor));
  std::unique_ptr<b200_engine> e(new b200_engine());
  e->cfg = *c;
  e->num_sms = prop.multiProcessorCount;
  const int tp = c->tp_size;
  e->H = c->hidden_size; e->nh = c->num_heads / tp; e->nkv = c->num_kv_heads / tp; e->G = c->num_heads / c->num_kv_heads;
  e->I = c->intermediate_size / tp; e->V = c->vocab_size; e->L = c->num_layers;
  e->E = c->num_experts;
  B200_REQUIRE(e->E == 0 || (e->E <= kMaxExperts && e->E >= 2 && c->num_experts_per_tok == kTopK), "MoE needs 2..16 experts and top-2 routing");
  const int vper = (c->vocab_size + tp - 1) / tp;
  e->v0 = vper * c->tp_rank;
  e->Vl = std::max(0, std::min(vper, c->vocab_size - e->v0));
  B200_REQUIRE(e->Vl > 0, "empty vocabulary shard");
  e->qkv_cols = (e->nh + 2 * e->nkv) * kHeadDim;
  B200_CUDA_OK(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
  B200_CUDA_OK(cudaStreamCreateWithFlags(&e->stream2, cudaStreamNonBlocking));
  B200_CUDA_OK(cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming));
  B200_CUDA_OK(cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming));
  if (getenv("B200_WAIT_TIMEOUT_MS")) {   // bound of the device-side waits (default 5 s), see common.cuh
    const unsigned long long ns = 1000000ull * (unsigned long long)std::max(1, atoi(getenv("B200_WAIT_TIMEOUT_MS")));
    B200_CUDA_OK(cudaMemcpyToSymbol(g_wait_timeout_ns, &ns, sizeof(ns)));
  }
  B200_CUDA_OK(cudaEventCreate(&e->ev0));
  B200_CUDA_OK(cudaEventCreate(&e->ev1));
  B200_CUDA_OK(cudaEventCreate(&e->ev2));
  int rc;
  const size_t H = e->H;
  // weights
  if ((rc = dmalloc(&e->embed, (size_t)e->V * H))) return rc;
  if ((rc = dmalloc(&e->lm_head, (size_t)e->Vl * H))) return rc;
  if ((rc = dmalloc(&e->final_norm, H))) return rc;
  e->layers.resize(e->L);
  for (auto& w : e->layers) {
    if ((rc = dmalloc(&w.wqkv, (size_t)e->qkv_cols * H))) return rc;
    if ((rc = dmalloc(&w.wo, H * e->nh * kHeadDim))) return rc;
    if (e->E == 0) {
      if ((rc = dmalloc(&w.wgu, (size_t)2 * e->I * H))) return rc;
      if ((rc = dmalloc(&w.wdown, H * e->I))) return rc;
    } else {
      if ((rc = dmalloc(&w.wr, (size_t)e->E * H))) return rc;
      if ((rc = dmalloc(&w.wgu_e, (size_t)e->E * 2 * e->I * H))) return rc;
      if ((rc = dmalloc(&w.wdown_e, (size_t)e->E * H * e->I))) return rc;
    }
    if ((rc = dmalloc(&w.ln1, H))) return rc;
    if ((rc = dmalloc(&w.ln2, H))) return rc;
  }
  // rope tables (engine default: double-precision angles; hosts that need bit parity with
  // LlamaRotaryEmbedding pass their own via b200_engine_set_rope_table)
  {
    const int R = c->max_position;
    std::vector<bf16> hc((size_t)R * 64), hs((size_t)R * 64);
    for (int i = 0; i < 64; ++i) {
      const float inv = 1.0f / powf(c->rope_theta, (float)(2 * i) / 128.0f);
      for (int pos = 0; pos < R; ++pos) {
        const float ang = (float)pos * inv;
        hc[(size_t)pos * 64 + i] = __float2bfloat16_rn(cosf(ang));
        hs[(size_t)pos * 64 + i] = __float2bfloat16_rn(sinf(ang));
      }
    }
    if ((rc = dmalloc(&e->cos_tab, (size_t)R * 64))) return rc;
    if ((rc = dmalloc(&e->sin_tab, (size_t)R * 64))) return rc;
    B200_CUDA_OK(cudaMemcpy(e->cos_tab, hc.data(), hc.size() * 2, cudaMemcpyHostToDevice));
    B200_CUDA_OK(cudaMemcpy(e->sin_tab, hs.data(), hs.size() * 2, cudaMemcpyHostToDevice));
  }
  // KV cache (zero-filled: masked-out V rows must be finite)
  e->max_pages = (c->max_seq_len + kPageTokens - 1) / kPageTokens;
  e->num_pages = c->num_kv_pages > 0 ? c->num_kv_pages : c->max_batch * e->max_pages;
  e->layer_stride = (long long)e->num_pages * e->nkv * kPageTokens * kHeadDim;
  if ((rc = dmalloc(&e->kcache, (size_t)e->layer_stride * e->L))) return rc;
  if ((rc = dmalloc(&e->vcache, (size_t)e->layer_stride * e->L))) return rc;
  B200_CUDA_OK(cudaMemset(e->kcache, 0, (size_t)e->layer_stride * e->L * 2));
  B200_CUDA_OK(cudaMemset(e->vcache, 0, (size_t)e->layer_stride * e->L * 2));
  if ((rc = dmalloc(&e->d_page_table, (size_t)c->max_batch * e->max_pages))) return rc;
  e->h_page_table.assign((size_t)c->max_batch * e->max_pages, 0);
  // activations
  e->cap_T = std::max(c->max_prefill_tokens, 128);
  const size_t T = e->cap_T;
  if ((rc = dmalloc(&e->x, T * H))) return rc;
  if ((rc = dmalloc(&e->xn, T * H))) return rc;
  if ((rc = dmalloc(&e->qkv, T * e->qkv_cols))) return rc;
  if ((rc = dmalloc(&e->attn, T * e->nh * kHeadDim))) return rc;
  if ((rc = dmalloc(&e->hbuf, T * e->I))) return rc;
  if (tp == 1 && (rc = dmalloc(&e->ybuf, T * H))) return rc;   // tp > 1: inside the IPC-shared exchange block (below)
  e->rows_cap = std::min(c->max_batch, kMaxRows);
  const size_t RC = (size_t)e->rows_cap;
  if ((rc = dmalloc(&e->xl, RC * H))) return rc;
  if ((rc = dmalloc(&e->qdec, RC * e->nh * kHeadDim))) return rc;
  if ((rc = dmalloc(&e->logits, RC * e->Vl))) return rc;
  B200_CUDA_OK(cudaMemset(e->x, 0, T * H * 2));
  B200_CUDA_OK(cudaMemset(e->xn, 0, T * H * 2));
  B200_CUDA_OK(cudaMemset(e->attn, 0, T * e->nh * kHeadDim * 2));
  B200_CUDA_OK(cudaMemset(e->hbuf, 0, T * e->I * 2));
  B200_CUDA_OK(cudaMemset(e->xl, 0, RC * H * 2));
  e->ws_elems = (size_t)16 * RC * std::max(std::max(e->qkv_cols, e->H), 2 * e->I);
  if (e->E) {
    e->g_rows = 2 * e->cap_T + 8 * e->E + 256;
    if ((rc = dmalloc(&e->tok_expert, (size_t)2 * T))) return rc;
    if ((rc = dmalloc(&e->tok_row, (size_t)2 * T))) return rc;
    if ((rc = dmalloc(&e->tok_weight, (size_t)2 * T))) return rc;
    if ((rc = dmalloc(&e->e_count, (size_t)kMaxExperts))) return rc;
    if ((rc = dmalloc(&e->e_off, (size_t)kMaxExperts + 1))) return rc;
    if ((rc = dmalloc(&e->xg, (size_t)e->g_rows * H))) return rc;
    if ((rc = dmalloc(&e->hg, (size_t)e->g_rows * e->I))) return rc;
    if ((rc = dmalloc(&e->yg, (size_t)e->g_rows * H))) return rc;
    B200_CUDA_OK(cudaMemset(e->xg, 0, (size_t)e->g_rows * H * 2));
    B200_CUDA_OK(cudaMemset(e->hg, 0, (size_t)e->g_rows * e->I * 2));
  }
  if ((rc = dmalloc(&e->ws, e->ws_elems))) return rc;
  e->sk_tiles = (std::max(2 * e->I, e->Vl) + kGemmBlockM - 1) / kGemmBlockM;
  e->sk_ws_floats = std::max<size_t>((size_t)e->sk_tiles * 2 * 64 * kGemmBlockM, (size_t)8 << 20);   // >= 32 MB
  if ((rc = dmalloc(&e->sk_ws, e->sk_ws_floats))) return rc;
  if ((rc = dmalloc(&e->sk_flags, (size_t)e->sk_tiles))) return rc;
  B200_CUDA_OK(cudaMemset(e->sk_flags, 0, (size_t)e->sk_tiles * sizeof(int)));
  if ((rc = dmalloc(&e->part_o, RC * e->nkv * 8 * e->G * kHeadDim))) return rc;
  if ((rc = dmalloc(&e->part_ml, RC * e->nkv * 8 * e->G * 2))) return rc;
  if ((rc = dmalloc(&e->attn_split_cnt, RC * e->nkv))) return rc;
  B200_CUDA_OK(cudaMemset(e->attn_split_cnt, 0, RC * e->nkv * sizeof(int)));
  if ((rc = dmalloc(&e->cand_val, RC * 16))) return rc;
  if ((rc = dmalloc(&e->cand_idx, RC * 16))) return rc;
  if ((rc = dmalloc(&e->cand_val_all, RC * tp))) return rc;
  if ((rc = dmalloc(&e->cand_idx_all, RC * tp))) return rc;
  // bookkeeping
  e->out_ld = c->max_seq_len;
  if ((rc = dmalloc(&e->d_tok, T))) return rc;
  if ((rc = dmalloc(&e->d_tok_seq, T))) return rc;
  if ((rc = dmalloc(&e->d_tok_pos, T))) return rc;
  if ((rc = dmalloc(&e->d_cu, 80))) return rc;
  if ((rc = dmalloc(&e->d_seq_slot, 80))) return rc;
  if ((rc = dmalloc(&e->d_last_rows, 80))) return rc;
  if ((rc = dmalloc(&e->d_cur_len, 80))) return rc;
  if ((rc = dmalloc(&e->d_next_tok, 80))) return rc;
  if ((rc = dmalloc(&e->d_dec_pos, 80))) return rc;
  if ((rc = dmalloc(&e->d_finished, 80))) return rc;
  if ((rc = dmalloc(&e->d_out_tokens, (size_t)c->max_batch * e->out_ld))) return rc;
  if ((rc = dmalloc(&e->d_forced, (size_t)c->max_batch * e->out_ld))) return rc;
  if ((rc = dmalloc(&e->d_eos, 16))) return rc;
  if ((rc = dmalloc(&e->d_stop_tok, 1024))) return rc;
  if ((rc = dmalloc(&e->d_stop_off, 32))) return rc;
  if ((rc = dmalloc(&e->d_state, 1))) return rc;
  e->h_stage_elems = 3 * T + 8 * 80;
  B200_CUDA_OK(cudaMallocHost(reinterpret_cast<void**>(&e->h_stage), e->h_stage_elems * 4));
  B200_CUDA_OK(cudaMallocHost(reinterpret_cast<void**>(&e->h_state), sizeof(StepState)));
  B200_CUDA_OK(cudaMallocHost(reinterpret_cast<void**>(&e->h_out_tokens), (size_t)c->max_batch * e->out_ld * 4));
  {
    const size_t raw = (size_t)c->max_batch * c->max_seq_len;
    if ((rc = dmalloc(&e->d_raw_ids, raw))) return rc;
    if ((rc = dmalloc(&e->d_raw_mask, raw))) return rc;
    if ((rc = dmalloc(&e->d_pred, raw))) return rc;
    if ((rc = dmalloc(&e->d_flat, T))) return rc;
    if ((rc = dmalloc(&e->d_offs, 80))) return rc;
    const size_t hraw = std::max(2 * raw, (T + 80) / 2 + 1);
    B200_CUDA_OK(cudaMallocHost(reinterpret_cast<void**>(&e->h_raw), hraw * 8));
    B200_CUDA_OK(cudaMallocHost(reinterpret_cast<void**>(&e->h_pred), raw * 8));
  }
  if (tp > 1) {
    B200_REQUIRE(tp <= kMaxTp && kMaxRows <= kArRows, "tp_size exceeds the peer-exchange layout");
    const ArLayout lay = ArLayout::make(e->H);
    // one allocation = one IPC handle: [decode LL packets | candidate exchange | flags | prefill exchange buffer y[T][H]]
    B200_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&e->ar_local), lay.total + T * H * sizeof(bf16)));
    B200_CUDA_OK(cudaMemset(e->ar_local, 0, lay.total + T * H * sizeof(bf16)));
    e->ybuf = reinterpret_cast<bf16*>(e->ar_local + lay.total);
    e->ybuf_in_block = true;
    if ((rc = dmalloc(&e->big_cnt, (size_t)2))) return rc;
    B200_CUDA_OK(cudaMemset(e->big_cnt, 0, 2 * sizeof(int)));
    if ((rc = dmalloc(&e->row_epoch, (size_t)kArRows))) return rc;
    if ((rc = dmalloc(&e->cand_epoch, (size_t)kArRows))) return rc;
    B200_CUDA_OK(cudaMemset(e->row_epoch, 0, kArRows * sizeof(int)));
    B200_CUDA_OK(cudaMemset(e->cand_epoch, 0, kArRows * sizeof(int)));
    e->p2p.tp = tp; e->p2p.rank = c->tp_rank; e->p2p.lay = lay; e->p2p.row_epoch = e->row_epoch; e->p2p.cand_epoch = e->cand_epoch;
    Nccl& n = Nccl::get();
    B200_REQUIRE(n.ok, "tp_size > 1 needs libnccl.so.2");
    B200_REQUIRE(nccl_id != nullptr, "tp_size > 1 needs an NCCL unique id");
    Nccl::UniqueId id;
    memcpy(&id, nccl_id, 128);
    B200_NCCL_OK(n.CommInitRank(&e->comm, tp, id, c->tp_rank));
  }
  B200_CUDA_OK(cudaDeviceSynchronize());
  *out = e.release();
  return 0;
}

int b200_engine_destroy(b200_engine_t* e) {
  if (!e) return 0;
  cudaSetDevice(e->cfg.device);
  cudaDeviceSynchronize();
  for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second);
  if (e->comm) Nccl::get().CommDestroy(e->comm);
  for (int r = 0; r < kMaxTp; ++r) if (e->ar_peer_map[r]) cudaIpcCloseMemHandle(e->ar_peer_map[r]);
  if (e->ar_local) cudaFree(e->ar_local);
  if (e->row_epoch) cudaFree(e->row_epoch);
  if (e->cand_epoch) cudaFree(e->cand_epoch);
  void* ptrs[] = {e->embed, e->lm_head, e->final_norm, e->cos_tab, e->sin_tab, e->kcache, e->vcache, e->d_page_table,
                  e->x, e->xn, e->qkv, e->attn, e->hbuf, e->ybuf_in_block ? nullptr : (void*)e->ybuf, e->big_cnt, e->xl, e->qdec, e->logits, e->ws, e->sk_ws, e->sk_flags,
                  e->tok_expert, e->tok_row, e->tok_weight, e->e_count, e->e_off, e->xg, e->hg, e->yg, e->part_o, e->part_ml, e->attn_split_cnt,
                  e->cand_val, e->cand_idx, e->cand_val_all, e->cand_idx_all, e->d_tok, e->d_tok_seq, e->d_tok_pos, e->d_cu,
                  e->d_seq_slot, e->d_last_rows, e->d_cur_len, e->d_next_tok, e->d_dec_pos, e->d_finished, e->d_out_tokens,
                  e->d_forced, e->d_eos, e->d_stop_tok, e->d_stop_off, e->d_state};
  for (void* p : ptrs) if (p) cudaFree(p);
  for (auto& w : e->layers) {
    void* lp[] = {w.wqkv, w.wo, w.wgu, w.wdown, w.ln1, w.ln2, w.wr, w.wgu_e, w.wdown_e};
    for (void* p : lp) if (p) cudaFree(p);
  }
  for (auto& kv : e->host_kv) cudaFreeHost(kv.second);
  if (e->h_stage) cudaFreeHost(e->h_stage);
  if (e->h_state) cudaFreeHost(e->h_state);
  if (e->h_out_tokens) cudaFreeHost(e->h_out_tokens);
  if (e->ev0) cudaEventDestroy(e->ev0);
  if (e->ev1) cudaEventDestroy(e->ev1);
  if (e->ev2) cudaEventDestroy(e->ev2);
  if (e->d_sample_cfg) cudaFree(e->d_sample_cfg);
  if (e->d_seen) cudaFree(e->d_seen);
  if (e->stream2) cudaStreamDestroy(e->stream2);
  if (e->ev_fork) cudaEventDestroy(e->ev_fork);
  if (e->ev_join) cudaEventDestroy(e->ev_join);
  if (e->stream) cudaStreamDestroy(e->stream);
  delete e;
  return 0;
}

int b200_engine_set_weight(b200_engine_t* e, const char* name, const void* data, int on_device, int ndim,
                           const int64_t* shape) {
  B200_REQUIRE(e && name && data && shape, "null argument");
  B200_CUDA_OK(cudaSetDevice(e->cfg.device));
  const std::string n(name);
  const bf16* src = reinterpret_cast<const bf16*>(data);
  const bool dev = on_device != 0;
  const long long H = e->H;
  const int r = e->cfg.tp_rank, tp = e->cfg.tp_size;
  auto expect = [&](long long d0, long long d1) -> bool {
    if (d1 < 0) return ndim == 1 && shape[0] == d0;
    return ndim == 2 && shape[0] == d0 && shape[1] == d1;
  };
  int rc = 0;
  if (n == "model.embed_tokens.weight") {
    B200_REQUIRE(expect(e->V, H), "shape mismatch for " + n);
    rc = copy_rows(e->embed, src, 0, e->V, H, dev);
  } else if (n == "lm_head.weight") {
    B200_REQUIRE(expect(e->V, H), "shape mismatch for " + n);
    rc = copy_rows(e->lm_head, src, e->v0, e->Vl, H, dev);
  } else if (n == "model.norm.weight") {
    B200_REQUIRE(expect(H, -1), "shape mismatch for " + n);
    rc = copy_rows(e->final_norm, src, 0, 1, H, dev);
  } else if (n.rfind("model.layers.", 0) == 0) {
    const size_t dot = n.find('.', 13);
    B200_REQUIRE(dot != std::string::npos, "bad weight name " + n);
    const int l = atoi(n.substr(13, dot - 13).c_str());
    B200_REQUIRE(l >= 0 && l < e->L, "layer index out of range in " + n);
    const std::string rest = n.substr(dot + 1);
    LayerW& w = e->layers[l];
    const long long QH = (long long)e->cfg.num_heads * kHeadDim, KH = (long long)e->cfg.num_kv_heads * kHeadDim;
    const long long ql = (long long)e->nh * kHeadDim, kl = (long long)e->nkv * kHeadDim;
    const long long If = e->cfg.intermediate_size, Il = e->I;
    if (rest == "input_layernorm.weight") {
      B200_REQUIRE(expect(H, -1), "shape mismatch for " + n);
      rc = copy_rows(w.ln1, src, 0, 1, H, dev);
    } else if (rest == "post_attention_layernorm.weight") {
      B200_REQUIRE(expect(H, -1), "shape mismatch for " + n);
      rc = copy_rows(w.ln2, src, 0, 1, H, dev);
    } else if (rest == "self_attn.q_proj.weight") {
      B200_REQUIRE(expect(QH, H), "shape mismatch for " + n);
      rc = copy_rows(w.wqkv, src, r * ql, ql, H, dev);
    } else if (rest == "self_attn.k_proj.weight") {
      B200_REQUIRE(expect(KH, H), "shape mismatch for " + n);
      rc = copy_rows(w.wqkv + ql * H, src, r * kl, kl, H, dev);
    } else if (rest == "self_attn.v_proj.weight") {
      B200_REQUIRE(expect(KH, H), "shape mismatch for " + n);
      rc = copy_rows(w.wqkv + (ql + kl) * H, src, r * kl, kl, H, dev);
    } else if (rest == "self_attn.o_proj.weight") {
      B200_REQUIRE(expect(H, QH), "shape mismatch for " + n);
      rc = copy_cols(w.wo, src, H, QH, r * ql, ql, dev);
    } else if (rest == "mlp.gate_proj.weight" || rest == "mlp.up_proj.weight") {
      B200_REQUIRE(expect(If, H), "shape mismatch for " + n);
      // interleave in groups of 16 rows: fused rows [32j, 32j+16) = gate[16j..], [32j+16, 32j+32) = up[16j..]
      bf16* dst = w.wgu + (rest == "mlp.up_proj.weight" ? 16 * H : 0);
      B200_CUDA_OK(cudaMemcpy2D(dst, 32 * H * 2, src + (long long)r * Il * H, 16 * H * 2, 16 * H * 2, Il / 16,
                                dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
    } else if (rest == "mlp.down_proj.weight") {
      B200_REQUIRE(expect(H, If), "shape mismatch for " + n);
      rc = copy_cols(w.wdown, src, H, If, r * Il, Il, dev);
    } else if (rest == "mlp.gate.weight") {
      B200_REQUIRE(e->E > 0 && expect(e->E, H), "shape mismatch for " + n);
      rc = copy_rows(w.wr, src, 0, e->E, H, dev);
    } else if (rest == "mlp.experts.gate_up_proj") {
      B200_REQUIRE(e->E > 0 && ndim == 3 && shape[0] == e->E && shape[1] == 2 * If && shape[2] == H, "shape mismatch for " + n);
      for (int x = 0; x < e->E; ++x) {   // per expert: rows [0,I) gate, [I,2I) up -> 16-row interleave of this rank's slice
        const bf16* g0 = src + ((long long)x * 2 * If + (long long)r * Il) * H;
        const bf16* u0 = src + ((long long)x * 2 * If + If + (long long)r * Il) * H;
        bf16* dst = w.wgu_e + (long long)x * 2 * Il * H;
        B200_CUDA_OK(cudaMemcpy2D(dst, 32 * H * 2, g0, 16 * H * 2, 16 * H * 2, Il / 16, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
        B200_CUDA_OK(cudaMemcpy2D(dst + 16 * H, 32 * H * 2, u0, 16 * H * 2, 16 * H * 2, Il / 16, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
      }
    } else if (rest == "mlp.experts.down_proj") {
      B200_REQUIRE(e->E > 0 && ndim == 3 && shape[0] == e->E && shape[1] == H && shape[2] == If, "shape mismatch for " + n);
      for (int x = 0; x < e->E && rc == 0; ++x)
        rc = copy_cols(w.wdown_e + (long long)x * H * Il, src + (long long)x * H * If, H, If, r * Il, Il, dev);
    } else if (rest == "self_attn.rotary_emb.inv_freq") {
      return 0;
    } else {
      set_last_error("unknown weight " + n);
      return -5;
    }
  } else {
    set_last_error("unknown weight " + n);
    return -5;
  }
  if (rc) return rc;
  e->seen[n] = 1;
  return 0;
}

int b200_engine_finalize_weights(b200_engine_t* e) {
  B200_REQUIRE(e, "null engine");
  const size_t want = 3 + (size_t)e->L * 9;
  B200_REQUIRE(e->seen.size() == want, "expected " + std::to_string(want) + " weight tensors, got " + std::to_string(e->seen.size()));
  B200_CUDA_OK(cudaDeviceSynchronize());
  e->finalized = true;
  return 0;
}

int b200_engine_set_rope_table(b200_engine_t* e, const void* cos_bf16, const void* sin_bf16, int32_t rows) {
  B200_REQUIRE(e && cos_bf16 && sin_bf16, "null argument");
  B200_REQUIRE(rows == e->cfg.max_position, "rope table must have max_position rows");
  B200_CUDA_OK(cudaMemcpy(e->cos_tab, cos_bf16, (size_t)rows * 64 * 2, cudaMemcpyHostToDevice));
  B200_CUDA_OK(cudaMemcpy(e->sin_tab, sin_bf16, (size_t)rows * 64 * 2, cudaMemcpyHostToDevice));
  return 0;
}

int b200_stage_prompt(b200_engine_t* e, const int64_t* ids, const int64_t* mask, int32_t B, int32_t S,
                      const b200_gen_params_t* gp) {
  B200_REQUIRE(e && ids && gp, "null argument");
  B200_CUDA_OK(cudaSetDevice(e->cfg.device));
  int rc = stage_prompt(e, ids, mask, B, S, gp);
  if (rc) return rc;
  B200_CUDA_OK(cudaStreamSynchronize(e->stream));
  return 0;
}

int b200_run_staged(b200_engine_t* e, int32_t do_prefill, int32_t decode_steps) {
  B200_REQUIRE(e, "null engine");
  B200_CUDA_OK(cudaSetDevice(e->cfg.device));
  int rc;
  if (do_prefill) {
    // reset the per-request device state so the same staged prompt can be replayed: the raw rows are still
    // resident on the device, so this re-runs the device-side concat and nothing crosses PCIe
    auto& st = e->st;
    if (st.S > 0) pack_padded_kernel<<<1, 1024, 0, e->stream>>>(e->d_raw_ids, e->staged_mask ? e->d_raw_mask : nullptr, st.B, st.S, pack_out(e));
    else pack_ragged_kernel<<<1, 1024, 0, e->stream>>>(e->d_flat, e->d_offs, st.B, pack_out(e));
    B200_CUDA_OK(cudaGetLastError());
    e->launches++;
    StepState init{0, 0, 0, st.max_new};
    *e->h_state = init;
    B200_CUDA_OK(cudaMemcpyAsync(e->d_state, e->h_state, sizeof(StepState), cudaMemcpyHostToDevice, e->stream));
    if ((rc = prefill(e))) return rc;
    st.prefilled = true;
  }
  B200_REQUIRE(e->st.prefilled, "run_staged: prefill has not run");
  for (int i = 0; i < decode_steps; ++i)
    if ((rc = decode_step(e, true))) return rc;
  return 0;
}

int b200_run_staged_timed(b200_engine_t* e, int32_t decode_steps, float* prefill_ms, float* decode_ms) {
  B200_REQUIRE(e && prefill_ms && decode_ms, "null argument");
  B200_CUDA_OK(cudaSetDevice(e->cfg.device));
  e->launches = 0;
  B200_CUDA_OK(cudaEventRecord(e->ev0, e->stream));
  int rc = b200_run_staged(e, 1, 0);
  if (rc) return rc;
  B200_CUDA_OK(cudaEventRecord(e->ev1, e->stream));
  if ((rc = b200_run_staged(e, 0, decode_steps))) return rc;
  B200_CUDA_OK(cudaEventRecord(e->ev2, e->stream));
  B200_CUDA_OK(cudaStreamSynchronize(e->stream));
  B200_CUDA_OK(cudaEventElapsedTime(prefill_ms, e->ev0, e->ev1));
  B200_CUDA_OK(cudaEventElapsedTime(decode_ms, e->ev1, e->ev2));
  e->timing.prefill_ms = *prefill_ms; e->timing.decode_ms = *decode_ms;
  e->timing.decode_steps = decode_steps; e->timing.kernel_launches = e->launches;
  return 0;
}

int b200_fetch_staged(b200_engine_t* e, int64_t* out_ids, int32_t* out_len, int32_t* stop_triggered) {
  B200_REQUIRE(e && out_ids && out_len, "null argument");
  B200_CUDA_OK(cudaSetDevice(e->cfg.device));
  return fetch_result(e, out_ids, out_len, stop_triggered);
}

int b200_generate(b200_engine_t* e, const int64_t* ids, const int64_t* mask, int32_t B, int32_t S,
                  const b200_gen_params_t* gp, int64_t* out_ids, int32_t* out_len, int32_t* stop_triggered,
                  uint16_t* logits_bf16, b200_token_callback cb, void* user) {
  B200_REQUIRE(e && ids && gp && out_ids && out_len, "null argument");
  B200_CUDA_OK(cudaSetDevice(e->cfg.device));
  cudaStream_t s = e->stream;
  e->launches = 0;
  B200_CUDA_OK(cudaEventRecord(e->ev0, s));
  int rc = stage_prompt(e, ids, mask, B, S, gp);
  if (rc) return rc;
  if ((rc = prefill(e))) return rc;
  e->st.prefilled = true;
  B200_CUDA_OK(cudaEventRecord(e->ev1, s));
  const bool record = logits_bf16 != nullptr;
  const bool eager = record;             // per-step logits copies -> no graph
  const size_t lrow = (size_t)e->Vl;     // logits of this rank's vocab shard
  // tensor parallel: every rank records the logits of ITS vocabulary shard ([max_new_tokens][B][ceil(V / tp)] rows,
  // the last rank's rows are shorter); the host concatenates the shards
  std::vector<int64_t> cbuf(B);
  auto after_step = [&](int step) -> int {
    if (record)
      B200_CUDA_OK(cudaMemcpyAsync(logits_bf16 + (size_t)step * B * lrow, e->logits, (size_t)B * lrow * 2, cudaMemcpyDeviceToHost, s));
    if (cb) {
      B200_CUDA_OK(cudaMemcpyAsync(e->h_out_tokens, e->d_out_tokens, (size_t)B * e->out_ld * 4, cudaMemcpyDeviceToHost, s));
      B200_CUDA_OK(cudaMemcpyAsync(e->h_state, e->d_state, sizeof(StepState), cudaMemcpyDeviceToHost, s));
      B200_CUDA_OK(cudaStreamSynchronize(s));
      if (e->h_state->step > step) {
        for (int b = 0; b < B; ++b) cbuf[b] = e->h_out_tokens[(size_t)b * e->out_ld + step];
        if (cb(user, step, cbuf.data(), B)) return 1;
      }
      return e->h_state->done ? 2 : 0;
    }
    return 0;
  };
  int steps = 0;
  int ar = after_step(0);
  // Tensor parallel: only the leader has a callback, so a `done` seen after the first token (EOS first / a stop sequence
  // that matches token 0) must not make it skip decode steps the followers still run — their all-reduces would wait for
  // it forever.  Every rank leaves at the shared i % 8 poll below; a user abort (ar == 1) is honoured there as well.
  bool aborted = ar == 1;
  if (e->cfg.tp_size > 1) ar = 0;
  if (ar == 0) {
    for (int i = 1; i < gp->max_new_tokens; ++i) {
      if ((rc = decode_step(e, !eager))) return rc;
      ++steps;
      ar = after_step(i);
      // under TP every rank must leave the loop at the same step (the next step contains collectives), so the
      // only exit points are the shared polling cadence below; a streaming leader just stops receiving tokens.
      if (ar && e->cfg.tp_size == 1) break;
      if (ar == 1) aborted = true;
      if (ar && e->cfg.tp_size > 1) ar = 0;
      if ((!cb || e->cfg.tp_size > 1) && (i % 8) == 0) {  // poll the device-side done flag without a per-token sync
        B200_CUDA_OK(cudaMemcpyAsync(e->h_state, e->d_state, sizeof(StepState), cudaMemcpyDeviceToHost, s));
        B200_CUDA_OK(cudaStreamSynchronize(s));
        if (e->h_state->done) break;
      }
    }
  }
  B200_CUDA_OK(cudaEventRecord(e->ev2, s));
  if ((rc = fetch_result(e, out_ids, out_len, stop_triggered))) return rc;
  B200_CUDA_OK(cudaEventElapsedTime(&e->timing.prefill_ms, e->ev0, e->ev1));
  B200_CUDA_OK(cudaEventElapsedTime(&e->timing.decode_ms, e->ev1, e->ev2));
  e->timing.decode_steps = steps;
  e->timing.kernel_launches = e->launches;
  return (ar == 1 || aborted) ? 1 : 0;
}

// Replaces the body of BatchHandler.batchPredict (pkg/batcher/handler.go:99-155): the instances of every
// waiting request (ragged token rows) are concatenated ON DEVICE, generated in one batch, and the predictions
// come back as one [n_rows][max_new_tokens] matrix in instance order, so each request's answer is the
// contiguous slice [first, first+count) the batcher recorded (handler.go:139-150).
int b200_batch_predict(b200_engine_t* e, const int64_t* const* rows, const int32_t* row_lens, int32_t n_rows,
                       const b200_gen_params_t* gp, int64_t* predictions, int32_t* n_generated,
                       int32_t* stop_triggered) {
  B200_REQUIRE(e && rows && row_lens && gp && predictions && n_generated, "null argument");
  B200_CUDA_OK(cudaSetDevice(e->cfg.device));
  cudaStream_t s = e->stream;
  e->launches = 0;
  B200_CUDA_OK(cudaEventRecord(e->ev0, s));
  int rc = stage_ragged(e, rows, row_lens, n_rows, gp);
  if (rc) return rc;
  if ((rc = prefill(e))) return rc;
  e->st.prefilled = true;
  B200_CUDA_OK(cudaEventRecord(e->ev1, s));
  int steps = 0;
  for (int i = 1; i < gp->max_new_tokens; ++i) {
    if ((rc = decode_step(e, true))) return rc;
    ++steps;
    if ((i % 8) == 0) {
      B200_CUDA_OK(cudaMemcpyAsync(e->h_state, e->d_state, sizeof(StepState), cudaMemcpyDeviceToHost, s));
      B200_CUDA_OK(cudaStreamSynchronize(s));
      if (e->h_state->done) break;
    }
  }
  B200_CUDA_OK(cudaEventRecord(e->ev2, s));
  B200_CUDA_OK(cudaMemcpyAsync(e->h_state, e->d_state, sizeof(StepState), cudaMemcpyDeviceToHost, s));
  B200_CUDA_OK(cudaStreamSynchronize(s));
  { int frc = check_fault(e); if (frc) return frc; }
  const int T = e->h_state->step;
  scatter_predictions_kernel<<<n_rows, 128, 0, s>>>(e->d_out_tokens, e->out_ld, n_rows, T, e->d_pred);
  B200_CUDA_OK(cudaGetLastError());
  e->launches++;
  B200_CUDA_OK(cudaMemcpyAsync(e->h_pred, e->d_pred, (size_t)n_rows * T * 8, cudaMemcpyDeviceToHost, s));
  B200_CUDA_OK(cudaStreamSynchronize(s));
  for (int b = 0; b < n_rows; ++b)
    for (int i = 0; i < gp->max_new_tokens; ++i)
      predictions[(size_t)b * gp->max_new_tokens + i] = i < T ? e->h_pred[(size_t)b * T + i] : gp->pad_token_id;
  *n_generated = T;
  if (stop_triggered) *stop_triggered = e->h_state->stop_triggered;
  B200_CUDA_OK(cudaEventElapsedTime(&e->timing.prefill_ms, e->ev0, e->ev1));
  B200_CUDA_OK(cudaEventElapsedTime(&e->timing.decode_ms, e->ev1, e->ev2));
  e->timing.decode_steps = steps;
  e->timing.kernel_launches = e->launches;
  return 0;
}

// ---- batcher trigger state machine (pkg/batcher/handler.go:157-199) ---------------------------------
struct b200_batcher { BatcherCore core; b200_batcher(int a, int b) : core(a, b) {} };

int b200_batcher_create(int32_t max_batch_size, int32_t max_latency_ms, b200_batcher_t** out) {
  B200_REQUIRE(out, "null argument");
  *out = new b200_batcher(max_batch_size, max_latency_ms);
  return 0;
}
int b200_batcher_destroy(b200_batcher_t* b) { delete b; return 0; }
int b200_batcher_config(b200_batcher_t* b, int32_t* max_batch_size, int32_t* max_latency_ms) {
  B200_REQUIRE(b && max_batch_size && max_latency_ms, "null argument");
  *max_batch_size = b->core.max_batch_size; *max_latency_ms = b->core.max_latency_ms;
  return 0;
}
int b200_batcher_add(b200_batcher_t* b, int64_t now_us, int32_t n_instances, int64_t* ticket) {
  B200_REQUIRE(b && ticket, "null argument");
  B200_REQUIRE(n_instances >= 1, "no instances in the request");
  *ticket = b->core.add(now_us, n_instances);
  return 0;
}
int b200_batcher_tick(b200_batcher_t* b, int64_t now_us, int32_t cap, int64_t* tickets, int32_t* first,
                      int32_t* count, int32_t* n_requests, int32_t* total_instances) {
  B200_REQUIRE(b && tickets && first && count && n_requests && total_instances, "null argument");
  long long* tk = reinterpret_cast<long long*>(tickets);
  const int n = b->core.tick(now_us, tk, first, count, cap, total_instances);
  B200_REQUIRE(n >= 0, "ticket buffer too small");
  *n_requests = n;
  return 0;
}

int b200_engine_fault(b200_engine_t* e, int32_t* code, int32_t reset) {
  B200_REQUIRE(e && code, "null argument");
  B200_CUDA_OK(cudaSetDevice(e->cfg.device));
  int c = 0;
  B200_CUDA_OK(cudaMemcpyFromSymbol(&c, g_fault_code, sizeof(int)));
  *code = c;
  if (reset) {
    const int zero = 0;
    B200_CUDA_OK(cudaMemcpyToSymbol(g_fault_code, &zero, sizeof(int)));
    e->faulted = false;
  }
  return 0;
}

int b200_engine_last_timing(b200_engine_t* e, b200_timing_t* out) {
  B200_REQUIRE(e && out, "null argument");
  *out = e->timing;
  return 0;
}

// ---- host-DRAM KV tier (BASELINE.json configs[3]: "paged-KV with host-DRAM KV-offload tier") ----------
// Moves every KV page of one staged sequence (all layers, K and V) to pinned host memory and back, asynchronously on
// the engine stream.  While a sequence is swapped out its device pages may be overwritten (scrub = 1 does so, for
// tests); after swap-in decoding continues bit-identically.
static int kv_swap(b200_engine_t* e, int32_t slot, bool out, int scrub) {
  auto& st = e->st;
  B200_REQUIRE(st.prefilled && slot >= 0 && slot < st.B, "no such staged sequence");
  B200_CUDA_OK(cudaSetDevice(e->cfg.device));
  const size_t page_elems = (size_t)e->nkv * kPageTokens * kHeadDim;
  const size_t seq_elems = (size_t)st.per_seq_pages * page_elems;          // per layer, per K or V
  const size_t bytes = seq_elems * 2 * 2 * e->L;
  if (out) {
    if (!e->host_kv.count(slot) || e->host_kv_bytes[slot] < bytes) {
      if (e->host_kv.count(slot)) cudaFreeHost(e->host_kv[slot]);
      bf16* h = nullptr;
      B200_CUDA_OK(cudaMallocHost(reinterpret_cast<void**>(&h), bytes));
      e->host_kv[slot] = h; e->host_kv_bytes[slot] = bytes;
    }
  } else {
    B200_REQUIRE(e->host_kv.count(slot), "sequence is not swapped out");
  }
  bf16* h = e->host_kv[slot];
  const size_t first = (size_t)slot * st.per_seq_pages * page_elems;
  for (int l = 0; l < e->L; ++l) {
    bf16* kd = e->kcache + (size_t)l * e->layer_stride + first;
    bf16* vd = e->vcache + (size_t)l * e->layer_stride + first;
    bf16* kh = h + ((size_t)l * 2) * seq_elems;
    bf16* vh = kh + seq_elems;
    if (out) {
      B200_CUDA_OK(cudaMemcpyAsync(kh, kd, seq_elems * 2, cudaMemcpyDeviceToHost, e->stream));
      B200_CUDA_OK(cudaMemcpyAsync(vh, vd, seq_elems * 2, cudaMemcpyDeviceToHost, e->stream));
      if (scrub) {
        B200_CUDA_OK(cudaMemsetAsync(kd, 0x7f, seq_elems * 2, e->stream));
        B200_CUDA_OK(cudaMemsetAsync(vd, 0x7f, seq_elems * 2, e->stream));
      }
    } else {
      B200_CUDA_OK(cudaMemcpyAsync(kd, kh, seq_elems * 2, cudaMemcpyHostToDevice, e->stream));
      B200_CUDA_OK(cudaMemcpyAsync(vd, vh, seq_elems * 2, cudaMemcpyHostToDevice, e->stream));
    }
  }
  return 0;
}
int b200_kv_swap_out(b200_engine_t* e, int32_t slot, int32_t scrub) { B200_REQUIRE(e, "null engine"); return kv_swap(e, slot, true, scrub); }
int b200_kv_swap_in(b200_engine_t* e, int32_t slot) { B200_REQUIRE(e, "null engine"); return kv_swap(e, slot, false, 0); }


// ---- continuous batching (include/kserve_b200.h) ---------------------------------------------------
int b200_cb_begin(b200_engine_t* e, int64_t pad_token_id, const int64_t* eos_token_ids, int32_t num_eos) {
  B200_REQUIRE(e, "null engine");
  B200_REQUIRE(e->finalized, "weights not finalized");
  B200_REQUIRE(num_eos >= 0 && num_eos <= 16, "too many eos tokens");
  B200_REQUIRE(e->max_pages <= e->num_pages, "KV page pool smaller than one full-length sequence");
  B200_CUDA_OK(cudaSetDevice(e->cfg.device));
  int rc = cb_alloc(e);
  if (rc) return rc;
  (void)pad_token_id;
  std::vector<int32_t> tmp(std::max(1, num_eos));
  for (int i = 0; i < num_eos; ++i) tmp[i] = (int32_t)eos_token_ids[i];
  if (num_eos) B200_CUDA_OK(cudaMemcpy(e->d_eos, tmp.data(), (size_t)num_eos * 4, cudaMemcpyHostToDevice));
  e->cb_num_eos = num_eos;
  // every page is free; slots get their page-table rows at admit
  e->cb_free_pages.clear();
  for (int pg = e->num_pages - 1; pg >= 0; --pg) e->cb_free_pages.push_back(pg);
  e->cb_page_ref.assign(e->num_pages, 0);
  e->cb_prefix.clear();
  e->cb_pending.clear();
  e->cb_slot_pages.assign(e->cfg.max_batch, {});
  e->cb_slot_sampling.assign(e->cfg.max_batch, 0);
  e->cb_swapped.assign(e->cfg.max_batch, 0);
  e->cb_swap_pages.assign(e->cfg.max_batch, 0);
  e->cb_sampling_slots = 0;
  e->cb_chunk_tokens = 0; e->cb_prefix_on = false;     // b200_cb_config applies to one begin .. end span
  for (auto& v : e->cb_stat) v = 0;
  e->cb_used.assign(e->cfg.max_batch, 0);
  e->cb_active.clear();
  e->cb_rows_dirty = true;
  e->cb_on = true;
  return 0;
}

int b200_cb_config(b200_engine_t* e, int32_t prefill_chunk_tokens, int32_t prefix_cache) {
  B200_REQUIRE(e, "null engine");
  B200_REQUIRE(prefill_chunk_tokens == 0 || prefill_chunk_tokens >= 128, "prefill chunks are multiples of 128 tokens (0 = whole prompts at admit)");
  e->cb_chunk_tokens = (prefill_chunk_tokens / 128) * 128;
  e->cb_prefix_on = prefix_cache != 0;
  return 0;
}

int b200_cb_stats(b200_engine_t* e, int64_t* out10) {
  B200_REQUIRE(e && out10, "null argument");
  int64_t evictable = 0;
  for (auto& kv : e->cb_prefix)
    if (e->cb_page_ref[kv.second.p0] == 1 && e->cb_page_ref[kv.second.p1] == 1) evictable += 2;
  out10[0] = e->cb_stat[0]; out10[1] = e->cb_stat[1]; out10[2] = e->cb_stat[2]; out10[3] = e->cb_stat[3]; out10[4] = e->cb_stat[4];
  out10[5] = (int64_t)e->cb_free_pages.size() + evictable;     // pages an admit could obtain right now
  out10[6] = (int64_t)e->cb_prefix.size();
  out10[7] = (int64_t)e->cb_pending.size();
  out10[8] = e->cb_stat[5]; out10[9] = e->cb_stat[6];      // sequences swapped out to / back in from host DRAM
  return 0;
}

int b200_cb_end(b200_engine_t* e) {
  B200_REQUIRE(e, "null engine");
  e->cb_on = false;
  e->cb_active.clear();
  e->cb_pending.clear();
  e->cb_prefix.clear();
  return 0;
}

int b200_cb_admit(b200_engine_t* e, int32_t n, const int64_t* const* rows, const int32_t* lens, const int32_t* max_new,
                  const int32_t* stop_count, const int32_t* stop_offsets, const int64_t* stop_tokens,
                  const b200_gen_params_t* sampling, int32_t* slots_out) {
  B200_REQUIRE(e && rows && lens && max_new && slots_out, "null argument");
  B200_CUDA_OK(cudaSetDevice(e->cfg.device));
  return cb_admit(e, n, rows, lens, max_new, stop_count, stop_offsets, stop_tokens, sampling, slots_out);
}

int b200_cb_step(b200_engine_t* e, int32_t n_steps) {
  B200_REQUIRE(e && e->cb_on, "b200_cb_begin was not called");
  B200_REQUIRE(!e->faulted, "engine fault: an earlier device-side wait timed out; re-create the engine");
  B200_CUDA_OK(cudaSetDevice(e->cfg.device));
  for (int i = 0; i < n_steps; ++i) {
    int rc;
    if (!e->cb_pending.empty() && (rc = cb_prefill_pending(e, e->cb_chunk_tokens > 0 ? e->cb_chunk_tokens : LLONG_MAX))) return rc;
    if ((rc = cb_decode_step(e))) return rc;
  }
  return 0;
}

int b200_cb_poll(b200_engine_t* e, int32_t* n_gen, int32_t* finished, int32_t* stop_hit) {
  B200_REQUIRE(e && e->cb_on && n_gen && finished, "null argument / not in continuous-batching mode");
  B200_CUDA_OK(cudaSetDevice(e->cfg.device));
  const size_t nb = (size_t)e->cfg.max_batch;
  cudaStream_t s = e->stream;
  B200_CUDA_OK(cudaMemcpyAsync(e->h_cb, e->cb.n_gen, nb * 4, cudaMemcpyDeviceToHost, s));
  B200_CUDA_OK(cudaMemcpyAsync(e->h_cb + nb, e->cb.finished, nb * 4, cudaMemcpyDeviceToHost, s));
  B200_CUDA_OK(cudaMemcpyAsync(e->h_cb + 2 * nb, e->cb.stop_hit, nb * 4, cudaMemcpyDeviceToHost, s));
  B200_CUDA_OK(cudaStreamSynchronize(s));
  { int frc = check_fault(e); if (frc) return frc; }
  for (size_t i = 0; i < nb; ++i) {
    const bool used = e->cb_used[i] != 0;
    n_gen[i] = used ? e->h_cb[i] : 0;
    finished[i] = used ? e->h_cb[nb + i] : 0;
    if (stop_hit) stop_hit[i] = used ? e->h_cb[2 * nb + i] : 0;
  }
  return 0;
}

int b200_cb_read(b200_engine_t* e, int32_t slot, int32_t first, int64_t* out, int32_t cap, int32_t* n_out) {
  B200_REQUIRE(e && e->cb_on && out && n_out, "null argument / not in continuous-batching mode");
  B200_REQUIRE(slot >= 0 && slot < e->cfg.max_batch && e->cb_used[slot], "slot is not in use");
  B200_CUDA_OK(cudaSetDevice(e->cfg.device));
  cudaStream_t s = e->stream;
  int32_t ng = 0;
  B200_CUDA_OK(cudaMemcpyAsync(&ng, e->cb.n_gen + slot, 4, cudaMemcpyDeviceToHost, s));
  B200_CUDA_OK(cudaStreamSynchronize(s));
  const int n = std::max(0, std::min(ng - first, cap));
  if (n > 0) {
    B200_CUDA_OK(cudaMemcpyAsync(e->h_cb, e->cb.out + (size_t)slot * e->out_ld + first, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
    B200_CUDA_OK(cudaStreamSynchronize(s));
    for (int i = 0; i < n; ++i) out[i] = e->h_cb[i];
  }
  *n_out = n;
  return 0;
}

// ---- host-DRAM KV tier of the continuous batcher (BASELINE.json configs[3]: "paged-KV with host-DRAM KV-offload tier") ----
// A running sequence is PREEMPTED to host memory when the page pool cannot serve a new admission: all of its KV pages (every
// layer, K and V) are copied to a pinned buffer on the engine stream, its pages go back to the pool (shared prefix pages
// merely lose a reference), and it leaves the decode batch; its per-sequence device state (length, generated tokens, next
// token, stop sequences) stays where it is.  swap-in takes fresh pages, copies the KV back and the sequence resumes with
// bit-identical results.  Policy (who, when) lives in the scheduler: kserve_b200/continuous.py preempts the most recently
// admitted request and resumes swapped requests before admitting new ones.
static int cb_swap(b200_engine_t* e, int32_t slot, bool out) {
  B200_REQUIRE(e && e->cb_on, "not in continuous-batching mode");
  B200_REQUIRE(slot >= 0 && slot < e->cfg.max_batch && e->cb_used[slot], "slot is not in use");
  B200_CUDA_OK(cudaSetDevice(e->cfg.device));
  const size_t page_elems = (size_t)e->nkv * kPageTokens * kHeadDim;      // per layer, per K or V
  const size_t page_bytes = page_elems * sizeof(bf16);
  cudaStream_t s = e->stream;
  if (out) {
    B200_REQUIRE(!e->cb_swapped[slot], "sequence is already swapped out");
    auto it = std::find(e->cb_active.begin(), e->cb_active.end(), (int)slot);
    B200_REQUIRE(it != e->cb_active.end(), "only a running sequence (prompt fully prefilled) can be swapped out");
    std::vector<int>& pages = e->cb_slot_pages[slot];
    const size_t bytes = pages.size() * page_bytes * 2 * e->L;
    if (!e->host_kv.count(slot) || e->host_kv_bytes[slot] < bytes) {
      if (e->host_kv.count(slot)) cudaFreeHost(e->host_kv[slot]);
      bf16* h = nullptr;
      B200_CUDA_OK(cudaMallocHost(reinterpret_cast<void**>(&h), bytes));
      e->host_kv[slot] = h; e->host_kv_bytes[slot] = bytes;
    }
    unsigned char* h = reinterpret_cast<unsigned char*>(e->host_kv[slot]);
    for (size_t i = 0; i < pages.size(); ++i) {     // one strided copy per page and cache: [L] rows of page_bytes
      unsigned char* hk = h + (i * 2) * page_bytes * e->L;
      B200_CUDA_OK(cudaMemcpy2DAsync(hk, page_bytes, e->kcache + (size_t)pages[i] * page_elems, (size_t)e->layer_stride * sizeof(bf16),
                                     page_bytes, e->L, cudaMemcpyDeviceToHost, s));
      B200_CUDA_OK(cudaMemcpy2DAsync(hk + page_bytes * e->L, page_bytes, e->vcache + (size_t)pages[i] * page_elems,
                                     (size_t)e->layer_stride * sizeof(bf16), page_bytes, e->L, cudaMemcpyDeviceToHost, s));
    }
    e->cb_swap_pages[slot] = (int)pages.size();
    for (int pg : pages) cb_unref_page(e, pg);       // reuse is stream-ordered after the copies above
    pages.clear();
    e->cb_active.erase(it);
    e->cb_rows_dirty = true;
    e->cb_swapped[slot] = 1;
    e->cb_stat[5]++;
    return 0;
  }
  B200_REQUIRE(e->cb_swapped[slot], "sequence is not swapped out");
  const int n = e->cb_swap_pages[slot];
  std::vector<int> got;
  for (int i = 0; i < n; ++i) {
    const int pg = cb_take_page(e);
    if (pg < 0) {
      for (int q : got) cb_unref_page(e, q);
      set_last_error("KV page pool exhausted: cannot swap the sequence back in yet");
      return -7;
    }
    got.push_back(pg);
  }
  const unsigned char* h = reinterpret_cast<const unsigned char*>(e->host_kv[slot]);
  for (int i = 0; i < n; ++i) {
    const unsigned char* hk = h + ((size_t)i * 2) * page_bytes * e->L;
    B200_CUDA_OK(cudaMemcpy2DAsync(e->kcache + (size_t)got[i] * page_elems, (size_t)e->layer_stride * sizeof(bf16), hk, page_bytes,
                                   page_bytes, e->L, cudaMemcpyHostToDevice, s));
    B200_CUDA_OK(cudaMemcpy2DAsync(e->vcache + (size_t)got[i] * page_elems, (size_t)e->layer_stride * sizeof(bf16), hk + page_bytes * e->L,
                                   page_bytes, page_bytes, e->L, cudaMemcpyHostToDevice, s));
  }
  e->cb_slot_pages[slot] = got;
  int32_t* row = e->h_page_table.data() + (size_t)slot * e->max_pages;
  for (int k = 0; k < e->max_pages; ++k) row[k] = k < n ? got[k] : got.back();
  B200_CUDA_OK(cudaMemcpyAsync(e->d_page_table + (size_t)slot * e->max_pages, row, (size_t)e->max_pages * 4, cudaMemcpyHostToDevice, s));
  B200_CUDA_OK(cudaStreamSynchronize(s));            // the page-table row is pageable host memory
  e->cb_swapped[slot] = 0;
  e->cb_active.push_back(slot);
  e->cb_rows_dirty = true;
  e->cb_stat[6]++;
  return 0;
}
int b200_cb_swap_out(b200_engine_t* e, int32_t slot) { return cb_swap(e, slot, true); }
int b200_cb_swap_in(b200_engine_t* e, int32_t slot) { return cb_swap(e, slot, false); }

int b200_cb_release(b200_engine_t* e, int32_t slot) {
  B200_REQUIRE(e && e->cb_on, "not in continuous-batching mode");
  B200_REQUIRE(slot >= 0 && slot < e->cfg.max_batch && e->cb_used[slot], "slot is not in use");
  e->cb_used[slot] = 0;
  auto it = std::find(e->cb_active.begin(), e->cb_active.end(), (int)slot);
  if (it != e->cb_active.end()) { e->cb_active.erase(it); e->cb_rows_dirty = true; }
  for (auto pd = e->cb_pending.begin(); pd != e->cb_pending.end(); ++pd)
    if (pd->slot == slot) { e->cb_pending.erase(pd); break; }      // cancelled before its prompt was in the cache
  for (int pg : e->cb_slot_pages[slot]) cb_unref_page(e, pg);       // shared prefix pages stay alive through the cache's reference
  e->cb_slot_pages[slot].clear();
  e->cb_swapped[slot] = 0;
  if (e->cb_slot_sampling[slot]) { e->cb_slot_sampling[slot] = 0; e->cb_sampling_slots--; }
  return 0;
}

// ---- peer-memory exchange setup (tensor parallel) --------------------------------------------------
int b200_engine_ipc_export(b200_engine_t* e, void* handle64) {
  B200_REQUIRE(e && handle64, "null argument");
  B200_REQUIRE(e->ar_local != nullptr, "engine was created with tp_size == 1");
  B200_CUDA_OK(cudaSetDevice(e->cfg.device));
  cudaIpcMemHandle_t h;
  B200_CUDA_OK(cudaIpcGetMemHandle(&h, e->ar_local));
  static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
  memcpy(handle64, &h, 64);
  return 0;
}

int b200_engine_ipc_import(b200_engine_t* e, const void* handles, int32_t n) {
  B200_REQUIRE(e && handles, "null argument");
  B200_REQUIRE(n == e->cfg.tp_size && e->ar_local != nullptr, "need one handle per rank");
  B200_CUDA_OK(cudaSetDevice(e->cfg.device));
  for (int r = 0; r < n; ++r) {
    if (r == e->cfg.tp_rank) { e->p2p.peer[r] = e->ar_local; continue; }
    cudaIpcMemHandle_t h;
    memcpy(&h, reinterpret_cast<const unsigned char*>(handles) + (size_t)r * 64, 64);
    void* p = nullptr;
    B200_CUDA_OK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    e->ar_peer_map[r] = p;
    e->p2p.peer[r] = reinterpret_cast<unsigned char*>(p);
  }
  e->p2p_ready = getenv("B200_NO_P2P") == nullptr;
  return 0;
}

// ---- debug timeline ---------------------------------------------------------------------------------
static TraceRec* g_trace_dev = nullptr;
int b200_debug_trace(int32_t capacity) {
  if (g_trace_dev) { cudaFree(g_trace_dev); g_trace_dev = nullptr; }
  TraceRec* nullp = nullptr;
  unsigned int zero = 0, cap = (unsigned int)std::max(capacity, 0);
  { int sp = getenv("B200_TRACE_SPLIT") ? 1 : 0; cudaMemcpyToSymbol(g_trace_split, &sp, sizeof(sp)); }
  if (capacity > 0) B200_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&g_trace_dev), sizeof(TraceRec) * capacity));
  B200_CUDA_OK(cudaMemcpyToSymbol(g_trace_cnt, &zero, sizeof(zero)));
  B200_CUDA_OK(cudaMemcpyToSymbol(g_trace_cap, &cap, sizeof(cap)));
  B200_CUDA_OK(cudaMemcpyToSymbol(g_trace_buf, capacity > 0 ? &g_trace_dev : &nullp, sizeof(TraceRec*)));
  return 0;
}
int b200_debug_trace_read(void* out, int32_t capacity, int32_t* n) {
  B200_REQUIRE(out && n, "null argument");
  B200_CUDA_OK(cudaDeviceSynchronize());
  unsigned int cnt = 0, zero = 0;
  B200_CUDA_OK(cudaMemcpyFromSymbol(&cnt, g_trace_cnt, sizeof(cnt)));
  const int m = std::min<int>((int)cnt, capacity);
  if (m > 0 && g_trace_dev) B200_CUDA_OK(cudaMemcpy(out, g_trace_dev, sizeof(TraceRec) * m, cudaMemcpyDeviceToHost));
  B200_CUDA_OK(cudaMemcpyToSymbol(g_trace_cnt, &zero, sizeof(zero)));
  *n = m;
  return 0;
}

// ---- single-kernel entry points ---------------------------------------------------------------------
static TmapCache g_op_tmaps;
static int g_op_sms = 0;
static int op_sms() {
  if (!g_op_sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_op_sms, cudaDevAttrMultiProcessorCount, dev);
  }
  return g_op_sms;
}

int b200_op_gemm(const void* A, const void* B, void* out, const void* residual, int M, int N, int K, int epi,
                 int block_n, int splits, int64_t ldo, void* stream) {
  g_op_tmaps.maps.clear();  // caller buffers may be reused at other shapes
  const bool t = epi >= EPI_T_STORE;
  int out_cols = (epi == EPI_SWIGLU) ? N / 2 : (epi == EPI_T_SWIGLU ? M / 2 : 0);
  GemmArgs a{(const bf16*)A, M, (const bf16*)B, N, M, N, K, epi, block_n, effective_splits(K, splits), out,
             (const bf16*)residual, ldo, (long long)N * ldo, out_cols, t};
  static float* op_sk_ws = nullptr;
  static int* op_sk_flags = nullptr;
  const int op_sk_tiles = 2048;
  if (t && !op_sk_ws) {
    B200_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&op_sk_ws), (size_t)op_sk_tiles * 2 * 64 * kGemmBlockM * sizeof(float)));
    B200_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&op_sk_flags), op_sk_tiles * sizeof(int)));
    B200_CUDA_OK(cudaMemset(op_sk_flags, 0, op_sk_tiles * sizeof(int)));
  }
  a.sk_ws = op_sk_ws; a.sk_flags = op_sk_flags; a.sk_tiles = op_sk_tiles; a.sk_ws_floats = (size_t)op_sk_tiles * 2 * 64 * kGemmBlockM;
  return launch_gemm(g_op_tmaps, a, op_sms(), (cudaStream_t)stream);
}

int b200_op_rmsnorm(void* x, const void* w, void* xn, int rows, int H, float eps, const float* partial, int splits,
                    const void* y, void* stream) {
  const int mode = partial ? 1 : (y ? 2 : 0);
  return launch_rmsnorm(mode, (bf16*)x, (const bf16*)w, (bf16*)xn, rows, H, eps, partial, splits, (long long)rows * H, H,
                        (const bf16*)y, (cudaStream_t)stream);
}

int b200_op_attn_prefill_tc(const void* q, int64_t ldq, int q_rows, void* out, int64_t ldo, const void* kcache,
                            const void* vcache, int num_pages, const int32_t* page_table, int max_pages,
                            const int32_t* cu_seqlens, const int32_t* seq_slot, int B, int max_len, int nh, int nkv,
                            void* stream) {
  g_op_tmaps.maps.clear();
  AttnTcParams p{};
  p.out = (bf16*)out; p.ldo = ldo; p.page_table = page_table; p.max_pages = max_pages; p.cu_seqlens = cu_seqlens;
  p.seq_slot = seq_slot; p.nh = nh; p.nkv = nkv; p.scale_log2 = (1.0f / sqrtf((float)kHeadDim)) * 1.4426950408889634f;
  return launch_attn_prefill_tc(g_op_tmaps, (const bf16*)q, q_rows, ldq, (const bf16*)kcache, (const bf16*)vcache, num_pages, p, B,
                                max_len, (cudaStream_t)stream);
}

int b200_op_attn_decode(const void* q, int64_t ldq, void* out, int64_t ldo, const void* kcache, const void* vcache,
                        const int32_t* page_table, int max_pages, const int32_t* seq_slot, const int32_t* tok_pos, int B,
                        int nh, int nkv, int splits, float* part_o, float* part_ml, void* stream) {
  AttnDecodeParams p{};
  p.q = (const bf16*)q; p.ldq = ldq; p.out = (bf16*)out; p.ldo = ldo; p.kcache = (const bf16*)kcache; p.vcache = (const bf16*)vcache;
  p.page_table = page_table; p.max_pages = max_pages; p.seq_slot = seq_slot; p.tok_pos = tok_pos; p.nh = nh; p.nkv = nkv;
  p.G = nh / nkv; p.splits = splits; p.part_o = part_o; p.part_ml = part_ml;
  p.scale_log2 = (1.0f / sqrtf((float)kHeadDim)) * 1.4426950408889634f;
  static int* op_split_cnt = nullptr;   // arrival counters of the last-CTA merge, left at zero by every merge
  static int op_split_cnt_len = 0;
  if (splits > 1 && B * nkv > op_split_cnt_len) {
    B200_CUDA_OK(cudaFree(op_split_cnt));
    op_split_cnt = nullptr;
    B200_CUDA_OK(cudaMalloc(reinterpret_cast<void**>(&op_split_cnt), (size_t)B * nkv * sizeof(int)));
    B200_CUDA_OK(cudaMemset(op_split_cnt, 0, (size_t)B * nkv * sizeof(int)));
    op_split_cnt_len = B * nkv;
  }
  p.split_counter = op_split_cnt;
  return launch_attn_decode(p, B, (cudaStream_t)stream);
}

int b200_op_rope_kv(const void* qkv, int64_t ld, void* q_out, int64_t ldq, void* kcache, void* vcache,
                    const int32_t* page_table, int max_pages, const int32_t* tok_seq, const int32_t* tok_pos,
                    const void* cos_tab, const void* sin_tab, int T, int nh, int nkv, void* stream) {
  RopeKvParams p{};
  p.qkv = (const bf16*)qkv; p.ld = ld; p.q_out = (bf16*)q_out; p.ldq = ldq; p.kcache = (bf16*)kcache; p.vcache = (bf16*)vcache;
  p.page_table = page_table; p.max_pages = max_pages; p.tok_seq = tok_seq; p.tok_pos = tok_pos;
  p.cos_tab = (const bf16*)cos_tab; p.sin_tab = (const bf16*)sin_tab; p.nh = nh; p.nkv = nkv;
  p.T = T;
  rope_kv_kernel<<<T, 512, 0, (cudaStream_t)stream>>>(p);
  B200_CUDA_OK(cudaGetLastError());
  return 0;
}

int b200_op_argmax(const void* logits, int64_t ld, int B, int V, float* out_val, int32_t* out_idx, void* stream) {
  argmax_kernel<<<dim3(B, 1), 1024, 0, (cudaStream_t)stream>>>((const bf16*)logits, ld, V, 0, out_val, out_idx, P2P{}, 0);
  B200_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // extern "C"
