/*
 * kserve_b200 — C ABI of the B200-native LLM predict path.
 *
 * This is the drop-in boundary for the reference's HF generative runtime: every entry point below
 * replaces one call the reference makes into its third-party compute backend (transformers/torch) or,
 * for the batcher, the body of one Go function.  Plain pointers and sizes only; no torch types.
 * All functions return 0 on success, non-zero on failure; b200_last_error() returns the message for the
 * calling thread.  One engine handle per GPU; calls on one handle must be serialised by the caller
 * (the reference serialises them too: generative_model.py:341-354 single worker thread).
 *
 * Reference citations are relative to /root/reference.
 */
#ifndef KSERVE_B200_H_
#define KSERVE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b200_engine b200_engine_t;

/* Model / runtime configuration. Mirrors the fields of the HF config the reference reads in
 * python/huggingfaceserver/huggingfaceserver/__main__.py:242-246 plus the serving limits of
 * generative_model.py:203-271 (max_length) and the TP layout of SURVEY.md §8e. */
typedef struct b200_model_config {
  int32_t vocab_size;          /* rows of embed_tokens / lm_head (after any [PAD] resize, :256-265) */
  int32_t hidden_size;
  int32_t intermediate_size;
  int32_t num_layers;
  int32_t num_heads;
  int32_t num_kv_heads;
  int32_t head_dim;            /* must be 128 */
  int32_t max_position;        /* rope table length */
  float rms_eps;
  float rope_theta;
  int32_t max_batch;           /* <= 64 sequences decoded together */
  int32_t max_seq_len;         /* prompt + generated tokens per sequence */
  int32_t max_prefill_tokens;  /* packed prompt tokens per generate() call */
  int32_t num_kv_pages;        /* 0 = max_batch * ceil(max_seq_len / 64) */
  int32_t tp_rank;
  int32_t tp_size;             /* 1, 2, 4 or 8; heads, kv heads and intermediate must divide */
  int32_t device;              /* CUDA device ordinal */
  int32_t num_experts;         /* 0 = dense MLP; > 0 = Mixtral-style sparse MoE (modeling_mixtral.py:62-135) */
  int32_t num_experts_per_tok; /* must be 2 when num_experts > 0 */
} b200_model_config_t;

/* Creates the engine on cfg->device. nccl_unique_id: 128 bytes shared by all ranks (from
 * b200_nccl_unique_id on rank 0, distributed by the host), or NULL when tp_size == 1. */
int b200_engine_create(const b200_model_config_t* cfg, const void* nccl_unique_id, b200_engine_t** out);
int b200_engine_destroy(b200_engine_t* e);
int b200_nccl_unique_id(void* out128);

/* Tensor parallel, optional fast path: every rank exports a 64-byte IPC handle of its exchange block and imports
 * the handles of all ranks (index = tp_rank; distributed by the host).  With it the per-layer all-reduce of the
 * decode step runs inside one kernel over NVLink peer memory (fused with the split-K reduce, residual add and
 * RMSNorm); without it the engine uses ncclAllReduce. */
int b200_engine_ipc_export(b200_engine_t* e, void* handle64);
int b200_engine_ipc_import(b200_engine_t* e, const void* handles, int32_t n);

/* Weights, by HF state_dict name (what AutoModelForCausalLM.from_pretrained would load,
 * generative_model.py:249-254).  `data` is the FULL (unsharded) bf16 tensor, row-major, on the host
 * (on_device=0) or on this engine's GPU (on_device=1); the engine copies the shard of its tp_rank and
 * fuses q/k/v and gate/up.  MoE checkpoints use the fused-expert names `mlp.gate.weight` [E,H],
 * `mlp.experts.gate_up_proj` [E,2I,H] and `mlp.experts.down_proj` [E,H,I].  b200_engine_finalize_weights fails if
 * a tensor is missing. */
int b200_engine_set_weight(b200_engine_t* e, const char* hf_name, const void* data, int on_device,
                           int ndim, const int64_t* shape);
int b200_engine_finalize_weights(b200_engine_t* e);
/* Optional: bf16 cos/sin tables [max_position][64] computed by the host exactly as
 * LlamaRotaryEmbedding.forward does (fp32 inv_freq * position -> cos/sin -> bf16).  Without this call the
 * engine computes the tables itself from rope_theta. */
int b200_engine_set_rope_table(b200_engine_t* e, const void* cos_bf16, const void* sin_bf16, int32_t rows);

/* Generation parameters == what the reference puts into GenerationConfig + StoppingCriteria
 * (generative_model.py:388-402, 576-593).  Greedy only this round (do_sample is never set there). */
typedef struct b200_gen_params {
  int32_t max_new_tokens;
  int64_t pad_token_id;          /* finished rows are padded with it (transformers utils.py:2796-2797) */
  const int64_t* eos_token_ids;  /* may be NULL */
  int32_t num_eos;
  const int64_t* stop_tokens;    /* flattened stop sequences (token ids) */
  const int32_t* stop_offsets;   /* [num_stop + 1] offsets into stop_tokens */
  int32_t num_stop;
  const int64_t* forced_tokens;  /* testing: [B][max_new_tokens] tokens to append instead of argmax, or NULL */
  /* Logits processors / sampling — what build_generation_config (generative_model.py:388-402) passes to transformers.
   * All-zero == greedy without processors.  tp_size must be 1 when any of them is active. */
  float repetition_penalty;      /* 0 or 1 = off; presence_penalty > 0 is mapped here by the reference (q8) */
  int32_t do_sample;             /* 0 = greedy (the reference default, q9); 1 = temperature / top-k / top-p sampling */
  float temperature;             /* 0 = 1.0 */
  float top_p;                   /* 0 = 1.0 (off) */
  int32_t top_k;                 /* 0 = 50, transformers' GenerationConfig default; at most 1024 */
  uint64_t seed;                 /* Philox key; the same seed reproduces the same tokens (not torch's stream) */
} b200_gen_params_t;

/* Per-step callback for streaming (TextIteratorStreamer in the reference, generative_model.py:307-322):
 * called on the calling thread after each step with the B new tokens. Return non-zero to abort. */
typedef int (*b200_token_callback)(void* user, int32_t step, const int64_t* tokens, int32_t batch);

/* Replaces `self._model.generate(**kwargs)` (generative_model.py:314,328).
 *   input_ids      host int64 [B][S] (left padded when attention_mask has leading zeros)
 *   attention_mask host int64 [B][S] or NULL (== all ones); must be left-contiguous padding
 *   out_ids        host int64 [B][S + max_new_tokens]; rows are the prompt followed by generated tokens
 *   out_len        S + number of generated tokens (same for every row, as in the reference)
 *   stop_triggered 1 iff a stop sequence ended generation (finish_reason "stop", :621-627)
 *   logits_bf16    NULL, or host uint16 [max_new_tokens][B][vocab_size] receiving each step's bf16 logits; under tensor
 *                  parallelism rank r receives its vocabulary shard [max_new_tokens][B][Vl], Vl = min(ceil(V / tp),
 *                  V - r * ceil(V / tp)) columns starting at column r * ceil(V / tp) */
int b200_generate(b200_engine_t* e, const int64_t* input_ids, const int64_t* attention_mask, int32_t B,
                  int32_t S, const b200_gen_params_t* params, int64_t* out_ids, int32_t* out_len,
                  int32_t* stop_triggered, uint16_t* logits_bf16, b200_token_callback cb, void* user);

/* Timing of the last b200_generate on this engine, measured with CUDA events on the engine stream. */
typedef struct b200_timing {
  float prefill_ms;       /* H2D of the prompt .. first token selected */
  float decode_ms;        /* all decode steps */
  int32_t decode_steps;
  int32_t kernel_launches;/* kernels of this library launched by the call (graph nodes included) */
} b200_timing_t;
int b200_engine_last_timing(b200_engine_t* e, b200_timing_t* out);

/* Failure handling of the device-side waits (peer-memory all-reduce packets / flags, candidate exchange, stream-K pieces):
 * a wait that times out — a tensor-parallel peer died or fell out of step — does NOT trap the CUDA context; it records a
 * code, the kernels run to completion with whatever data they have, and the entry point that next synchronises
 * (b200_generate, b200_batch_predict, b200_fetch_staged, b200_cb_poll) returns -8 with the text in b200_last_error();
 * the engine then refuses further work until it is re-created (or the fault is reset for a diagnostic retry).
 * code: 0 none, 1 peer flag, 2 all-reduce packet, 3 candidate exchange, 4 stream-K piece. */
int b200_engine_fault(b200_engine_t* e, int32_t* code, int32_t reset);

/* Device-resident variant for benchmarking the kernels alone: prompt already staged with
 * b200_stage_prompt (no H2D/D2H inside), runs prefill + `steps` decode steps, no result copy. */
int b200_stage_prompt(b200_engine_t* e, const int64_t* input_ids, const int64_t* attention_mask, int32_t B,
                      int32_t S, const b200_gen_params_t* params);
int b200_run_staged(b200_engine_t* e, int32_t do_prefill, int32_t decode_steps);
/* prefill + decode_steps decode steps of the staged prompt, each phase bracketed by CUDA events on the
 * engine's own stream (the stream every kernel of the engine is launched on); synchronises at the end. */
int b200_run_staged_timed(b200_engine_t* e, int32_t decode_steps, float* prefill_ms, float* decode_ms);
int b200_fetch_staged(b200_engine_t* e, int64_t* out_ids, int32_t* out_len, int32_t* stop_triggered);

/* ---- batcher ----------------------------------------------------------------------------------------
 * Replaces BatchHandler.batchPredict (pkg/batcher/handler.go:99-155).  rows[i] / row_lens[i] are the token
 * ids of instance i of the formed batch (all waiting requests' instances, in arrival order); they are
 * concatenated on the device, generated as ONE batch and returned as predictions[n_rows][max_new_tokens]
 * (instance order, rows padded with pad_token_id after *n_generated tokens), so request r's answer is rows
 * [first_r, first_r + count_r) exactly as handler.go:139-150 scatters them. */
int b200_batch_predict(b200_engine_t* e, const int64_t* const* rows, const int32_t* row_lens, int32_t n_rows,
                       const b200_gen_params_t* params, int64_t* predictions, int32_t* n_generated,
                       int32_t* stop_triggered);

/* The trigger / index bookkeeping of BatchHandler.batch (handler.go:157-188) as a clock-driven state machine
 * (the host keeps its own concurrency: goroutines+channels in Go, asyncio in Python).
 *   create: <=0 selects the reference defaults 32 instances / 5000 ms (handler.go:190-196).
 *   add   : a request with n_instances arrived at now_us -> ticket (the `case req := <-channelIn` arm).
 *   tick  : the check made after every select iteration (handler.go:180-186): fires when
 *           instances >= max_batch_size, or whole ms since the first instance >= max_latency and > 0 waiting.
 *           On fire returns the waiting requests (ticket, first index, count) and resets. */
typedef struct b200_batcher b200_batcher_t;
int b200_batcher_create(int32_t max_batch_size, int32_t max_latency_ms, b200_batcher_t** out);
int b200_batcher_destroy(b200_batcher_t* b);
int b200_batcher_config(b200_batcher_t* b, int32_t* max_batch_size, int32_t* max_latency_ms);
int b200_batcher_add(b200_batcher_t* b, int64_t now_us, int32_t n_instances, int64_t* ticket);
int b200_batcher_tick(b200_batcher_t* b, int64_t now_us, int32_t cap, int64_t* tickets, int32_t* first,
                      int32_t* count, int32_t* n_requests, int32_t* total_instances);

/* ---- single kernels on caller-provided device pointers (unit tests / micro-benchmarks) ------------- */
/* D = A[M,K] * B[N,K]^T, bf16, fp32 accumulate. epi: 0 store, 1 store+residual, 2 swiglu (B rows
 * interleaved 16 gate/16 up), 3 transposed store, 4 transposed swiglu (A rows interleaved),
 * 5 transposed fp32 split-K partials.  block_n: 256 for epi 0-2, 16/32/64 for epi 3-5. */
int b200_op_gemm(const void* A, const void* B, void* out, const void* residual, int M, int N, int K, int epi,
                 int block_n, int splits, int64_t ldo, void* stream);
int b200_op_rmsnorm(void* x, const void* w, void* xn, int rows, int H, float eps, const float* partial,
                    int splits, const void* y, void* stream);
/* tcgen05/TMEM prefill attention (the engine's); q_rows = rows of the q buffer, num_pages = pages of the caches */
int b200_op_attn_prefill_tc(const void* q, int64_t ldq, int q_rows, void* out, int64_t ldo, const void* kcache,
                            const void* vcache, int num_pages, const int32_t* page_table, int max_pages,
                            const int32_t* cu_seqlens, const int32_t* seq_slot, int B, int max_len, int nh, int nkv,
                            void* stream);
/* split-KV decode attention; with splits > 1 the last CTA of each (row, kv head) merges the part_o / part_ml partials */
int b200_op_attn_decode(const void* q, int64_t ldq, void* out, int64_t ldo, const void* kcache,
                        const void* vcache, const int32_t* page_table, int max_pages, const int32_t* seq_slot,
                        const int32_t* tok_pos, int B, int nh, int nkv, int splits, float* part_o, float* part_ml,
                        void* stream);
int b200_op_rope_kv(const void* qkv, int64_t ld, void* q_out, int64_t ldq, void* kcache, void* vcache,
                    const int32_t* page_table, int max_pages, const int32_t* tok_seq, const int32_t* tok_pos,
                    const void* cos_tab, const void* sin_tab, int T, int nh, int nkv, void* stream);
int b200_op_argmax(const void* logits, int64_t ld, int B, int V, float* out_val, int32_t* out_idx, void* stream);

/* Host-DRAM KV tier (BASELINE.json configs[3]): move all KV pages of staged sequence `slot` to pinned host memory /
 * back to the device, asynchronously on the engine stream.  scrub != 0 overwrites the device pages after the copy
 * (tests).  Decoding after swap_in continues exactly as if the sequence had stayed resident. */
int b200_kv_swap_out(b200_engine_t* e, int32_t slot, int32_t scrub);
int b200_kv_swap_in(b200_engine_t* e, int32_t slot);

/* Continuous (iteration-level) batching — SURVEY.md §8(f) ranks 1 and 4.  Replaces the reference's strictly serial
 * request loop (python/huggingfaceserver/huggingfaceserver/generative_model.py:341-354: one `generate` at a time) and the
 * throughput role of the Go batcher (pkg/batcher/handler.go:157-188): sequences join and leave the running batch between
 * decode steps.  One engine per GPU, one scheduler thread (calls are not re-entrant); under tensor parallelism every rank
 * makes the same calls in the same order (kserve_b200/tp.py replicates them), all host-side decisions are deterministic.
 *
 *   b200_cb_begin   enter the mode: every KV page goes to the free pool; eos ids apply to every sequence, as
 *                   `generation_config.eos_token_id` does in the reference
 *   b200_cb_config  prefill_chunk_tokens: 0 = a prompt is prefilled completely inside b200_cb_admit; >= 128 = prompts
 *                   are prefilled in chunks of at most that many packed tokens (multiples of 128 per prompt), ONE chunk
 *                   pass before every decode step of b200_cb_step, so an admit never stalls the running sequences for
 *                   longer than a chunk.  prefix_cache != 0: full 128-token blocks of a finished prefill stay in the
 *                   pool (reference counted, least-recently-used eviction) keyed by the chain hash of the tokens up to
 *                   and including the block; a later prompt with the same leading blocks shares those pages and only
 *                   its remaining tokens are computed (greedy results are identical to a full prefill).
 *   b200_cb_admit   n new prompts (host int64 token rows) into free slots: KV pages for len + max_new tokens each (rc -7
 *                   and "KV page pool exhausted" when the pool, after evicting unused cached blocks, cannot supply
 *                   them: nothing is admitted), per-sequence max_new, up to 4 stop sequences of <= 8 tokens each
 *                   (stop_count[i] sequences for prompt i, stop_offsets = running offsets, sum(stop_count) + 1 entries,
 *                   into stop_tokens) and, optionally, per-sequence logits processors / sampling: `sampling[i]` uses the
 *                   repetition_penalty / do_sample / temperature / top_p / top_k / seed fields of b200_gen_params_t
 *                   (NULL = greedy; tp_size must be 1 when any is active); slots_out[i] receives the slot of prompt i
 *   b200_cb_step    n iterations; each = one prefill chunk pass if prompts are pending, then one decode step over every
 *                   running slot (CUDA graph per row count); finished sequences are frozen on the device until released
 *   b200_cb_poll    per slot: tokens generated so far, finished flag, stop-sequence flag ([max_batch] each)
 *   b200_cb_read    generated tokens [first, first + cap) of a slot (for streaming reads as well as final results)
 *   b200_cb_release free the slot and drop its page references (its row leaves the decode batch at the next step)
 *   b200_cb_stats   out10 = {prompt tokens admitted, of those served from shared pages, prefilled tokens, cache evictions,
 *                   prefill passes, pages an admit could obtain now, cached blocks, prompts still being prefilled,
 *                   sequences swapped out to host DRAM, swapped back in}
 *   b200_cb_end     leave the mode
 * Greedy results per sequence are identical to b200_generate on that prompt alone. */
int b200_cb_begin(b200_engine_t* e, int64_t pad_token_id, const int64_t* eos_token_ids, int32_t num_eos);
int b200_cb_config(b200_engine_t* e, int32_t prefill_chunk_tokens, int32_t prefix_cache);
int b200_cb_admit(b200_engine_t* e, int32_t n, const int64_t* const* rows, const int32_t* lens, const int32_t* max_new,
                  const int32_t* stop_count, const int32_t* stop_offsets, const int64_t* stop_tokens,
                  const b200_gen_params_t* sampling, int32_t* slots_out);
int b200_cb_step(b200_engine_t* e, int32_t n_steps);
int b200_cb_poll(b200_engine_t* e, int32_t* n_gen, int32_t* finished, int32_t* stop_hit);
int b200_cb_read(b200_engine_t* e, int32_t slot, int32_t first, int64_t* out, int32_t cap, int32_t* n_out);
int b200_cb_release(b200_engine_t* e, int32_t slot);
int b200_cb_stats(b200_engine_t* e, int64_t* out10);
int b200_cb_end(b200_engine_t* e);
/* Host-DRAM KV tier (BASELINE.json configs[3]) for the continuous batcher: preempt a RUNNING sequence to pinned host memory
 * (all of its KV pages, asynchronously on the engine stream; its pages return to the pool, it leaves the decode batch, its
 * per-sequence state stays on the device) and bring it back later (fresh pages; rc -7 while the pool cannot supply them).
 * Decoding resumes bit-identically.  The policy is the scheduler's: kserve_b200/continuous.py preempts the most recently
 * admitted request when an admission finds the pool exhausted and resumes swapped requests before admitting new ones. */
int b200_cb_swap_out(b200_engine_t* e, int32_t slot);
int b200_cb_swap_in(b200_engine_t* e, int32_t slot);

/* Debug timeline: capacity > 0 enables per-CTA {t0, t1 (globaltimer ns), kind, block} records (24 bytes each),
 * 0 disables; read drains up to `capacity` records into `out`. */
int b200_debug_trace(int32_t capacity);
int b200_debug_trace_read(void* out, int32_t capacity, int32_t* n);

const char* b200_last_error(void);
const char* b200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* KSERVE_B200_H_ */
