/*
 * b200serve.h -- C ABI of libb200serve.so, the B200-native (sm_100a) hot path that replaces the
 * Triton engine path of clearml-serving.
 *
 * The reference has NO FFI for this path (it is 100% Python): a request crosses into the model
 * runtime as a gRPC ModelInfer message built in
 *     clearml_serving/serving/preprocess_service.py:374-422   (collate: np.array + protobuf contents)
 * and comes back through
 *     clearml_serving/serving/preprocess_service.py:430-446   (scatter: np.frombuffer + np.resize),
 * with tritonserver (third-party) doing queue -> batch -> H2D -> model -> D2H -> split, configured by
 *     clearml_serving/engines/triton/triton_helper.py:291-409 (config.pbtxt: dims, dtypes, max_batch).
 * For the in-process CPU engines the same boundary is `self._model.predict(data)`
 *     preprocess_service.py:459-464 (sklearn), :478-483 (xgboost).
 * Each entry point below names the reference interface it stands in for.  INTEGRATION.md shows the
 * ctypes binding a maintainer adds to the reference to call it.
 *
 * Conventions: every function returns 0 on success or a negative b2s_status; the message of the
 * last failure on the calling thread is b2s_last_error().  There is no CPU fallback: without a
 * CUDA device b2s_init fails and every other call returns B2S_ERR_NOT_INITIALISED.
 * A device out-of-memory message contains the literal "CUDA out of memory. " so that the reference's
 * restart logic (clearml_serving/serving/main.py:116-123) keeps working.
 * Plain pointers and sizes only; no torch / C++ types cross this boundary.
 */
#ifndef B200SERVE_H
#define B200SERVE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define B2S_API __attribute__((visibility("default")))
#else
#define B2S_API
#endif

#define B2S_ABI_VERSION 2

typedef enum b2s_status {
    B2S_OK = 0,
    B2S_ERR_INVALID = -1,         /* bad argument / malformed model blob / shape or dtype mismatch */
    B2S_ERR_CUDA = -2,            /* CUDA runtime error (message carries the CUDA error string)    */
    B2S_ERR_OOM = -3,             /* device or pinned arena exhausted: "CUDA out of memory. ..."    */
    B2S_ERR_NOT_INITIALISED = -4, /* b2s_init not called / no CUDA device                           */
    B2S_ERR_BUSY = -5,            /* all staging slots of the stream are in flight                  */
    B2S_ERR_NOT_READY = 1         /* b2s_event_query: batch still running (not an error)            */
} b2s_status;

/* numpy-compatible element types: the dtype universe of the reference's Triton client
 * (_content_lookup, preprocess_service.py:271-282) plus fp16 for on-device compute. */
typedef enum b2s_dtype {
    B2S_F32 = 0, B2S_F64 = 1, B2S_I32 = 2, B2S_I64 = 3, B2S_U8 = 4, B2S_I8 = 5,
    B2S_BOOL = 6, B2S_U64 = 7, B2S_F16 = 8, B2S_U32 = 9
} b2s_dtype;

typedef enum b2s_model_kind {
    B2S_MODEL_FOREST = 1, /* GBDT / random forest: replaces Booster.predict / sklearn predict      */
    B2S_MODEL_LINEAR = 2, /* linear / logistic decision function + argmax                          */
    B2S_MODEL_GRAPH = 3   /* op-list DL graph (ResNet / BERT class), fp16 compute                  */
} b2s_model_kind;

#define B2S_MAX_DIMS 8

/* One host tensor of one request.  `data` is caller-owned host memory (need not be pinned).
 * Stands in for InferInputTensor (name/shape/typed contents, preprocess_service.py:395-409) on the
 * way in and for raw_output_contents[i] + shape (preprocess_service.py:432-442) on the way out. */
typedef struct b2s_tensor {
    void *data;
    int32_t dtype;                 /* b2s_dtype */
    int32_t ndim;
    int64_t shape[B2S_MAX_DIMS];   /* leading dim = the request's own batch dim (usually 1) */
} b2s_tensor;

typedef uint64_t b2s_model_t;
typedef uint64_t b2s_stream_t;
typedef uint64_t b2s_event_t;

/* Static description of a loaded model's I/O (what triton_helper.py:342-360 writes into
 * config.pbtxt as input/output dims + data_type). */
typedef struct b2s_model_info {
    int32_t kind;
    int32_t n_inputs;
    int32_t n_outputs;
    int32_t in_dtype[4];
    int32_t out_dtype[4];
    int64_t in_row_elems[4];   /* elements per batch row of input i  (-1 = variable length)   */
    int64_t out_row_elems[4];  /* elements per batch row of output i                          */
    int64_t weight_bytes;      /* bytes resident in HBM for this model                        */
    int64_t algo_bytes_fixed;  /* algorithmic bytes per launch independent of batch rows      */
    int64_t algo_bytes_per_row;/* algorithmic bytes per batch row (in + out)                  */
} b2s_model_info;

/* ---- library / device lifetime ------------------------------------------------------------- */

/* Bind `device`, create the shared pinned staging arena (`pinned_arena_bytes`, 0 = default 64 MiB).
 * Replaces: tritonserver start-up (triton_helper.py:245-261; --pinned-memory-pool-byte-size). */
B2S_API int b2s_init(int device, size_t pinned_arena_bytes);
B2S_API int b2s_shutdown(void);
B2S_API int b2s_abi_version(void);
B2S_API const char *b2s_last_error(void);
/* kernels launched by this library since b2s_init (the bench's `gpu_launches` evidence) */
B2S_API uint64_t b2s_launch_count(void);
B2S_API int b2s_device_count(void);

/* ---- models -------------------------------------------------------------------------------- */

/* Load a model from a packed blob (built by clearml_serving_b200.formats from the same files the
 * reference loads: XGBoost JSON via Booster.load_model preprocess_service.py:475-476, joblib pickles
 * via joblib.load :457, TorchScript/ONNX placed by triton_helper.py:159-186) onto `device`.
 * `cfg_json` may be NULL. */
B2S_API int b2s_model_load(int device, int kind, const void *blob, size_t blob_bytes,
                   const char *cfg_json, b2s_model_t *out_model);
B2S_API int b2s_model_free(b2s_model_t model);
B2S_API int b2s_model_get_info(b2s_model_t model, b2s_model_info *out_info);
/* developer aid: 64 int64 phase stamps of the model's last launch (forest: needs B2S_FOREST_TIMING=1) */
B2S_API int b2s_debug_read(b2s_model_t model, long long *out64);

/* ---- streams: one CUDA stream + staging slots per endpoint ----------------------------------- */

/* One stream per endpoint (north_star: "one CUDA stream per endpoint with a shared pinned staging
 * arena").  `max_rows` = the endpoint's max_batch_size (auxiliary_cfg, examples/huggingface/
 * readme.md:113); `n_slots` batches may be in flight at once (0 = default 4).  `max_row_elems`
 * bounds variable-length inputs (ignored for fixed-width models, pass 0). */
B2S_API int b2s_stream_create(b2s_model_t model, int64_t max_rows, int64_t max_row_elems, int n_slots,
                      b2s_stream_t *out_stream);
B2S_API int b2s_stream_destroy(b2s_stream_t stream);
B2S_API int b2s_stream_synchronize(b2s_stream_t stream);
/* raw cudaStream_t, for callers that record their own CUDA events on it (bench.py) */
B2S_API void *b2s_stream_cuda_handle(b2s_stream_t stream);

/* ---- the hot path ---------------------------------------------------------------------------- */

/* Collate n_req requests (each with model.n_inputs tensors, row-major in[req * n_inputs + i]) into
 * the stream's next pinned slot, H2D, run the model's kernels, D2H; all asynchronous on the stream.
 * `out[req * n_outputs + o].data` must point at caller-owned host buffers large enough for the
 * request's rows; they are filled by b2s_event_wait (scatter).  Shapes of `out` are written back.
 * Replaces: the whole TritonPreprocessRequest.process round trip (preprocess_service.py:385-446)
 * plus tritonserver's dynamic-batch execution. */
B2S_API int b2s_infer_batch(b2s_model_t model, b2s_stream_t stream, int32_t n_req,
                    const b2s_tensor *in, b2s_tensor *out, b2s_event_t *out_done);

/* Zero-copy variant for hosts that collate straight into the pinned slot (the Python scheduler):
 * acquire a free slot, write rows into in_ptr[i] (row-major, model dtype), submit, then read
 * out_ptr[o] after b2s_event_wait and release.  For variable-length inputs `row_offsets`
 * (int64[n_rows+1], element offsets into each ragged input) is passed at submit. */
B2S_API int b2s_slot_acquire(b2s_stream_t stream, int32_t *out_slot, void **in_ptr /*[n_inputs]*/,
                     void **out_ptr /*[n_outputs]*/);
B2S_API int b2s_slot_submit(b2s_model_t model, b2s_stream_t stream, int32_t slot, int64_t n_rows,
                    const int64_t *row_offsets, b2s_event_t *out_done);
/* Collate INSIDE the library (no GIL, worker pool for large batches) into an acquired slot and submit it:
 * in_ptrs[req * n_inputs + i] = host pointer of request `req`'s input i (C-contiguous, the model's dtype),
 * req_rows[req] = that request's own batch rows, req_row_len[req] = elements per row of its variable-length inputs
 * (NULL for fixed-width models).  Rows are packed back to back in request order; for variable-length models the
 * slot's row-offset table (cu_seqlens) is written too.  The outputs are read from the slot's out_ptr after
 * b2s_event_wait, then b2s_slot_release.  This is what the Python dynamic batcher calls per batch: it replaces
 * the per-request np.array(...).flatten() -> protobuf of preprocess_service.py:393-406 and tritonserver's batch
 * gather. */
B2S_API int b2s_slot_collate(b2s_model_t model, b2s_stream_t stream, int32_t slot, int32_t n_req,
                             const void *const *in_ptrs, const int64_t *req_rows, const int64_t *req_row_len,
                             b2s_event_t *out_done);
B2S_API int b2s_slot_release(b2s_stream_t stream, int32_t slot);

/* Completion: wait (blocking, no GIL needed) / poll.  b2s_event_wait performs the scatter of
 * b2s_infer_batch outputs into the per-request buffers and frees the slot. */
B2S_API int b2s_event_wait(b2s_event_t ev);
B2S_API int b2s_event_query(b2s_event_t ev);

/* Device-resident execution (inputs/outputs already in HBM; used for kernel-only timing and by
 * hosts that own device memory).  d_in[i] / d_out[o] are device pointers on the model's device. */
B2S_API int b2s_infer_device(b2s_model_t model, b2s_stream_t stream, int64_t n_rows,
                     const void *const *d_in, void *const *d_out, const int64_t *d_row_offsets);

/* Plain device memory helpers so a host needs no other CUDA binding. */
B2S_API int b2s_device_malloc(int device, size_t bytes, void **out_ptr);
B2S_API int b2s_device_free(int device, void *ptr);
B2S_API int b2s_memcpy_h2d(int device, void *dst, const void *src, size_t bytes);
B2S_API int b2s_memcpy_d2h(int device, void *dst, const void *src, size_t bytes);
/* Overwrite a buffer larger than L2 (benchmark hygiene: cold-cache timing). */
B2S_API int b2s_flush_l2(int device);
/* Same, but enqueued asynchronously on a library stream: the GPU stays busy while the host queues
 * the timed launch behind it, so CUDA-event timing of a microsecond-scale kernel carries no host
 * launch gap. */
B2S_API int b2s_stream_flush_l2(b2s_stream_t stream);

/* CUDA-event timers on a library stream (device time, not wall clock). */
typedef uint64_t b2s_timer_t;
B2S_API int b2s_timer_create(b2s_stream_t stream, b2s_timer_t *out_timer);
B2S_API int b2s_timer_start(b2s_timer_t timer);
B2S_API int b2s_timer_stop(b2s_timer_t timer);
B2S_API int b2s_timer_elapsed_ms(b2s_timer_t timer, float *out_ms); /* synchronises on the stop event */
B2S_API int b2s_timer_destroy(b2s_timer_t timer);

/* ---- operator-level entry points (device pointers) ------------------------------------------------
 * The building blocks of B2S_MODEL_GRAPH models, exported so that parity tests can check each kernel
 * against its oracle through the C ABI.  `cuda_stream` is a raw cudaStream_t (b2s_stream_cuda_handle)
 * or NULL for the default stream.  Stand in for the cuBLAS/cuDNN calls of tritonserver's libtorch /
 * ONNX-Runtime backends (selected by triton_helper.py:378-385). */

/* C[M,N] = act(A[M,K] . B[N,K]^T + bias[N]) + residual[M,N]; A,B,residual 16-bit (fp16 or bf16),
 * bias fp32, C 16-bit or fp32.  act: 0 none, 1 GELU(erf), 2 ReLU, 3 tanh, 4 SwiGLU (the LLM gate/up projection: columns
 * [64j, 64j+32) of A.B^T are gate, [64j+32, 64j+64) up; C[M, N/2] 16-bit = silu(gate) * up, N % 64 == 0, no bias /
 * residual).  tcgen05 + TMA + TMEM. */
B2S_API int b2s_op_gemm(int device, void *cuda_stream, const void *A, const void *B, void *C, int M, int N,
                        int K, const float *bias, const void *residual, int act, int is_bf16, int out_f32);

/* y[n_img,OH,OW,Cout] = act(conv2d(x[n_img,H,W,C], w[Cout,KS,KS,C]) + bias[Cout]) (+ residual[n_img,OH,OW,Cout], with the
 * activation after the add when act_after): fp16 NHWC activations (C % 64 == 0), square filter, symmetric
 * stride / zero padding.  Implicit GEMM: the A tiles are gathered by im2col-mode TMA, no patch matrix exists.
 * Stands in for the cuDNN convolutions of tritonserver's backends (triton_helper.py:378-385, examples/pytorch). */
B2S_API int b2s_op_conv(int device, void *cuda_stream, const void *x, int64_t n_img, int H, int W, int C,
                        const void *w, int Cout, int KS, int stride, int pad, const float *bias,
                        const void *residual, void *y, int act, int act_after);

/* y[n_img,OH,OW,Cout] = act(conv2d(x, w, stride 2, pad 3) + bias) for the 7x7 network stem, straight from the request
 * pixels x[n_img,C,H,W] (NCHW, float32 or uint8 -- the dtypes the reference's Triton client can send,
 * preprocess_service.py:271-282; C <= 4).  The pixels are rearranged 2x2 space-to-depth into `z_scratch`
 * (n_img*(OH+3)*(OW+3)*32 bytes) and the convolution runs as a 4x4 stride-1 implicit GEMM; `w2` is the filter packed to
 * [Cout,256] fp16 (clearml_serving_b200/formats.py: stem_s2d_weight).  Cout <= 128, OW <= 128. */
B2S_API int b2s_op_conv_stem(int device, void *cuda_stream, const void *x_nchw, int in_dtype, int64_t n_img, int C,
                             int H, int W, const void *w2, int Cout, const float *bias, void *z_scratch, void *y,
                             int act);

/* LayerNorm over the last dim of fp32 in[rows,H] (torch.nn.LayerNorm numerics): writes an fp16 copy
 * (next GEMM operand) and/or an fp32 copy (residual stream); either output may be NULL. */
B2S_API int b2s_op_layernorm(int device, void *cuda_stream, const float *in, int64_t rows, int H,
                             const float *gamma, const float *beta, float eps, void *out16, float *out32);
/* BERT embeddings for packed (ragged) tokens: word[id] + position[idx in sequence] + type[tt] -> LayerNorm.
 * cu_seqlens int64[n_seq+1]; tables fp16 [vocab|max_pos|n_types, H]. */
B2S_API int b2s_op_embed_layernorm(int device, void *cuda_stream, const int32_t *ids, const int32_t *types,
                                   const int64_t *cu_seqlens, int n_seq, int64_t n_tokens, int H,
                                   const void *word, const void *pos, const void *type, int vocab, int max_pos,
                                   int n_types, const float *gamma, const float *beta, float eps, void *out16,
                                   float *out32);

/* Variable-length non-causal self-attention over packed tokens: qkv fp16 [T, 3*heads*64] (Q|K|V),
 * out fp16 [T, heads*64]; key_mask int32[T] (0 = masked key) or NULL.  Sequences of <= 384 tokens run on tcgen05
 * (S and O accumulators in tensor memory, K / V by TMA, thread-per-row exact softmax); longer ones on the
 * mma.sync flash form.  total_tokens = T = cu_seqlens[n_seq] (<= 0: read back from the device, which synchronises). */
B2S_API int b2s_op_attention(int device, void *cuda_stream, const void *qkv, const int64_t *cu_seqlens,
                             const int32_t *key_mask, void *out, int n_seq, int max_seqlen, int heads,
                             int head_dim, int64_t total_tokens);

/* developer aid: SM-clock stamps of the tcgen05 attention kernel's first work items (needs B2S_ATTN_TIMING=1) */
B2S_API int b2s_debug_attention_stamps(long long *out256);

/* ---- decoder-only LLM endpoint (BASELINE.json configs[4]) -------------------------------------------
 * Replaces the vLLM engine the reference wraps in `VllmPreprocessRequest`
 * (clearml_serving/serving/preprocess_service.py:1097-1348; engine args from `auxiliary_cfg`,
 * examples/vllm/preprocess.py): a Llama-family model (RMSNorm, RoPE, grouped-query attention, SwiGLU) with
 * a slot-based KV cache, greedy sampling, and optional 2-way tensor parallelism as ONE PROCESS PER GPU.
 * The two ranks exchange row-parallel partial sums through peer memory: each exports a handle with
 * b2s_llm_comm_export(), the host side swaps the 64 bytes (torch.distributed / any channel) and calls
 * b2s_llm_comm_attach() on both before the first step; both ranks then issue the same call sequence.
 * Every call enqueues on the model's own CUDA stream and returns; b2s_llm_get_tokens synchronises. */
typedef struct b2s_llm b2s_llm;
typedef struct b2s_llm_config {
    int32_t vocab, hidden, inter, n_layers, n_heads, n_kv_heads, head_dim; /* head_dim must be 128 */
    int32_t max_batch;   /* KV slots = sequences per wave, <= 32 */
    int32_t max_ctx;     /* positions per slot (prompt + generated) */
    int32_t max_tokens;  /* prompt tokens of one prefill wave (workspace size) */
    int32_t tp_size, tp_rank; /* 1 or 2 */
    float rope_theta, rms_eps;
    int32_t kv_pages;    /* pages (64 tokens x all kv heads of this rank, every layer) of the paged KV pool;
                            0 = max_batch * ceil(max_ctx / 64), i.e. every slot can reach max_ctx */
} b2s_llm_config;

B2S_API int b2s_llm_create(int device, const b2s_llm_config *cfg, b2s_llm **out);
B2S_API int b2s_llm_free(b2s_llm *llm);
/* deterministic on-device initialisation N(0, std) of every projection / embedding (configs[4] "random-init");
 * a pure function of (seed, tensor, global row, global col): all tensor-parallel layouts hold the same model */
B2S_API int b2s_llm_init_random(b2s_llm *llm, uint64_t seed, float std);
/* device pointer + shape of this rank's shard of a weight: "embed", "lm_head", "final_norm" (layer ignored),
 * "wqkv" [(hq+2hkv)*128/tp, H], "wo" [H, hq*128/tp], "wgu" [2*I/tp, H] (gate and up rows interleaved in
 * blocks of 32: fused row 64j+w = gate row 32j+w for w < 32, up row 32j+w-32 otherwise),
 * "wdown" [H, I/tp], "ln1", "ln2"; elem_bytes 2 = bf16, 4 = fp32.  Upload with b2s_memcpy_h2d. */
B2S_API int b2s_llm_tensor(b2s_llm *llm, const char *name, int layer, void **dptr, int64_t *rows, int64_t *cols,
                           int *elem_bytes);
B2S_API int b2s_llm_comm_export(b2s_llm *llm, unsigned char *handle64, uint64_t *bytes);
B2S_API int b2s_llm_comm_attach(b2s_llm *llm, const unsigned char *peer_handle64);
/* prompt wave: tokens[offsets[n_seq]] int32 (host), offsets[n_seq + 1]; sequence b takes KV slot b; samples
 * the first generated token of every sequence */
B2S_API int b2s_llm_prefill(b2s_llm *llm, int n_seq, const int32_t *tokens, const int32_t *offsets);
/* ---- continuous batching over the PAGED KV cache (what vLLM's scheduler + block manager do behind the reference's
 * engine, preprocess_service.py:1097-1348).  The cache is a pool of pages of 64 tokens; a sequence occupies a KV slot
 * (< max_batch) whose page-table row names its pages.  The HOST scheduler (clearml_serving_b200/llm_service.py) owns
 * slot / page allocation: it admits new prompts into free slots while other sequences are mid-generation
 * (b2s_llm_prefill_slots), then declares which sequences the next decode steps advance (b2s_llm_set_rows: any subset,
 * any order, state carried by the host: context length and the last sampled token), runs 1..k steps (b2s_llm_decode)
 * and reads the new tokens (b2s_llm_get_tokens: row r = r-th sequence given to set_rows / prefill_slots). */
B2S_API int b2s_llm_kv_info(b2s_llm *llm, int32_t *n_pages, int32_t *page_tokens, int32_t *pages_per_seq);
/* page-table row of `slot`: logical pages [first, first + n) -> pool pages `pages[i]`; ordered on the model's stream */
B2S_API int b2s_llm_set_pages(b2s_llm *llm, int slot, int first, int n, const int32_t *pages);
/* like b2s_llm_prefill, sequence b into KV slot slots[b] (distinct); sequences in other slots are untouched */
B2S_API int b2s_llm_prefill_slots(b2s_llm *llm, int n_seq, const int32_t *tokens, const int32_t *offsets, const int32_t *slots);
/* the rows of the next decode steps: row r = the sequence in KV slot slots[r] with ctx_len[r] cached tokens whose
 * last sampled token is next_tok[r]; the rows' generated-token buffers restart at position 0 */
B2S_API int b2s_llm_set_rows(b2s_llm *llm, int n_rows, const int32_t *slots, const int32_t *ctx_len, const int32_t *next_tok);
/* n_steps greedy decode steps for the current wave (use_graph: replay one captured CUDA graph per step) */
B2S_API int b2s_llm_decode(b2s_llm *llm, int n_steps, int use_graph);
/* out[n_seq][n] int32 (host): the first n generated tokens of each sequence; synchronises */
B2S_API int b2s_llm_get_tokens(b2s_llm *llm, int32_t *out, int n);
B2S_API int b2s_llm_keep_logits(b2s_llm *llm, int on);
B2S_API int b2s_llm_get_logits(b2s_llm *llm, float *out); /* [n_seq][vocab / tp] fp32 of the last step */
B2S_API int b2s_llm_synchronize(b2s_llm *llm);
B2S_API int b2s_llm_event_record(b2s_llm *llm, int which);             /* which in 0..7 */
B2S_API int b2s_llm_elapsed_ms(b2s_llm *llm, int from, int to, float *ms);
B2S_API int b2s_llm_flush_l2(b2s_llm *llm);
/* y[m][n_out] fp32 += X[m<=32, K] . W[n_out, K]^T (bf16 operands): the weight-streaming decode GEMM */
B2S_API int b2s_op_skinny_gemm(int device, void *cuda_stream, const void *W, const void *X, float *y, int n_out,
                               int K, int m);
/* Decode attention of one layer, fused with RoPE and the KV append (the kernels b2s_llm_decode runs).  ws_qkv fp32
 * [n_seq, (n_heads + 2 n_kv_heads) * 128] is the QKV projection (q heads | k heads | v heads) and is left all zero;
 * k_pool / v_pool bf16 [n_pages][n_kv_heads][64][128]; sequence b (<= 32) has ctx_len[b] cached tokens in the pages of
 * page_table[slots[b] * pages_per_seq ...], its new k / v row is appended at position ctx_len[b] (clamped to max_ctx - 1);
 * rope_cos / rope_sin fp32 [max_ctx][64]; out bf16 [n_seq, n_heads * 128].  stream_form 0: one CTA per (sequence, kv head);
 * 1: 64-key blocks dealt over n_cta SMs (2 CTAs per SM when n_heads / n_kv_heads <= 4), partials in part_ws
 * (2 * n_cta * 2 * 8 * 132 floats, no initial value needed) and arrival counters part_cnt (int [n_seq * n_kv_heads], zero
 * before, left zero). */
B2S_API int b2s_op_llm_attn_decode(int device, void *cuda_stream, float *ws_qkv, void *k_pool, void *v_pool, int n_pages,
                                   const int32_t *ctx_len, const int32_t *slots, const int32_t *page_table, int pages_per_seq,
                                   const float *rope_cos, const float *rope_sin, int max_ctx, void *out, int n_seq, int n_heads,
                                   int n_kv_heads, int stream_form, int n_cta, float *part_ws, int *part_cnt);
/* Prefill attention of one layer as b2s_llm_prefill runs it: RoPE on q (in place) and k, K / V rows written to the pages
 * of each sequence's slot, then causal grouped-query attention.  qkv bf16 [T, (n_heads + 2 n_kv_heads) * 128];
 * cu_seqlens int32 [n_seq + 1] (T = cu_seqlens[n_seq], read back: synchronises); token t is sequence tok_seq[t] at
 * position tok_pos[t] (0, 1, ... within its sequence); out bf16 [T, n_heads * 128]. */
B2S_API int b2s_op_llm_attn_prefill(int device, void *cuda_stream, void *qkv, void *k_pool, void *v_pool, const int32_t *cu_seqlens,
                                    const int32_t *tok_seq, const int32_t *tok_pos, const int32_t *slots, const int32_t *page_table,
                                    int pages_per_seq, const float *rope_cos, const float *rope_sin, int max_ctx, void *out, int n_seq,
                                    int max_seqlen, int n_heads, int n_kv_heads);
/* Greedy sampling: tokens[b] = index of the first maximum of logits fp32 [n_seq, vocab], the row split over n_split CTAs.
 * logits are left zero, keep (or NULL) receives a copy; row_key / row_cnt ([n_seq], zero before) are left zero.
 * Synchronises. */
B2S_API int b2s_op_llm_argmax(int device, void *cuda_stream, float *logits, float *keep, int n_seq, int vocab, int n_split,
                              unsigned long long *row_key, int *row_cnt, int32_t *tokens);

#ifdef __cplusplus
}
#endif
#endif /* B200SERVE_H */
