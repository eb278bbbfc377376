/* tensorlink_b200 — C ABI of the B200-native shard executor.
 *
 * The reference (tensorlink-lab/tensorlink) has no FFI: its shard operator is Python
 * (`LayerGroupModule.forward(**kwargs)`, tensorlink/ml/injector.py:154-281) and the arithmetic is
 * whatever Hugging Face `transformers` does inside `decoder_layer(...)`.  This header is the plain-C
 * boundary that sits UNDER that operator: every entry point replaces one group of ATen library calls
 * the reference's worker makes per layer (`module(**kwargs)`, tensorlink/ml/worker.py:333) or its
 * autograd (`assoc_output.backward(loss)`, tensorlink/ml/worker.py:271).  INTEGRATION.md shows the
 * ctypes binding a maintainer would add on the reference side.
 *
 * Conventions
 *  - all pointers are DEVICE pointers on the current device unless the name ends in `_host`;
 *    bf16 tensors are `void*`; row-major, innermost dimension contiguous, 16-byte aligned.
 *  - `stream` is a `cudaStream_t` passed as `void*`; every call is asynchronous on that stream.
 *  - no entry point allocates or frees device memory; workspaces are passed in.
 *  - return value: 0 on success, a negative `tl_status` otherwise; `tl_last_error()` gives the
 *    (thread-local) message.  There is no CPU fallback: on a machine without an sm_100 device
 *    compute calls return TL_ERR_NO_DEVICE.
 *  - rounding points replicate the reference's bf16 pipeline (each HF op output is rounded to bf16
 *    before the next op consumes it); accumulation is fp32.
 */
#ifndef TENSORLINK_B200_H
#define TENSORLINK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TL_ABI_VERSION 1

typedef enum {
    TL_OK = 0,
    TL_ERR_INVALID = -1,   /* bad shape / alignment / flag combination */
    TL_ERR_CUDA = -2,      /* a CUDA runtime / driver call failed       */
    TL_ERR_NO_DEVICE = -3, /* no sm_100 device visible                  */
    TL_ERR_WORKSPACE = -4  /* workspace too small                       */
} tl_status;

/* epilogue / operand flags for tl_gemm_bf16 and tl_gemv_bf16 */
#define TL_EPI_BIAS 1      /* + bias[N] (bf16), added in fp32 before the output rounding (oneDNN post-op)  */
#define TL_EPI_RESIDUAL 2  /* out = bf16(bf16(acc) + residual[M,N])  — HF `residual + hidden_states`        */
#define TL_EPI_SWIGLU 4    /* rows of B interleave gate/up (2j, 2j+1); out[M,N/2] = silu(gate)*up, HF rounding */
#define TL_EPI_OUT_F32 8   /* C is fp32 instead of bf16                                                     */
#define TL_EPI_ACCUM 16    /* C += result (bf16 read-modify-write; gradient accumulation)                   */
#define TL_A_MN_MAJOR 32   /* A is given as [K, M] row-major (contraction dim outermost)                     */
#define TL_B_MN_MAJOR 64   /* B is given as [K, N] row-major                                                 */

int tl_abi_version(void);
const char* tl_last_error(void);
/* sm_count / compute capability of the current device; TL_ERR_NO_DEVICE if none */
int tl_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- K1  Qwen2RMSNorm.forward (site-packages/transformers/models/qwen2/modeling_qwen2.py:258-263)
 * y[r,:] = w * bf16(x[r,:] * rsqrt(mean(x[r,:]^2) + eps)); rstd_out (fp32[rows]) optional, for backward */
int tl_rmsnorm_fwd(const void* x, const void* w, void* y, float* rstd_out, int rows, int H, float eps, void* stream);

/* ---- K7  embed_tokens gather (modeling_qwen2.py:367): out[n,:] = table[ids[n],:] */
int tl_embed_fwd(const int64_t* ids, const void* table, void* out, int n_tokens, int H, int vocab, void* stream);

/* ---- K2/K5/K6/K7  nn.Linear as one tcgen05 GEMM: C[M,N] = A[M,K] * B[N,K]^T (+ epilogue flags above).
 * lda/ldb/ldc in elements.  Replaces q/k/v_proj (modeling_qwen2.py:217-219, fused into one B), o_proj (:244),
 * gate/up/down_proj (:46-48), lm_head (:474-476) and, with the MN-major flags, their dgrad/wgrad. */
int tl_gemm_bf16(const void* A, const void* B, void* C, int M, int N, int K, int lda, int ldb, int ldc,
                 const void* bias, const void* residual, int flags, void* stream);

/* same contract with a caller-provided workspace (>= tl_gemm_splitk_ws(M, N) bytes): batched-decode shapes (M <= 128) whose
 * few output tiles cannot occupy every SM are split along K (fp32 partials + one reduce/epilogue pass) */
size_t tl_gemm_splitk_ws(int M, int N);
int tl_gemm_bf16_ws(const void* A, const void* B, void* C, int M, int N, int K, int lda, int ldb, int ldc,
                    const void* bias, const void* residual, int flags, void* workspace, size_t ws_bytes, void* stream);
/* ... and the RMSNorm that follows this Linear in the decoder layer (modeling_qwen2.py:296 / :280 of the next layer):
 * with norm_w != NULL also writes H_out[M,N] = norm_w * bf16(C * rstd(C)), C being the bf16 result above (ldc == N,
 * bias / residual epilogue only).  Fused into the split-K reduce pass when that path runs, otherwise one extra
 * tl_rmsnorm_fwd launch (C identical either way; H may differ in a last bf16 bit: the row's sum of squares is reduced
 * in another order). */
int tl_gemm_bf16_ws_norm(const void* A, const void* B, void* C, int M, int N, int K, int lda, int ldb, int ldc,
                         const void* bias, const void* residual, int flags, void* workspace, size_t ws_bytes,
                         const void* norm_w, float eps, void* H_out, void* stream);

/* ---- decode-shaped Linear (M <= 8 tokens), HBM-bound weight streaming:
 * y[M,N] = f(norm(x)[M,K] * W[N,K]^T).  norm_w != NULL fuses the preceding RMSNorm (K1) as a prologue. */
int tl_gemv_bf16(const void* x, const void* W, void* y, int M, int N, int K, const void* bias,
                 const void* residual, const void* norm_w, float eps, int flags, void* stream);
/* same, plus a hint: once its own weight loads are issued the kernel queues L2 prefetches of the first next_bytes of
 * next_W (the weights the NEXT launch on this stream will read; 16-byte aligned, may be NULL), so HBM keeps streaming
 * across the launch boundary and the next kernel starts from L2.  Purely a performance hint: results are identical. */
int tl_gemv_bf16_pf(const void* x, const void* W, void* y, int M, int N, int K, const void* bias,
                    const void* residual, const void* norm_w, float eps, int flags, const void* next_W,
                    size_t next_bytes, void* stream);

/* ---- K3  rotary tables (modeling_qwen2.py:102-113): cos/sin[pos, d/2] = bf16(cos/sin(pos * inv_freq)) */
int tl_rope_table(const float* inv_freq, void* cos_tab, void* sin_tab, int max_pos, int half_dim, void* stream);

/* ---- K3 + KV-cache append (+ Qwen3 q/k RMSNorm, modeling_qwen3.py:248-264):
 * qkv[n, (n_h+2n_kv)*d] (post-bias) -> q_out[n, n_h*d] rotated; K/V written to
 * cache[b, kv_head, pos, d] with b = n / S, pos = pos0[b or 0] + n % S (pos0 read from device memory so a
 * captured CUDA graph can be replayed while the position advances). q_norm_w/k_norm_w may be NULL. */
int tl_rope_kv_fwd(const void* qkv, void* q_out, void* k_cache, void* v_cache, const int32_t* pos0_dev,
                   const void* cos_tab, const void* sin_tab, const void* q_norm_w, const void* k_norm_w,
                   float eps, int n_tokens, int S, int n_h, int n_kv, int d, int T_max, void* stream);

/* ---- K4  causal GQA attention, prefill / training forward (modeling_qwen2.py:161-184 SDPA contract).
 * q[B,S,n_h,d]; caches [B,n_kv,T_max,d] hold keys 0..past_len+S-1; out[B,S,n_h*d];
 * lse (fp32 [B,n_h,S], natural log) optional, kept for backward. */
int tl_attn_prefill_fwd(const void* q, const void* k_cache, const void* v_cache, void* out, float* lse, int B,
                        int S, int past_len, int n_h, int n_kv, int d, int T_max, float scale, void* stream);

/* ---- K4  decode attention, one query token per batch row, split over the KV length.
 * kv_len_dev: device int32, number of valid keys (same for all rows).  workspace >= tl_attn_decode_ws(...) */
size_t tl_attn_decode_ws(int B, int n_h, int d, int T_max);
int tl_attn_decode_fwd(const void* q, const void* k_cache, const void* v_cache, void* out,
                       const int32_t* kv_len_dev, void* workspace, size_t ws_bytes, int B, int n_h, int n_kv,
                       int d, int T_max, float scale, void* stream);

/* ---- K3 + K4 fused for decode, T_max <= 2048: RoPE (+q/k-norm) of the new token, KV-cache append at *pos_dev and
 * single-pass attention over keys 0..*pos_dev, one launch per layer.  qkv[B, (n_h+2n_kv)*d] post-bias; out[B, n_h*d] */
int tl_attn_decode_fused(const void* qkv, void* k_cache, void* v_cache, void* out, const int32_t* pos_dev,
                         const void* cos_tab, const void* sin_tab, const void* q_norm_w, const void* k_norm_w,
                         float eps, int B, int n_h, int n_kv, int d, int T_max, float scale, void* stream);

/* ---- K7  final norm + lm_head + greedy argmax for M <= 8 rows: ids[m] = argmax_v bf16(norm(x)[m,:]·W[v,:])
 * (lowest index wins ties, as torch.argmax).  logits_out (bf16 [M,V]) optional.
 * workspace >= tl_lmhead_ws(M, V) bytes. */
size_t tl_lmhead_ws(int M, int V);
int tl_lmhead_argmax(const void* x, const void* W, const void* norm_w, float eps, int64_t* ids_out,
                     void* logits_out, void* workspace, size_t ws_bytes, int M, int V, int H, void* stream);

/* argmax over bf16 logits[M,V] (any M); workspace >= M*64*8 bytes */
int tl_argmax_bf16(const void* logits, int64_t* ids_out, void* workspace, size_t ws_bytes, int M, int V, void* stream);

/* ---- token sampling on the device (csrc/sample.cu): what HF `generate(do_sample=True)` does on the host's copy of the
 * logits (the reference delegates to it, tensorlink/ml/module.py:763-769, ml/worker.py:403-404): temperature -> top-k
 * (every logit >= the k-th largest is kept; 0 = off) -> top-p (a token is kept while the probability mass above it is
 * < top_p; ties at the threshold are kept) -> one multinomial draw per row from Philox4x32-10(seed; row, counter).
 * counters_dev: int32[M] in device memory, advanced by the kernel (a captured graph draws a fresh number per replay).
 * workspace >= tl_sample_ws(M) bytes.  logits bf16 [M,V] row-major; ids_out int64[M]. */
size_t tl_sample_ws(int M);
int tl_sample(const void* logits, int64_t* ids_out, int M, int V, float temperature, int top_k, float top_p,
              unsigned long long seed, int32_t* counters_dev, void* workspace, size_t ws_bytes, void* stream);

/* ---- small device-side helpers used by the captured decode graph */
int tl_advance_pos(int32_t* pos_dev, int32_t* kv_len_dev, int delta, void* stream); /* pos += delta; kv_len = pos */
/* out_tokens[b, *step_dev] = ids[b] for b < B (row pitch ld), then ++*step_dev: the generated-token log
 * (replaces the per-token TOKEN packet, tensorlink/p2p/torch_node.py:543-551) */
int tl_append_token(const int64_t* ids, int64_t* out_tokens, int32_t* step_dev, int B, int ld, void* stream);

/* ---- a chain of dependent decode-step jobs as ONE persistent kernel (csrc/decode_chain.cu) ----------------
 * The job list replaces the per-layer launch sequence of `DistributedWorker._handle_forward` ->
 * `module(**kwargs)` (tensorlink/ml/worker.py:297-357) for single-token rows (M <= 4): one CTA per SM walks the
 * list; the producer warp streams the weights of EVERY GEMV job through one shared-memory ring without ever waiting
 * for a dependency, a dependency between jobs is one release/acquire counter, the attention job is split-KV over
 * all CTAs (one group per row and kv head).  Typical chain = one decoder layer:
 *   ATTN(j) -> GEMV o(j) -> GEMV gate/up(j) -> GEMV down(j) -> GEMV qkv(j+1). */
#define TL_JOB_GEMV 0     /* y[M,N or N/2] = f(norm(x)[M,K] W[N,K]^T): same semantics and flags as tl_gemv_bf16 */
#define TL_JOB_ATTN 1     /* RoPE (+ q/k norm) + KV append + attention for one new token per row: x = qkv[M,(n_h+2n_kv)d]
                           * (post-bias), y = out[M,n_h*d]; reads the position from *pos_dev (cached keys 0..pos-1) */
#define TL_ATTN_POS_PER_ROW 1   /* flags of an ATTN job: pos_dev is int32[M], one position per row (ragged batches) */
#define TL_DECODE_CHAIN_MAX_JOBS 16
#define TL_DECODE_CHAIN_SYNC_BYTES 1024   /* per launch site, zero-initialised once; the kernel leaves it zeroed */
typedef struct tl_decode_job {
    int32_t type, N, K, flags;
    int32_t n_h, n_kv, d, T_max;
    float eps, scale;
    const void* W;
    const void* x;
    void* y;
    const void* bias;
    const void* residual;
    const void* norm_w;
    const void* pos_dev;
    const void* cos_tab;
    const void* sin_tab;
    const void* q_norm_w;
    const void* k_norm_w;
    void* k_cache;
    void* v_cache;
} tl_decode_job;
/* bytes of the attention-partials workspace shared by every chain launch of a stage */
size_t tl_decode_chain_ws(int M, int n_h, int n_kv, int d);
/* jobs: HOST array (copied into kernel parameter space).  sync_slot: TL_DECODE_CHAIN_SYNC_BYTES of device memory
 * private to this launch site (consecutive launches under programmatic dependent launch must not share one); word 2
 * is an error flag the kernel raises instead of hanging when a dependency wait exceeds 2 s.  pf_ptr/pf_bytes:
 * optional L2 prefetch hint = the weights the NEXT launch streams first. */
int tl_decode_chain(const tl_decode_job* jobs, int n_jobs, int M, void* sync_slot, void* attn_ws, size_t attn_ws_bytes,
                    const void* pf_ptr, size_t pf_bytes, void* stream);
/* debugging aid: device buffer of n_slots * 2*(TL_DECODE_CHAIN_MAX_JOBS+1)*4 uint64; every later chain launch takes the
 * next slot and stamps it with globaltimer values (CTA 0 and the last CTA; per job: start / input staged / work done /
 * dependency passed; last row: kernel entry / previous grid done / exit); NULL = off */
int tl_decode_chain_trace(void* buf, int n_slots);

/* ---- peer-memory mailboxes: the inter-shard hop of a decode step (csrc/peer.cu) ---------------------------
 * Replace the per-hop send of `DistributedModel.forward` (tensorlink/ml/module.py:438-462: tensor -> bytes ->
 * shared memory -> node process -> socket) and the worker's pickup (tensorlink/ml/worker.py:297-305) on one
 * NVSwitch node: the receiver's input buffer is mapped into the sender (CUDA IPC), the sender's last kernel stores
 * its rows there over NVLink, and a sequence number published with release/acquire at system scope hands it over.
 * All counters are device-resident and advance inside the kernels, so a captured CUDA graph replays unchanged. */
/* cudaMalloc + zero `bytes` and export the allocation: handle64 = the 64-byte cudaIpcMemHandle_t */
int tl_peer_alloc(size_t bytes, void** ptr, unsigned char* handle64);
/* map another process's allocation (peer access enabled lazily); *ptr is valid on this process's device */
int tl_peer_open(const unsigned char* handle64, void** ptr);
int tl_peer_close(void* ptr);   /* unmap a tl_peer_open mapping */
int tl_peer_free(void* ptr);    /* free a tl_peer_alloc allocation */
/* ++*want_dev, then wait until *flag_local >= *want_dev (mod 2^32).  After timeout_ns (0 = 10 s) sets *err_dev = 1
 * and returns instead of hanging; once *err_dev is set every later wait returns at once.  wait_ns_dev (optional) accumulates the nanoseconds spent waiting. */
int tl_peer_wait(const uint32_t* flag_local, uint32_t* want_dev, uint32_t* err_dev, uint64_t* wait_ns_dev,
                 uint64_t timeout_ns, int32_t* bump_dev, void* stream);   /* bump_dev (optional): ++*bump_dev as well */
/* ++*sent_dev, then publish it in the peer's flag after every earlier write of this stream (release, system scope) */
int tl_peer_signal(uint32_t* flag_peer, uint32_t* sent_dev, int32_t* bump_dev, void* stream);   /* bump_dev as above */
/* copy `bytes` (multiple of 16, both 16-byte aligned) into the peer buffer, then signal as above */
int tl_peer_put(void* dst_peer, const void* src, size_t bytes, uint32_t* flag_peer, uint32_t* sent_dev, void* stream);

/* ---- training-only pieces (K8/K9/K10): replace the autograd graph of `assoc_output.backward(loss)`
 * (tensorlink/ml/worker.py:271) and `optimizer.step()` (tensorlink/ml/worker.py:1317) ------------------------- */
/* SwiGLU on interleaved gate/up pre-activations gu[M,2I] (col 2j = gate_j, 2j+1 = up_j): h[M,I], HF rounding */
int tl_swiglu_fwd(const void* gu, void* h, int M, int I, void* stream);
/* dgu[M,2I] from dh[M,I] */
int tl_swiglu_bwd(const void* gu, const void* dh, void* dgu, int M, int I, void* stream);
/* RMSNorm backward: dx = rstd*(dy*w - n*mean(dy*w*n)) (+ dx_add if non-NULL); dw_accum (fp32 [H]) += sum dy*n */
int tl_rmsnorm_bwd(const void* x, const void* w, const void* dy, const float* rstd, const void* dx_add, void* dx,
                   float* dw_accum, int rows, int H, void* stream);
/* RoPE backward + KV gather: dqkv[n, (n_h+2n_kv)*d] from dq[n, n_h*d] and dk/dv[B, n_h, T_max, d] (one partial per
 * query head as written by tl_attn_bwd; the n_h/n_kv partials of a kv head are summed in fp32) */
int tl_rope_kv_bwd(const void* dq, const void* dk, const void* dv, void* dqkv, const void* cos_tab,
                   const void* sin_tab, int n_tokens, int S, int n_h, int n_kv, int d, int T_max, void* stream);
/* Qwen3 q/k-norm backward, in place on the q and k slices of dqkv[n, (n_h+2n_kv)*d] (gradient w.r.t. the
 * normalised vectors on entry, w.r.t. the pre-norm vectors on exit); gain gradients accumulate in fp32 [d] */
int tl_qk_norm_bwd(const void* qkv_pre, void* dqkv, const void* q_norm_w, const void* k_norm_w, float* dqn_accum,
                   float* dkn_accum, float eps, int n_tokens, int n_h, int n_kv, int d, void* stream);
/* attention backward (recompute P from lse): dq[B,S,n_h,d]; dk/dv[B,n_h,T_max,d] rows < S, one partial per query head */
size_t tl_attn_bwd_ws(int B, int S, int n_h);
int tl_attn_bwd(const void* q, const void* k_cache, const void* v_cache, const void* out, const void* dout,
                const float* lse, void* dq, void* dk, void* dv, void* workspace, size_t ws_bytes, int B, int S,
                int n_h, int n_kv, int d, int T_max, float scale, void* stream);
/* cross-entropy on bf16 logits[M,V] (fp32 math): *loss_sum += sum_rows (lse - logit[label]); *n_valid += rows
 * with a valid label; dlogits = (softmax - onehot) * grad_scale (may alias logits); label outside [0,V) ignored */
int tl_ce_fwd_bwd(const void* logits, const int64_t* labels, float* loss_sum, int32_t* n_valid, void* dlogits,
                  float grad_scale, int M, int V, void* stream);
/* embedding backward: dtable[id,:] += sum of dout[n,:] over the tokens n with ids[n] == id, summed in fp32 in token
 * order and rounded once into the bf16 row (deterministic, no atomics).  Takes the ids stably sorted (sorted_ids) and
 * the token index of each (order); ids outside [0, vocab) are skipped.  H %% 8 == 0, dout / dtable 16-byte aligned */
int tl_embed_bwd(const int64_t* sorted_ids, const int64_t* order, const void* dout, void* dtable, int n_tokens, int H,
                 int vocab, void* stream);
/* bias gradient: db_accum[N] (fp32) += sum_m dy[m,:N] (row pitch ld) */
int tl_colsum(const void* dy, float* db_accum, int M, int N, int ld, void* stream);
/* dst[n] (+)= src[n]: fp32 accumulator into a bf16 gradient */
int tl_f32_to_bf16_accum(const float* src, void* dst, size_t n, int accumulate, void* stream);
/* a[n] += b[n] over bf16 (n %% 8 == 0) */
int tl_add_inplace(void* a, const void* b, size_t n, void* stream);
/* a[n] = (accumulate ? a[n] : 0) + scale * b[n]: commits a pending gradient with the upstream gradient's scale
 * (the reference gets this from autograd: ml/worker.py:271 `assoc_output.backward(loss)`); bf16 (n %% 8 == 0) / fp32 */
int tl_scale_add_bf16(void* a, const void* b, float scale, int accumulate, size_t n, void* stream);
int tl_scale_add_f32(float* a, const float* b, float scale, int accumulate, size_t n, void* stream);
/* fused Adam / AdamW (torch.optim update rule, fp32 math and moments) over a flat bf16 parameter arena
 * (all four arrays 16-byte aligned; n arbitrary) */
int tl_adamw_step(void* param, const void* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                  float beta1, float beta2, float eps, float weight_decay, int step, int decoupled,
                  void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TENSORLINK_B200_H */
