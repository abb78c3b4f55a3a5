/* libb200_train - C ABI of the B200-native sharded-data-parallel Llama training step.
 *
 * Drop-in boundary for the device work that NVIDIA-NeMo/Automodel's recipe
 * (nemo_automodel/recipes/llm/train_ft.py:1357-1473 `_forward_backward_step`, :1482-1635 `_run_train_optim_step`)
 * reaches through torch ATen/cuBLAS/flash-attn/FSDP2.  The reference has no native code on this path; each entry
 * below names the Python call site whose device work it replaces.
 *
 * Conventions: every entry returns 0 on success or a negative B200_ERR_* code (message via b200_last_error());
 * no exceptions, no allocation (callers pass device pointers and workspaces), no implicit synchronisation,
 * every launch goes to the explicit `stream`.  All activations/weights are bf16 (uint16 storage), token-major
 * row-major [rows, cols] with an explicit leading dimension where a view is allowed.  Re-entrant: forward
 * entries are called from the rank's main thread, backward entries may be called from any thread of the process.
 */
#ifndef B200_TRAIN_H_
#define B200_TRAIN_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* b200_stream_t; /* == cudaStream_t */

#define B200_ERR_ARG (-1)
#define B200_ERR_CUDA (-2)
#define B200_ERR_DRIVER (-3)
#define B200_ERR_UNSUPPORTED (-4)
#define B200_ERR_NCCL (-5)

const char* b200_last_error(void);
int b200_abi_version(void);
/* 0 when the current device is sm_100 (B200); B200_ERR_UNSUPPORTED otherwise. */
int b200_device_check(void);
/* options; "attn_impl": 1 = tcgen05/TMEM attention (default), 0 = mma.sync v1 kernels (bisecting only); "attn_fwd_variant", "gemm_bn",
 * "gemm_2cta": kernel selection for A/B runs; "gemm_sched": 0 = static persistent tile striding (default), 1 = cluster launch control
 * (clusterlaunchcontrol.try_cancel: running clusters absorb pending tiles) for the CTA-pair GEMM; "side_blocks_per_sm": k > 0 caps b200_adamw_step / b200_sumsq_bf16 at k 256-thread CTAs per
 * SM so that they co-reside with a GEMM CTA when issued on a side stream (0 = full occupancy). */
int b200_set_option(const char* name, int value);

/* ---- dense contractions: nn.Linear fwd/dgrad/wgrad (components/models/llama/model.py:113-115,151,170,511)
 * kind 0 (NT): C[M,N] = A[M,K] * B[N,K]^T      forward   y = x W^T
 * kind 1 (NN): C[M,N] = A[M,K] * B[K,N]        dgrad     dx = dy W
 * kind 2 (TN): C[M,N] = A[K,M]^T * B[K,N]      wgrad     dW = dy^T x
 * flags bit0: C = acc + R (R bf16 [M,N], may alias C);  bit1: round acc to bf16 before the add (reference numerics:
 * residual add after the o_proj/down_proj output was materialised, model.py:227,233; also grad accumulation).
 * tcgen05 tensor cores, TMA, TMEM accumulators.  group_m: L2 rasterisation group (0 = default).
 * flags bit 2 (4, experimental): SwiGLU epilogue for kind NT with B = [W_gate; W_up] (N = 2F, F % 128 == 0, M >= 256):
 * C = [gate | up] as usual and R (an OUTPUT here, [M, F], pitch ldr) = bf16(bf16(silu(gate)) * up)  (model.py:155-170 act_fn(gate) * up).
 */
#define B200_GEMM_NT 0
#define B200_GEMM_NN 1
#define B200_GEMM_TN 2
#define B200_GEMM_RESIDUAL 1
#define B200_GEMM_ROUND_BEFORE_ADD 2
#define B200_GEMM_SWIGLU 4
int b200_gemm_bf16(int kind, const void* A, int lda, const void* B, int ldb, void* C, int ldc, const void* R, int ldr,
                   int M, int N, int K, int flags, int group_m, int max_ctas, b200_stream_t stream);
/* cuBLASLt on the same operands: the bar to beat (bench/tests only, never on the training path). */
int b200_gemm_bf16_cublaslt(int kind, const void* A, int lda, const void* B, int ldb, void* C, int ldc, int M, int N,
                            int K, void* workspace, size_t workspace_bytes, b200_stream_t stream);

/* ---- Float32RMSNorm (components/models/common/utils.py:250-276) */
int b200_rmsnorm_fwd(const void* x, const void* w, void* y, float* rstd, int rows, int cols, float eps, b200_stream_t stream);
int b200_rmsnorm_bwd_workspace_floats(int rows, int cols);
/* dx = rmsnorm'(dy) (+ dres, the residual-stream gradient);  dw (bf16 [cols]) = or += column sums */
int b200_rmsnorm_bwd(const void* dy, const void* x, const void* w, const float* rstd, const void* dres, void* dx, void* dw,
                     int accumulate_dw, float* workspace, int rows, int cols, b200_stream_t stream);

/* ---- RoPE, rotate-half convention, bf16 cos/sin tables [max_pos, head_dim] (components/models/llama/rope_utils.py:39-67)
 * in place on `heads` consecutive heads of a token-major buffer; backward = adjoint rotation. */
int b200_rope_inplace(void* qk, const void* cos_table, const void* sin_table, const int* position_ids, int tokens, int heads,
                      int head_dim, int ld, int backward, b200_stream_t stream);

/* ---- qkv projection bias (Qwen2: components/models/qwen2/model.py:80-82, nn.Linear(bias=True) for q/k/v)
 * forward: in place on the fused [tokens, heads*head_dim] qkv rows: y = bf16(x + bias) for every head, then RoPE (as b200_rope_inplace)
 * on the first rope_heads heads (q and k).  backward: b200_rope_inplace(backward=1) on dq/dk as without bias, then the bias gradient is
 * the column sum of dqkv: out[c] (=|+=) bf16(sum_t x[t, c]) with fp32 accumulation (deterministic two-stage reduction). */
int b200_bias_rope_inplace(void* qkv, const void* bias, const void* cos_table, const void* sin_table, const int* position_ids, int tokens,
                           int rope_heads, int heads, int head_dim, int ld, b200_stream_t stream);
int b200_colsum_workspace_floats(int rows, int cols);
int b200_colsum_bf16(const void* x, void* out, float* workspace, int rows, int cols, int64_t ld, int accumulate, b200_stream_t stream);

/* ---- SwiGLU (components/models/llama/model.py:170); gu = [gate | up] columns */
int b200_swiglu_fwd(const void* gu, void* a, int64_t tokens, int ffn, b200_stream_t stream);
int b200_swiglu_bwd(const void* da, const void* gu, void* dgu, int64_t tokens, int ffn, b200_stream_t stream);

/* ---- embedding gather / deterministic scatter-add (model.py:320).  workspace: 2*tokens ints */
int b200_embed_fwd(const int* ids, const void* W, void* out, int tokens, int hidden, b200_stream_t stream);
int b200_embed_bwd(const int* ids, const void* dh, void* dW, int* workspace, int tokens, int hidden, int accumulate,
                   b200_stream_t stream);

/* ---- causal GQA flash attention, varlen via cu_seqlens[nseq+1] (model.py:135-148) */
int b200_attn_fwd(const void* q, const void* k, const void* v, void* o, float* lse, const int* cu_seqlens, int nseq,
                  int max_seqlen, int64_t ldq, int64_t ldk, int64_t ldv, int64_t ldo, int Hq, int Hkv, int head_dim,
                  int total_tokens, float scale, b200_stream_t stream);
/* Workspace for batches of `total_tokens` tokens whose sequences are at most `max_seqlen` long.  With max_seqlen <= 512 it includes a
 * second fp32 dQ accumulator, and dQ of sequences of 257..512 tokens is then bit-reproducible; otherwise dQ may differ from launch to
 * launch in its last bits (fp32 additions in the order the CTAs finish).  b200_attn_bwd takes the size it was given. */
size_t b200_attn_bwd_workspace_bytes(int total_tokens, int Hq, int head_dim, int max_seqlen);
int b200_attn_bwd(const void* q, const void* k, const void* v, const void* o, const void* dout, const float* lse, void* dq,
                  void* dk, void* dv, void* workspace, size_t workspace_bytes, const int* cu_seqlens, int nseq, int max_seqlen, int64_t ldq,
                  int64_t ldk, int64_t ldv, int64_t ldo, int64_t lddo, int64_t lddq, int64_t lddk, int64_t lddv, int Hq,
                  int Hkv, int head_dim, int total_tokens, float scale, b200_stream_t stream);

/* ---- MaskedCrossEntropy fwd+bwd fused (components/loss/masked_ce.py:73-89): logits [rows, V] bf16 are overwritten
 * with dlogits = (softmax - onehot)/num_label_tokens; loss_out[0] (=|+=) sum_rows(nll)/num_label_tokens. */
int b200_ce_fwd_bwd(void* logits, const int* labels, float* row_loss, float* loss_out, int rows, int vocab, int64_t ld,
                    int64_t num_label_tokens, int accumulate_loss, b200_stream_t stream);

/* ---- grad-norm (components/training/utils.py:122-141): out[0] (=|+=) sum(g^2) over n bf16 values */
int b200_sumsq_workspace_floats(void);
int b200_sumsq_bf16(const void* g, int64_t n, float* out, float* workspace, int accumulate, b200_stream_t stream);

/* ---- fused AdamW on the local shard incl. on-device clip coefficient (train_ft.py:1556-1558, utils.py:168-169)
 * mode 0: fp32 math (optional fp32 master weights); mode 1: torch.optim.AdamW op-by-op bf16 rounding sequence. */
int b200_adamw_step(void* p, const void* g, void* m, void* v, float* master, int64_t n, float lr, float beta1, float beta2,
                    float eps, float weight_decay, int step, float max_grad_norm, const float* grad_norm_sq, int mode,
                    b200_stream_t stream);

/* dst += src (bf16), gradient accumulation helper */
int b200_add_inplace_bf16(void* dst, const void* src, int64_t n, b200_stream_t stream);

/* ---- per-unit collectives of the sharded step on NVLink 5 / NVSwitch (replace FSDP2's NCCL all_gather_into_tensor / reduce_scatter_tensor,
 * torch/distributed/fsdp/_fully_shard/_fsdp_collectives.py:237-291,448-664, as set up by components/distributed/parallelizer.py:858-872
 * with MixedPrecisionPolicy(param bf16, reduce fp32), components/distributed/config.py:121-132).
 * b200_ctx: one per rank; owns no memory.  The caller registers SYMMETRIC buffers (the same allocation on every rank of one NVSwitch
 * box, e.g. from torch.distributed._symmetric_memory): peer_ptrs[j] = this rank's mapping of rank j's buffer (peer_ptrs[rank] = the
 * local pointer), multicast_ptr = the NVLS multicast mapping of the buffer or NULL, plus one zero-initialised symmetric signal pad of
 * b200_ctx_signal_pad_bytes() bytes.  A unit is world*shard_elems bf16 values at byte_offset of a registered buffer; rank r owns
 * elements [r*shard_elems, (r+1)*shard_elems).
 *   b200_reducescatter_layer: in place; the owner's slice := bf16(sum over ranks, fp32 accumulation, ONE rounding) - NVLS
 *       multimem.ld_reduce(.acc::f32) when the buffer has a multicast mapping (mode 0), 16-byte peer loads summed in rank order otherwise
 *       (or mode 1).  The other slices of the local buffer are left as they were.
 *   b200_allgather_layer: in place; every rank's slice is replicated into every rank's buffer (NVLS multimem.st, or peer pulls).
 * Cross-rank ordering is inside the kernels (CTA-to-CTA release/acquire flags on the signal pad): each rank launches the entry on its
 * own stream behind the work that produces its contribution; all ranks must launch the same entries in the same order with the same
 * `ctas` (1..64).  No host synchronisation, no NCCL.  A rank that never arrives makes the peers' kernels trap after the ctx timeout
 * (default 60 s) instead of hanging. */
typedef struct b200_ctx b200_ctx;
int b200_ctx_create(b200_ctx** ctx, int rank, int world); /* world <= 8 */
int b200_ctx_destroy(b200_ctx* ctx);
int b200_ctx_set_timeout_ms(b200_ctx* ctx, int64_t ms);
size_t b200_ctx_signal_pad_bytes(void);
int b200_ctx_set_signal_pad(b200_ctx* ctx, void* const* pads, size_t bytes);
int b200_ctx_register_buffer(b200_ctx* ctx, int slot, void* const* peer_ptrs, void* multicast_ptr, size_t bytes); /* slot 0..3 */
int b200_ctx_has_multicast(const b200_ctx* ctx, int slot);
int b200_reducescatter_layer(b200_ctx* ctx, int slot, size_t byte_offset, int64_t shard_elems, int mode, int ctas, b200_stream_t stream);
int b200_allgather_layer(b200_ctx* ctx, int slot, size_t byte_offset, int64_t shard_elems, int mode, int ctas, b200_stream_t stream);
/* vals[0..n) (n <= 16 fp32 values in device memory) := their sum over all ranks, added in rank order on every rank (identical bits
 * everywhere): the grad-norm^2 and reported-loss reductions of the step (components/training/utils.py:150-160 all_reduce of the norm,
 * recipes/llm/train_ft.py:1608-1610 _dp_allreduce of the loss) without an NCCL kernel.  Same launch rules as the entries above; issue it
 * on the same stream as them so that every cross-rank wait of the step belongs to one sequence. */
int b200_allreduce_scalars(b200_ctx* ctx, float* vals, int n, b200_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* B200_TRAIN_H_ */
