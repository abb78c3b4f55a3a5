// extern "C" surface of libb200_train (declared in include/b200_train.h).
#include <cuda_runtime.h>
#include <cublasLt.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <mutex>

#include "../../include/b200_train.h"
#include "common.h"

namespace b200 {

static thread_local char g_err[512] = "";

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

// implemented in elementwise.cu / attention.cu
int rmsnorm_fwd(const void*, const void*, void*, float*, int, int, float, cudaStream_t);
int rmsnorm_bwd_workspace_floats(int, int);
int rmsnorm_bwd(const void*, const void*, const void*, const float*, const void*, void*, void*, int, float*, int, int, cudaStream_t);
int rope_inplace(void*, const void*, const void*, const int*, int, int, int, int, int, cudaStream_t);
int bias_rope_inplace(void*, const void*, const void*, const void*, const int*, int, int, int, int, int, cudaStream_t);
int colsum_workspace_floats(int, int);
int colsum_bf16(const void*, void*, float*, int, int, int64_t, int, cudaStream_t);
int swiglu_fwd(const void*, void*, int64_t, int, cudaStream_t);
int swiglu_bwd(const void*, const void*, void*, int64_t, int, cudaStream_t);
int embed_fwd(const int*, const void*, void*, int, int, cudaStream_t);
int embed_bwd(const int*, const void*, void*, int*, int, int, int, cudaStream_t);
int ce_fwd_bwd(void*, const int*, float*, float*, int, int, int64_t, int64_t, int, cudaStream_t);
int sumsq_workspace_floats();
int sumsq_bf16(const void*, int64_t, float*, float*, int, cudaStream_t);
int adamw_step(void*, const void*, void*, void*, float*, int64_t, float, float, float, float, float, int, float, const float*, int,
               cudaStream_t);
int add_inplace_bf16(void*, const void*, int64_t, cudaStream_t);
int attn_fwd(const void*, const void*, const void*, void*, float*, const int*, int, int, int64_t, int64_t, int64_t, int64_t, int, int,
             int, int, float, cudaStream_t);
size_t attn_bwd_workspace_bytes(int, int, int, int);
int attn_bwd(const void*, const void*, const void*, const void*, const void*, const float*, void*, void*, void*, void*, size_t, const int*, int,
             int, int64_t, int64_t, int64_t, int64_t, int64_t, int64_t, int64_t, int64_t, int, int, int, int, float, cudaStream_t);

int attn_fwd_tc(const void*, const void*, const void*, void*, float*, const int*, int, int, int64_t, int64_t, int64_t, int64_t, int, int,
                int, int, float, cudaStream_t);
int attn_bwd_tc(const void*, const void*, const void*, const void*, const void*, const float*, void*, void*, void*, void*, size_t, const int*, int,
                int, int64_t, int64_t, int64_t, int64_t, int64_t, int64_t, int64_t, int64_t, int, int, int, int, float, cudaStream_t);

struct CommCtx;
int ctx_create(CommCtx**, int, int);
int ctx_destroy(CommCtx*);
int ctx_set_timeout_ms(CommCtx*, int64_t);
int ctx_set_signal_pad(CommCtx*, void* const*, size_t);
int ctx_register_buffer(CommCtx*, int, void* const*, void*, size_t);
int ctx_has_multicast(const CommCtx*, int);
int reducescatter_layer(CommCtx*, int, size_t, int64_t, int, int, cudaStream_t);
int allgather_layer(CommCtx*, int, size_t, int64_t, int, int, cudaStream_t);
int allreduce_scalars(CommCtx*, float*, int, cudaStream_t);
size_t ctx_signal_pad_bytes();

int attn_fwd_tc64(const void*, const void*, const void*, void*, float*, const int*, int, int, int64_t, int64_t, int64_t, int64_t, int, int,
                  int, int, float, cudaStream_t);
int attn_fwd_ts(const void*, const void*, const void*, void*, float*, const int*, int, int, int64_t, int64_t, int64_t, int64_t, int, int,
                int, int, float, int, cudaStream_t);
static int g_attn_fwd_variant = 2;  // 2 (default): P kept in tensor memory, packed-fp32 softmax (attention_fwd_ts.cu: 869 TFLOP/s, 0 of 6000 launches differ); 1: attention_fwd64.cu (627 TFLOP/s); 0: attention_tc.cu forward (510)

// debug option: 1 (default) = tcgen05/TMEM attention, 0 = the mma.sync v1 kernels (kept for bisecting only)
static int g_attn_impl = 1;
extern int forced_bn;
extern int use_pair;
extern int side_blocks_per_sm;
namespace pair { extern int sched_mode; }

// ---------------------------------------------------------------- cuBLASLt comparator (bench / tests only)
int gemm_bf16_cublaslt(int kind, const void* A, int lda, const void* B, int ldb, void* C, int ldc, int M, int N, int K, void* ws,
                       size_t ws_bytes, cudaStream_t stream) {
  static cublasLtHandle_t handle = nullptr;
  static std::mutex mu;
  {
    std::lock_guard<std::mutex> lk(mu);
    if (!handle && cublasLtCreate(&handle) != CUBLAS_STATUS_SUCCESS) return set_error(B200_ERR_CUDA, "cublasLtCreate failed");
  }
  // Row-major C[M,N] == column-major C^T[N,M] with ld = ldc.  C^T = op(Bc) * op(Ac) in column-major terms.
  // NT: C^T[N,M] = W(col-major view of B[N,K] row-major is B^T [K,N], ld=ldb) -> opT ; A row-major [M,K] is col-major [K,M] -> opN
  cublasLtMatmulDesc_t desc = nullptr;
  cublasLtMatrixLayout_t la = nullptr, lb = nullptr, lc = nullptr;
  cublasLtMatmulPreference_t pref = nullptr;
  cublasOperation_t opa, opb;  // for the column-major product  C^T = op(X) * op(Y),  X from B, Y from A
  int xr, xc, yr, yc;          // stored column-major shapes of X (from B) and Y (from A)
  if (kind == GEMM_NT) {        // B row-major [N,K] -> col-major [K,N]; need [N,K] -> T.   A row-major [M,K] -> col-major [K,M]; need [K,M] -> N
    opa = CUBLAS_OP_T; xr = K; xc = N; opb = CUBLAS_OP_N; yr = K; yc = M;
  } else if (kind == GEMM_NN) {  // B row-major [K,N] -> col-major [N,K]; need [N,K] -> N.   A as above -> N
    opa = CUBLAS_OP_N; xr = N; xc = K; opb = CUBLAS_OP_N; yr = K; yc = M;
  } else if (kind == GEMM_TN) {  // B row-major [K,N] -> col-major [N,K] -> N.  A row-major [K,M] -> col-major [M,K]; need [K,M] -> T
    opa = CUBLAS_OP_N; xr = N; xc = K; opb = CUBLAS_OP_T; yr = M; yc = K;
  } else {
    return set_error(B200_ERR_ARG, "unknown gemm kind %d", kind);
  }
  int rc = 0;
  cublasStatus_t s;
  const float alpha = 1.f, beta = 0.f;
  cublasLtMatmulHeuristicResult_t heur;
  int found = 0;
  s = cublasLtMatmulDescCreate(&desc, CUBLAS_COMPUTE_32F, CUDA_R_32F);
  if (s != CUBLAS_STATUS_SUCCESS) { rc = set_error(B200_ERR_CUDA, "cublasLtMatmulDescCreate %d", (int)s); goto done; }
  cublasLtMatmulDescSetAttribute(desc, CUBLASLT_MATMUL_DESC_TRANSA, &opa, sizeof(opa));
  cublasLtMatmulDescSetAttribute(desc, CUBLASLT_MATMUL_DESC_TRANSB, &opb, sizeof(opb));
  cublasLtMatrixLayoutCreate(&la, CUDA_R_16BF, xr, xc, ldb);
  cublasLtMatrixLayoutCreate(&lb, CUDA_R_16BF, yr, yc, lda);
  cublasLtMatrixLayoutCreate(&lc, CUDA_R_16BF, N, M, ldc);
  cublasLtMatmulPreferenceCreate(&pref);
  cublasLtMatmulPreferenceSetAttribute(pref, CUBLASLT_MATMUL_PREF_MAX_WORKSPACE_BYTES, &ws_bytes, sizeof(ws_bytes));
  s = cublasLtMatmulAlgoGetHeuristic(handle, desc, la, lb, lc, lc, pref, 1, &heur, &found);
  if (s != CUBLAS_STATUS_SUCCESS || found == 0) { rc = set_error(B200_ERR_CUDA, "cublasLt heuristic failed (%d)", (int)s); goto done; }
  s = cublasLtMatmul(handle, desc, &alpha, B, la, A, lb, &beta, C, lc, C, lc, &heur.algo, ws, ws_bytes, stream);
  if (s != CUBLAS_STATUS_SUCCESS) rc = set_error(B200_ERR_CUDA, "cublasLtMatmul failed (%d)", (int)s);
done:
  if (pref) cublasLtMatmulPreferenceDestroy(pref);
  if (la) cublasLtMatrixLayoutDestroy(la);
  if (lb) cublasLtMatrixLayoutDestroy(lb);
  if (lc) cublasLtMatrixLayoutDestroy(lc);
  if (desc) cublasLtMatmulDescDestroy(desc);
  return rc;
}

}  // namespace b200

using namespace b200;
static inline cudaStream_t S(b200_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

extern "C" {

const char* b200_last_error(void) { return g_err; }
int b200_abi_version(void) { return 2; }
int b200_set_option(const char* name, int value) {
  if (name && !strcmp(name, "attn_impl")) { g_attn_impl = value; return 0; }
  if (name && !strcmp(name, "attn_fwd_variant")) { g_attn_fwd_variant = value; return 0; }
  if (name && !strcmp(name, "gemm_bn")) { b200::forced_bn = value; return 0; }
  if (name && !strcmp(name, "gemm_2cta")) { b200::use_pair = value; return 0; }
  if (name && !strcmp(name, "gemm_sched")) { b200::pair::sched_mode = value; return 0; }
  if (name && !strcmp(name, "side_blocks_per_sm")) { b200::side_blocks_per_sm = value; return 0; }
  return set_error(B200_ERR_ARG, "unknown option %s", name ? name : "(null)");
}

int b200_device_check(void) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return set_error(B200_ERR_CUDA, "cudaGetDevice: %s", cudaGetErrorString(e));
  int major = 0, minor = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
  if (major != 10) return set_error(B200_ERR_UNSUPPORTED, "device is sm_%d%d; libb200_train is built for sm_100a only", major, minor);
  return 0;
}

int b200_gemm_bf16(int kind, const void* A, int lda, const void* B, int ldb, void* C, int ldc, const void* R, int ldr, int M, int N, int K,
                   int flags, int group_m, int max_ctas, b200_stream_t stream) {
  return gemm_bf16_tcgen05(kind, A, lda, B, ldb, C, ldc, R, ldr, M, N, K, flags, group_m, max_ctas, S(stream));
}
int b200_gemm_bf16_cublaslt(int kind, const void* A, int lda, const void* B, int ldb, void* C, int ldc, int M, int N, int K,
                            void* workspace, size_t workspace_bytes, b200_stream_t stream) {
  return gemm_bf16_cublaslt(kind, A, lda, B, ldb, C, ldc, M, N, K, workspace, workspace_bytes, S(stream));
}
int b200_rmsnorm_fwd(const void* x, const void* w, void* y, float* rstd, int rows, int cols, float eps, b200_stream_t stream) {
  return rmsnorm_fwd(x, w, y, rstd, rows, cols, eps, S(stream));
}
int b200_rmsnorm_bwd_workspace_floats(int rows, int cols) { return rmsnorm_bwd_workspace_floats(rows, cols); }
int b200_rmsnorm_bwd(const void* dy, const void* x, const void* w, const float* rstd, const void* dres, void* dx, void* dw,
                     int accumulate_dw, float* workspace, int rows, int cols, b200_stream_t stream) {
  return rmsnorm_bwd(dy, x, w, rstd, dres, dx, dw, accumulate_dw, workspace, rows, cols, S(stream));
}
int b200_rope_inplace(void* qk, const void* cos_table, const void* sin_table, const int* position_ids, int tokens, int heads,
                      int head_dim, int ld, int backward, b200_stream_t stream) {
  return rope_inplace(qk, cos_table, sin_table, position_ids, tokens, heads, head_dim, ld, backward, S(stream));
}
int b200_bias_rope_inplace(void* qkv, const void* bias, const void* cos_table, const void* sin_table, const int* position_ids, int tokens,
                           int rope_heads, int heads, int head_dim, int ld, b200_stream_t stream) {
  return bias_rope_inplace(qkv, bias, cos_table, sin_table, position_ids, tokens, rope_heads, heads, head_dim, ld, S(stream));
}
int b200_colsum_workspace_floats(int rows, int cols) { return colsum_workspace_floats(rows, cols); }
int b200_colsum_bf16(const void* x, void* out, float* workspace, int rows, int cols, int64_t ld, int accumulate, b200_stream_t stream) {
  return colsum_bf16(x, out, workspace, rows, cols, ld, accumulate, S(stream));
}
int b200_swiglu_fwd(const void* gu, void* a, int64_t tokens, int ffn, b200_stream_t stream) { return swiglu_fwd(gu, a, tokens, ffn, S(stream)); }
int b200_swiglu_bwd(const void* da, const void* gu, void* dgu, int64_t tokens, int ffn, b200_stream_t stream) {
  return swiglu_bwd(da, gu, dgu, tokens, ffn, S(stream));
}
int b200_embed_fwd(const int* ids, const void* W, void* out, int tokens, int hidden, b200_stream_t stream) {
  return embed_fwd(ids, W, out, tokens, hidden, S(stream));
}
int b200_embed_bwd(const int* ids, const void* dh, void* dW, int* workspace, int tokens, int hidden, int accumulate, b200_stream_t stream) {
  return embed_bwd(ids, dh, dW, workspace, tokens, hidden, accumulate, S(stream));
}
int b200_attn_fwd(const void* q, const void* k, const void* v, void* o, float* lse, const int* cu_seqlens, int nseq, int max_seqlen,
                  int64_t ldq, int64_t ldk, int64_t ldv, int64_t ldo, int Hq, int Hkv, int head_dim, int total_tokens, float scale,
                  b200_stream_t stream) {
  if (g_attn_impl == 1 && g_attn_fwd_variant >= 2)
    return attn_fwd_ts(q, k, v, o, lse, cu_seqlens, nseq, max_seqlen, ldq, ldk, ldv, ldo, Hq, Hkv, head_dim, total_tokens, scale, 1, S(stream));
  if (g_attn_impl == 1 && g_attn_fwd_variant == 1)
    return attn_fwd_tc64(q, k, v, o, lse, cu_seqlens, nseq, max_seqlen, ldq, ldk, ldv, ldo, Hq, Hkv, head_dim, total_tokens, scale, S(stream));
  if (g_attn_impl == 1)
    return attn_fwd_tc(q, k, v, o, lse, cu_seqlens, nseq, max_seqlen, ldq, ldk, ldv, ldo, Hq, Hkv, head_dim, total_tokens, scale, S(stream));
  return attn_fwd(q, k, v, o, lse, cu_seqlens, nseq, max_seqlen, ldq, ldk, ldv, ldo, Hq, Hkv, head_dim, total_tokens, scale, S(stream));
}
size_t b200_attn_bwd_workspace_bytes(int total_tokens, int Hq, int head_dim, int max_seqlen) {
  return attn_bwd_workspace_bytes(total_tokens, Hq, head_dim, max_seqlen);
}
int b200_attn_bwd(const void* q, const void* k, const void* v, const void* o, const void* dout, const float* lse, void* dq, void* dk,
                  void* dv, void* workspace, size_t workspace_bytes, const int* cu_seqlens, int nseq, int max_seqlen, int64_t ldq,
                  int64_t ldk, int64_t ldv, int64_t ldo, int64_t lddo, int64_t lddq, int64_t lddk, int64_t lddv, int Hq, int Hkv,
                  int head_dim, int total_tokens, float scale, b200_stream_t stream) {
  if (g_attn_impl == 1)
    return attn_bwd_tc(q, k, v, o, dout, lse, dq, dk, dv, workspace, workspace_bytes, cu_seqlens, nseq, max_seqlen, ldq, ldk, ldv, ldo, lddo, lddq, lddk,
                       lddv, Hq, Hkv, head_dim, total_tokens, scale, S(stream));
  return attn_bwd(q, k, v, o, dout, lse, dq, dk, dv, workspace, workspace_bytes, cu_seqlens, nseq, max_seqlen, ldq, ldk, ldv, ldo, lddo, lddq, lddk, lddv,
                  Hq, Hkv, head_dim, total_tokens, scale, S(stream));
}
int b200_ce_fwd_bwd(void* logits, const int* labels, float* row_loss, float* loss_out, int rows, int vocab, int64_t ld,
                    int64_t num_label_tokens, int accumulate_loss, b200_stream_t stream) {
  return ce_fwd_bwd(logits, labels, row_loss, loss_out, rows, vocab, ld, num_label_tokens, accumulate_loss, S(stream));
}
int b200_sumsq_workspace_floats(void) { return sumsq_workspace_floats(); }
int b200_sumsq_bf16(const void* g, int64_t n, float* out, float* workspace, int accumulate, b200_stream_t stream) {
  return sumsq_bf16(g, n, out, workspace, accumulate, S(stream));
}
int b200_adamw_step(void* p, const void* g, void* m, void* v, float* master, int64_t n, float lr, float beta1, float beta2, float eps,
                    float weight_decay, int step, float max_grad_norm, const float* grad_norm_sq, int mode, b200_stream_t stream) {
  return adamw_step(p, g, m, v, master, n, lr, beta1, beta2, eps, weight_decay, step, max_grad_norm, grad_norm_sq, mode, S(stream));
}
int b200_add_inplace_bf16(void* dst, const void* src, int64_t n, b200_stream_t stream) { return add_inplace_bf16(dst, src, n, S(stream)); }

int b200_ctx_create(b200_ctx** ctx, int rank, int world) { return ctx_create(reinterpret_cast<CommCtx**>(ctx), rank, world); }
int b200_ctx_destroy(b200_ctx* ctx) { return ctx_destroy(reinterpret_cast<CommCtx*>(ctx)); }
int b200_ctx_set_timeout_ms(b200_ctx* ctx, int64_t ms) { return ctx_set_timeout_ms(reinterpret_cast<CommCtx*>(ctx), ms); }
int b200_ctx_set_signal_pad(b200_ctx* ctx, void* const* pads, size_t bytes) {
  return ctx_set_signal_pad(reinterpret_cast<CommCtx*>(ctx), pads, bytes);
}
int b200_ctx_register_buffer(b200_ctx* ctx, int slot, void* const* peer_ptrs, void* multicast_ptr, size_t bytes) {
  return ctx_register_buffer(reinterpret_cast<CommCtx*>(ctx), slot, peer_ptrs, multicast_ptr, bytes);
}
int b200_ctx_has_multicast(const b200_ctx* ctx, int slot) { return ctx_has_multicast(reinterpret_cast<const CommCtx*>(ctx), slot); }
size_t b200_ctx_signal_pad_bytes(void) { return ctx_signal_pad_bytes(); }
int b200_allreduce_scalars(b200_ctx* ctx, float* vals, int n, b200_stream_t stream) {
  return allreduce_scalars(reinterpret_cast<CommCtx*>(ctx), vals, n, S(stream));
}
int b200_reducescatter_layer(b200_ctx* ctx, int slot, size_t byte_offset, int64_t shard_elems, int mode, int ctas, b200_stream_t stream) {
  return reducescatter_layer(reinterpret_cast<CommCtx*>(ctx), slot, byte_offset, shard_elems, mode, ctas, S(stream));
}
int b200_allgather_layer(b200_ctx* ctx, int slot, size_t byte_offset, int64_t shard_elems, int mode, int ctas, b200_stream_t stream) {
  return allgather_layer(reinterpret_cast<CommCtx*>(ctx), slot, byte_offset, shard_elems, mode, ctas, S(stream));
}

}  // extern "C"
