"""Tensor-level wrappers over the C ABI.  torch supplies device memory and streams only; every op below is one or
more launches of the hand-written sm_100a kernels in csrc/.  Inputs must be CUDA bf16 (unless noted) and contiguous
in the last dimension."""
import os

import torch

from ._lib import lib, check

NT, NN, TN = 0, 1, 2
GEMM_RESIDUAL, GEMM_ROUND_BEFORE_ADD, GEMM_SWIGLU = 1, 2, 4

# number of kernels of THIS library launched so far (bench.py reports the count inside its timed region)
LAUNCHES = 0
# optional hook: callable(kind, M, N, K) -> context manager, used by bench.py to time every GEMM launch with CUDA events
GEMM_TIMER = None


def _count(n):
    global LAUNCHES
    LAUNCHES += n


def _st():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return 0 if t is None else t.data_ptr()


def _chk2d(t, name):
    assert t.is_cuda and t.dtype == torch.bfloat16 and t.dim() == 2 and t.stride(1) == 1, f"{name}: need CUDA bf16 [rows, cols] with unit inner stride"


def set_option(name, value):
    """Debug switches of the library ("attn_impl": 1 = tcgen05 attention (default), 0 = mma.sync v1)."""
    check(lib().b200_set_option(name.encode(), int(value)), "b200_set_option")


def device_check():
    check(lib().b200_device_check(), "b200_device_check")


def _apply_env_options():
    """A/B switches from the environment (B200_GEMM_SCHED=1: cluster-launch-control tile scheduler of the CTA-pair GEMM)."""
    import os
    v = os.environ.get("B200_GEMM_SCHED")
    if v is not None:
        set_option("gemm_sched", int(v))


_apply_env_options()


def gemm(kind, a, b, out=None, residual=None, round_before_add=True, group_m=0, max_ctas=0):
    """kind NT: a[M,K] b[N,K] -> [M,N];  NN: a[M,K] b[K,N];  TN: a[K,M] b[K,N].  Views with a row pitch are fine."""
    _chk2d(a, "a"); _chk2d(b, "b")
    if kind == NT:
        M, K = a.shape; N, K2 = b.shape
    elif kind == NN:
        M, K = a.shape; K2, N = b.shape
    else:
        K, M = a.shape; K2, N = b.shape
    assert K == K2, (a.shape, b.shape, kind)
    if out is None:
        out = torch.empty(M, N, dtype=torch.bfloat16, device=a.device)
    _chk2d(out, "out")
    assert out.shape == (M, N)
    flags = 0
    ldr = 0
    if residual is not None:
        _chk2d(residual, "residual")
        assert residual.shape == (M, N)
        flags |= GEMM_RESIDUAL | (GEMM_ROUND_BEFORE_ADD if round_before_add else 0)
        ldr = residual.stride(0)
    if GEMM_TIMER is not None:
        with GEMM_TIMER(kind, M, N, K):
            check(lib().b200_gemm_bf16(kind, a.data_ptr(), a.stride(0), b.data_ptr(), b.stride(0), out.data_ptr(), out.stride(0),
                                       _p(residual), ldr, M, N, K, flags, group_m, max_ctas, _st()), "b200_gemm_bf16")
        _count(1)
        return out
    check(lib().b200_gemm_bf16(kind, a.data_ptr(), a.stride(0), b.data_ptr(), b.stride(0), out.data_ptr(), out.stride(0),
                               _p(residual), ldr, M, N, K, flags, group_m, max_ctas, _st()), "b200_gemm_bf16")
    _count(1)
    return out


_lt_ws = {}


def gemm_swiglu(x, w_gu, gu=None, a=None):
    """x[M,K] @ w_gu[2F,K]^T with the SwiGLU epilogue: returns (gu [M,2F] = [gate | up], a [M,F] = silu(gate) * up), both bf16, from ONE
    GEMM launch (CTA-pair kernel; M >= 256, F % 128 == 0).  Bit-identical to gemm(NT) followed by swiglu_fwd."""
    _chk2d(x, "x"); _chk2d(w_gu, "w_gu")
    M, K = x.shape
    N = w_gu.shape[0]
    assert w_gu.shape[1] == K and N % 2 == 0
    if gu is None:
        gu = torch.empty(M, N, dtype=torch.bfloat16, device=x.device)
    if a is None:
        a = torch.empty(M, N // 2, dtype=torch.bfloat16, device=x.device)
    _chk2d(gu, "gu"); _chk2d(a, "a")

    def launch():
        check(lib().b200_gemm_bf16(NT, x.data_ptr(), x.stride(0), w_gu.data_ptr(), w_gu.stride(0), gu.data_ptr(), gu.stride(0), a.data_ptr(),
                                   a.stride(0), M, N, K, GEMM_SWIGLU, 0, 0, _st()), "b200_gemm_bf16(swiglu)")

    if GEMM_TIMER is not None:
        with GEMM_TIMER(NT, M, N, K):
            launch()
    else:
        launch()
    _count(1)
    return gu, a


def gemm_cublaslt(kind, a, b, out=None):
    """cuBLASLt on the same operands (comparator for tests/bench; not used by the training path)."""
    if kind == NT:
        M, K = a.shape; N, _ = b.shape
    elif kind == NN:
        M, K = a.shape; _, N = b.shape
    else:
        K, M = a.shape; _, N = b.shape
    if out is None:
        out = torch.empty(M, N, dtype=torch.bfloat16, device=a.device)
    ws = _lt_ws.get(a.device)
    if ws is None:
        ws = _lt_ws[a.device] = torch.empty(64 << 20, dtype=torch.uint8, device=a.device)
    check(lib().b200_gemm_bf16_cublaslt(kind, a.data_ptr(), a.stride(0), b.data_ptr(), b.stride(0), out.data_ptr(), out.stride(0),
                                        M, N, K, ws.data_ptr(), ws.numel(), _st()), "b200_gemm_bf16_cublaslt")
    return out


def rmsnorm_fwd(x, w, eps, out=None, rstd=None):
    rows, cols = x.shape
    assert x.is_contiguous() and w.is_contiguous()
    if out is None:
        out = torch.empty_like(x)
    if rstd is None:
        rstd = torch.empty(rows, dtype=torch.float32, device=x.device)
    check(lib().b200_rmsnorm_fwd(x.data_ptr(), w.data_ptr(), out.data_ptr(), rstd.data_ptr(), rows, cols, float(eps), _st()), "b200_rmsnorm_fwd")
    _count(1)
    return out, rstd


def rmsnorm_bwd(dy, x, w, rstd, dres=None, dx=None, dw=None, accumulate_dw=False, workspace=None):
    rows, cols = x.shape
    assert dy.is_contiguous() and x.is_contiguous()
    if dx is None:
        dx = torch.empty_like(x)
    if dw is None:
        assert not accumulate_dw
        dw = torch.empty(cols, dtype=torch.bfloat16, device=x.device)
    need = lib().b200_rmsnorm_bwd_workspace_floats(rows, cols)
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(need, dtype=torch.float32, device=x.device)
    check(lib().b200_rmsnorm_bwd(dy.data_ptr(), x.data_ptr(), w.data_ptr(), rstd.data_ptr(), _p(dres), dx.data_ptr(), dw.data_ptr(),
                                 int(accumulate_dw), workspace.data_ptr(), rows, cols, _st()), "b200_rmsnorm_bwd")
    _count(2)
    return dx, dw


def rope_(qk, cos, sin, pos, heads, head_dim, backward=False):
    """In place on the first `heads` heads of each row of qk [T, >=heads*head_dim] (row pitch = qk.stride(0))."""
    assert qk.dtype == torch.bfloat16 and qk.stride(1) == 1 and pos.dtype == torch.int32
    check(lib().b200_rope_inplace(qk.data_ptr(), cos.data_ptr(), sin.data_ptr(), pos.data_ptr(), qk.shape[0], heads, head_dim,
                                  qk.stride(0), int(backward), _st()), "b200_rope_inplace")
    _count(1)
    return qk


def bias_rope_(qkv, bias, cos, sin, pos, rope_heads, heads, head_dim):
    """In place on qkv [T, heads*head_dim]: += bias on every head, RoPE on the first `rope_heads` heads (Qwen2 q/k/v bias)."""
    assert qkv.dtype == torch.bfloat16 and qkv.stride(1) == 1 and pos.dtype == torch.int32 and bias.numel() == heads * head_dim
    check(lib().b200_bias_rope_inplace(qkv.data_ptr(), bias.data_ptr(), cos.data_ptr(), sin.data_ptr(), pos.data_ptr(), qkv.shape[0], rope_heads,
                                       heads, head_dim, qkv.stride(0), _st()), "b200_bias_rope_inplace")
    _count(1)
    return qkv


_cs_ws = {}


def colsum_(x, out, accumulate=False):
    """out[c] (=|+=) bf16(sum_t x[t, c]) with fp32 accumulation: the bias gradient."""
    T, C = x.shape
    assert x.stride(1) == 1 and out.numel() == C
    need = lib().b200_colsum_workspace_floats(T, C)
    ws = _cs_ws.get(x.device)
    if ws is None or ws.numel() < need:
        ws = _cs_ws[x.device] = torch.empty(need, dtype=torch.float32, device=x.device)
    check(lib().b200_colsum_bf16(x.data_ptr(), out.data_ptr(), ws.data_ptr(), T, C, x.stride(0), int(accumulate), _st()), "b200_colsum_bf16")
    _count(2)
    return out


def swiglu_fwd(gu, out=None):
    T, F2 = gu.shape
    assert gu.is_contiguous()
    if out is None:
        out = torch.empty(T, F2 // 2, dtype=torch.bfloat16, device=gu.device)
    check(lib().b200_swiglu_fwd(gu.data_ptr(), out.data_ptr(), T, F2 // 2, _st()), "b200_swiglu_fwd")
    _count(1)
    return out


def swiglu_bwd(da, gu, out=None):
    T, F2 = gu.shape
    assert gu.is_contiguous() and da.is_contiguous()
    if out is None:
        out = torch.empty_like(gu)
    check(lib().b200_swiglu_bwd(da.data_ptr(), gu.data_ptr(), out.data_ptr(), T, F2 // 2, _st()), "b200_swiglu_bwd")
    _count(1)
    return out


def embed_fwd(ids, W, out=None):
    assert ids.dtype == torch.int32 and W.is_contiguous()
    T = ids.numel()
    if out is None:
        out = torch.empty(T, W.shape[1], dtype=torch.bfloat16, device=W.device)
    check(lib().b200_embed_fwd(ids.data_ptr(), W.data_ptr(), out.data_ptr(), T, W.shape[1], _st()), "b200_embed_fwd")
    _count(1)
    return out


def embed_bwd(ids, dh, dW, accumulate=False, workspace=None):
    T = ids.numel()
    if workspace is None:
        workspace = torch.empty(2 * T, dtype=torch.int32, device=dh.device)
    check(lib().b200_embed_bwd(ids.data_ptr(), dh.data_ptr(), dW.data_ptr(), workspace.data_ptr(), T, dh.shape[1], int(accumulate), _st()),
          "b200_embed_bwd")
    _count(2)
    return dW


def attn_fwd(q, k, v, cu_seqlens, max_seqlen, Hq, Hkv, D, scale=None, out=None, lse=None):
    """q [T, Hq*D] / k, v [T, Hkv*D] views (row pitch free).  Returns o [T, Hq*D], lse [Hq, T] fp32."""
    T = q.shape[0]
    scale = scale if scale is not None else D ** -0.5
    if out is None:
        out = torch.empty(T, Hq * D, dtype=torch.bfloat16, device=q.device)
    if lse is None:
        lse = torch.empty(Hq, T, dtype=torch.float32, device=q.device)
    check(lib().b200_attn_fwd(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), lse.data_ptr(), cu_seqlens.data_ptr(),
                              cu_seqlens.numel() - 1, max_seqlen, q.stride(0), k.stride(0), v.stride(0), out.stride(0), Hq, Hkv, D, T,
                              float(scale), _st()), "b200_attn_fwd")
    _count(1)
    return out, lse


def attn_bwd(q, k, v, o, dout, lse, cu_seqlens, max_seqlen, Hq, Hkv, D, dq, dk, dv, scale=None, workspace=None):
    T = q.shape[0]
    scale = scale if scale is not None else D ** -0.5
    if workspace is None:
        workspace = torch.empty(lib().b200_attn_bwd_workspace_bytes(T, Hq, D, max_seqlen), dtype=torch.uint8, device=q.device)
    check(lib().b200_attn_bwd(q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(), dout.data_ptr(), lse.data_ptr(), dq.data_ptr(),
                              dk.data_ptr(), dv.data_ptr(), workspace.data_ptr(), workspace.numel(), cu_seqlens.data_ptr(), cu_seqlens.numel() - 1,
                              max_seqlen, q.stride(0), k.stride(0), v.stride(0), o.stride(0), dout.stride(0), dq.stride(0),
                              dk.stride(0), dv.stride(0), Hq, Hkv, D, T, float(scale), _st()), "b200_attn_bwd")
    _count(3)
    return dq, dk, dv


def ce_fwd_bwd_(logits, labels, num_label_tokens, loss_out, accumulate=False, row_loss=None):
    """logits [T, V] bf16 is overwritten with dlogits.  loss_out: fp32[1] device tensor."""
    T, V = logits.shape
    assert labels.dtype == torch.int32 and logits.stride(1) == 1
    if row_loss is None:
        row_loss = torch.empty(T, dtype=torch.float32, device=logits.device)
    check(lib().b200_ce_fwd_bwd(logits.data_ptr(), labels.data_ptr(), row_loss.data_ptr(), loss_out.data_ptr(), T, V, logits.stride(0),
                                int(num_label_tokens), int(accumulate), _st()), "b200_ce_fwd_bwd")
    _count(2)
    return loss_out


_ss_ws = {}


def sumsq_(g, out, accumulate=False):
    ws = _ss_ws.get(g.device)
    if ws is None:
        ws = _ss_ws[g.device] = torch.empty(lib().b200_sumsq_workspace_floats(), dtype=torch.float32, device=g.device)
    check(lib().b200_sumsq_bf16(g.data_ptr(), g.numel(), out.data_ptr(), ws.data_ptr(), int(accumulate), _st()), "b200_sumsq_bf16")
    _count(2)
    return out


def adamw_step_(p, g, m, v, lr, beta1, beta2, eps, wd, step, max_grad_norm=0.0, grad_norm_sq=None, mode=0, master=None):
    check(lib().b200_adamw_step(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), _p(master), p.numel(), lr, beta1, beta2, eps, wd,
                                int(step), float(max_grad_norm or 0.0), _p(grad_norm_sq), int(mode), _st()), "b200_adamw_step")
    _count(1)


def add_(dst, src):
    check(lib().b200_add_inplace_bf16(dst.data_ptr(), src.data_ptr(), dst.numel(), _st()), "b200_add_inplace_bf16")
    _count(1)
    return dst


if os.environ.get("B200_ATTN_FWD_VARIANT"):       # A/B and bisecting knob (see include/b200_train.h b200_set_option "attn_fwd_variant")
    set_option("attn_fwd_variant", int(os.environ["B200_ATTN_FWD_VARIANT"]))


def reducescatter_layer(ctx, slot, byte_offset, shard_elems, mode=0, ctas=32, stream=None):
    """In-place reduce-scatter of one unit of a registered symmetric buffer (fp32 accumulation, one rounding); see include/b200_train.h."""
    check(lib().b200_reducescatter_layer(ctx, int(slot), int(byte_offset), int(shard_elems), int(mode), int(ctas),
                                         stream if stream is not None else _st()), "b200_reducescatter_layer")
    _count(1)


def allgather_layer(ctx, slot, byte_offset, shard_elems, mode=0, ctas=32, stream=None):
    """In-place all-gather of one unit of a registered symmetric buffer."""
    check(lib().b200_allgather_layer(ctx, int(slot), int(byte_offset), int(shard_elems), int(mode), int(ctas),
                                     stream if stream is not None else _st()), "b200_allgather_layer")
    _count(1)


def allreduce_scalars_(ctx, vals, stream=None):
    """vals (fp32, <= 16 elements, contiguous) := sum over the ranks of the symmetric-memory context, in rank order."""
    assert vals.dtype == torch.float32 and vals.is_contiguous() and vals.numel() <= 16
    check(lib().b200_allreduce_scalars(ctx, vals.data_ptr(), vals.numel(), stream if stream is not None else _st()), "b200_allreduce_scalars")
    _count(1)
    return vals
