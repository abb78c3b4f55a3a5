"""Sharded-data-parallel Llama training step on B200: host orchestration over the sm_100a kernels.

This is the replacement for what the reference's `_forward_backward_step` / `_run_train_optim_step`
(/root/reference/nemo_automodel/recipes/llm/train_ft.py:1357-1473, 1482-1635) reach through
torch FSDP2 + DTensor + ATen/cuBLAS/flash-attn:

  per-unit parameter all-gather  ->  transformer-block forward/backward  ->  gradient reduce-scatter
  ->  grad-norm + clip  ->  AdamW on the local shard.

Design (B200-first, 180 GB HBM per GPU):
  * flat bf16 storage per unit (layout.py); a rank's parameter shard is a slice *inside* the unsharded buffer, so the
    all-gather is in place and happens ONCE per optimizer step (parameters stay gathered through forward and backward:
    16 GB for Llama-3-8B), halving the reference's all-gather traffic (it re-gathers every layer in backward,
    parallelizer.py:860-871);
  * gradients are produced by the wgrad GEMMs directly into the unit's flat gradient buffer; the reduce-scatter is in
    place on that buffer and overlaps the backward of the next unit on a side stream;
  * explicit forward/backward over pre-allocated activation arenas - no autograd graph, no caching-allocator churn;
  * grad-norm is one fused reduction per unit + one scalar all-reduce; the clip coefficient never visits the host.
All device math is in csrc/ (via ops); torch provides memory, streams and torch.distributed only.
"""
import math
import os
from typing import Dict, List, Optional

import numpy as np
import torch
import torch.distributed as dist

from .layout import LlamaDims, UnitLayout, build_layout, total_params

IGNORE_INDEX = -100


def _rope_inv_freq(d: LlamaDims) -> torch.Tensor:
    """inv_freq as the reference computes it (components/models/llama/rope_utils.py:108-150), fp32 on the host."""
    D = d.head_dim
    inv = 1.0 / (torch.tensor(float(d.rope_theta), dtype=torch.float32) ** (torch.arange(0, D, 2, dtype=torch.int64).float() / D))
    sc = d.rope_scaling or {}
    rtype = sc.get("rope_type", sc.get("type", "default"))
    if rtype == "default":
        return inv
    if rtype != "llama3":
        raise ValueError(f"rope_type {rtype!r} is not supported (default and llama3 are; rope_utils.py:152-190 of the reference)")
    factor = sc.get("factor", 1.0)
    lo, hi = sc.get("low_freq_factor", 1.0), sc.get("high_freq_factor", 4.0)
    old = sc.get("original_max_position_embeddings", d.max_pos)
    low_wl, high_wl = old / lo, old / hi
    wavelen = 2 * math.pi / inv
    inv_l = torch.where(wavelen > low_wl, inv / factor, inv)
    smooth = (old / wavelen - lo) / (hi - lo)
    smoothed = (1 - smooth) * inv_l / factor + smooth * inv_l
    med = (~(wavelen < high_wl)) & (~(wavelen > low_wl))
    return torch.where(med, smoothed, inv_l)


def rope_tables(d: LlamaDims, n_pos: int, device) -> (torch.Tensor, torch.Tensor):
    """bf16 cos/sin tables [n_pos, head_dim] (rope_utils.py:191-205: fp32 math, rounded to the model dtype)."""
    # inv_freq on the host (the reference's module computes it at construction, device=None), the angle table on the target device:
    # `_build_cache` runs cos/sin on x.device (rope_utils.py:191-205), and CUDA's cosf differs from glibc's by an ulp on some entries.
    inv = _rope_inv_freq(d).to(device)
    t = torch.arange(n_pos, device=device, dtype=torch.float32)
    freqs = torch.outer(t, inv)
    emb = torch.cat((freqs, freqs), dim=-1)
    return emb.cos().to(torch.bfloat16), emb.sin().to(torch.bfloat16)


def cu_seqlens_from_position_ids(position_ids: np.ndarray):
    """Packed batches restart position_ids at every document (components/datasets/llm/packed_sequence.py:37-110).
    position_ids [b,S] (host) -> (cu_seqlens int32 [nseq+1] over the flattened b*S tokens, max_seqlen)."""
    b, S = position_ids.shape
    flat = position_ids.reshape(-1)
    starts = np.flatnonzero(flat == 0)
    row_starts = np.arange(b) * S
    starts = np.union1d(starts, row_starts)
    cu = np.concatenate([starts, [b * S]]).astype(np.int32)
    return cu, int(np.diff(cu).max())


class _Streams:
    """CUDA streams/events; no-ops on CPU (CPU execution exists only for the orchestration tests)."""

    def __init__(self, device):
        self.cuda = device.type == "cuda"
        # high priority: a pending communication CTA (small: 512 threads, <= 64 registers, no smem) is placed before the next compute kernel's
        # CTAs, next to which it then co-resides
        self.comm = torch.cuda.Stream(device, priority=-1) if self.cuda else None
        self.opt = torch.cuda.Stream(device) if self.cuda else None
        self.wg = torch.cuda.Stream(device) if self.cuda else None    # weight-gradient GEMMs (see backward_from_dlogits)

    def event(self):
        return torch.cuda.Event() if self.cuda else None

    def record(self, ev, stream=None):
        if self.cuda:
            ev.record(stream if stream is not None else torch.cuda.current_stream())

    def wait(self, ev, stream=None):
        if self.cuda and ev is not None:
            (stream if stream is not None else torch.cuda.current_stream()).wait_event(ev)


class ShardedLlamaEngine:
    """One rank of the sharded-DP training step.  `ops` is automodel_b200.ops (CUDA); tests inject a CPU stand-in to
    exercise the orchestration over gloo without a GPU."""

    def __init__(self, cfg, device, process_group=None, max_tokens=4096, lr=1e-5, betas=(0.9, 0.95), eps=1e-8, weight_decay=0.1,
                 adam_mode=0, master_weights=False, ops=None, max_positions=None, reference_rounding=True, activation_checkpointing=False,
                 replica_group=None, reduce_dtype=None, comm=None, reshard_after_forward=False):
        if ops is None:
            from . import ops as _ops  # raises if libb200_train.so is missing: no fallback
            ops = _ops
        self.ops = ops
        self.dims = cfg if isinstance(cfg, LlamaDims) else LlamaDims.from_hf(cfg)
        d = self.dims
        self.device = torch.device(device)
        if self.device.type == "cuda" and self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())   # comparable with tensor.device
        self.pg = process_group
        if process_group is not None:
            self.world = dist.get_world_size(process_group)
            self.rank = dist.get_rank(process_group)
        else:
            self.world, self.rank = 1, 0
        # HSDP (reference: dp_replicate_size > 1, mesh (dp_replicate, dp_shard), distributed/mesh_utils.py:116-190): parameters and
        # optimizer state are sharded inside `process_group` and replicated across `replica_group`; a unit's gradient shard is
        # all-reduced across the replicas right after its reduce-scatter.
        self.rpg = replica_group
        self.replicas = dist.get_world_size(replica_group) if replica_group is not None else 1
        self.replica_rank = dist.get_rank(replica_group) if replica_group is not None else 0
        # Optional: run the persistent GEMMs on (SMs - comm_sms) CTAs while NCCL kernels overlap them (B200_COMM_SMS, default 0).
        self.comm_sms = 0
        if self.world > 1 and self.device.type == "cuda":
            self.comm_sms = int(os.environ.get("B200_COMM_SMS", "0"))  # measured at N=2 (profiles/r1_n2_comm_sms.md): 0 is best
        self.gemm_ctas = 0  # 0 = one CTA per SM
        if self.comm_sms > 0:
            self.gemm_ctas = torch.cuda.get_device_properties(self.device).multi_processor_count - self.comm_sms
        self.units: List[UnitLayout] = build_layout(d, self.world)
        self.n_params = total_params(self.units)
        self.max_tokens = max_tokens
        self.lr, self.betas, self.eps, self.wd = lr, betas, eps, weight_decay
        if master_weights and adam_mode == 1:
            # mode 1 reproduces torch.optim.AdamW on bf16 parameters op by op (every intermediate rounded to bf16): an fp32 master copy would
            # be overwritten with the rounded value each step - it only makes sense with the fp32-math update
            raise ValueError("master_weights=True needs adam_mode=0 (fp32 update math); adam_mode=1 is the bf16 torch.optim.AdamW sequence")
        self.adam_mode = adam_mode
        self.round_before_add = bool(reference_rounding)
        self.step_count = 0
        self.streams = _Streams(self.device)
        # Weight-gradient GEMMs on their own stream: they are off the dgrad dependency chain, so they fill the tensor pipes while the
        # chain runs its HBM-bound kernels (SwiGLU', RMSNorm', RoPE', attention pre/post passes) and the tail waves of the dgrad GEMMs.
        # Default: on for one GPU (measured +2.3..3.4 %); with N > 1 it is opt-in until it has been measured next to the NCCL kernels.
        self._wg_on = self.streams.cuda and os.environ.get("B200_WGRAD_STREAM", "1" if self.world == 1 else "0") == "1"
        self.opt_overlap = self.streams.cuda and os.environ.get("B200_OPT_OVERLAP", "1") != "0"   # optimizer sweep on its own stream
        self._overlap_cfg = (self._wg_on, self.opt_overlap)     # what set_stream_overlap(True) restores
        self._wg_pending = {}     # tmp buffer name -> event of the last side-stream GEMM that reads it (WAR guard for the next writer)
        self._wg_last = None
        # B200_FUSE_SWIGLU=1: SwiGLU computed in the epilogue of the gate/up GEMM (b200_gemm_bf16 flag 4) instead of a separate HBM pass
        self._fuse_swiglu = self.streams.cuda and os.environ.get("B200_FUSE_SWIGLU", "0") == "1" and d.ffn % 128 == 0
        if self.streams.cuda:
            # side-stream HBM-bound sweeps (AdamW, grad-norm partials) leave register/thread room for a co-resident GEMM CTA
            self.ops.set_option("side_blocks_per_sm", int(os.environ.get("B200_SIDE_BLOCKS", "0")))
        bf, dev = torch.bfloat16, self.device

        # ---- persistent flat storage
        self._rs_started = False
        # Gradient reduction precision (reference: MixedPrecisionPolicy.reduce_dtype, default float32, components/distributed/config.py:121-132):
        # "float32" = fp32 accumulation across ranks with ONE rounding to the bf16 gradient, "bfloat16" = NCCL's bf16 ring (rounds per hop).
        self.reduce_dtype = reduce_dtype or os.environ.get("B200_REDUCE_DTYPE", "float32")
        if self.reduce_dtype not in ("float32", "bfloat16"):
            raise ValueError(f"reduce_dtype {self.reduce_dtype!r}: float32 or bfloat16")
        # Per-unit collectives.  "nvls": this repository's kernels on symmetric memory (b200_allgather_layer / b200_reducescatter_layer).
        # The all-gather is the NVSwitch multicast store (bit-exact).  The reduce-scatter follows reduce_dtype: float32 = peer loads summed
        # in fp32 in rank order + ONE round-to-nearest-even (what the reference's fp32 reduce-scatter followed by the cast to the bf16
        # gradient computes); bfloat16 = the NVSwitch in-fabric reduction (multimem.ld_reduce .acc::f32), measured at <= 1 bf16 ulp of the
        # exact sum but NOT correctly rounded (ties away from zero and worse: profiles/r2_nvls_collectives.md) - the precision class of a
        # bf16 reduction, at the lowest SM cost.  "p2p": both collectives on the peer-load variants (no multicast needed).  "nccl":
        # torch.distributed in-place collectives (multi-node groups; fp32 reduction goes through an fp32 staging buffer).
        # Default "auto": the symmetric-memory kernels whenever the shard group is one NVSwitch box (<= 8 CUDA ranks, no replica groups),
        # NCCL otherwise or when the symmetric allocation / rendezvous is not available on the platform.
        self.comm = comm or os.environ.get("B200_COMM", "auto")
        if self.comm not in ("auto", "nccl", "nvls", "p2p"):
            raise ValueError(f"comm {self.comm!r}: auto, nccl, nvls or p2p")
        self.sym = None
        self._comm_ctas = int(os.environ.get("B200_COMM_CTAS", "32"))
        want_sym = self.comm in ("nvls", "p2p") or (self.comm == "auto" and self.world <= 8 and self.replicas == 1)
        if reshard_after_forward:
            if self.comm in ("nvls", "p2p"):
                raise NotImplementedError("reshard_after_forward runs on the torch.distributed collectives (comm='nccl'); the symmetric-memory pool is not built")
            want_sym = False
        if self.world > 1 and dev.type == "cuda" and want_sym:
            if self.world > 8:
                raise NotImplementedError("the symmetric-memory data path spans one NVSwitch box (<= 8 ranks per shard group); use comm='nccl'")
            try:
                self._setup_symmetric(process_group, dev, bf)
            except Exception as e:  # noqa: BLE001 - platform without symmetric memory / peer access
                if self.comm != "auto":
                    raise
                import sys
                sys.stderr.write(f"[automodel_b200] symmetric-memory collectives unavailable ({type(e).__name__}: {e}); using NCCL\n")
                self.sym = None
        if self.sym is None:
            self.comm_kind = "nccl" if self.world > 1 else "none"
            pooled = (lambda ui: reshard_after_forward and 1 <= ui <= d.layers)      # layer units live in the reshard pool (set up below)
            self.p_full = [None if pooled(ui) else torch.zeros(u.padded, dtype=bf, device=dev) for ui, u in enumerate(self.units)]   # unsharded params (shard lives inside)
            self.g_full = [None if pooled(ui) else torch.zeros(u.padded, dtype=bf, device=dev) for ui, u in enumerate(self.units)]   # unsharded grads (RS in place)
        # ---- reshard_after_forward (the reference's FSDP2 schedule, components/distributed/parallelizer.py:858-872: a decoder layer's
        # parameters are unsharded only while the layer computes).  Persistent state of a layer unit is its 1/N parameter shard and a 1/N
        # gradient shard; the unsharded parameters / gradients of the layers rotate through a pool of POOL buffers (all-gather before the
        # layer's forward and again before its backward, reduce-scatter right after its backward, every micro-batch).  Memory O(P/N + POOL
        # layers) instead of O(P): what the 70B config needs.  The embed and head units stay resident, as the reference's root unit does.
        self.reshard = bool(reshard_after_forward)
        if self.reshard:
            self._setup_reshard_pool(dev, bf)
        self._rs32 = self._rs32_out = None
        if self.world > 1 and self.sym is None and self.reduce_dtype == "float32":
            big = max(u.padded for u in self.units)
            self._rs32 = torch.empty(big, dtype=torch.float32, device=dev)
            self._rs32_out = torch.empty(big // self.world, dtype=torch.float32, device=dev)
        self.m = [torch.zeros(u.padded // self.world, dtype=bf, device=dev) for u in self.units]
        self.v = [torch.zeros(u.padded // self.world, dtype=bf, device=dev) for u in self.units]
        self.master = [torch.zeros(u.padded // self.world, dtype=torch.float32, device=dev) for u in self.units] if master_weights else None
        self.P: Dict[str, torch.Tensor] = {}
        self.G: Dict[str, torch.Tensor] = {}
        for ui, u in enumerate(self.units):
            for s in u.slots:
                self.P[s.name] = self.p_full[ui][s.offset:s.offset + s.numel].view(s.shape)
                self.G[s.name] = self.g_full[ui][s.offset:s.offset + s.numel].view(s.shape)
        self._mk_fused_views()
        self.ev_opt = [None] * len(self.units)  # AdamW of unit done (optimizer side stream)
        self.ev_opt_all = None
        self.ev_ag = [None] * len(self.units)   # all-gather of unit done
        self.ev_rs = [None] * len(self.units)   # reduce-scatter of unit done

        n_pos = max_positions or max(d.max_pos, 1)
        self.cos, self.sin = rope_tables(d, n_pos, dev)

        # ---- activation arenas (allocated once for max_tokens)
        T, h, F, L = max_tokens, d.hidden, d.ffn, d.layers
        e = lambda *shape, dtype=bf: torch.empty(*shape, dtype=dtype, device=dev)
        # Activation checkpointing (distributed/parallelizer.py:237-268 wraps every decoder layer in checkpoint_wrapper): only the layer
        # inputs h[l] are kept; the layer's other activations live in ONE buffer set shared by all layers and are recomputed from h[l]
        # (same kernels, bit-identical values) right before the layer's backward.  8B, 4096 tokens: 18.3 GB -> 0.57 GB of activations.
        self.recompute = bool(activation_checkpointing)
        per = (lambda mk: [mk()] * L) if self.recompute else (lambda mk: [mk() for _ in range(L)])
        self.act = {
            "h": [e(T, h) for _ in range(L + 1)],            # residual stream: h[l] = input of layer l, h[L] = output
            "x1": per(lambda: e(T, h)),
            "rstd1": per(lambda: e(T, dtype=torch.float32)),
            "qkv": per(lambda: e(T, d.qkv_cols)),
            "lse": per(lambda: e(d.heads, T, dtype=torch.float32)),
            "o2": per(lambda: e(T, d.q_cols)),
            "h1": per(lambda: e(T, h)),
            "x2": per(lambda: e(T, h)),
            "rstd2": per(lambda: e(T, dtype=torch.float32)),
            "gu": per(lambda: e(T, 2 * F)),
            "a": per(lambda: e(T, F)),
        }
        self.xf, self.rstdf = e(T, h), e(T, dtype=torch.float32)
        self.logits = e(T, d.vocab)
        self.row_loss = e(T, dtype=torch.float32)
        self.tmp = {
            "dh_a": e(T, h), "dh_b": e(T, h), "dxf": e(T, h), "da": e(T, F), "dgu": e(T, 2 * F), "dx": e(T, h),
            "do2": e(T, d.q_cols), "dqkv": e(T, d.qkv_cols),
        }
        # token inputs: two (pinned host, device) buffer sets used alternately, so the host can stage micro-batch i+1 while
        # the device still reads micro-batch i (embed_bwd at the very end of backward needs the ids)
        pin = self.device.type == "cuda"
        self._in_dev = [torch.empty(4 * T + 1, dtype=torch.int32, device=dev) for _ in range(2)]   # ids | labels | pos | cu
        self._in_host = [torch.empty(4 * T + 1, dtype=torch.int32, pin_memory=pin) for _ in range(2)]
        self._in_ev = [None, None]
        self._in_idx = 0
        self.h2d_bytes = 0
        self.embed_ws = torch.empty(2 * T, dtype=torch.int32, device=dev)
        if self.device.type == "cuda":
            from ._lib import lib
            self.norm_ws = torch.empty(lib().b200_rmsnorm_bwd_workspace_floats(T, h), dtype=torch.float32, device=dev)
            # sized for the longest sequence this engine can see (the RoPE tables bound it)
            self.attn_ws = torch.empty(lib().b200_attn_bwd_workspace_bytes(T, d.heads, d.head_dim, min(T, n_pos)), dtype=torch.uint8, device=dev)
        else:
            self.norm_ws = self.attn_ws = None
        self.loss_dev = torch.zeros(1, dtype=torch.float32, device=dev)
        self.norm_sq = torch.zeros(1, dtype=torch.float32, device=dev)
        self._grads_dirty = False
        self._unsynced = False    # gradients accumulated but not yet reduce-scattered (backward ran with last_micro=False)

    def _setup_symmetric(self, process_group, dev, bf):
        """Parameter and gradient storage of all units in two symmetric slabs + the b200_ctx that the collectives entries take."""
        from .symm import SymmetricSlab, CommContext
        offs, tot = [], 0
        for u in self.units:
            offs.append(tot)
            tot += u.padded
        self._unit_off = offs
        self._p_slab, self._g_slab = SymmetricSlab(tot, bf, dev, process_group), SymmetricSlab(tot, bf, dev, process_group)
        self.p_full = [self._p_slab.tensor[o:o + u.padded] for o, u in zip(offs, self.units)]
        self.g_full = [self._g_slab.tensor[o:o + u.padded] for o, u in zip(offs, self.units)]
        sym = CommContext(process_group, dev)
        sym.register(CommContext.PARAMS, self._p_slab)
        sym.register(CommContext.GRADS, self._g_slab)
        mc = self.comm != "p2p" and sym.has_multicast(CommContext.GRADS) and sym.has_multicast(CommContext.PARAMS)
        self._ag_mode = 0 if mc else 1
        self._rs_mode = 0 if (mc and self.reduce_dtype == "bfloat16") else 1
        self._rs_ctas = self._comm_ctas if self._rs_mode == 0 else int(os.environ.get("B200_P2P_RS_CTAS", "64"))
        self.comm_kind = ("nvls" if self._rs_mode == 0 else "nvls-ag+p2p-rs") if mc else "p2p"
        self.sym = sym

    # ------------------------------------------------------------------ reshard_after_forward
    POOL = 2

    def _setup_reshard_pool(self, dev, bf):
        d, K = self.dims, self.POOL
        L = d.layers
        big = max(self.units[1 + l].padded for l in range(L)) if L else 0
        self._pool_p = [torch.zeros(big, dtype=bf, device=dev) for _ in range(K)]
        self._pool_g = [torch.zeros(big, dtype=bf, device=dev) for _ in range(K)]
        self.p_shard, self.g_shard = [None] * len(self.units), [None] * len(self.units)
        for ui, u in enumerate(self.units):
            a, b = u.shard_range(self.rank, self.world)
            if 1 <= ui <= L:
                # the full-size buffers allocated above are dropped: layer units live as shards + pool slots
                self.p_full[ui] = self._pool_p[(ui - 1) % K][:u.padded]
                self.g_full[ui] = self._pool_g[(ui - 1) % K][:u.padded]
                self.p_shard[ui] = torch.zeros(b - a, dtype=bf, device=dev)
                self.g_shard[ui] = torch.zeros(b - a, dtype=bf, device=dev)
            else:
                self.p_shard[ui] = self.p_full[ui][a:b]
                self.g_shard[ui] = self.g_full[ui][a:b]
        self._slot_layer = [None] * K        # which layer's parameters pool slot k holds (None: stale)
        self._slot_free = [None] * K         # event: the last compute that read parameter slot k has finished
        self._gslot_rs = [None] * K          # event: the reduce-scatter that read gradient slot k has finished
        self._rs_tmp = torch.zeros(big // max(self.world, 1) if big else 0, dtype=bf, device=dev)
        self._micro = (True, True)           # (first_micro, last_micro) of the backward in progress

    def _is_pooled(self, ui):
        return self.reshard and 1 <= ui <= self.dims.layers

    def _ensure_layer(self, l, prefetch_only=False):
        """Unsharded parameters of layer l in its pool slot: copy the local shard into its place and all-gather in place (communication
        stream on the GPU; the compute stream waits for the event unless this is a prefetch)."""
        K = self.POOL
        k, ui = l % K, 1 + l
        st = self.streams
        if self._slot_layer[k] != l:
            u = self.units[ui]
            a, b = u.shard_range(self.rank, self.world)
            slot = self.p_full[ui]

            def issue():
                slot[a:b].copy_(self.p_shard[ui])
                if self.world > 1:
                    if st.cuda:
                        dist.all_gather_into_tensor(slot, slot[a:b], group=self.pg)
                    else:
                        dist.all_gather_into_tensor(slot, slot[a:b].clone(), group=self.pg)

            if st.cuda:
                ev = st.event()
                st.record(ev)                       # the shard (AdamW) and everything that read the slot before, as far as issued here
                with torch.cuda.stream(st.comm):
                    st.wait(ev, st.comm)
                    st.wait(self._slot_free[k], st.comm)
                    if self.ev_opt[ui] is not None:
                        st.wait(self.ev_opt[ui], st.comm)
                    issue()
                    done = st.event()
                    st.record(done, st.comm)
                    self.ev_ag[ui] = done
            else:
                issue()
            self._slot_layer[k] = l
        if not prefetch_only and self.ev_ag[ui] is not None:
            st.wait(self.ev_ag[ui])
            self.ev_ag[ui] = None

    def _release_layer(self, l):
        """The compute stream is done reading layer l's parameter slot (end of its forward / backward)."""
        if self.streams.cuda:
            ev = self.streams.event()
            self.streams.record(ev)
            self._slot_free[l % self.POOL] = ev

    def _reduce_scatter_pooled(self, ui):
        """Reduce-scatter of a pooled layer unit's gradient slot into the persistent gradient shard (= on the first micro-batch, += after)."""
        first, last = self._micro
        st = self.streams
        k = (ui - 1) % self.POOL
        n = self.units[ui].padded
        per = n // self.world
        gslot, gsh = self.g_full[ui], self.g_shard[ui]
        a, b = self.units[ui].shard_range(self.rank, self.world)
        wide = self.reduce_dtype == "float32" and self.world > 1

        def body():
            if self.world == 1:
                red = gslot[a:b]
            elif wide:
                g32 = gslot.float() if self._rs32 is None else self._rs32[:n].copy_(gslot)
                o32 = torch.empty(per, dtype=torch.float32, device=gslot.device) if self._rs32_out is None else self._rs32_out[:per]
                dist.reduce_scatter_tensor(o32, g32, op=dist.ReduceOp.SUM, group=self.pg)
                if self.replicas > 1:
                    dist.all_reduce(o32, op=dist.ReduceOp.SUM, group=self.rpg)
                red = self._rs_tmp[:per].copy_(o32)
            else:
                red = self._rs_tmp[:per]
                dist.reduce_scatter_tensor(red, gslot if st.cuda else gslot.clone(), op=dist.ReduceOp.SUM, group=self.pg)
                if self.replicas > 1:
                    dist.all_reduce(red, op=dist.ReduceOp.SUM, group=self.rpg)
            if first:
                gsh.copy_(red)
            else:
                self.ops.add_(gsh, red)
            if last and st.cuda:      # grad-norm partial under the rest of the backward (the CPU path sums every shard in compute_grad_norm_sq)
                self.ops.sumsq_(gsh, self.norm_sq, accumulate=self._rs_started)
                self._rs_started = True

        if st.cuda:
            # N = 1 has no collective: the copy and the grad-norm partial go to the stream where _reduce_scatter_unit takes the resident
            # units' partials.  Every partial then adds into norm_sq in issue order (the resident engine's order), and no two sumsq_ calls
            # share the device's sumsq workspace from different streams at once.
            side = st.opt if self.world == 1 and self.replicas == 1 else st.comm
            ev = st.event()
            st.record(ev)
            wg = self._wg_last if self._wg_on else None
            with torch.cuda.stream(side):
                st.wait(ev, side)
                st.wait(wg, side)
                body()
                done = st.event()
                st.record(done, side)
                self.ev_rs[ui] = done
                self._gslot_rs[k] = done
        else:
            body()

    def _before_grad_slot_write(self, l):
        """Layer l's backward is about to overwrite gradient slot l % POOL: the reduce-scatter of the layer that used it last must be done."""
        k = l % self.POOL
        ev = self._gslot_rs[k]
        if ev is not None:
            self.streams.wait(ev)
            if self._wg_on:
                self.streams.wait(ev, self.streams.wg)
            self._gslot_rs[k] = None

    # ------------------------------------------------------------------ parameter plumbing
    def _mk_fused_views(self):
        d = self.dims
        self.W = []
        for l in range(d.layers):
            ui = 1 + l
            u = self.units[ui]
            off = {s.name.split(".", 3)[3]: s.offset for s in u.slots}
            pf, gf = self.p_full[ui], self.g_full[ui]

            def view(buf, o, r, c):
                return buf[o:o + r * c].view(r, c)

            self.W.append({
                "qkv": view(pf, off["self_attn.q_proj.weight"], d.qkv_cols, d.hidden),
                "o": view(pf, off["self_attn.o_proj.weight"], d.hidden, d.q_cols),
                "gu": view(pf, off["mlp.gate_proj.weight"], 2 * d.ffn, d.hidden),
                "down": view(pf, off["mlp.down_proj.weight"], d.hidden, d.ffn),
                "n1": pf[off["input_layernorm.weight"]:off["input_layernorm.weight"] + d.hidden],
                "n2": pf[off["post_attention_layernorm.weight"]:off["post_attention_layernorm.weight"] + d.hidden],
                "d_qkv": view(gf, off["self_attn.q_proj.weight"], d.qkv_cols, d.hidden),
                "d_o": view(gf, off["self_attn.o_proj.weight"], d.hidden, d.q_cols),
                "d_gu": view(gf, off["mlp.gate_proj.weight"], 2 * d.ffn, d.hidden),
                "d_down": view(gf, off["mlp.down_proj.weight"], d.hidden, d.ffn),
                "d_n1": gf[off["input_layernorm.weight"]:off["input_layernorm.weight"] + d.hidden],
                "d_n2": gf[off["post_attention_layernorm.weight"]:off["post_attention_layernorm.weight"] + d.hidden],
            })
            if d.qkv_bias:
                ob = off["self_attn.q_proj.bias"]
                self.W[-1]["qkv_b"] = pf[ob:ob + d.qkv_cols]
                self.W[-1]["d_qkv_b"] = gf[ob:ob + d.qkv_cols]
        # lm_head matrix and its gradient: the embed unit's when the embeddings are tied
        head = "model.embed_tokens.weight" if d.tied else "lm_head.weight"
        self.lm_head_w, self.lm_head_g = self.P[head], self.G[head]

    def load_state_dict(self, sd):
        """sd: HF-named full tensors (torch or numpy, any float dtype).  Every rank loads the full model (the metric's
        random-init / a from_pretrained snapshot); optimizer shards start at zero."""
        self.sync_params()      # a pending side-stream optimizer sweep / all-gather must not overwrite the freshly loaded weights
        if self.streams.cuda:
            torch.cuda.synchronize(self.device)
        with torch.no_grad():
            for ui, u in enumerate(self.units):
                for sl in u.slots:
                    src, dst = sd[sl.name], self.P[sl.name]
                    if isinstance(src, np.ndarray):
                        src = torch.from_numpy(np.ascontiguousarray(src))
                    if src is not dst:
                        dst.copy_(src.to(dst.dtype).reshape(dst.shape))
                if self._is_pooled(ui):      # the unit was assembled in its pool slot: keep this rank's shard
                    a, b = u.shard_range(self.rank, self.world)
                    self.p_shard[ui].copy_(self.p_full[ui][a:b])
            if self.reshard:
                self._slot_layer = [None] * self.POOL
            if self.master is not None:
                for ui, u in enumerate(self.units):
                    self.master[ui].copy_(self.shard(self.p_full, ui).float())
        for t in self.m + self.v:
            t.zero_()
        self.step_count = 0

    # ------------------------------------------------------------------ optimizer state in per-parameter (HF-named) form
    def gather_optimizer_state(self):
        """{name: (exp_avg, exp_avg_sq)} as FULL HF-shaped tensors.  World 1: views of the flat shards (live, zero copy).  World N: every
        unit's shards are all-gathered into temporaries (checkpoint time only; 2 x model size of extra memory)."""
        self.sync_params()
        out = {}
        for ui, u in enumerate(self.units):
            if self.world == 1:
                mf, vf = self.m[ui], self.v[ui]
            else:
                mf, vf = torch.empty_like(self.p_full[ui]), torch.empty_like(self.p_full[ui])
                dist.all_gather_into_tensor(mf, self.m[ui].contiguous(), group=self.pg)
                dist.all_gather_into_tensor(vf, self.v[ui].contiguous(), group=self.pg)
            for sl in u.slots:
                out[sl.name] = (mf[sl.offset:sl.offset + sl.numel].view(sl.shape), vf[sl.offset:sl.offset + sl.numel].view(sl.shape))
        return out

    def load_optimizer_state(self, named, step_count):
        """Inverse of gather_optimizer_state: copy this rank's slice of every full (exp_avg, exp_avg_sq) into the flat shards."""
        self.sync_params()
        if self.streams.cuda:
            torch.cuda.synchronize(self.device)
        with torch.no_grad():
            for ui, u in enumerate(self.units):
                a, b = u.shard_range(self.rank, self.world)
                for sl in u.slots:
                    lo, hi = max(sl.offset, a), min(sl.offset + sl.numel, b)
                    if lo >= hi or sl.name not in named:
                        continue
                    m_src, v_src = named[sl.name]
                    self.m[ui][lo - a:hi - a].copy_(m_src.reshape(-1)[lo - sl.offset:hi - sl.offset])
                    self.v[ui][lo - a:hi - a].copy_(v_src.reshape(-1)[lo - sl.offset:hi - sl.offset])
        self.step_count = int(step_count)

    def refresh_master_(self):
        """fp32 master copies (if kept) := the current bf16 weights of this rank's shards (after an external in-place weight load)."""
        if self.master is not None:
            with torch.no_grad():
                for ui, u in enumerate(self.units):
                    self.master[ui].copy_(self.shard(self.p_full, ui).float())

    def init_random_(self, seed=0, std=0.02):
        """Random init of the metric config, on device: N(0, std) linears/embeddings, ones for norms
        (HF initialize_weights semantics, components/checkpoint/checkpointing.py:574-676).  Same values on every rank."""
        g = torch.Generator(device=self.device).manual_seed(seed)
        self.sync_params()
        with torch.no_grad():
            for ui, u in enumerate(self.units):      # unit order = the order of self.P: the same random stream as a resident engine draws
                for sl in u.slots:
                    name, p = sl.name, self.P[sl.name]
                    if name.endswith("norm.weight") or "layernorm" in name:
                        p.fill_(1.0)
                    elif name.endswith(".bias"):
                        p.zero_()
                    else:
                        p.copy_((torch.randn(p.shape, generator=g, device=self.device, dtype=torch.float32) * std).to(p.dtype))
                if self._is_pooled(ui):
                    a, b = u.shard_range(self.rank, self.world)
                    self.p_shard[ui].copy_(self.p_full[ui][a:b])
        if self.reshard:
            self._slot_layer = [None] * self.POOL
        self.load_state_dict(self.P) if not self.reshard else self._reset_optimizer_state()

    def _reset_optimizer_state(self):
        self.refresh_master_()
        for t in self.m + self.v:
            t.zero_()
        self.step_count = 0

    def state_dict(self):
        self.sync_params()
        if not self.reshard:
            return dict(self.P)
        # reshard mode: the layers exist only as shards; gather every layer unit into a temporary (checkpoint / inspection time only)
        out = {}
        for ui, u in enumerate(self.units):
            if self._is_pooled(ui):
                full = torch.empty(u.padded, dtype=self.p_shard[ui].dtype, device=self.device)
                if self.world > 1:
                    dist.all_gather_into_tensor(full, self.p_shard[ui].contiguous(), group=self.pg)
                else:
                    full.copy_(self.p_shard[ui])
            else:
                full = self.p_full[ui]
            for sl in u.slots:
                out[sl.name] = full[sl.offset:sl.offset + sl.numel].view(sl.shape)
        return out

    def named_grads(self):
        return dict(self.G)

    def shard(self, bufs, ui):
        if self.reshard:
            if bufs is self.p_full:
                return self.p_shard[ui]
            if bufs is self.g_full:
                return self.g_shard[ui]
        a, b = self.units[ui].shard_range(self.rank, self.world)
        return bufs[ui][a:b]

    # ------------------------------------------------------------------ collectives (NCCL over NVLink via torch.distributed)
    def _all_gather_unit(self, ui):
        if self.world == 1:
            return
        st = self.streams
        ev = st.event()
        st.record(ev)                       # shard update (AdamW) issued on the compute stream
        if st.cuda and self.sym is not None:
            # our kernel on the symmetric parameter slab: NVLS multimem.st of the updated slice (or peer pulls); the cross-rank
            # "everybody's slice has landed" barrier is inside the kernel
            n_shard = self.units[ui].padded // self.world
            with torch.cuda.stream(st.comm):
                st.wait(ev, st.comm)
                self.ops.allgather_layer(self.sym.ptr, 0, self._unit_off[ui] * 2, n_shard, self._ag_mode, self._comm_ctas, st.comm.cuda_stream)
                done = st.event()
                st.record(done, st.comm)
                self.ev_ag[ui] = done
        elif st.cuda:
            with torch.cuda.stream(st.comm):
                st.wait(ev, st.comm)
                dist.all_gather_into_tensor(self.p_full[ui], self.shard(self.p_full, ui), group=self.pg)
                done = st.event()
                st.record(done, st.comm)
                self.ev_ag[ui] = done
        else:
            dist.all_gather_into_tensor(self.p_full[ui], self.shard(self.p_full, ui).clone(), group=self.pg)

    def _reduce_scatter_unit(self, ui):
        wg = self._wg_last if self._wg_on else None   # the unit's weight gradients written on the wgrad stream
        if self.world == 1 and self.replicas > 1:
            # replicas only (no sharding): all-reduce the whole unit across the replicas
            st = self.streams
            if st.cuda:
                ev = st.event()
                st.record(ev)
                with torch.cuda.stream(st.comm):
                    st.wait(ev, st.comm)
                    st.wait(wg, st.comm)
                    dist.all_reduce(self.g_full[ui], op=dist.ReduceOp.SUM, group=self.rpg)
                    self.ops.sumsq_(self.g_full[ui], self.norm_sq, accumulate=self._rs_started)
                    self._rs_started = True
                    done = st.event()
                    st.record(done, st.comm)
                    self.ev_rs[ui] = done
            else:
                dist.all_reduce(self.g_full[ui], op=dist.ReduceOp.SUM, group=self.rpg)
            return
        if self.world == 1:
            st = self.streams
            if st.cuda:
                # N = 1: nothing to reduce; the unit's grad-norm partial is taken now on the side stream, under the rest of the backward
                ev = st.event()
                st.record(ev)
                with torch.cuda.stream(st.opt):
                    st.wait(ev, st.opt)
                    st.wait(wg, st.opt)
                    self.ops.sumsq_(self.g_full[ui], self.norm_sq, accumulate=self._rs_started)
                    self._rs_started = True
                    done = st.event()
                    st.record(done, st.opt)
                    self.ev_rs[ui] = done
            return
        st = self.streams
        ev = st.event()
        st.record(ev)                       # this unit's gradients are complete on the compute stream
        if st.cuda and self.sym is not None:
            # ONE kernel: meets the peers (in-kernel barrier = "unit ui's gradients are complete on every rank"), reduces this rank's
            # slice across all ranks with fp32 accumulation (NVSwitch multimem.ld_reduce, or peer loads in rank order) and writes the
            # bf16 shard in place
            n_shard = self.units[ui].padded // self.world
            with torch.cuda.stream(st.comm):
                st.wait(ev, st.comm)
                st.wait(wg, st.comm)
                self.ops.reducescatter_layer(self.sym.ptr, 1, self._unit_off[ui] * 2, n_shard, self._rs_mode, self._rs_ctas, st.comm.cuda_stream)
                if self.replicas > 1:
                    dist.all_reduce(self.shard(self.g_full, ui), op=dist.ReduceOp.SUM, group=self.rpg)
                self.ops.sumsq_(self.shard(self.g_full, ui), self.norm_sq, accumulate=self._rs_started)
                self._rs_started = True
                done = st.event()
                st.record(done, st.comm)
                self.ev_rs[ui] = done
        elif st.cuda:
            with torch.cuda.stream(st.comm):
                st.wait(ev, st.comm)
                st.wait(wg, st.comm)
                if self._rs32 is not None:
                    # fp32 reduction as the reference's MixedPrecisionPolicy(reduce_dtype=float32): widen, reduce-scatter, ONE rounding
                    n = self.units[ui].padded
                    g32, o32 = self._rs32[:n], self._rs32_out[:n // self.world]
                    g32.copy_(self.g_full[ui])
                    dist.reduce_scatter_tensor(o32, g32, op=dist.ReduceOp.SUM, group=self.pg)
                    if self.replicas > 1:
                        dist.all_reduce(o32, op=dist.ReduceOp.SUM, group=self.rpg)
                    self.shard(self.g_full, ui).copy_(o32)
                else:
                    dist.reduce_scatter_tensor(self.shard(self.g_full, ui), self.g_full[ui], op=dist.ReduceOp.SUM, group=self.pg)
                    if self.replicas > 1:
                        dist.all_reduce(self.shard(self.g_full, ui), op=dist.ReduceOp.SUM, group=self.rpg)
                self.ops.sumsq_(self.shard(self.g_full, ui), self.norm_sq, accumulate=self._rs_started)  # grad-norm partial, off the critical path
                self._rs_started = True
                done = st.event()
                st.record(done, st.comm)
                self.ev_rs[ui] = done
        else:
            wide = self.reduce_dtype == "float32"
            src = self.g_full[ui].float() if wide else self.g_full[ui].clone()
            out = torch.empty(src.numel() // self.world, dtype=src.dtype, device=src.device)
            dist.reduce_scatter_tensor(out, src, op=dist.ReduceOp.SUM, group=self.pg)
            if self.replicas > 1:
                dist.all_reduce(out, op=dist.ReduceOp.SUM, group=self.rpg)
            self.shard(self.g_full, ui).copy_(out)

    def _wait_params(self, ui):
        """Unit ui's parameters are current: its AdamW (side stream) and, with N > 1, its all-gather have completed."""
        if self._is_pooled(ui):
            self._ensure_layer(ui - 1)
            if self.ev_opt[ui] is not None:      # consumed by the gather (communication stream); nothing else reads the shard here
                self.ev_opt[ui] = None
            return
        if self.ev_opt[ui] is not None:
            self.streams.wait(self.ev_opt[ui])
            self.ev_opt[ui] = None
        if self.ev_ag[ui] is not None:
            self.streams.wait(self.ev_ag[ui])
            self.ev_ag[ui] = None

    def close(self):
        """Drain the side streams.  The flat buffers are ordinary caching-allocator blocks owned by the allocating stream: if they were
        released while an optimizer sweep, wgrad GEMM or collective of this engine is still in flight on another stream, the next
        allocation could be handed memory those kernels are about to write."""
        if self.streams.cuda:
            torch.cuda.synchronize(self.device)

    def __del__(self):
        try:
            self.close()
        except Exception as e:  # noqa: BLE001 - a destructor must not raise, but a failed drain (sticky CUDA error) must not vanish either
            import sys
            sys.stderr.write(f"ShardedLlamaEngine.close() failed during destruction: {type(e).__name__}: {e}\n")

    def set_stream_overlap(self, on: bool):
        """Measurement aid: with overlap off every kernel of the step runs back to back on the compute stream (weight-gradient GEMMs and
        the optimizer sweep included), so per-kernel CUDA-event durations are the kernels' own; on = back to the schedule this engine was
        configured with (B200_WGRAD_STREAM / B200_OPT_OVERLAP and their world-size defaults).  Results are identical either way."""
        self.sync_params()
        if self.streams.cuda:
            torch.cuda.synchronize(self.device)
        self._wg_on, self.opt_overlap = self._overlap_cfg if on else (False, False)   # on = the configured schedule, not "everything"

    def sync_params(self):
        """Make the current stream wait for every pending parameter update (state_dict readers, checkpointing)."""
        for ui in range(len(self.units)):
            if self._is_pooled(ui):      # no gather here: just order the current stream behind the shard's AdamW / a gather in flight
                for evs in (self.ev_opt, self.ev_ag):
                    if evs[ui] is not None:
                        self.streams.wait(evs[ui])
                continue
            self._wait_params(ui)

    # ------------------------------------------------------------------ forward + backward of one micro-batch
    def _stage_inputs(self, input_ids, labels, position_ids):
        """Host int64 [b,S] tensors -> pinned int32 staging -> ONE async H2D copy of [ids | labels | pos | cu_seqlens].
        Tensors already on the engine's device (the recipe moves each batch there before calling the model, train_ft.py:1403-1420)
        are converted in place on the device: no host round trip unless the batch is packed (position_ids given), where the number of
        documents and the longest one size the attention grids and must be known on the host."""
        b, S = input_ids.shape
        T = b * S
        if T > self.max_tokens:
            raise ValueError(f"micro-batch of {T} tokens exceeds max_tokens={self.max_tokens}")
        if S > self.cos.shape[0]:
            # the RoPE kernel indexes the cos/sin tables by the position inside the row; the reference regrows its cache instead
            # (rope_utils.py:224-226) - here the tables are sized once, from max_positions / max_position_embeddings
            raise ValueError(f"rows of {S} tokens exceed the RoPE tables ({self.cos.shape[0]} positions): raise max_positions")
        if self.streams.cuda and input_ids.device == self.device:
            k = self._in_idx
            self._in_idx ^= 1
            nseq, max_len = self._fill_input_buffer(self._in_dev[k], input_ids, labels, position_ids)
            return (k, T, nseq, max_len)
        # RoPE rotates by the index inside the row, as the reference's LlamaRotaryEmbedding does (it takes only the length from position_ids,
        # rope_utils.py:212-235); position_ids only delimit the documents of a packed row (cu_seqlens for the varlen attention).
        pos_np = np.tile(np.arange(S, dtype=np.int64), (b, 1))
        cu_np, max_len = cu_seqlens_from_position_ids(pos_np if position_ids is None else position_ids.cpu().numpy())
        nseq = cu_np.size - 1
        k = self._in_idx
        self._in_idx ^= 1
        if self._in_ev[k] is not None:
            self._in_ev[k].synchronize()      # the copy that last used this pinned buffer has completed
        host, devb = self._in_host[k], self._in_dev[k]
        host[0:T].copy_(input_ids.reshape(-1))
        if labels is None:
            host[T:2 * T].fill_(IGNORE_INDEX)
        else:
            host[T:2 * T].copy_(labels.reshape(-1))
        host[2 * T:3 * T].copy_(torch.from_numpy(pos_np).reshape(-1))
        host[3 * T:3 * T + nseq + 1].copy_(torch.from_numpy(cu_np))
        n = 3 * T + nseq + 1
        devb[:n].copy_(host[:n], non_blocking=True)
        self.h2d_bytes += n * 4
        if self.streams.cuda:
            ev = self.streams.event()
            self.streams.record(ev)
            self._in_ev[k] = ev
        return (k, T, nseq, max_len)

    @staticmethod
    def _fill_input_buffer(devb, input_ids, labels, position_ids):
        """[ids | labels | pos | cu_seqlens] (int32) written into `devb` from tensors that already live on its device."""
        b, S = input_ids.shape
        T = b * S
        dev = devb.device
        devb[0:T].copy_(input_ids.reshape(-1))
        if labels is None:
            devb[T:2 * T].fill_(IGNORE_INDEX)
        else:
            devb[T:2 * T].copy_(labels.reshape(-1))
        devb[2 * T:3 * T].view(b, S).copy_(torch.arange(S, dtype=torch.int32, device=dev))     # RoPE positions = index inside the row
        if position_ids is None:
            devb[3 * T:3 * T + b + 1].copy_(torch.arange(0, T + 1, S, dtype=torch.int32, device=dev))
            return b, S
        cu_np, max_len = cu_seqlens_from_position_ids(position_ids.cpu().numpy())
        nseq = cu_np.size - 1
        devb[3 * T:3 * T + nseq + 1].copy_(torch.from_numpy(cu_np).to(dev, non_blocking=True))
        return nseq, max_len

    def stage(self, input_ids, labels, position_ids=None):
        """Copy one micro-batch to the device ahead of time; pass the returned handle to forward_backward(staged=...).
        At most two micro-batches can be resident (two buffer sets)."""
        return self._stage_inputs(input_ids, labels, position_ids)

    def set_labels(self, handle, labels):
        """Replace the labels of a staged micro-batch (the recipe pops `labels` from the batch before calling the model and hands them
        to the loss function instead, train_ft.py:1436-1460)."""
        k, T, _, _ = handle
        lab = labels.reshape(-1)
        if lab.numel() != T:
            raise ValueError(f"labels have {lab.numel()} tokens, the staged micro-batch {T}")
        self._in_dev[k][T:2 * T].copy_(lab.to(torch.int32), non_blocking=True)
        self.h2d_bytes += 0 if lab.device == self.device else T * 4

    def forward_backward(self, input_ids, labels, position_ids, num_label_tokens, first_micro=True, last_micro=True, staged=None):
        """One micro-batch.  Loss (already divided by the GLOBAL label-token count, train_ft.py:1449-1473) accumulates in
        self.loss_dev; parameter gradients (= or +=) land in the flat gradient buffers; on the last micro-batch each unit's
        gradients are reduce-scattered as soon as its backward is done."""
        handle = staged if staged is not None else self._stage_inputs(input_ids, labels, position_ids)
        self.forward_logits(handle)
        self.fused_loss(handle, num_label_tokens)
        self.backward_from_dlogits(handle, first_micro=first_micro, last_micro=last_micro)

    def _views(self, handle):
        k, T, nseq, max_len = handle
        devb = self._in_dev[k]
        return T, nseq, max_len, devb[0:T], devb[T:2 * T], devb[2 * T:3 * T], devb[3 * T:3 * T + nseq + 1]

    def fused_loss(self, handle, num_label_tokens):
        """MaskedCrossEntropy fused with its backward (components/loss/masked_ce.py:73-89): the loss accumulates on the device,
        the logits buffer becomes dlogits in place."""
        T, _, _, _, lab, _, _ = self._views(handle)
        self.ops.ce_fwd_bwd_(self.logits[:T], lab, num_label_tokens, self.loss_dev, accumulate=True, row_loss=self.row_loss[:T])

    def forward_logits(self, handle):
        """Forward of one staged micro-batch up to the bf16 logits [T, V] (a view of the engine's logits buffer); every activation the
        backward needs stays in the arenas."""
        ops, d, A = self.ops, self.dims, self.act
        ctas = self.gemm_ctas

        def G(*a, **k):
            return ops.gemm(*a, max_ctas=ctas, **k)

        T, nseq, max_len, ids, lab, pos, cu = self._views(handle)
        L, Hq, Hkv, D = d.layers, d.heads, d.kv_heads, d.head_dim
        qc, kc = d.q_cols, d.kv_cols
        rba = self.round_before_add
        sl = lambda t: t[:T]

        # ---------------- forward (models/llama/model.py:293-388, 203-234)
        self._wait_params(0)
        ops.embed_fwd(ids, self.P["model.embed_tokens.weight"], out=sl(A["h"][0]))
        for l in range(L):
            self._wait_params(1 + l)
            if self.reshard and l + 1 < L:
                self._ensure_layer(l + 1, prefetch_only=True)     # next layer's all-gather under this layer's compute
            self._layer_forward(l, T, pos, cu, max_len)
            if self.reshard:
                self._release_layer(l)
        self._wait_params(1 + L)
        hL = sl(A["h"][L])
        xf = sl(self.xf)
        ops.rmsnorm_fwd(hL, self.P["model.norm.weight"], d.eps, out=xf, rstd=sl(self.rstdf))
        logits = sl(self.logits)
        G(ops.NT, xf, self.lm_head_w, out=logits)
        return logits

    def _layer_forward(self, l, T, pos, cu, max_len):
        """Decoder layer l: h[l] -> h[l+1] (models/llama/model.py:203-234), every intermediate the backward needs written to the arenas.
        Also the recompute step of activation checkpointing (called again from the backward, when the arenas are shared)."""
        ops, d, A = self.ops, self.dims, self.act
        ctas = self.gemm_ctas

        def G(*a, **k):
            return ops.gemm(*a, max_ctas=ctas, **k)

        Hq, Hkv, D = d.heads, d.kv_heads, d.head_dim
        qc, kc = d.q_cols, d.kv_cols
        rba = self.round_before_add
        sl = lambda t: t[:T]
        W = self.W[l]
        h = sl(A["h"][l])
        x1 = sl(A["x1"][l]); qkv = sl(A["qkv"][l]); o2 = sl(A["o2"][l]); h1 = sl(A["h1"][l])
        x2 = sl(A["x2"][l]); gu = sl(A["gu"][l]); a = sl(A["a"][l])
        ops.rmsnorm_fwd(h, W["n1"], d.eps, out=x1, rstd=sl(A["rstd1"][l]))
        G(ops.NT, x1, W["qkv"], out=qkv)
        if d.qkv_bias:
            ops.bias_rope_(qkv, W["qkv_b"], self.cos, self.sin, pos, Hq + Hkv, Hq + 2 * Hkv, D)
        else:
            ops.rope_(qkv, self.cos, self.sin, pos, Hq + Hkv, D)
        ops.attn_fwd(qkv[:, :qc], qkv[:, qc:qc + kc], qkv[:, qc + kc:], cu, max_len, Hq, Hkv, D, out=o2, lse=A["lse"][l])
        G(ops.NT, o2, W["o"], out=h1, residual=h, round_before_add=rba)
        ops.rmsnorm_fwd(h1, W["n2"], d.eps, out=x2, rstd=sl(A["rstd2"][l]))
        if self._fuse_swiglu and T >= 256 and ctas == 0:
            ops.gemm_swiglu(x2, W["gu"], gu, a)
        else:
            G(ops.NT, x2, W["gu"], out=gu)
            ops.swiglu_fwd(gu, out=a)
        G(ops.NT, a, W["down"], out=sl(A["h"][l + 1]), residual=h1, round_before_add=rba)

    def backward_from_dlogits(self, handle, first_micro=True, last_micro=True):
        """Backward of one staged micro-batch; self.logits[:T] must hold d(loss)/d(logits) in bf16."""
        ops, d, A, tmp = self.ops, self.dims, self.act, self.tmp
        ctas = self.gemm_ctas

        def G(*a, **k):
            return ops.gemm(*a, max_ctas=ctas, **k)

        st = self.streams

        def WG(reads, x, y, out, accumulate=None):
            """Weight-gradient GEMM out (+)= x^T y.  With the wgrad stream on it is issued there, behind an event that marks its inputs
            complete on the compute stream; `reads` names the scratch buffers it reads so their next writer can wait for it."""
            accf = acc if accumulate is None else accumulate
            if not self._wg_on:
                return G(ops.TN, x, y, out=out, residual=out if accf else None)
            ev = st.event()
            st.record(ev)
            with torch.cuda.stream(st.wg):
                st.wait(ev, st.wg)
                G(ops.TN, x, y, out=out, residual=out if accf else None)
                done = st.event()
                st.record(done, st.wg)
            for r in reads:
                self._wg_pending[r] = done
            self._wg_last = done

        def before_write(name):
            ev = self._wg_pending.pop(name, None)
            if ev is not None:
                st.wait(ev)

        T, nseq, max_len, ids, lab, pos, cu = self._views(handle)
        L, Hq, Hkv, D = d.layers, d.heads, d.kv_heads, d.head_dim
        qc, kc = d.q_cols, d.kv_cols
        acc = not first_micro
        # reshard_after_forward: a layer's gradients are produced into a fresh pool slot and reduce-scattered every micro-batch; the
        # accumulation over micro-batches happens on the 1/N gradient shard (the reference's FSDP2 does the same when it reshards)
        lacc = acc and not self.reshard
        if self.reshard:
            self._micro = (first_micro, last_micro)
        if first_micro:
            self._rs_started = False   # a new accumulation window: grad-norm partials of an abandoned backward (no optimizer step) are dropped
        sl = lambda t: t[:T]
        hL, xf, logits = sl(A["h"][L]), sl(self.xf), sl(self.logits)
        if self.ev_opt_all is not None:   # the previous optimizer sweep (side stream) has consumed the gradient buffers / norm
            st.wait(self.ev_opt_all)
            if self._wg_on:
                st.wait(self.ev_opt_all, st.wg)
            self.ev_opt_all = None
        head_ui = 1 + L
        WG((), logits, xf, self.lm_head_g)
        head_wg = self._wg_last if self._wg_on else None   # tied embeddings: the scatter-add at the end of backward accumulates on top of it
        dxf = sl(tmp["dxf"])
        G(ops.NN, logits, self.lm_head_w, out=dxf)
        dh = sl(tmp["dh_a"]); dh_next = sl(tmp["dh_b"])
        dh_name, dh_next_name = "dh_a", "dh_b"
        ops.rmsnorm_bwd(dxf, hL, self.P["model.norm.weight"], sl(self.rstdf), dx=dh, dw=self.G["model.norm.weight"],
                        accumulate_dw=acc, workspace=self.norm_ws)
        if last_micro:
            self._reduce_scatter_unit(head_ui)
        for l in reversed(range(L)):
            W = self.W[l]
            if self.reshard:
                self._ensure_layer(l)                                  # unsharded parameters for the dgrad GEMMs (and the recompute)
                if l > 0:
                    self._ensure_layer(l - 1, prefetch_only=True)      # next layer's all-gather under this layer's backward
                self._before_grad_slot_write(l)
            if self.recompute and l != L - 1:
                # the shared arenas hold layer l+1 (or, for the top layer, already this layer: the forward ended there).  The previous
                # layer's wgrad GEMMs (side stream) still read them: wait, then rebuild layer l's activations from h[l].
                if self._wg_on and self._wg_last is not None:
                    st.wait(self._wg_last)
                self._layer_forward(l, T, pos, cu, max_len)
            h = sl(A["h"][l]); x1 = sl(A["x1"][l]); qkv = sl(A["qkv"][l]); o2 = sl(A["o2"][l]); h1 = sl(A["h1"][l])
            x2 = sl(A["x2"][l]); gu = sl(A["gu"][l]); a = sl(A["a"][l])
            da = sl(tmp["da"]); dgu = sl(tmp["dgu"]); dx = sl(tmp["dx"]); do2 = sl(tmp["do2"]); dqkv = sl(tmp["dqkv"])
            # MLP
            WG((dh_name,), dh, a, W["d_down"], lacc)
            G(ops.NN, dh, W["down"], out=da)
            before_write("dgu")
            ops.swiglu_bwd(da, gu, out=dgu)
            WG(("dgu",), dgu, x2, W["d_gu"], lacc)
            G(ops.NN, dgu, W["gu"], out=dx)
            # dh1 = dh + rmsnorm'(dx2)
            before_write(dh_next_name)
            ops.rmsnorm_bwd(dx, h1, W["n2"], sl(A["rstd2"][l]), dres=dh, dx=dh_next, dw=W["d_n2"], accumulate_dw=lacc, workspace=self.norm_ws)
            dh, dh_next = dh_next, dh
            dh_name, dh_next_name = dh_next_name, dh_name
            # attention
            WG((dh_name,), dh, o2, W["d_o"], lacc)
            G(ops.NN, dh, W["o"], out=do2)
            before_write("dqkv")
            ops.attn_bwd(qkv[:, :qc], qkv[:, qc:qc + kc], qkv[:, qc + kc:], o2, do2, A["lse"][l], cu, max_len, Hq, Hkv, D,
                         dqkv[:, :qc], dqkv[:, qc:qc + kc], dqkv[:, qc + kc:], workspace=self.attn_ws)
            ops.rope_(dqkv, self.cos, self.sin, pos, Hq + Hkv, D, backward=True)
            if d.qkv_bias:
                ops.colsum_(dqkv, W["d_qkv_b"], accumulate=lacc)
            WG(("dqkv",), dqkv, x1, W["d_qkv"], lacc)
            G(ops.NN, dqkv, W["qkv"], out=dx)
            before_write(dh_next_name)
            ops.rmsnorm_bwd(dx, h, W["n1"], sl(A["rstd1"][l]), dres=dh, dx=dh_next, dw=W["d_n1"], accumulate_dw=lacc, workspace=self.norm_ws)
            dh, dh_next = dh_next, dh
            dh_name, dh_next_name = dh_next_name, dh_name
            if self.reshard:
                self._release_layer(l)
                self._reduce_scatter_pooled(1 + l)
            elif last_micro:
                self._reduce_scatter_unit(1 + l)
        if d.tied:
            st.wait(head_wg)       # the lm_head weight gradient (= or += above) is in the shared matrix; the token rows add to it
        elif first_micro:
            self.G["model.embed_tokens.weight"].zero_()
        ops.embed_bwd(ids, dh, self.G["model.embed_tokens.weight"], accumulate=True, workspace=self.embed_ws)
        if last_micro:
            self._reduce_scatter_unit(0)
        self._unsynced = not last_micro
        if self._wg_on and self._wg_last is not None:
            # join: whatever follows on the compute stream (the next forward overwrites the saved activations and the logits buffer the
            # wgrad GEMMs read; gradient accumulation / hooks read the flat gradient buffers) is ordered after the last wgrad GEMM
            st.wait(self._wg_last)
            self._wg_pending.clear()
        self._grads_dirty = True

    # ------------------------------------------------------------------ grad-norm, clip, AdamW, parameter all-gather
    def optimizer_step(self, max_grad_norm: Optional[float] = 1.0, lr: Optional[float] = None):
        """components/training/utils.py:65-171 + train_ft.py:1556-1558 on the flat shards.  Returns the device scalar
        holding the squared global grad norm (sqrt on the host only for logging)."""
        self.compute_grad_norm_sq()
        return self.apply_adamw(max_grad_norm, lr)

    def compute_grad_norm_sq(self):
        """Global squared gradient norm over the (reduce-scattered) shards -> self.norm_sq (device scalar)."""
        ops = self.ops
        nu = len(self.units)
        if self._unsynced:
            # the caller never announced the last micro-batch (recipe without the get_sync_ctx hook, INTEGRATION.md §3): the gradients of
            # every unit are complete but still local - reduce-scatter them now (correct; only the overlap with the backward is lost)
            for ui in reversed(range(nu)):
                if self._is_pooled(ui):
                    # already reduce-scattered after every micro-batch; only the grad-norm partial of the summed shard is missing
                    if self.ev_rs[ui] is not None:
                        self.streams.wait(self.ev_rs[ui])
                        self.ev_rs[ui] = None
                    if self.streams.cuda:     # (the CPU path sums every shard below)
                        ops.sumsq_(self.g_shard[ui], self.norm_sq, accumulate=self._rs_started)
                        self._rs_started = True
                else:
                    self._reduce_scatter_unit(ui)
            self._unsynced = False
        fused_norm = self._rs_started   # the per-unit partials were already accumulated as each unit's gradients completed
        for ui in range(nu):
            if self.ev_rs[ui] is not None:
                self.streams.wait(self.ev_rs[ui])
                self.ev_rs[ui] = None
            if not fused_norm:
                ops.sumsq_(self.shard(self.g_full, ui), self.norm_sq, accumulate=ui > 0)
        if fused_norm:
            self._rs_started = False
        if self.world > 1:
            if not self._sym_allreduce(self.norm_sq):
                dist.all_reduce(self.norm_sq, op=dist.ReduceOp.SUM, group=self.pg)
        return self.norm_sq

    def apply_adamw(self, max_grad_norm: Optional[float] = 1.0, lr: Optional[float] = None):
        """Fused AdamW (+ clip by the norm in self.norm_sq) on every unit shard, then the in-place parameter all-gather."""
        ops = self.ops
        if lr is not None:
            self.lr = lr
        self.step_count += 1
        st = self.streams

        def run():
            for ui in range(len(self.units)):
                ops.adamw_step_(self.shard(self.p_full, ui), self.shard(self.g_full, ui), self.m[ui], self.v[ui], self.lr, self.betas[0],
                                self.betas[1], self.eps, self.wd, self.step_count, max_grad_norm=max_grad_norm or 0.0,
                                grad_norm_sq=self.norm_sq, mode=self.adam_mode, master=None if self.master is None else self.master[ui])
                if st.cuda:
                    ev = st.event()
                    st.record(ev)
                    self.ev_opt[ui] = ev
                if not self._is_pooled(ui):      # pooled layers are gathered on demand, before their next forward / backward
                    self._all_gather_unit(ui)
            if self.reshard:
                self._slot_layer = [None] * self.POOL      # every pool slot now holds parameters of the previous step

        if self.opt_overlap:
            # The HBM-bound optimizer sweep runs on its own stream, unit by unit in forward order: the next step's forward (tensor-bound)
            # starts as soon as the first units are updated and overlaps the rest (per-unit events gate each layer).
            ready = st.event()
            st.record(ready)
            with torch.cuda.stream(st.opt):
                st.wait(ready, st.opt)
                run()
                self.ev_opt_all = st.event()
                st.record(self.ev_opt_all, st.opt)
        else:
            run()
        self._grads_dirty = False
        return self.norm_sq

    def train_step(self, micro_batches, max_grad_norm: Optional[float] = 1.0, num_label_tokens: Optional[int] = None, staged=None):
        """micro_batches: list of dicts with host tensors input_ids / labels [/ position_ids] of shape [b,S].
        staged: optional list of handles from stage() (inputs already resident on the device; needs num_label_tokens).
        Returns (loss, grad_norm) as 0-d device tensors (no host sync here)."""
        if staged is not None:
            assert num_label_tokens is not None
            self.loss_dev.zero_()
            for i, hd in enumerate(staged):
                self.forward_backward(None, None, None, num_label_tokens, first_micro=(i == 0), last_micro=(i == len(staged) - 1), staged=hd)
            nsq = self.optimizer_step(max_grad_norm)
            loss = self._allreduce_dp(self.loss_dev.clone())
            return loss[0], nsq.sqrt()[0]
        if num_label_tokens is None:
            n = sum(int((mb["labels"] != IGNORE_INDEX).sum()) for mb in micro_batches)
            if self.world * self.replicas > 1:
                n = int(self._allreduce_dp(torch.tensor([n], dtype=torch.int64, device=self.device)).item())
            num_label_tokens = n
        self.loss_dev.zero_()
        for i, mb in enumerate(micro_batches):
            self.forward_backward(mb["input_ids"], mb["labels"], mb.get("position_ids"), num_label_tokens,
                                  first_micro=(i == 0), last_micro=(i == len(micro_batches) - 1))
        nsq = self.optimizer_step(max_grad_norm)
        loss = self._allreduce_dp(self.loss_dev.clone())
        return loss[0], nsq.sqrt()[0]

    def _sym_allreduce(self, t):
        """Scalar SUM over the shard group with b200_allreduce_scalars on the communication stream (the stream of the reduce-scatter /
        all-gather kernels: every cross-rank wait of the step then belongs to ONE sequence that is the same on all ranks, and no NCCL kernel
        sits on the step's dependency chain).  Returns False when the symmetric-memory path does not apply."""
        if self.sym is None or not self.streams.cuda or t.dtype != torch.float32 or t.numel() > 16 or not t.is_contiguous():
            return False
        st = self.streams
        ev = st.event()
        st.record(ev)                              # producers of `t` on the current stream
        with torch.cuda.stream(st.comm):
            st.wait(ev, st.comm)
            self.ops.allreduce_scalars_(self.sym.ptr, t, stream=st.comm.cuda_stream)
            done = st.event()
            st.record(done, st.comm)
        st.wait(done)
        return True

    def _allreduce_dp(self, t):
        """SUM over every data-parallel rank: the shard group, then (HSDP) the replica group."""
        if self.world > 1 and not self._sym_allreduce(t):
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.pg)
        if self.replicas > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.rpg)
        return t
