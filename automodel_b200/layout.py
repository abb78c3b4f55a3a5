"""Flat sharded parameter layout of the B200 sharded-DP step.

Replaces the reference's per-parameter DTensor Shard(0) plan
(/root/reference/nemo_automodel/components/distributed/parallelizer.py:137-319, 791-903: one FSDP unit per decoder
layer + a root unit) with contiguous flat bf16 buffers: one per unit, each rank owning the contiguous 1/N slice
[rank*n/N, (rank+1)*n/N).  No padding per parameter, one collective per unit, no copy-in/copy-out: the all-gather
output *is* the unsharded parameter storage and the reduce-scatter input *is* the gradient storage.
Inside a unit the HF parameters are laid out so that fused contractions see one matrix:
    [q_proj; k_proj; v_proj] -> one [(Hq+2Hkv)*d, h] weight,   [gate_proj; up_proj] -> one [2F, h] weight.
HF names/shapes (models/llama/model.py:85-101,162-166) are preserved as views for state_dict / checkpoint export.
"""
from dataclasses import dataclass, field
from typing import List, Tuple

ALIGN = 8  # elements: 16-byte vector / TMA base alignment for bf16


@dataclass
class LlamaDims:
    hidden: int
    ffn: int
    layers: int
    heads: int
    kv_heads: int
    head_dim: int
    vocab: int
    eps: float = 1e-5
    rope_theta: float = 10000.0
    rope_scaling: dict = None
    max_pos: int = 4096
    qkv_bias: bool = False        # Qwen2: q/k/v projections carry a bias (components/models/qwen2/model.py:80-82)
    tied: bool = False            # tie_word_embeddings: lm_head shares model.embed_tokens.weight (Qwen2 <= 1.5B, Llama-3.2-1B/3B)

    @staticmethod
    def from_hf(cfg) -> "LlamaDims":
        g = (lambda k, d=None: cfg.get(k, d)) if isinstance(cfg, dict) else (lambda k, d=None: getattr(cfg, k, d))
        heads = g("num_attention_heads")
        hidden = g("hidden_size")
        mt = g("model_type")
        if mt not in (None, "llama", "mistral", "qwen2"):
            raise ValueError(f"model_type {mt!r}: the B200 sharded step implements the Llama-family decoder (llama, qwen2, and mistral without "
                             "sliding window)")
        if mt == "qwen2":
            # Qwen2Config always carries a sliding_window size; it only applies when use_sliding_window is set (layer_types "sliding_attention")
            if g("use_sliding_window", False) or any(t != "full_attention" for t in (g("layer_types") or [])):
                raise ValueError("sliding-window attention is not supported")
        elif g("sliding_window"):
            raise ValueError("sliding-window attention is not supported")
        if g("hidden_act", "silu") not in (None, "silu"):
            raise ValueError(f"hidden_act {g('hidden_act')!r}: the MLP kernels implement SwiGLU (silu) only")
        if (g("attention_dropout", 0.0) or 0.0) != 0.0:
            raise ValueError("attention_dropout != 0 is not supported")
        if g("mlp_bias", False):
            raise ValueError("mlp_bias is not supported")
        if mt != "qwen2" and g("attention_bias", False):
            raise ValueError("attention_bias (bias on q/k/v AND o_proj) is not supported; Qwen2's q/k/v-only bias is")
        # RoPE base and scaling as the reference resolves them (components/models/llama/rope_utils.py:90-109): transformers >= 5 keeps both
        # in `rope_parameters` ({"rope_theta", "rope_type", "factor", ...}); older configs have `rope_theta` + `rope_scaling`.
        rp = g("rope_parameters")
        if rp:
            theta, scaling = rp.get("rope_theta", 10000.0), dict(rp)
        else:
            theta, scaling = g("rope_theta", 10000.0) or 10000.0, g("rope_scaling")
        if (g("partial_rotary_factor", 1.0) or 1.0) != 1.0:
            raise ValueError("partial_rotary_factor != 1 is not supported")
        return LlamaDims(hidden=hidden, ffn=g("intermediate_size"), layers=g("num_hidden_layers"), heads=heads,
                         kv_heads=g("num_key_value_heads") or heads, head_dim=g("head_dim") or hidden // heads,
                         vocab=g("vocab_size"), eps=g("rms_norm_eps", 1e-5), rope_theta=theta,
                         rope_scaling=scaling, max_pos=g("max_position_embeddings", 4096), qkv_bias=(mt == "qwen2"),
                         tied=bool(g("tie_word_embeddings", False)))

    @property
    def q_cols(self):
        return self.heads * self.head_dim

    @property
    def kv_cols(self):
        return self.kv_heads * self.head_dim

    @property
    def qkv_cols(self):
        return self.q_cols + 2 * self.kv_cols


@dataclass
class ParamSlot:
    name: str           # HF name
    shape: Tuple[int, ...]
    offset: int         # element offset inside the unit's flat buffer

    @property
    def numel(self):
        n = 1
        for s in self.shape:
            n *= s
        return n


@dataclass
class UnitLayout:
    name: str
    slots: List[ParamSlot] = field(default_factory=list)
    numel: int = 0        # un-padded
    padded: int = 0       # multiple of world*ALIGN

    def shard_range(self, rank: int, world: int) -> Tuple[int, int]:
        per = self.padded // world
        return rank * per, (rank + 1) * per


def _mk_unit(name: str, entries: List[Tuple[str, Tuple[int, ...]]], world: int) -> UnitLayout:
    u = UnitLayout(name)
    off = 0
    for pname, shape in entries:
        slot = ParamSlot(pname, tuple(shape), off)
        if slot.numel % ALIGN:
            raise ValueError(f"{pname}: numel {slot.numel} is not a multiple of {ALIGN}")
        u.slots.append(slot)
        off += slot.numel
    u.numel = off
    q = world * ALIGN
    u.padded = (off + q - 1) // q * q
    return u


def build_layout(d: LlamaDims, world: int) -> List[UnitLayout]:
    """Units in forward order: embed, layer 0..L-1, head (final norm + lm_head)."""
    units = [_mk_unit("embed", [("model.embed_tokens.weight", (d.vocab, d.hidden))], world)]
    for l in range(d.layers):
        p = f"model.layers.{l}."
        units.append(_mk_unit(f"layer{l}", [
            (p + "self_attn.q_proj.weight", (d.q_cols, d.hidden)),
            (p + "self_attn.k_proj.weight", (d.kv_cols, d.hidden)),
            (p + "self_attn.v_proj.weight", (d.kv_cols, d.hidden)),
            (p + "self_attn.o_proj.weight", (d.hidden, d.q_cols)),
            (p + "mlp.gate_proj.weight", (d.ffn, d.hidden)),
            (p + "mlp.up_proj.weight", (d.ffn, d.hidden)),
            (p + "mlp.down_proj.weight", (d.hidden, d.ffn)),
            (p + "input_layernorm.weight", (d.hidden,)),
            (p + "post_attention_layernorm.weight", (d.hidden,)),
        ] + ([(p + "self_attn.q_proj.bias", (d.q_cols,)), (p + "self_attn.k_proj.bias", (d.kv_cols,)), (p + "self_attn.v_proj.bias", (d.kv_cols,))]
             if d.qkv_bias else []), world))     # q;k;v biases contiguous: one fused [(Hq+2Hkv)*d] vector
    # tied embeddings: the head unit is the final norm alone; the lm_head GEMMs read / write the embed unit's matrix and gradient
    units.append(_mk_unit("head", [("model.norm.weight", (d.hidden,))] + ([] if d.tied else [("lm_head.weight", (d.vocab, d.hidden))]), world))
    return units


def total_params(units: List[UnitLayout]) -> int:
    return sum(u.numel for u in units)


def memory_plan(d: LlamaDims, world: int, tokens: int, reshard_after_forward: bool = False, activation_checkpointing: bool = False,
                master_weights: bool = False, pool: int = 2) -> dict:
    """Bytes of HBM per rank that ShardedLlamaEngine allocates for a configuration (what its constructor sums up to; no allocation
    here).  Used to decide between the resident layout (every unit's parameters and full-size gradients live for the whole step) and
    reshard_after_forward (layers as 1/N shards + a `pool`-slot buffer pool), and documented for the 70B config in DESIGN.md."""
    units = build_layout(d, world)
    L, h, F, T = d.layers, d.hidden, d.ffn, tokens
    padded = [u.padded for u in units]
    layer = max(padded[1:1 + L]) if L else 0
    root = padded[0] + padded[-1]
    P = sum(padded)
    if reshard_after_forward:
        params = 2 * (root + (P - root) // world + pool * layer)
        grads = 2 * (root + (P - root) // world + pool * layer + layer // world)
    else:
        params = grads = 2 * P
    optim = (2 + 2 + (4 if master_weights else 0)) * (P // world)
    per_layer = 2 * T * (h * 5 + d.qkv_cols + d.q_cols + 3 * F) + 4 * T * (2 + d.heads)      # x1, h1, x2, (h counted below) qkv, o2, gu (2F), a (F); rstd x2, lse
    acts = 2 * T * h * (L + 1) + (per_layer if activation_checkpointing else per_layer * L)
    dq_accs = 2 if min(T, d.max_pos) <= 512 else 1        # attention dQ accumulators (fp32, Hq*D = h): two for sequences of <= 512 tokens
    tmp = 2 * T * (4 * h + 3 * F + d.q_cols + d.qkv_cols) + 2 * T * d.vocab + 4 * T * h * dq_accs     # backward scratch, logits, dQ
    staging = 4 * (max(padded) + max(padded) // world) if world > 1 else 0                   # fp32 reduce staging of the NCCL path
    total = params + grads + optim + acts + tmp + staging
    return {"params": params, "grads": grads, "optimizer": optim, "activations": acts, "scratch_logits": tmp, "fp32_reduce_staging": staging, "total": total}
