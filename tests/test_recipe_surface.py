"""The reference-facing facade (automodel_b200/recipe.py) driven exactly the way the reference recipe drives its model
(recipes/llm/train_ft.py:1357-1473, 1482-1635): model(**batch).logits -> loss_fn(logits, labels, num_label_tokens) ->
(loss * dp).backward() -> clip -> optimizer.step().  Runs on CPU with the stand-in kernels; parity target = the reference fixtures.
The reference's MaskedCrossEntropy is the loss function, restated and pinned to the reference's own outputs
(tests/golden/surface_golden.npz, written by tests/golden/gen_surface_golden.py)."""
import os
import numpy as np
import pytest
import torch

from automodel_b200.recipe import B200ShardedConfig, B200ShardedManager, B200MaskedCrossEntropy, B200FusedAdamW, B200CausalLM
from tests import cpu_kernels
from tests.golden_utils import load, model_cfg, init_params, batches

SURFACE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "surface_golden.npz")


class _TorchMaskedCE(torch.nn.Module):
    """components/loss/masked_ce.py:73-89 restated."""

    def forward(self, logits, labels, mask=None, num_label_tokens=None):
        loss = torch.nn.functional.cross_entropy(logits.view(-1, logits.size(-1)).float(), labels.view(-1), reduction="sum", ignore_index=-100)
        return loss / num_label_tokens


@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
def test_restated_masked_ce_equals_the_reference_golden(dtype):
    """The restatement returns, bit for bit, what the reference's MaskedCrossEntropy returned on the same logits and labels."""
    z = np.load(SURFACE)
    logits = torch.from_numpy(z["ce/logits"]).to(getattr(torch, dtype))
    loss = _TorchMaskedCE()(logits, torch.from_numpy(z["ce/labels"]), num_label_tokens=int(z["ce/num_label_tokens"]))
    assert float(loss) == float(z[f"ce/loss_{dtype}"]), (float(loss), float(z[f"ce/loss_{dtype}"]))


class _Cfg:
    def __init__(self, d):
        self._d = d

    def to_dict(self):
        return dict(self._d)


@pytest.mark.parametrize("loss_kind", ["reference_loss", "fused_loss"])
def test_recipe_loop_over_facade_matches_reference_fixture(loss_kind):
    _run_recipe_loop(loss_kind, torch.device("cpu"), cpu_kernels)


@pytest.mark.gpu
@pytest.mark.parametrize("loss_kind", ["reference_loss", "fused_loss"])
def test_recipe_loop_over_facade_on_gpu(loss_kind):
    """Same loop on the B200 through the real kernels (C ABI)."""
    _run_recipe_loop(loss_kind, torch.device("cuda", 0), None)


def _run_recipe_loop(loss_kind, device, ops):
    z, meta = load("hd128_fp32")          # 2 micro-batches per step: exercises set_requires_gradient_sync / accumulation
    cfg = model_cfg(meta)
    oc = meta["optimizer"]
    mgr = B200ShardedManager(B200ShardedConfig(max_tokens=meta["config"]["lbs"] * meta["config"]["seq"], adam_mode=1), device=device, ops=ops)
    model = mgr.parallelize(_Cfg(cfg))
    assert isinstance(model, B200CausalLM)
    model.engine.load_state_dict(init_params(meta))
    names = [n for n, _ in model.named_parameters()]
    assert "model.layers.1.self_attn.k_proj.weight" in names and len(names) == 2 + 9 * cfg["num_hidden_layers"] + 1
    opt = B200FusedAdamW(model.parameters(), lr=oc["lr"], betas=tuple(oc["betas"]), eps=oc["eps"], weight_decay=oc["weight_decay"]).attach(model)
    if loss_kind == "fused_loss":
        loss_fn = B200MaskedCrossEntropy()
    else:
        loss_fn = _TorchMaskedCE()
    dp = 1
    for s in range(len(meta["loss"])):
        mbs = batches(z, meta, s)
        n = sum(int((b["labels"] != -100).sum()) for b in mbs)
        total = 0.0
        for i, b in enumerate(mbs):
            model.set_requires_gradient_sync(i == len(mbs) - 1)
            labels = torch.from_numpy(b["labels"])
            if loss_kind == "fused_loss":
                out = model(input_ids=torch.from_numpy(b["input_ids"]), labels=labels)
            else:
                out = model(input_ids=torch.from_numpy(b["input_ids"]))
            loss = loss_fn(out.logits, labels.to(out.logits.device), num_label_tokens=n)
            (loss * dp).backward()
            total += float(loss.detach())
        gn = float(model.b200_clip_grad_norm(meta["max_grad_norm"]))
        opt.step(); opt.zero_grad()
        assert abs(total - meta["loss"][s]) < 4e-3, (s, total, meta["loss"][s])
        assert abs(gn - meta["grad_norm"][s]) < 2e-2 * meta["grad_norm"][s], (s, gn, meta["grad_norm"][s])
    # parameters exposed to the recipe are live views of the flat buffers
    p = dict(model.named_parameters())["lm_head.weight"]
    assert p.data_ptr() == model.engine.P["lm_head.weight"].data_ptr()
    assert p.grad.data_ptr() == model.engine.G["lm_head.weight"].data_ptr()


def test_position_ids_are_document_delimiters_only():
    """B200ShardedConfig.packed_sequences: position_ids reach the engine only as document delimiters (None = one document per row)."""
    z, meta = load("hd128_fp32")
    cfg = model_cfg(meta)
    S = meta["config"]["seq"]
    plain = torch.arange(S)[None]
    packed = torch.cat([torch.arange(100), torch.arange(S - 100)])[None]
    for mode, want_plain, want_packed in ((None, True, True), (True, True, True), (False, False, False)):
        mgr = B200ShardedManager(B200ShardedConfig(max_tokens=S, packed_sequences=mode), device=torch.device("cpu"), ops=cpu_kernels)
        model = mgr.parallelize(_Cfg(cfg))
        assert (model._document_position_ids(plain) is not None) == want_plain
        assert (model._document_position_ids(packed) is not None) == want_packed
        assert model._document_position_ids(None) is None
    # and they change the result exactly when they delimit documents
    mgr = B200ShardedManager(B200ShardedConfig(max_tokens=S), device=torch.device("cpu"), ops=cpu_kernels)
    model = mgr.parallelize(_Cfg(cfg))
    model.engine.load_state_dict(init_params(meta))
    ids = torch.from_numpy(batches(z, meta, 0)[0]["input_ids"])
    with torch.no_grad():
        a = model(input_ids=ids).logits.float().clone()
        b = model(input_ids=ids, position_ids=plain).logits.float().clone()
        c = model(input_ids=ids, position_ids=packed).logits.float().clone()
    assert torch.equal(a, b)
    assert torch.equal(a[:, :100], c[:, :100]) and not torch.equal(a[:, 100:], c[:, 100:])


def test_parallelize_rejects_models_it_would_not_train_faithfully():
    """PEFT adapters (extra parameters) and frozen parameters must fail at parallelize time, before any memory is taken."""
    import transformers
    z, meta = load("hd128_fp32")
    c = meta["config"]
    hf_cfg = transformers.LlamaConfig(vocab_size=c["vocab"], hidden_size=c["hidden"], intermediate_size=c["ffn"], num_hidden_layers=c["layers"],
                                      num_attention_heads=c["heads"], num_key_value_heads=c["kv"], max_position_embeddings=c["seq"],
                                      rope_theta=c["theta"], tie_word_embeddings=False)
    mgr = B200ShardedManager(B200ShardedConfig(max_tokens=c["seq"]), device=torch.device("cpu"), ops=cpu_kernels)
    with torch.device("meta"):
        ok = transformers.LlamaForCausalLM(hf_cfg)
    assert isinstance(mgr.parallelize(ok), B200CausalLM)            # a meta model of the right family is accepted (initialised later)
    with torch.device("meta"):
        lora = transformers.LlamaForCausalLM(hf_cfg)
    lora.model.layers[0].self_attn.q_proj.lora_A = torch.nn.Parameter(torch.empty(8, c["hidden"], device="meta"))
    with pytest.raises(NotImplementedError, match="PEFT"):
        mgr.parallelize(lora)
    with torch.device("meta"):
        frozen = transformers.LlamaForCausalLM(hf_cfg)
    frozen.model.embed_tokens.weight.requires_grad_(False)
    with pytest.raises(NotImplementedError, match="frozen"):
        mgr.parallelize(frozen)


def test_fallback_routes_unsupported_models_to_the_reference_manager():
    """With a fallback (what integration.register() installs: the reference's FSDP2Manager over the same mesh) the same rejections
    become a hand-over instead of an error, and the B200 optimizer / loss targets keep working on the foreign model."""
    import transformers
    from automodel_b200.recipe import B200FusedAdamW, B200MaskedCrossEntropy
    z, meta = load("hd128_fp32")
    c = meta["config"]
    hf_cfg = transformers.LlamaConfig(vocab_size=c["vocab"], hidden_size=c["hidden"], intermediate_size=c["ffn"], num_hidden_layers=c["layers"],
                                      num_attention_heads=c["heads"], num_key_value_heads=c["kv"], max_position_embeddings=c["seq"],
                                      rope_theta=c["theta"], tie_word_embeddings=False, attention_bias=True)

    class _RefManager:
        def parallelize(self, model):
            model.handled_by_reference = True
            return model

    mgr = B200ShardedManager(B200ShardedConfig(max_tokens=c["seq"]), device=torch.device("cpu"), ops=cpu_kernels, fallback=_RefManager)
    ref_model = transformers.LlamaForCausalLM(hf_cfg)
    out = mgr.parallelize(ref_model)
    assert out is ref_model and out.handled_by_reference and "attention_bias" in mgr.used_fallback
    opt = B200FusedAdamW(params=out.parameters(), lr=1e-3, betas=(0.9, 0.95), weight_decay=0.1)
    assert type(opt) is torch.optim.AdamW and opt.param_groups[0]["betas"] == (0.9, 0.95)
    logits = torch.randn(2, 8, 32)
    lab = torch.randint(0, 32, (2, 8)); lab[0, :3] = -100
    n = int((lab != -100).sum())
    got = B200MaskedCrossEntropy()(logits=logits, labels=lab, num_label_tokens=n)
    torch.testing.assert_close(got, _TorchMaskedCE()(logits=logits, labels=lab, num_label_tokens=n))


def test_foreign_optimizer_is_detected():
    """torch.optim.AdamW on the facade's parameter views would skip the clip and, sharded, read reduce-scattered buffers: the next
    training forward after a clip that was not followed by B200FusedAdamW.step() fails loudly."""
    z, meta = load("hd128_fp32")
    mgr = B200ShardedManager(B200ShardedConfig(max_tokens=meta["config"]["seq"]), device=torch.device("cpu"), ops=cpu_kernels)
    model = mgr.parallelize(_Cfg(model_cfg(meta)))
    model.engine.load_state_dict(init_params(meta))
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
    b = batches(z, meta, 0)[0]
    ids, lab = torch.from_numpy(b["input_ids"]), torch.from_numpy(b["labels"])
    out = model(input_ids=ids)
    loss = _TorchMaskedCE()(logits=out.logits, labels=lab, num_label_tokens=int((lab != -100).sum()))
    loss.backward()
    model.b200_clip_grad_norm(1.0)
    opt.step()
    with pytest.raises(RuntimeError, match="B200FusedAdamW"):
        model(input_ids=ids)


def test_strategy_config_accepts_an_fsdp2_yaml_and_refuses_what_it_cannot_honour():
    """Every FSDP2Config key is a B200ShardedConfig key (so `_validate_strategy_kwargs`, recipes/_dist_setup.py:44-54, lets an FSDP2 YAML
    through with only `strategy:` changed); keys that would change the computation raise.  FSDP2Config's field names: golden data."""
    import dataclasses
    theirs = set(np.load(SURFACE)["fsdp2_config_fields"].tolist())
    assert len(theirs) == 14 and {"mp_policy", "tp_plan", "defer_fsdp_grad_sync"} <= theirs
    ours = {f.name for f in dataclasses.fields(B200ShardedConfig)}
    assert theirs <= ours, sorted(theirs - ours)
    B200ShardedConfig(defer_fsdp_grad_sync=False, enable_fsdp2_prefetch=True, fsdp2_backward_prefetch_depth=1, backend="gloo")
    for bad in (dict(sequence_parallel=True), dict(enable_compile=True), dict(tp_plan={"a": 1}), dict(offload_policy=object())):
        with pytest.raises(ValueError):
            B200ShardedConfig(**bad)


def test_reduce_dtype_is_honoured_or_refused():
    """FSDP2Config's default MixedPrecisionPolicy reduces gradients in fp32 (components/distributed/config.py:121-132).  The strategy
    config maps `mp_policy.reduce_dtype` / `reduce_dtype` onto the engine's reduction kind (round 1 silently reduced in bf16) and refuses
    what it cannot do."""
    from torch.distributed.fsdp import MixedPrecisionPolicy
    assert B200ShardedConfig().reduce_dtype == "float32"
    assert B200ShardedConfig(mp_policy=MixedPrecisionPolicy(param_dtype=torch.bfloat16, reduce_dtype=torch.float32)).reduce_dtype == "float32"
    assert B200ShardedConfig(mp_policy=MixedPrecisionPolicy(param_dtype=torch.bfloat16, reduce_dtype=torch.bfloat16)).reduce_dtype == "bfloat16"
    assert B200ShardedConfig(reduce_dtype="bf16").reduce_dtype == "bfloat16"
    assert B200ShardedConfig(mp_policy=MixedPrecisionPolicy(reduce_dtype=torch.float32), reduce_dtype="bfloat16").reduce_dtype == "bfloat16"   # explicit key wins
    for bad in (dict(reduce_dtype="float16"), dict(mp_policy=MixedPrecisionPolicy(reduce_dtype=torch.float16)),
                dict(mp_policy=MixedPrecisionPolicy(param_dtype=torch.float32)), dict(mp_policy=MixedPrecisionPolicy(output_dtype=torch.float32)),
                dict(reshard_after_forward=True)):
        with pytest.raises(ValueError):
            B200ShardedConfig(**bad)
    z, meta = load("hd128_fp32")
    for rd in ("float32", "bfloat16"):
        mgr = B200ShardedManager(B200ShardedConfig(max_tokens=meta["config"]["seq"], reduce_dtype=rd, comm="nccl"), device=torch.device("cpu"), ops=cpu_kernels)
        model = mgr.parallelize(_Cfg(model_cfg(meta)))
        assert model.engine.reduce_dtype == rd and model.engine.comm == "nccl"
