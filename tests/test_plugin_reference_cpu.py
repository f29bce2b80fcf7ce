"""Engine-level drop-in check on CPU: the reference's OWN Qwen3-style MoE
model (xtuner.v1.model.moe.moe.MoE: embeddings, attention, MoEDecoderLayer, aux losses, lm_head + CE loss) runs a
forward+backward with this package's plugin classes installed by ``xtuner_b200.plugin.convert_model`` — FusedDispatcher,
GreedyRouter, permute/unpermute/group_gemm/swiglu autograd wrappers — and must reproduce the unconverted model's loss and
gradients exactly.  The CUDA kernels cannot run here, so the *raw kernel entry points* (the torch custom ops that call the
C-ABI) are replaced by oracle-backed stand-ins inside this test; everything above them (autograd formulas, protocol
plumbing, dtype/shape conventions, what the reference's layer and losses consume) is the shipped code.

The engine-level tests run the reference's model code and so run only where a reference tree is given
(``XTUNER_REFERENCE_ROOT``).  The last two tests need none: they drive ``plugin`` against stand-ins of the reference modules
it rebinds and compare with what the reference's functions returned (``tests/golden/reference_seams.pt``)."""
import hashlib
import os
import sys
import types

import pytest
import torch
from torch import nn

from tests.conftest import load_golden

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import ref_shim  # noqa: E402

needs_reference = pytest.mark.skipif(not ref_shim.reference_available(),
                                     reason="runs the reference's model code: set XTUNER_REFERENCE_ROOT to a reference tree")


def _install_cpu_kernel_standins(monkeypatch):
    from oracle import moe_oracle as O
    from xtuner_b200 import ops, router

    monkeypatch.setattr(ops, "_require_cuda", lambda *a: None)
    from xtuner_b200 import plugin as _plugin

    monkeypatch.setattr(_plugin, "_gg_eligible", lambda x, w: True)  # host tensors / tiny widths: still route to our op

    def permute_op(input_act, indices, n_experts):
        perm, sorted_idx = O.permute(input_act, indices)
        rmap = torch.empty_like(sorted_idx)
        rmap[sorted_idx] = torch.arange(sorted_idx.numel())
        return perm, rmap.to(torch.int32), sorted_idx, O.tokens_per_expert_hist(indices, n_experts)

    def unpermute_op(input_act, row_id_map, probs, num_tokens, topk):
        gathered = input_act[row_id_map.long()].view(num_tokens, topk, -1)
        if probs is not None:
            return (gathered * probs.unsqueeze(-1)).sum(1).to(input_act.dtype)
        return gathered.float().sum(1).to(input_act.dtype) if topk > 1 else gathered[:, 0]

    def unpermute_bwd_op(grad_out, input_fwd, row_id_map, probs, topk, need_prob_grad):
        T = grad_out.shape[0]
        p = probs if probs is not None else torch.ones(T, topk)
        act = torch.empty_like(input_fwd)
        rows = row_id_map.long().view(T, topk)
        g32 = grad_out.float()
        act[rows.reshape(-1)] = (g32.unsqueeze(1) * p.unsqueeze(-1)).to(input_fwd.dtype).reshape(T * topk, -1)
        pg = (g32.unsqueeze(1) * input_fwd[rows.reshape(-1)].view(T, topk, -1).float()).sum(-1)
        return act, pg

    def gg_nt(x, w, tpe):
        return O.group_gemm(x, w, tpe)

    def gg_nn(dy, w, tpe):
        outs, s = [], 0
        for i, n in enumerate(tpe.tolist()):
            outs.append(dy[s : s + n] @ w[i])
            s += n
        return torch.cat(outs)

    def gg_tn(dy, x, tpe):
        outs, s = [], 0
        for n in tpe.tolist():
            outs.append(dy[s : s + n].T @ x[s : s + n])
            s += n
        return torch.stack(outs)

    def swiglu_op(h):
        return O.swiglu(h)

    def swiglu_bwd_op(g, h):
        with torch.enable_grad():  # called from inside an autograd backward (grad mode is off there)
            hh = h.detach().clone().requires_grad_(True)
            (gh,) = torch.autograd.grad(O.swiglu(hh), hh, g)
        return gh

    def router_op(logits, top_k, scoring, norm, scaling):
        r = O.greedy_router(logits, top_k, norm, scaling, "softmax" if scoring == 0 else "sigmoid")
        return r["router_weights"], r["topk_weights"], r["topk_ids"], r["topk_ids"].to(torch.int32), r["topkens_per_expert"]

    def router_bwd_op(rw, tw, ids, g_tw, g_rw, scoring, norm, scaling):
        # rebuild logits-independent graph: softmax backward needs only rw; use autograd on a surrogate with the same Jacobian
        with torch.enable_grad():
            lg = torch.log(rw.clamp_min(1e-30)).detach().requires_grad_(True)  # softmax(log p) == p
            r = O.greedy_router(lg, tw.shape[1], norm, scaling, "softmax" if scoring == 0 else "sigmoid")
            loss = 0
            if g_tw is not None:
                loss = loss + (r["topk_weights"] * g_tw).sum()
            if g_rw is not None:
                loss = loss + (r["router_weights"] * g_rw).sum()
            (gl,) = torch.autograd.grad(loss, lg)
        return gl

    monkeypatch.setattr(ops, "_permute_op", permute_op)
    monkeypatch.setattr(ops, "_unpermute_op", unpermute_op)
    monkeypatch.setattr(ops, "_unpermute_bwd_op", unpermute_bwd_op)
    monkeypatch.setattr(ops, "_gg_nt", gg_nt)
    monkeypatch.setattr(ops, "_gg_nn", gg_nn)
    monkeypatch.setattr(ops, "_gg_tn", gg_tn)
    monkeypatch.setattr(ops, "_swiglu_op", swiglu_op)
    monkeypatch.setattr(ops, "_swiglu_bwd_op", swiglu_bwd_op)
    monkeypatch.setattr(router, "_router_greedy_op", router_op)
    monkeypatch.setattr(router, "_router_greedy_bwd_op", router_bwd_op)
    def _route_impl(logits, top_k, norm_topk_prob=True, router_scaling_factor=1.0, scoring_func="softmax"):
        if logits.dtype != torch.float32:
            logits = logits.float()
        rw, tw, ids, ids32, tpe = router._GreedyRoute.apply(logits.contiguous(), top_k, router.SCORING[scoring_func], norm_topk_prob,
                                                            router_scaling_factor)
        return {"logits": logits, "router_weights": rw, "topk_weights": tw, "topk_ids": ids, "topkens_per_expert": tpe}, ids32

    monkeypatch.setattr(router, "greedy_route", _route_impl)


def _build_reference_model(seed, noaux=False, hidden=64):
    ref_shim.apply_cpu_patches()
    from xtuner.v1.model.moe.moe import MoE, MoEConfig
    from xtuner.v1.module.attention import MHAConfig
    from xtuner.v1.module.router import GreedyRouterConfig

    if noaux:  # DeepSeek-V3 style layer: sigmoid no-aux router with group-limited top-k, one shared expert
        import xtuner.v1.module.router.noaux_router as _nr
        from xtuner.v1.module.router import NoAuxRouterConfig

        _nr.get_device = lambda: "cpu"
        cfg = MoEConfig(
            vocab_size=512, max_position_embeddings=256, pad_token_id=0, eos_token_id=0, num_hidden_layers=2, hidden_size=64,
            intermediate_size=128, rms_norm_eps=1e-6, rope_theta=1e6, hidden_act="silu",
            attention=MHAConfig(num_attention_heads=4, num_key_value_heads=2, head_dim=16, attn_impl="eager_attention"),
            tie_word_embeddings=False, n_routed_experts=32, n_shared_experts=1, num_experts_per_tok=4, first_k_dense_replace=0,
            hidden_factor=1.0, moe_intermediate_size=32,
            router=NoAuxRouterConfig(scoring_func="sigmoid", router_scaling_factor=2.5, norm_topk_prob=True, n_group=4, topk_group=2),
            compile_cfg=False,
        )
        torch.manual_seed(seed)
        model = MoE(config=cfg)
        model.init_weights()
        with torch.no_grad():
            for m in model.modules():
                if hasattr(m, "e_score_correction_bias"):
                    m.e_score_correction_bias.copy_(torch.randn_like(m.e_score_correction_bias) * 0.05)
        return model.to(torch.bfloat16), cfg
    cfg = MoEConfig(
        vocab_size=512, max_position_embeddings=256, pad_token_id=0, eos_token_id=0, num_hidden_layers=2, hidden_size=hidden,
        intermediate_size=128, rms_norm_eps=1e-6, rope_theta=1e6, hidden_act="silu",
        attention=MHAConfig(num_attention_heads=4, num_key_value_heads=2, head_dim=16, attn_impl="eager_attention"),
        tie_word_embeddings=False, n_routed_experts=8, n_shared_experts=0, num_experts_per_tok=2, first_k_dense_replace=0,
        hidden_factor=1.0, moe_intermediate_size=32,
        router=GreedyRouterConfig(scoring_func="softmax", router_scaling_factor=1.0, norm_topk_prob=True), compile_cfg=False,
    )
    torch.manual_seed(seed)
    model = MoE(config=cfg)
    model.init_weights()
    model = model.to(torch.bfloat16)  # the accelerated path is bf16 (as under FSDP's MixedPrecisionPolicy)
    return model, cfg


def _loss_and_grads(model, cfg):
    from xtuner.v1.loss.ce_loss import CELossConfig
    from xtuner.v1.model.moe.moe import SequenceContext

    torch.manual_seed(123)
    input_ids = torch.randint(0, cfg.vocab_size, (1, 65), dtype=torch.int64)
    seq_ctx = SequenceContext.from_input_ids(input_ids=(input_ids[:, :-1],), device="cpu")
    loss_cfg = CELossConfig()
    lctx = loss_cfg.build(data={"shifted_labels": input_ids[:, 1:]}, sp_mesh=None)
    lctx = loss_cfg.loss_ctx_cls.build_batches([lctx])[0]
    model.zero_grad(set_to_none=True)
    out = model(seq_ctx=seq_ctx, loss_ctx={"lm": lctx})
    fields = {k: getattr(out, k) for k in type(out).model_fields} if hasattr(type(out), "model_fields") else dict(out)
    # TrainEngine._get_total_loss: the sum of every output field whose name contains "loss" (train_engine.py:601-613)
    total = sum(v for k, v in fields.items() if "loss" in k and isinstance(v, torch.Tensor) and v.requires_grad)
    total.backward()
    grads = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}
    return {k: v.detach().clone() for k, v in fields.items() if isinstance(v, torch.Tensor) and v.numel() == 1}, grads


@needs_reference
def test_reference_moe_model_with_plugin_matches_unconverted(monkeypatch):
    import torch.distributed as dist

    if not dist.is_initialized():
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT="29688", RANK="0", WORLD_SIZE="1", LOCAL_RANK="0")
        dist.init_process_group("gloo", rank=0, world_size=1)
    try:
        model, cfg = _build_reference_model(0)
        ref_out, ref_grads = _loss_and_grads(model, cfg)
        assert "loss" in ref_out and torch.isfinite(ref_out["loss"])

        from xtuner_b200 import plugin
        from xtuner_b200.dispatcher import FusedDispatcher

        _install_cpu_kernel_standins(monkeypatch)
        n = plugin.convert_model(model)
        assert n == cfg.num_hidden_layers
        layers = [m for m in model.modules() if hasattr(m, "dispatcher")]
        assert all(isinstance(m.dispatcher, FusedDispatcher) for m in layers)
        our_out, our_grads = _loss_and_grads(model, cfg)
        for k, v in ref_out.items():
            torch.testing.assert_close(our_out[k], v, rtol=1e-6, atol=1e-7, msg=lambda m, k=k: f"{k}: {m}")
        assert set(our_grads) == set(ref_grads)
        for k in ref_grads:
            torch.testing.assert_close(our_grads[k], ref_grads[k], rtol=1e-4, atol=1e-6, msg=lambda m, k=k: f"grad {k}: {m}")
        plugin.restore_model(model)
        back_out, _ = _loss_and_grads(model, cfg)
        assert torch.equal(back_out["loss"], ref_out["loss"])
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()


@needs_reference
def test_reference_moe_model_with_fused_layer_mode(monkeypatch):
    """``convert_model(fused=True)``: the layer's MoE half goes through ``fused.fused_moe_block`` (one autograd node on
    the GPU).  Here that node is an oracle stand-in; what is checked is the glue — which tensors of the reference layer
    are handed over, the returned tuple the reference's MoE model consumes (aux losses included), gradient flow to
    ``post_attention_layernorm.weight`` / ``gate.weight`` / expert weights, and ``restore_model``."""
    import torch.distributed as dist
    from torch.nn import functional as F

    from oracle import moe_oracle as O

    if not dist.is_initialized():
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT="29690", RANK="0", WORLD_SIZE="1", LOCAL_RANK="0")
        dist.init_process_group("gloo", rank=0, world_size=1)
    calls = []

    def fused_block_standin(h, norm_weight, eps, gate_weight, w13, w2, *, top_k, norm_topk_prob=True,
                            router_scaling_factor=1.0, hidden_factor=1.0, scoring_func="softmax"):
        calls.append(tuple(h.shape))
        assert scoring_func == "softmax" and h.dtype == torch.bfloat16
        shape = h.shape
        h2 = h.view(-1, shape[-1])
        x = F.rms_norm(h2, norm_weight.shape, norm_weight, eps)
        r = O.moe_layer_forward(x, gate_weight, w13, w2, top_k, norm_topk_prob, router_scaling_factor, hidden_factor, residual=h2)
        rr = {"logits": r["router.logits"], "router_weights": r["router.router_weights"], "topk_weights": None,
              "topk_ids": r["router.topk_ids"], "topkens_per_expert": r["router.topkens_per_expert"]}
        return r["hidden_states"].view(shape), rr

    try:
        model, cfg = _build_reference_model(0)
        ref_out, ref_grads = _loss_and_grads(model, cfg)

        from xtuner_b200 import fused, plugin

        _install_cpu_kernel_standins(monkeypatch)
        monkeypatch.setattr(fused, "fused_moe_block", fused_block_standin)
        assert plugin.convert_model(model, fused=True) == cfg.num_hidden_layers
        our_out, our_grads = _loss_and_grads(model, cfg)
        assert len(calls) == cfg.num_hidden_layers and calls[0] == (1, 64, cfg.hidden_size)
        for k, v in ref_out.items():
            torch.testing.assert_close(our_out[k], v, rtol=1e-6, atol=1e-7, msg=lambda m, k=k: f"{k}: {m}")
        assert set(our_grads) == set(ref_grads)
        for k in ref_grads:
            torch.testing.assert_close(our_grads[k], ref_grads[k], rtol=1e-4, atol=1e-6, msg=lambda m, k=k: f"grad {k}: {m}")
        plugin.restore_model(model)
        assert not any("_forward" in vars(m) for m in model.modules())
        back_out, _ = _loss_and_grads(model, cfg)
        assert torch.equal(back_out["loss"], ref_out["loss"])
        assert len(calls) == cfg.num_hidden_layers  # restored model no longer reaches the fused node
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()


def _install_emulated_cabi(monkeypatch):
    """Keep the shipped custom ops (``ops.py`` / ``router.py`` bodies: buffer allocation, argument order) and emulate
    only the library underneath them in host memory."""
    from tests.cabi_emulator import EmulatedLib
    from xtuner_b200 import _capi, ops, router

    lib = EmulatedLib(_capi.load())
    monkeypatch.setattr(_capi, "ensure_init", lambda: lib)
    for mod in (ops, router):
        monkeypatch.setattr(mod, "current_stream", lambda: None)
    monkeypatch.setattr(ops, "_require_cuda", lambda *a: None)
    monkeypatch.setattr(ops, "permute_workspace", lambda T, K, E, dev: torch.zeros(int(lib.xtb_moe_permute_workspace_bytes(T, K, E)), dtype=torch.uint8))
    monkeypatch.setattr(ops, "_scratch", lambda tag, n, dev: torch.empty(max(int(n), 16), dtype=torch.uint8))
    import functools

    monkeypatch.setattr(router, "greedy_route", functools.partial(_greedy_route_nocheck, router))  # minus the is_cuda guard
    from xtuner_b200 import plugin

    monkeypatch.setattr(plugin, "_gg_eligible", lambda x, w: True)  # host tensors / tiny widths: still route to our op
    return lib


def _greedy_route_nocheck(router, logits, top_k, norm_topk_prob=True, router_scaling_factor=1.0, scoring_func="softmax"):
    if logits.dtype != torch.float32:
        logits = logits.float()
    rw, tw, ids, ids32, tpe = router._GreedyRoute.apply(logits.contiguous(), top_k, router.SCORING[scoring_func], norm_topk_prob,
                                                        router_scaling_factor)
    return {"logits": logits, "router_weights": rw, "topk_weights": tw, "topk_ids": ids, "topkens_per_expert": tpe}, ids32


@needs_reference
def test_reference_moe_model_with_plugin_through_emulated_cabi(monkeypatch):
    """Same engine-level check, one level lower: the shipped custom-op bodies run and only the C-ABI is emulated."""
    import torch.distributed as dist

    if not dist.is_initialized():
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT="29691", RANK="0", WORLD_SIZE="1", LOCAL_RANK="0")
        dist.init_process_group("gloo", rank=0, world_size=1)
    try:
        model, cfg = _build_reference_model(0)
        ref_out, ref_grads = _loss_and_grads(model, cfg)
        from xtuner_b200 import plugin

        lib = _install_emulated_cabi(monkeypatch)
        assert plugin.convert_model(model) == cfg.num_hidden_layers
        our_out, our_grads = _loss_and_grads(model, cfg)
        for name in ("xtb_router_greedy", "xtb_moe_permute", "xtb_group_gemm_nt", "xtb_swiglu", "xtb_moe_unpermute",
                     "xtb_moe_unpermute_bwd", "xtb_group_gemm_nn", "xtb_group_gemm_tn", "xtb_swiglu_bwd", "xtb_router_greedy_bwd"):
            assert name in lib.calls, f"{name} was not reached"
        for k, v in ref_out.items():
            torch.testing.assert_close(our_out[k], v, rtol=1e-6, atol=1e-7, msg=lambda m, k=k: f"{k}: {m}")
        assert set(our_grads) == set(ref_grads)
        for k in ref_grads:
            torch.testing.assert_close(our_grads[k], ref_grads[k], rtol=1e-4, atol=1e-6, msg=lambda m, k=k: f"grad {k}: {m}")
        plugin.restore_model(model)
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()


@needs_reference
def test_reference_deepseek_style_model_with_plugin_through_emulated_cabi(monkeypatch):
    """Row a2' at engine level: the reference's MoE model with NoAuxRouterConfig (sigmoid, group-limited top-k, bias) and
    a shared expert, converted by the plugin (NoAuxRouter incl. its new backward, FusedDispatcher, grouped GEMM ops) with
    the C-ABI emulated, reproduces the unconverted model's losses and gradients."""
    import torch.distributed as dist

    if not dist.is_initialized():
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT="29692", RANK="0", WORLD_SIZE="1", LOCAL_RANK="0")
        dist.init_process_group("gloo", rank=0, world_size=1)
    try:
        model, cfg = _build_reference_model(1, noaux=True)
        ref_out, ref_grads = _loss_and_grads(model, cfg)
        assert torch.isfinite(ref_out["loss"])
        from xtuner_b200 import plugin, router

        lib = _install_emulated_cabi(monkeypatch)
        monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))  # NoAuxRouter.forward's guard
        assert plugin.convert_model(model) == cfg.num_hidden_layers
        assert all(isinstance(m.gate.router, router.NoAuxRouter) for m in model.modules() if hasattr(m, "dispatcher"))
        our_out, our_grads = _loss_and_grads(model, cfg)
        assert "xtb_router_noaux" in lib.calls and "xtb_router_noaux_bwd" in lib.calls
        for k, v in ref_out.items():
            torch.testing.assert_close(our_out[k], v, rtol=1e-5, atol=1e-6, msg=lambda m, k=k: f"{k}: {m}")
        assert set(our_grads) == set(ref_grads)
        for k in ref_grads:
            torch.testing.assert_close(our_grads[k], ref_grads[k], rtol=2e-3, atol=2e-5, msg=lambda m, k=k: f"grad {k}: {m}")
        plugin.restore_model(model)
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()


@needs_reference
def test_reference_moe_model_fused_mode_through_emulated_cabi(monkeypatch):
    """``convert_model(fused=True)`` with the REAL fused node (``fused.FusedMoEBlockFunction``: RMSNorm + gate + route +
    dispatch + experts + combine + residual, and its hand-written backward chain) over the emulated C-ABI, inside the
    reference's own model: losses and every parameter gradient against the unconverted model."""
    import torch.distributed as dist

    if not dist.is_initialized():
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT="29693", RANK="0", WORLD_SIZE="1", LOCAL_RANK="0")
        dist.init_process_group("gloo", rank=0, world_size=1)
    try:
        model, cfg = _build_reference_model(0, hidden=256)  # a width the fused norm kernels support
        ref_out, ref_grads = _loss_and_grads(model, cfg)
        from xtuner_b200 import fused, plugin

        lib = _install_emulated_cabi(monkeypatch)
        monkeypatch.setattr(fused, "current_stream", lambda: None)
        monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))  # fused_moe_block's guard
        assert plugin.convert_model(model, fused=True) == cfg.num_hidden_layers
        our_out, our_grads = _loss_and_grads(model, cfg)
        assert lib.calls.count("xtb_rmsnorm_gate") == cfg.num_hidden_layers and "xtb_moe_dispatch_bwd_rmsnorm" in lib.calls
        for k, v in ref_out.items():
            torch.testing.assert_close(our_out[k], v, rtol=2e-4, atol=1e-5, msg=lambda m, k=k: f"{k}: {m}")
        assert set(our_grads) == set(ref_grads)
        for k in ref_grads:
            a, b = our_grads[k].float(), ref_grads[k].float()
            bad = ((a - b).abs() > 3e-2 * (b.abs() + b.abs().mean())).float().mean()
            assert bad < 5e-3, f"grad {k}: {bad:.4f} of elements off"
        plugin.restore_model(model)
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()



class NaiveDispatcher:
    """Stand-in for the reference's ep=1 dispatcher: ``convert_model`` recognises it by name and reads these attributes."""

    def __init__(self, n_routed_experts):
        self._n_routed_experts, self._process_group = n_routed_experts, None
        self._training_dtype = self._generate_dtype = "bf16"


class GreedyRouter(nn.Module):
    """Stand-in for the reference's GreedyRouter (recognised by name; the attributes ``_convert_router`` copies)."""

    def __init__(self, n_routed_experts, top_k):
        super().__init__()
        self.n_routed_experts, self.top_k, self.norm_topk_prob = n_routed_experts, top_k, True
        self.scoring_func, self.router_scaling_factor = "softmax", 1.0


def _standin_moe_model(n_layers=2, E=8, K=2):
    """Modules laid out like the reference's MoE decoder layers where ``convert_model`` looks: a ``dispatcher`` attribute
    and ``gate`` (holding ``router``) / ``experts`` sub-modules."""
    layers = nn.ModuleList()
    for _ in range(n_layers):
        layer = nn.Module()
        layer.dispatcher = NaiveDispatcher(E)
        layer.gate = nn.Module()
        layer.gate.router = GreedyRouter(E, K)
        layer.experts = nn.Module()
        layers.append(layer)
    return layers


def _standin_module(monkeypatch, ref, name, **globals_):
    """A stand-in of the reference module ``name`` carrying the globals the reference module has."""
    assert sorted(ref["module_globals"][name]) == sorted(globals_)
    mod = types.ModuleType(name)
    for k, v in globals_.items():
        setattr(mod, k, v)
    monkeypatch.setitem(sys.modules, name, mod)
    return mod


def test_convert_model_leaves_unsupported_layers_whole_and_group_gemm_falls_back(monkeypatch):
    """ADVICE r1: (1) a layer whose router has no counterpart must not be half-converted (dispatcher swapped, router not);
    (2) the process-wide ``group_gemm`` rebind must hand inputs our kernels do not cover back to the reference's op."""
    from xtuner_b200 import plugin
    from xtuner_b200.dispatcher import FusedDispatcher
    from xtuner_b200.router import GreedyRouter as OurGreedyRouter

    ref = load_golden("reference_seams")
    calls = []

    def ref_group_gemm(x, w, tpe):  # the reference's op as GroupGemmProtocol describes it: one product per expert
        calls.append(tuple(x.shape))
        return torch.cat([a @ w[i].T for i, a in enumerate(x.split(tpe.tolist()))])

    mgl = _standin_module(monkeypatch, ref, "xtuner.v1.module.grouped_linear.moe_group_linear", group_gemm=ref_group_gemm)
    model = _standin_moe_model()
    layers = [m for m in model.modules() if hasattr(m, "dispatcher")]

    class GreedyGroupedRouter(GreedyRouter):  # a router class the plugin does not know
        pass

    layers[0].gate.router.__class__ = GreedyGroupedRouter
    before = [(m.dispatcher, m.gate.router) for m in layers]
    assert plugin.convert_model(model) == len(layers) - 1
    assert layers[0].dispatcher is before[0][0] and layers[0].gate.router is before[0][1]
    assert not hasattr(layers[0], plugin._SAVED)
    assert isinstance(layers[1].dispatcher, FusedDispatcher) and isinstance(layers[1].gate.router, OurGreedyRouter)
    original = getattr(mgl, plugin._SAVED)
    assert original is ref_group_gemm
    x = torch.randn(6, 64).to(torch.bfloat16)  # CPU, width 64: not eligible -> the reference's own op answers
    w = torch.randn(2, 32, 64).to(torch.bfloat16)
    tpe = torch.tensor([2, 4])
    assert torch.equal(mgl.group_gemm(x, w, tpe), original(x, w, tpe))
    assert calls == [(6, 64), (6, 64)]
    plugin.restore_model(model)
    assert mgl.group_gemm is original
    assert layers[1].dispatcher is before[1][0] and layers[1].gate.router is before[1][1]


def test_fp8_cast_rebind_matches_the_reference_functions(monkeypatch):
    """``plugin.install_fp8_cast()``: the reference's ``cast_to_per_block_fp8_with_scales`` / ``tensor_to_per_block_fp8_scales``
    (float8/fsdp_utils.py:75-116,196-223 — what ``fsdp_pre_all_gather`` calls on the local shard) routed through the shipped
    wrappers (``ops.fp8_block_cast`` / ``ops.fp8_block_scales``: shape checks, buffer allocation, argument order) over the
    host-memory emulation of the C-ABI must return the reference's own bits (its scales, and the sha256 of its casts, as
    stored from the reference); shapes the kernels do not take (shard rows % 128 == 64, fewer than 128 rows) must stay on
    the reference's code."""
    from xtuner_b200 import plugin

    ref = load_golden("reference_seams")
    want = ref["fp8"]
    fallback = []

    def ref_cast(tensor, scales, block_size=128, float8_dtype=torch.float8_e4m3fn):
        fallback.append("cast")
        return torch.zeros(tensor.shape, dtype=float8_dtype)

    def ref_scales(tensor, reduce_mesh=None, float8_dtype=torch.float8_e4m3fn, block_size=128):
        fallback.append("scales")
        return torch.ones(1)

    fu = _standin_module(monkeypatch, ref, "xtuner.v1.float8.fsdp_utils", cast_to_per_block_fp8_with_scales=ref_cast,
                         tensor_to_per_block_fp8_scales=ref_scales)
    lib = _install_emulated_cabi(monkeypatch)
    monkeypatch.setattr(plugin, "_on_device", lambda t: True)  # host tensors: the eligibility predicate's only device question
    plugin.install_fp8_cast()
    try:
        g = torch.Generator().manual_seed(5)  # the inputs the stored reference results were computed from
        for dtype in (torch.float32, torch.bfloat16):
            w = (torch.randn(3, 256, 384, generator=g) * 2).to(dtype)
            w[0, :128, :128] = 0  # an all-zero block: scale = EPS / 448
            want_s = want[str(dtype)]["scales"]
            got_s = fu.tensor_to_per_block_fp8_scales(w)
            assert torch.equal(got_s, want_s) and got_s.shape == (3, 2, 3)
            for i in range(3):
                got = fu.cast_to_per_block_fp8_with_scales(w[i], want_s[i])
                assert got.dtype == torch.float8_e4m3fn
                assert hashlib.sha256(got.view(torch.uint8).numpy().tobytes()).hexdigest() == want[str(dtype)]["cast_sha256"][i]
        n_ours = len(lib.calls)
        assert lib.calls.count("xtb_fp8_block_cast") == 6 and lib.calls.count("xtb_fp8_block_scales") == 2
        assert fallback == []
        # shapes outside the kernels' domain stay on the reference path (no library call)
        small = torch.randn(64, 256, generator=g)
        s_small = torch.rand(2, 1, generator=g) + 0.5
        fu.cast_to_per_block_fp8_with_scales(small, s_small)
        assert fallback == ["cast"] and len(lib.calls) == n_ours
    finally:
        plugin.uninstall_fp8_cast()
    assert fu.cast_to_per_block_fp8_with_scales is ref_cast and fu.tensor_to_per_block_fp8_scales is ref_scales
