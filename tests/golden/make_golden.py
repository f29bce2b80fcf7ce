"""Generate golden input/output vectors for the MoE hot path by running the REFERENCE'S OWN CODE
(imported from /root/reference through ``ref_shim``) on CPU with seeded inputs.

Run in the authoring container only (the GPU box has no /root/reference):

    python tests/golden/make_golden.py

Outputs: ``tests/golden/*.pt`` (small, committed).  Each fixture is a flat ``dict[str, Tensor|int|float|str]``.
The reference objects exercised are named in each section; nothing here comes from ``oracle/``.
Inputs are tie-free by construction (fp32 logits from a continuous RNG; SURVEY.md §7 "bit-exact routing").
"""
from __future__ import annotations

import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_shim  # noqa: E402

ref_shim.apply_cpu_patches()

from xtuner.v1.module.decoder_layer.moe_decoder_layer import MoEActFnConfig, MoEBlock, MoEGate  # noqa: E402
from xtuner.v1.module.dispatcher.base import NaiveDispatcher  # noqa: E402
from xtuner.v1.module.router.greedy import GreedyRouter, GreedyRouterConfig  # noqa: E402
from xtuner.v1.module.router.noaux_router import NoAuxRouter  # noqa: E402
from xtuner.v1.ops.comm.all_to_all import ulysses_all_to_all  # noqa: E402,F401  (imported to pin the module)
from xtuner.v1.ops.moe.cuda.permute_unpermute import (  # noqa: E402
    cuda_token_permute_torch,
    cuda_token_unpermute_torch,
)


def save(name: str, obj: dict) -> None:
    obj = {k: (v.detach().clone() if isinstance(v, torch.Tensor) else v) for k, v in obj.items()}
    path = os.path.join(HERE, name + ".pt")
    torch.save(obj, path)
    print(f"wrote {path}  ({os.path.getsize(path) / 1024:.1f} KiB)")


def run_naive_dispatcher(disp, hidden_states, topk_ids, topk_weights, experts):
    """Same call sequence as MoEDecoderLayer._forward (moe_decoder_layer.py:411-464)."""
    pre = disp.dispatch_preprocess(hidden_states=hidden_states, topk_ids=topk_ids, topk_weights=topk_weights)
    dis = disp.dispatch(pre_dispatched=pre, topk_weights=topk_weights, decoding=False)
    post = disp.dispatch_postprocess(pre_dispatched=pre, dispatched=dis)
    y = experts(post["hidden_states"], post["tokens_per_expert"])
    prec = disp.combine_preprocess(hidden_states=y, pre_dispatched=pre, dispatched=dis, post_dispatched=post)
    comb = disp.combine(pre_dispatched=pre, dispatched=dis, post_dispatched=post, pre_combined=prec, decoding=False)
    out = disp.combine_postprocess(
        pre_dispatched=pre, dispatched=dis, post_dispatched=post, pre_combined=prec, combined=comb
    )
    return post, y, out["hidden_states"]


# ---------------------------------------------------------------------------------------------
# 1. The reference's only exact KAT on the dispatch path: tests/module/dispatcher/test_noep.py:19-87
#    (run on CPU instead of "cuda"; integers, so device-independent)
# ---------------------------------------------------------------------------------------------
def gen_noep_kat():
    disp = NaiveDispatcher(n_routed_experts=4)
    hidden = torch.arange(4).unsqueeze(1).to(torch.bfloat16).repeat(1, 32)
    topk_ids = torch.tensor([[0, 1], [1, 2], [2, 3], [3, 0]])
    topk_weights = torch.ones_like(topk_ids, dtype=torch.float32)
    target = torch.tensor([[0], [2], [4], [6]]).to(torch.bfloat16).repeat(1, 32)
    post, _, out = run_naive_dispatcher(disp, hidden, topk_ids, topk_weights, lambda h, tpe: h)
    assert torch.equal(out, target), "reference KAT failed on CPU?!"
    save(
        "noep_kat",
        dict(
            hidden_states=hidden,
            topk_ids=topk_ids,
            topk_weights=topk_weights,
            target=target,
            permuted=post["hidden_states"],
            row_id_map=post["row_ids_map"],
            tokens_per_expert=post["tokens_per_expert"],
            out=out,
        ),
    )


# ---------------------------------------------------------------------------------------------
# 2. GreedyRouter (module/router/greedy.py:47-98), softmax + renorm; two geometries
# ---------------------------------------------------------------------------------------------
def gen_greedy_router():
    for tag, (T, E, K, norm, scale, skew) in {
        "c2": (192, 8, 2, True, 1.0, 0.0),  # config-2 geometry (8 experts, top-2)
        "q3": (96, 128, 8, True, 1.0, 0.0),  # Qwen3-30B-A3B real geometry (128 experts, top-8)
        "skew": (160, 8, 2, False, 2.5, 2.0),  # imbalanced, no renorm, scaling factor
    }.items():
        g = torch.Generator().manual_seed(1234 + T)
        logits = torch.randn(T, E, generator=g, dtype=torch.float32) * 2.0
        if skew:
            logits = logits + skew * torch.log(1.0 / torch.arange(1, E + 1, dtype=torch.float32))  # Zipf popularity
        router = GreedyRouterConfig(scoring_func="softmax", router_scaling_factor=scale, norm_topk_prob=norm).build(
            n_routed_experts=E, num_experts_per_tok=K
        )
        assert isinstance(router, GreedyRouter)
        lg = logits.clone().requires_grad_(True)
        out = router(lg)
        # a scalar that touches all three differentiable outputs (Appendix B "three routes")
        gw = torch.randn(T, K, generator=g)
        gr = torch.randn(T, E, generator=g)
        loss = (out["topk_weights"] * gw).sum() + (out["router_weights"] * gr).sum()
        loss.backward()
        save(
            f"greedy_router_{tag}",
            dict(
                logits=logits,
                top_k=K,
                norm_topk_prob=norm,
                router_scaling_factor=scale,
                router_weights=out["router_weights"],
                topk_weights=out["topk_weights"],
                topk_ids=out["topk_ids"],
                tokens_per_expert=out["topkens_per_expert"],
                grad_topk_weights=gw,
                grad_router_weights=gr,
                grad_logits=lg.grad,
            ),
        )


# ---------------------------------------------------------------------------------------------
# 3. NoAuxRouter (module/router/noaux_router.py:50-150), DeepSeek-V3 geometry
# ---------------------------------------------------------------------------------------------
def gen_noaux_router():
    T, E, K, NG, TG, scale = 64, 256, 8, 8, 4, 2.5
    g = torch.Generator().manual_seed(77)
    logits = torch.randn(T, E, generator=g, dtype=torch.float32)
    import xtuner.v1.module.router.noaux_router as _nr

    _nr.get_device = lambda: "cpu"
    router = NoAuxRouter(
        n_routed_experts=E,
        num_experts_per_tok=K,
        router_scaling_factor=scale,
        scoring_func="sigmoid",
        n_group=NG,
        topk_group=TG,
        norm_topk_prob=True,
    )
    bias = torch.randn(E, generator=g) * 0.1
    router.e_score_correction_bias.copy_(bias)
    out = router(logits)
    save(
        "noaux_router_dsv3",
        dict(
            logits=logits,
            e_score_correction_bias=bias,
            top_k=K,
            n_group=NG,
            topk_group=TG,
            router_scaling_factor=scale,
            router_weights=out["router_weights"],
            topk_weights=out["topk_weights"],
            topk_ids=out["topk_ids"],
            tokens_per_expert=out["topkens_per_expert"],
        ),
    )


def gen_noaux_router_bwd():
    """Backward of the reference NoAuxRouter through BOTH differentiable outputs (topk_weights feeds the combine,
    router_weights the balancing loss): grads from the reference's own autograd.  Two cases: group-limited
    (n_group 8 / topk_group 4) and ungrouped (n_group == topk_group, no mask branch, noaux_router.py:91)."""
    import xtuner.v1.module.router.noaux_router as _nr

    _nr.get_device = lambda: "cpu"
    out = {}
    for tag, (T, E, K, NG, TG, scale, norm) in {
        "grouped": (48, 256, 8, 8, 4, 2.5, True),
        "ungrouped": (40, 64, 6, 1, 1, 1.0, True),
        "nonorm": (24, 128, 4, 4, 2, 1.5, False),
    }.items():
        g = torch.Generator().manual_seed(177 + T)
        logits = torch.randn(T, E, generator=g, dtype=torch.float32).requires_grad_(True)
        router = NoAuxRouter(
            n_routed_experts=E, num_experts_per_tok=K, router_scaling_factor=scale, scoring_func="sigmoid",
            n_group=NG, topk_group=TG, norm_topk_prob=norm,
        )
        bias = torch.randn(E, generator=g) * 0.1
        router.e_score_correction_bias.copy_(bias)
        res = router(logits)
        g_tw = torch.randn(T, K, generator=g)
        g_rw = torch.randn(T, E, generator=g)
        (gl_tw,) = torch.autograd.grad(res["topk_weights"], logits, g_tw, retain_graph=True)
        (gl_rw,) = torch.autograd.grad(res["router_weights"], logits, g_rw, retain_graph=True)
        (gl_both,) = torch.autograd.grad([res["topk_weights"], res["router_weights"]], logits, [g_tw, g_rw])
        out[tag] = dict(
            logits=logits.detach(), e_score_correction_bias=bias, top_k=K, n_group=NG, topk_group=TG,
            router_scaling_factor=scale, norm_topk_prob=norm, router_weights=res["router_weights"].detach(),
            topk_weights=res["topk_weights"].detach(), topk_ids=res["topk_ids"], grad_topk_weights=g_tw,
            grad_router_weights=g_rw, grad_logits_from_topk=gl_tw, grad_logits_from_router_weights=gl_rw,
            grad_logits=gl_both,
        )
    save("noaux_router_bwd", out)


# ---------------------------------------------------------------------------------------------
# 4. permute / unpermute with autograd: ops/moe/cuda/permute_unpermute.py:205-248 (in-tree fallbacks,
#    the pinned definition — SURVEY.md §8c "we pin to the in-tree fallback (fp32 accumulate)")
# ---------------------------------------------------------------------------------------------
def gen_dispatch():
    for tag, (T, H, E, K) in {"c2": (96, 64, 8, 2), "k8": (40, 32, 16, 8), "empty_expert": (24, 32, 8, 2)}.items():
        g = torch.Generator().manual_seed(99 + T)
        x = torch.randn(T, H, generator=g).to(torch.bfloat16)
        scores = torch.randn(T, E, generator=g)
        if tag == "empty_expert":
            scores[:, 3] = -1e9  # expert 3 receives nothing
            scores[:, 7] = -1e9
        topk_ids = scores.topk(K, dim=-1)[1]
        probs = torch.rand(T, K, generator=g) + 0.1
        probs = probs / probs.sum(-1, keepdim=True)

        xr = x.clone().requires_grad_(True)
        permuted, row_id_map = cuda_token_permute_torch(xr, topk_ids.to(torch.int32))
        g_perm = torch.randn(T * K, H, generator=g).to(torch.bfloat16)
        (grad_x,) = torch.autograd.grad(permuted, xr, g_perm)

        y = torch.randn(T * K, H, generator=g).to(torch.bfloat16)
        yr = y.clone().requires_grad_(True)
        pr = probs.clone().requires_grad_(True)
        out = cuda_token_unpermute_torch(yr, row_id_map, pr)
        g_out = torch.randn(T, H, generator=g).to(torch.bfloat16)
        grad_y, grad_probs = torch.autograd.grad(out, (yr, pr), g_out)
        out_noprob = cuda_token_unpermute_torch(y, torch.arange(T * K), None)
        save(
            f"dispatch_{tag}",
            dict(
                x=x,
                topk_ids=topk_ids,
                n_experts=E,
                permuted=permuted,
                row_id_map=row_id_map,
                tokens_per_expert=torch.bincount(topk_ids.reshape(-1), minlength=E),
                grad_permuted=g_perm,
                grad_x=grad_x,
                y=y,
                probs=probs,
                out=out,
                grad_out=g_out,
                grad_y=grad_y,
                grad_probs=grad_probs,
                out_noprob_identity=out_noprob,
            ),
        )


# ---------------------------------------------------------------------------------------------
# 5. MoE half of MoEDecoderLayer._forward (moe_decoder_layer.py:392-488) built from the reference's
#    MoEGate (:93-141) + NaiveDispatcher (dispatcher/base.py:222-539) + MoEBlock (:150-200), bf16
#    activations/weights, fp32 gate; forward + backward
# ---------------------------------------------------------------------------------------------
def gen_moe_layer():
    for tag, (T, H, I, E, K) in {"c2_small": (256, 128, 128, 8, 2), "ragged": (77, 128, 128, 4, 2)}.items():
        torch.manual_seed(2024 + T)
        router_cfg = GreedyRouterConfig(scoring_func="softmax", router_scaling_factor=1.0, norm_topk_prob=True)
        gate = MoEGate(hidden_size=H, n_routed_experts=E, num_experts_per_tok=K, router_config=router_cfg)
        experts = MoEBlock(
            hidden_size=H, moe_intermediate_size=I, n_routed_experts=E, moe_act_fn_cfg=MoEActFnConfig()
        )
        disp = NaiveDispatcher(n_routed_experts=E)
        with torch.no_grad():
            gate.weight.normal_(0, 0.5)
            experts.fused_w1w3.weight.normal_(0, H**-0.5)
            experts.fused_w2.weight.normal_(0, I**-0.5)
        # compute-dtype copies as FSDP's MixedPrecisionPolicy(param_dtype=bf16) would hand them over
        gate_w = gate.weight.detach().clone()  # gate runs in fp32 (router_compute_dtype="float32")
        w13 = experts.fused_w1w3.weight.detach().to(torch.bfloat16)
        w2 = experts.fused_w2.weight.detach().to(torch.bfloat16)
        experts.fused_w1w3.weight.data = w13.clone()
        experts.fused_w2.weight.data = w2.clone()

        x = (torch.randn(1, T, H) * 1.0).to(torch.bfloat16)
        residual = torch.randn(1, T, H).to(torch.bfloat16)
        xr = x.clone().requires_grad_(True)

        router_results = gate(xr)
        post, y_perm, combined = run_naive_dispatcher(
            disp,
            xr.view(-1, H),
            router_results["topk_ids"],
            router_results["topk_weights"],
            lambda h, tpe: experts(h, tpe, decoding=False),
        )
        out = combined.view(1, T, H) * 1.0 + residual  # _post_moe_forward :705, hidden_factor = 1.0
        g_out = torch.randn(1, T, H).to(torch.bfloat16)
        grads = torch.autograd.grad(
            out, (xr, gate.weight, experts.fused_w1w3.weight, experts.fused_w2.weight), g_out
        )
        save(
            f"moe_layer_{tag}",
            dict(
                x=x,
                residual=residual,
                gate_weight=gate_w,
                w13=w13,
                w2=w2,
                top_k=K,
                n_experts=E,
                logits=router_results["logits"],
                router_weights=router_results["router_weights"],
                topk_ids=router_results["topk_ids"],
                topk_weights=router_results["topk_weights"],
                tokens_per_expert=post["tokens_per_expert"],
                row_id_map=post["row_ids_map"],
                x_perm=post["hidden_states"],
                y_perm=y_perm,
                combined=combined,
                out=out,
                grad_out=g_out,
                grad_x=grads[0],
                grad_gate_weight=grads[1],
                grad_w13=grads[2],
                grad_w2=grads[3],
            ),
        )


def gen_variants():
    """More corners of the same reference code, in ONE new file (existing fixtures stay byte-identical):
    router — sigmoid scoring with/without renormalisation (greedy.py:73-86); layer — top-4 of 16 experts with
    hidden_factor 0.5 and an un-normalised scaled router (top-4 of 8), and a sigmoid-scored layer."""
    out = {}
    for tag, (T, E, K, scoring, norm, scale) in {
        "router_sigmoid_norm": (100, 8, 2, "sigmoid", True, 1.0),
        "router_sigmoid_raw": (90, 64, 6, "sigmoid", False, 2.0),
        "router_softmax_k1": (70, 8, 1, "softmax", True, 1.0),
    }.items():
        g = torch.Generator().manual_seed(4321 + T)
        logits = torch.randn(T, E, generator=g, dtype=torch.float32) * 1.5
        router = GreedyRouterConfig(scoring_func=scoring, router_scaling_factor=scale, norm_topk_prob=norm).build(
            n_routed_experts=E, num_experts_per_tok=K)
        lg = logits.clone().requires_grad_(True)
        res = router(lg)
        gw = torch.randn(T, K, generator=g)
        gr = torch.randn(T, E, generator=g)
        ((res["topk_weights"] * gw).sum() + (res["router_weights"] * gr).sum()).backward()
        out[tag] = dict(logits=logits, top_k=K, scoring_func=scoring, norm_topk_prob=norm, router_scaling_factor=scale,
                        router_weights=res["router_weights"].detach(), topk_weights=res["topk_weights"].detach(),
                        topk_ids=res["topk_ids"], tokens_per_expert=res["topkens_per_expert"], grad_topk_weights=gw,
                        grad_router_weights=gr, grad_logits=lg.grad)
    for tag, (T, H, I, E, K, scoring, norm, scale, hf) in {
        "layer_k4_hf": (60, 128, 128, 8, 4, "softmax", False, 1.5, 0.5),
        "layer_sigmoid": (40, 128, 128, 4, 2, "sigmoid", True, 1.0, 1.0),
    }.items():
        torch.manual_seed(777 + T)
        router_cfg = GreedyRouterConfig(scoring_func=scoring, router_scaling_factor=scale, norm_topk_prob=norm)
        gate = MoEGate(hidden_size=H, n_routed_experts=E, num_experts_per_tok=K, router_config=router_cfg)
        experts = MoEBlock(hidden_size=H, moe_intermediate_size=I, n_routed_experts=E, moe_act_fn_cfg=MoEActFnConfig())
        disp = NaiveDispatcher(n_routed_experts=E)
        with torch.no_grad():
            gate.weight.normal_(0, 0.5)
            experts.fused_w1w3.weight.normal_(0, H**-0.5)
            experts.fused_w2.weight.normal_(0, I**-0.5)
        gate_w = gate.weight.detach().clone()
        w13 = experts.fused_w1w3.weight.detach().to(torch.bfloat16)
        w2 = experts.fused_w2.weight.detach().to(torch.bfloat16)
        experts.fused_w1w3.weight.data = w13.clone()
        experts.fused_w2.weight.data = w2.clone()
        x = torch.randn(1, T, H).to(torch.bfloat16)
        residual = torch.randn(1, T, H).to(torch.bfloat16)
        xr = x.clone().requires_grad_(True)
        rr = gate(xr)
        post, y_perm, combined = run_naive_dispatcher(
            disp, xr.view(-1, H), rr["topk_ids"], rr["topk_weights"], lambda h, tpe: experts(h, tpe, decoding=False))
        res = combined.view(1, T, H) * hf + residual  # _post_moe_forward :705
        g_out = torch.randn(1, T, H).to(torch.bfloat16)
        grads = torch.autograd.grad(res, (xr, gate.weight, experts.fused_w1w3.weight, experts.fused_w2.weight), g_out)
        out[tag] = dict(x=x, residual=residual, gate_weight=gate_w, w13=w13, w2=w2, top_k=K, n_experts=E,
                        scoring_func=scoring, norm_topk_prob=norm, router_scaling_factor=scale, hidden_factor=hf,
                        logits=rr["logits"].detach(), topk_ids=rr["topk_ids"], topk_weights=rr["topk_weights"].detach(),
                        tokens_per_expert=post["tokens_per_expert"], combined=combined.detach(), out=res.detach(),
                        grad_out=g_out, grad_x=grads[0], grad_gate_weight=grads[1], grad_w13=grads[2], grad_w2=grads[3])
    save("variants", out)


# ---------------------------------------------------------------------------------------------
# 6. ulysses_all_to_all layout (ops/comm/all_to_all.py:6-51) — real collective, gloo, sp=4, spawned
# ---------------------------------------------------------------------------------------------
def _ulysses_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    from torch.distributed.device_mesh import init_device_mesh

    sys.path.insert(0, HERE)
    import ref_shim as _rs

    _rs.import_reference()
    from xtuner.v1.ops.comm.all_to_all import ulysses_all_to_all as a2a

    dist.init_process_group("gloo", rank=rank, world_size=world)
    mesh = init_device_mesh("cpu", (world,))
    g = torch.Generator().manual_seed(500 + rank)
    q_in = torch.randn(1, 8, 6, 4, generator=g)  # [1, Hq, S/sp, D] (mha.py:373)
    o_in = torch.randn(1, 24, 2, 4, generator=g)  # [1, S, Hq/sp, D] (mha.py:421)
    q_out = a2a(q_in, scatter_dim=1, gather_dim=2, mesh=mesh)
    o_out = a2a(o_in, scatter_dim=1, gather_dim=2, mesh=mesh)
    q.put((rank, q_in, q_out, o_in, o_out))
    dist.barrier()
    dist.destroy_process_group()


def gen_ulysses():
    import torch.multiprocessing as mp

    world, port = 4, 29611
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_ulysses_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in range(world)], key=lambda t: t[0])
    for p in procs:
        p.join()
    save(
        "ulysses_a2a_sp4",
        dict(
            sp=world,
            q_in=torch.stack([r[1] for r in res]),
            q_out=torch.stack([r[2] for r in res]),
            o_in=torch.stack([r[3] for r in res]),
            o_out=torch.stack([r[4] for r in res]),
        ),
    )


# ---------------------------------------------------------------------------------------------
# 7. fp8 tile-wise quantisation (float8/fsdp_utils.py:75-116,195-223; triton_kernels/per_tile_quant.py:145-155)
# ---------------------------------------------------------------------------------------------
def gen_fp8():
    from xtuner.v1.float8.fsdp_utils import cast_to_per_block_fp8_with_scales, tensor_to_per_block_fp8_scales
    from xtuner.v1.float8.triton_kernels.per_tile_quant import per_tile_quant_torch

    g = torch.Generator().manual_seed(808)
    w = torch.randn(2, 256, 384, generator=g) * torch.logspace(-3, 1, 384)  # wide dynamic range across blocks
    w[0, :128, :128] = 0.0  # an all-zero block exercises EPS
    scales = tensor_to_per_block_fp8_scales(w)
    q0 = cast_to_per_block_fp8_with_scales(w[0], scales[0])
    q1 = cast_to_per_block_fp8_with_scales(w[1], scales[1])
    x = (torch.randn(48, 512, generator=g) * 3).to(torch.bfloat16)
    x[3] = 0
    x[5, 7] = 1e4  # saturating element inside one tile
    fn = getattr(per_tile_quant_torch, "_torchdynamo_orig_callable", per_tile_quant_torch)
    xq, xs = fn(x)
    save("fp8_quant", dict(w=w, w_scales=scales, w_q=torch.stack([q0, q1]).view(torch.uint8), x=x, x_q=xq.view(torch.uint8),
                           x_scales=xs))


# ---------------------------------------------------------------------------------------------
# 8. the reference's seams the plugin plugs into: signatures, result keys, state-dict layout, module globals the
#    plugin rebinds, and what the fp8 cast functions return (tests/test_dropin_conformance.py,
#    tests/test_plugin_reference_cpu.py)
# ---------------------------------------------------------------------------------------------
def _params(fn):
    import inspect

    return [(n, int(p.kind), p.default is not inspect.Parameter.empty) for n, p in inspect.signature(fn).parameters.items()
            if n != "self"]


def _sha256(t: torch.Tensor) -> str:
    import hashlib

    return hashlib.sha256(t.contiguous().view(torch.uint8).numpy().tobytes()).hexdigest()


def gen_seams():
    import inspect

    import xtuner.v1.float8.fsdp_utils as fu
    import xtuner.v1.module.attention.mha as mha
    import xtuner.v1.module.grouped_linear.moe_group_linear as mgl
    from xtuner.v1.module.dispatcher.base import GenericDispatcher
    from xtuner.v1.module.router.noaux_router import NoAuxRouter as RefNoAux
    from xtuner.v1.module.router.protocol import RouterResults
    from xtuner.v1.ops.comm.all_to_all import ulysses_all_to_all as ref_a2a
    from xtuner.v1.ops.moe.protocol import GroupGemmProtocol, MoePermuteProtocol, MoeUnpermuteProtocol

    def positional(fn):
        return [n for n, p in inspect.signature(fn).parameters.items() if n != "self" and p.kind != inspect.Parameter.KEYWORD_ONLY]

    abstract = sorted(GenericDispatcher.__abstractmethods__)
    out = dict(
        dispatcher_abstract=abstract,
        dispatcher_params={name: _params(getattr(NaiveDispatcher, name)) for name in abstract},
        dispatcher_init=_params(NaiveDispatcher.__init__),
        protocol_positional=dict(group_gemm=positional(GroupGemmProtocol.__call__), permute=positional(MoePermuteProtocol.__call__),
                                 unpermute=positional(MoeUnpermuteProtocol.__call__)),
        router_results_keys=sorted(RouterResults.__annotations__),
        greedy_router_init=_params(GreedyRouter.__init__),
        noaux_router_init=_params(RefNoAux.__init__),
        greedy_router_forward=_params(GreedyRouter.forward),
        ulysses_all_to_all=list(inspect.signature(ref_a2a).parameters),
        module_globals={"xtuner.v1.module.attention.mha": ["ulysses_all_to_all"] if hasattr(mha, "ulysses_all_to_all") else [],
                        "xtuner.v1.module.grouped_linear.moe_group_linear": ["group_gemm"] if hasattr(mgl, "group_gemm") else [],
                        "xtuner.v1.float8.fsdp_utils": [n for n in ("cast_to_per_block_fp8_with_scales", "tensor_to_per_block_fp8_scales")
                                                        if hasattr(fu, n)]},
    )
    H, I, E, K = 64, 32, 4, 2
    gate = MoEGate(hidden_size=H, n_routed_experts=E, num_experts_per_tok=K,
                   router_config=GreedyRouterConfig(scoring_func="softmax", router_scaling_factor=1.0, norm_topk_prob=True))
    experts = MoEBlock(hidden_size=H, moe_intermediate_size=I, n_routed_experts=E, moe_act_fn_cfg=MoEActFnConfig())
    keys = {f"gate.{k}": tuple(v.shape) for k, v in gate.state_dict().items()}
    keys.update({f"experts.{k}": tuple(v.shape) for k, v in experts.state_dict().items()})
    out["state_dict_shapes_h64_i32_e4_k2"] = keys
    # fp8 block scales and casts of seeded weights (the stored scales exactly, the e4m3 casts as sha256 of their bytes)
    g = torch.Generator().manual_seed(5)
    fp8 = {}
    for dtype in (torch.float32, torch.bfloat16):
        w = (torch.randn(3, 256, 384, generator=g) * 2).to(dtype)
        w[0, :128, :128] = 0
        s = fu.tensor_to_per_block_fp8_scales(w)
        fp8[str(dtype)] = dict(scales=s, cast_sha256=[_sha256(fu.cast_to_per_block_fp8_with_scales(w[i], s[i])) for i in range(3)])
    small = torch.randn(64, 256, generator=g)
    s_small = torch.rand(2, 1, generator=g) + 0.5
    fp8["small_cast_sha256"] = _sha256(fu.cast_to_per_block_fp8_with_scales(small, s_small))
    out["fp8"] = fp8
    save("reference_seams", out)


if __name__ == "__main__":
    which = sys.argv[1:] or ["noep", "greedy", "noaux", "noaux_bwd", "dispatch", "layer", "variants", "ulysses", "fp8", "seams"]
    fns = dict(
        noep=gen_noep_kat,
        greedy=gen_greedy_router,
        noaux=gen_noaux_router,
        noaux_bwd=gen_noaux_router_bwd,
        dispatch=gen_dispatch,
        layer=gen_moe_layer,
        variants=gen_variants,
        ulysses=gen_ulysses,
        fp8=gen_fp8,
        seams=gen_seams,
    )
    for w in which:
        fns[w]()
