"""Drop-in conformance (CPU): the host-side mirror must expose the reference's seams with the same names, keyword arguments
and result keys (SURVEY.md §8b).  What the reference exposes is stored in ``tests/golden/reference_seams.pt``, read from the
reference's own classes by ``tests/golden/make_golden.py seams``."""
import inspect
import os
import sys
import types

import pytest

from tests.conftest import load_golden


@pytest.fixture(scope="module")
def ref():
    return load_golden("reference_seams")


def _params(fn):
    return [(n, p.kind, p.default is not inspect.Parameter.empty) for n, p in inspect.signature(fn).parameters.items() if n != "self"]


def test_dispatcher_methods_match_generic_dispatcher(ref):
    from xtuner_b200.dispatcher import FusedDispatcher

    abstract = ref["dispatcher_abstract"]
    assert abstract == ["combine", "combine_postprocess", "combine_preprocess", "dispatch", "dispatch_postprocess", "dispatch_preprocess"]
    for name in abstract:
        op, tp = _params(getattr(FusedDispatcher, name)), ref["dispatcher_params"][name]
        assert [n for n, _, _ in op] == [n for n, _, _ in tp], (name, op, tp)
        assert all(k == inspect.Parameter.KEYWORD_ONLY for _, k, _ in op), f"{name}: keyword-only like the reference"
    # constructor keywords accepted by build_dispatcher (dispatcher/__init__.py:30-96) for the ep=1 case
    ctor = [n for n, _, _ in _params(FusedDispatcher.__init__)]
    for kw in ("n_routed_experts", "process_group", "training_dtype", "generate_dtype"):
        assert kw in ctor and kw in [n for n, _, _ in ref["dispatcher_init"]]


def test_op_protocol_signatures(ref):
    from xtuner_b200 import ops

    def names(fn):
        return [n for n, p in inspect.signature(fn).parameters.items() if n != "self" and p.kind != inspect.Parameter.KEYWORD_ONLY]

    want = ref["protocol_positional"]
    assert names(ops.group_gemm) == want["group_gemm"]
    assert names(ops.permute) == want["permute"]
    assert names(ops.unpermute) == want["unpermute"]


def test_router_results_keys_and_ctor(ref):
    from xtuner_b200.router import GreedyRouter, NoAuxRouter, RouterResults

    assert sorted(RouterResults.__annotations__) == ref["router_results_keys"]
    assert [n for n, _, _ in _params(GreedyRouter.__init__)] == [n for n, _, _ in ref["greedy_router_init"]]
    assert [n for n, _, _ in _params(NoAuxRouter.__init__)] == [n for n, _, _ in ref["noaux_router_init"]]
    assert [n for n, _, _ in _params(GreedyRouter.forward)] == [n for n, _, _ in ref["greedy_router_forward"]]


def test_ulysses_all_to_all_signature(ref):
    from xtuner_b200.comm import ulysses_all_to_all

    assert list(inspect.signature(ulysses_all_to_all).parameters) == ref["ulysses_all_to_all"]


def test_state_dict_keys_match_reference_modules(ref):
    import torch

    from xtuner_b200.moe import MoELayer

    H, I, E, K = 64, 32, 4, 2
    ours = MoELayer(hidden_size=H, moe_intermediate_size=I, n_routed_experts=E, num_experts_per_tok=K)
    our_keys = {k: v.shape for k, v in ours.state_dict().items()}
    ref_keys = {k: torch.Size(v) for k, v in ref["state_dict_shapes_h64_i32_e4_k2"].items()}
    assert our_keys == ref_keys, (our_keys, ref_keys)
    assert all(isinstance(v, torch.Size) for v in our_keys.values())


def test_install_ulysses_rebinds_mha_global(ref, monkeypatch):
    """``install_ulysses`` rebinds the module global the reference's attention calls; here that module is a stand-in with
    the global the reference module has."""
    from xtuner_b200 import comm, plugin

    name = "xtuner.v1.module.attention.mha"
    assert ref["module_globals"][name] == ["ulysses_all_to_all"]
    mha = types.ModuleType(name)

    def orig(input, scatter_dim, gather_dim, mesh):  # noqa: A002
        raise AssertionError("not called")

    mha.ulysses_all_to_all = orig
    monkeypatch.setitem(sys.modules, name, mha)
    plugin.install_ulysses()
    try:
        assert mha.ulysses_all_to_all is comm.ulysses_all_to_all
    finally:
        plugin.uninstall_ulysses()
    assert mha.ulysses_all_to_all is orig


def test_install_fsdp_comm_on_fully_sharded_module():
    """FSDP2 wiring on CPU (gloo, 1 rank): every FSDPModule gets our comm objects through torch's own setters."""
    import torch
    import torch.distributed as dist
    from torch import nn
    from torch.distributed.device_mesh import init_device_mesh
    from torch.distributed.fsdp import fully_shard

    from xtuner_b200 import comm, plugin

    created = False
    if not dist.is_initialized():
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT="29689", RANK="0", WORLD_SIZE="1", LOCAL_RANK="0")
        dist.init_process_group("gloo", rank=0, world_size=1)
        created = True
    try:
        mesh = init_device_mesh("cpu", (1,))
        model = nn.Sequential(nn.Linear(16, 16), nn.Linear(16, 16))
        for blk in model:
            fully_shard(blk, mesh=mesh)
        fully_shard(model, mesh=mesh)
        n = plugin.install_fsdp_comm(model)
        assert n == 3
        for m in model.modules():
            state = getattr(m, "_get_fsdp_state", None)
            if state is None:
                continue
            pg = m._get_fsdp_state()._fsdp_param_group
            if pg is not None:
                assert isinstance(pg._all_gather_comm, comm.P2PAllGather)
                assert isinstance(pg._reduce_scatter_comm, comm.P2PReduceScatter)
    finally:
        if created:
            dist.destroy_process_group()
