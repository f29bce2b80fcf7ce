"""CPU checks of bench.py's pure parts: work model, profile post-processing (roofline objects) and the reference arm."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_layer_work_matches_baseline_md():
    import bench

    w = bench.layer_work(8192, 2048, 768, 8, 2)
    assert w["dispatch_bytes_fwd"] == 8192 * 2048 * 2 * 3 + 8192 * 2 * 8  # BASELINE.md §5: 100.8 MB
    assert abs(w["dispatch_bytes_fwd"] / 1e6 - 100.8) < 0.1
    assert abs(w["gemm_flops_fwd"] / 1e9 - 154.6) < 0.1 and abs(w["gemm_flops_fwd_bwd"] / 1e9 - 463.9) < 0.1
    assert abs(w["unpermute_bwd_bytes"] / 1e6 - 167.8) < 0.1


def test_summarize_profile_rooflines():
    import bench

    cfg = dict(bench.C2)
    # one layer-step worth of fake event times (ms)
    prof = [("xtb_group_gemm_nt_swiglu", 0.105), ("xtb_group_gemm_nt", 0.056), ("xtb_group_gemm_nn", 0.050),
            ("xtb_group_gemm_nn", 0.090), ("xtb_group_gemm_tn", 0.052), ("xtb_group_gemm_tn", 0.095),
            ("xtb_moe_permute_prepared", 0.021), ("xtb_router_greedy_dispatch", 0.0127), ("xtb_moe_combine", 0.029),
            ("xtb_swiglu_bwd", 0.029)]
    roof, disp, kus = bench.summarize_profile(prof, cfg, L=48, ms_step=32.0, n_prof_layer_steps=1)
    gemm_ms = 0.105 + 0.056 + 0.05 + 0.09 + 0.052 + 0.095
    assert abs(roof["achieved"] - 463.856467968e9 / (gemm_ms * 1e-3) / 1e12) < 1e-6
    assert roof["bound"] == "tensor" and roof["unit"] == "TFLOP/s" and 0 < roof["frac"] < 1.2
    assert abs(roof["share_of_step"] - gemm_ms * 48 / 32.0) < 1e-9
    assert disp["bound"] == "hbm" and disp["unit"] == "GB/s"
    assert abs(disp["gather_only_GBs"] - 100794368 / 0.021e-3 / 1e9) < 1e-3
    assert kus["xtb_group_gemm_nn"] == 70.0 and kus["xtb_moe_combine"] == 29.0
    json.dumps({"roofline": roof, "roofline_dispatch": disp})  # serialisable
    if os.path.exists(os.path.join(ROOT, "profiles", "ncu_traffic.json")):
        assert roof["traffic"] and roof["traffic"] > 5e7
        assert disp["traffic"]["gather"] and disp["traffic"]["combine"]


def test_dispatch_roofline_with_fused_gate_route():
    """With the one-launch gate+router+bucketing the whole kernel is charged to the dispatch and the gate's bytes are
    added to the numerator (no free lunch in the figure)."""
    import bench

    cfg = dict(bench.C2)
    T, H, E = cfg["T"], cfg["H"], cfg["E"]
    base = [("xtb_group_gemm_nt", 0.056), ("xtb_moe_permute_prepared", 0.021), ("xtb_moe_combine", 0.029)]
    _, two, _ = bench.summarize_profile(base + [("xtb_gate_logits", 0.022), ("xtb_router_greedy_dispatch", 0.0127)], cfg, 48, 32.0, 1)
    _, one, _ = bench.summarize_profile(base + [("xtb_gate_route_dispatch", 0.010)], cfg, 48, 32.0, 1)
    assert one["bytes_route_plus_dispatch"] == two["bytes_route_plus_dispatch"] + T * H * 2 + E * H * 4
    assert one["route_us"] == 10.0 and two["route_us"] == 12.7
    assert "xtb_gate_route_dispatch" in one["kernel"] and one["route_plus_dispatch_GBs"] > two["route_plus_dispatch_GBs"]


def test_kernel_table_models():
    import bench

    cfg = dict(bench.C2)
    T, H, I, E, K = (cfg[k] for k in "THIEK")
    M = T * K
    # two profiled layer-steps of the block path (ms per call)
    one = [("xtb_rmsnorm_gate", 0.020), ("xtb_gate_logits", 0.022), ("xtb_router_greedy_dispatch", 0.0127),
           ("xtb_moe_permute_prepared", 0.021), ("xtb_group_gemm_nt_swiglu", 0.105), ("xtb_group_gemm_nt", 0.056),
           ("xtb_moe_combine", 0.029), ("xtb_moe_unpermute_bwd", 0.039), ("xtb_group_gemm_tn", 0.060),
           ("xtb_group_gemm_nn", 0.052), ("xtb_swiglu_bwd", 0.029), ("xtb_group_gemm_tn", 0.094), ("xtb_group_gemm_nn", 0.090),
           ("xtb_router_greedy_bwd", 0.0097), ("xtb_gate_logits_bwd", 0.036), ("xtb_moe_dispatch_bwd_rmsnorm", 0.055)]
    rows = {r["entry"]: r for r in bench.kernel_table(one + one, cfg, hbm_peak=6490.0, tf_peak=1471.0)}
    assert rows["xtb_group_gemm_nn"]["calls_per_layer"] == 2 and rows["xtb_group_gemm_nn"]["us_per_layer"] == 142.0
    assert rows["xtb_group_gemm_nn"]["flops_per_layer"] == 2 * M * H * I + 2 * M * 2 * I * H
    assert abs(rows["xtb_group_gemm_nt_swiglu"]["achieved_TFLOPs"] - 2 * M * 2 * I * H / 105e-6 / 1e12) < 0.1
    assert rows["xtb_moe_permute_prepared"]["bytes_per_layer"] == 100794368
    assert abs(rows["xtb_moe_permute_prepared"]["frac"] - 100794368 / 21e-6 / 1e9 / 6490.0) < 1e-3
    assert rows["xtb_moe_dispatch_bwd_rmsnorm"]["bound"] == "hbm" and 0.5 < rows["xtb_moe_dispatch_bwd_rmsnorm"]["frac"] < 0.8
    assert rows["xtb_moe_combine"]["bytes_per_layer"] == T * H * 2 * (K + 1) + T * K * 8 + T * H * 2
    flops_total = sum(r["flops_per_layer"] for r in rows.values() if r.get("bound") == "tensor")
    assert flops_total == bench.layer_work(T, H, I, E, K)["gemm_flops_fwd_bwd"]
    json.dumps(list(rows.values()))
    assert bench.kernel_table([], cfg) == []


def test_reference_arm_prints_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--cpu-sample-tokens", "256", "--layers", "48"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["value"] > 0 and d["cpu_baseline"]["kind"] == "port"
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    # under torchrun only rank 0 prints; other ranks exit 0 without work
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r2 = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True,
                        text=True, timeout=120, cwd=ROOT, env=env)
    assert r2.returncode == 0 and r2.stdout.strip() == ""


def test_dump_outputs_budget_and_fixed_sample(tmp_path, monkeypatch):
    """``--dump-outputs``: float32 files, the whole set within the byte budget, arrays above their share sampled at the
    same positions on every call (two builds dumped with the same arguments compare element for element)."""
    import numpy as np
    import torch

    import bench

    monkeypatch.setattr(bench, "DUMP_BYTES", 3 * 4 * 1000)  # three arrays: 1000 elements each at most
    g = torch.Generator().manual_seed(0)
    arrays = {"loss": torch.tensor(2.5), "small": torch.randn(10, 20, generator=g).to(torch.bfloat16),
              "big": torch.randn(300, 70, generator=g)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    total = 0
    for name, t in arrays.items():
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, b)
        total += a.nbytes
        if t.numel() <= 1000:
            assert a.shape == tuple(t.shape) and np.array_equal(a, t.float().numpy())
        else:
            assert a.shape == (1000,) and np.isin(a, t.numpy().reshape(-1)).all()
    assert total <= bench.DUMP_BYTES


def test_bench_rejects_zero_steps_and_dump_of_the_cpu_arm():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120,
                           cwd=ROOT)
        assert r.returncode == 2 and "error" in r.stderr, (extra, r.stderr[-500:])
