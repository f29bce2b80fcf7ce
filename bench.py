#!/usr/bin/env python
"""bench.py — throughput of the MoE hot path (BASELINE.json north_star) on B200.

A *step* is one pass of the hot path over one batch of synthetic input: forward + backward of ``--layers``
MoE layers (gate GEMM -> router -> dispatch/permute -> grouped expert GEMM w13 -> SwiGLU -> grouped GEMM
w2 -> combine/unpermute -> residual, and every backward kernel), at config C2 of BASELINE.md:
T=8192 tokens, H=2048, I=768, E=8, top-2, bf16 (Qwen3-30B-A3B geometry with 8 experts).  Attention, the
optimizer and FSDP collectives are outside this path at N=1 (SURVEY.md §8e: ep=1 data parallel — ranks
do not exchange anything on the MoE path), so N>1 runs shard tokens across ranks ("weak" scaling).

Prints ONE JSON line (rank 0).  ``--impl reference`` times the CPU oracle (the reference's eager algorithm
restated in torch CPU ops, oracle/moe_oracle.py) on the host cores instead.
"""
from __future__ import annotations

import argparse
import atexit
import datetime
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C2 = dict(T=8192, H=2048, I=768, E=8, K=2)
METRIC = "tokens/sec (MoE hot path fwd+bwd, Qwen3-MoE 8e top-2 bf16, seq=8k, per-step tokens / step time)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--layers", type=int, default=48, help="MoE layers per step (Qwen3-30B-A3B has 48)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--skew", type=float, default=0.0, help="Zipf exponent of expert popularity (0 = near-uniform)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--mode", default="graph", choices=["graph", "eager"],
                    help="graph: capture the whole fwd+bwd step in a CUDA graph and replay it (falls back to eager)")
    ap.add_argument("--path", default="block", choices=["block", "fused", "modules"],
                    help="block: FusedMoEBlock (RMSNorm + MoE + residual as one autograd node); fused: FusedMoELayer after "
                         "torch's RMSNorm; modules: op-by-op dispatcher protocol after torch's RMSNorm")
    ap.add_argument("--cpu-sample-tokens", type=int, default=8192)
    ap.add_argument("--reshard", type=int, default=0,
                    help="FSDPConfig.reshard_after_forward for the sharded expert parameters: 0 = gathered bf16 parameters stay "
                         "resident between forward and backward (3.6 GB at 48 layers), 1 = the reference's default (re-gather in "
                         "backward, two rotating buffers)")
    ap.add_argument("--fsdp", type=int, default=-1,
                    help="N>1: 1 = expert parameters FSDP-sharded over the ranks (fp32 master shards, cast+push all-gather with "
                         "prefetch, re-gather in backward, reduce-scatter of the gradients: xtuner_b200/fsdp_experts.py) inside "
                         "the timed step; 0 = independent replicas (no inter-rank traffic); -1 = 1 when N>1")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (loss, output of the last layer, "
                         "gradient of the step input, every parameter gradient) as DIR/<name>.npy in float32; arrays larger "
                         "than an equal share of 64 MB are replaced by a fixed seeded sample of their elements")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    return args


# ----------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md "clocks line")
# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,"
         "timestamp")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.lines: list[str] = []
        self.windows: list[list[float]] = []  # [begin, end] host times of the timed regions
        self.t_load = 0.0

    # nvidia-smi needs several hundred ms before its first line (longer with 8 ranks starting one each), more than a short
    # timed region lasts: the sampler is started ahead of the warm-up replays and the samples are attributed to the timed
    # regions by their timestamps.
    def load_begins(self):
        self.t_load = time.time()  # from here on the GPU runs the timed step back to back (warm-up replays, then timed)

    def begin(self):
        self.windows.append([time.time(), float("inf")])

    def end(self):
        self.windows[-1][1] = time.time()

    def _in_window(self, stamp: str, strict: bool = True) -> bool:
        try:
            t = datetime.datetime.strptime(stamp.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except ValueError:
            return True
        if not strict:
            return t >= self.t_load - 0.02
        return not self.windows or any(b - 0.02 <= t <= e + 0.02 for b, e in self.windows)

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.idx)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
            atexit.register(self._kill)  # an exception on the way must not leave nvidia-smi -lms running
        except Exception:
            self.proc = None

    def _kill(self):
        try:
            if self.proc is not None and self.proc.poll() is None:
                self.proc.kill()
        except Exception:
            pass

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        def collect(only_windows: bool):
            sm, mx, reasons, pw = [], [], set(), []
            for ln in self.lines:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 9 or (len(f) > 9 and not self._in_window(f[9], strict=only_windows)):
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            return sm, mx, reasons, pw

        sm, mx, reasons, pw = collect(True)
        window = ("nvidia-smi -lms 100 samples whose timestamp falls inside the timed regions (device-resident steps and "
                  "end-to-end steps: the same step)")
        if not sm:  # timed regions shorter than the sampling period (few steps / few layers)
            sm, mx, reasons, pw = collect(False)
            window = ("the timed regions are shorter than the 100 ms sampling period: all samples from the warm-up replays of "
                      "the same step to the end of the end-to-end region")
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm),
                "reasons": sorted(reasons), "window": window}


# ----------------------------------------------------------------------------------------------------
# algorithmic work per MoE layer (BASELINE.md §5)
# ----------------------------------------------------------------------------------------------------
def layer_work(T, H, I, E, K):
    s = 2
    return dict(
        gemm_flops_fwd=2 * T * K * H * 3 * I,
        gemm_flops_fwd_bwd=3 * 2 * T * K * H * 3 * I,
        dispatch_bytes_fwd=T * H * s * (1 + K) + T * K * 8,
        combine_bytes_fwd=T * H * s * (K + 1) + T * K * 8,
        permute_bwd_bytes=T * H * s * (K + 1) + T * K * 4,
        unpermute_bwd_bytes=T * H * s + 2 * T * K * H * s + T * K * 4,
    )


# ----------------------------------------------------------------------------------------------------
# CPU oracle arm (cpu_baseline and --impl reference)
# ----------------------------------------------------------------------------------------------------
def cpu_oracle_rate(cfg, layers, sample_tokens, reps, warmup):
    """tokens/sec of the CPU oracle, scaled to the same definition as the GPU arm: one step = `layers`
    layers fwd+bwd.  Measured on ONE layer over `sample_tokens` tokens (cost is linear in both).

    The thread count is chosen by a short probe (the eager per-expert matmuls of the reference algorithm do not
    scale to 128 threads; oversubscription made the 128-thread run ~6x slower than 8 threads) so the CPU arm gets
    its best configuration; `cores` in the JSON is the thread count actually used."""
    import torch

    from oracle import moe_oracle as O

    ncpu = os.cpu_count() or 1
    H, I, E, K = cfg["H"], cfg["I"], cfg["E"], cfg["K"]
    g = torch.Generator().manual_seed(0)

    def make(n_tok):
        x = torch.randn(n_tok, H, generator=g).to(torch.bfloat16).requires_grad_(True)
        gw = (torch.randn(E, H, generator=g) * 0.02).requires_grad_(True)
        w13 = (torch.randn(E * 2 * I, H, generator=g) * H**-0.5).to(torch.bfloat16).requires_grad_(True)
        w2 = (torch.randn(E * H, I, generator=g) * I**-0.5).to(torch.bfloat16).requires_grad_(True)
        nw = torch.ones(H).requires_grad_(True)
        return x, gw, w13, w2, nw

    def one(t):
        # the same unit the GPU arm times: post_attention_layernorm -> MoE -> + residual (moe_decoder_layer.py:664-705)
        h, gw, w13, w2, nw = t
        x = torch.nn.functional.rms_norm(h, (H,), nw.to(h.dtype), 1e-6)
        out = O.moe_layer_forward(x, gw, w13, w2, K, residual=h)["hidden_states"]
        out.float().square().mean().backward()

    # probe: 1024 tokens, candidate thread counts
    probe = make(min(1024, sample_tokens))
    cands = sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu})
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        one(probe)
        t0 = time.perf_counter()
        one(probe)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    data = make(sample_tokens)
    for _ in range(warmup):
        one(data)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        one(data)
        ts.append(time.perf_counter() - t0)
    t_layer = statistics.median(ts)
    return sample_tokens / (t_layer * layers), best, t_layer


def summarize_profile(prof_ms, cfg, L, ms_step, n_prof_layer_steps):
    """Pure post-processing (unit-tested on CPU): per-kernel averages and the two roofline objects from the list of
    (kernel name, milliseconds) measured with CUDA events."""
    T, H, I, E, K = (cfg[k] for k in "THIEK")
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    tf_peak = peaks.get("bf16_tflops_sustained") or 1400.0
    peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained: kernel timed inside a long step)" if peaks else "fallback"
    M = T * K
    work = layer_work(T, H, I, E, K)
    # DRAM traffic per launch from the committed ncu --set full captures (profiles/ncu_traffic.json)
    ncu_traffic = {}
    try:
        ncu_traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))["kernels"]
    except Exception:
        pass

    def traffic_of(*names):
        vals = [ncu_traffic[n]["dram_bytes_per_launch"] for n in names if n in ncu_traffic]
        return (sum(vals) / len(vals)) if vals and len(vals) == len(names) else None

    # 5 launches per layer: w13+SwiGLU, w2, dA, dX, and both weight gradients in one (xtb_group_gemm_tn_pair)
    gemm_traffic = traffic_of("group_gemm2_kernel<0, 1, 1>", "group_gemm2_kernel<0, 0, 1>", "group_gemm2_kernel<1, 0, 1>",
                              "group_gemm2_kernel<1, 0, 1>", "group_gemm2_kernel<2, 0, 1>")
    kt: dict = {}
    for name, ms_ in prof_ms:
        d = kt.setdefault(name, [0.0, 0])
        d[0] += ms_
        d[1] += 1
    n_layer_steps = n_prof_layer_steps
    gemm_names = [n for n in kt if "group_gemm" in n]
    gemm_ms = sum(kt[n][0] for n in gemm_names)
    flops = work["gemm_flops_fwd_bwd"] * n_layer_steps
    achieved = flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    roofline = {
        "kernel": "group_gemm2_kernel<NT|NN|TN, EPI, STORE=1> (tcgen05 CTA-pair grouped expert GEMMs; NT-w13 has the SwiGLU epilogue)",
        "bound": "tensor", "achieved": achieved, "peak": tf_peak, "unit": "TFLOP/s", "frac": achieved / tf_peak,
        "peak_source": peak_src, "traffic": gemm_traffic,
        "traffic_note": "average DRAM bytes per GEMM launch (5 launches per layer, the two weight gradients share one) from "
                        "profiles/ncu_traffic.json; algorithmic operand+output bytes average 152 MB per launch — outputs "
                        "largely stay in the 126 MB L2",
        "share_of_step": (gemm_ms / n_prof_layer_steps) * L / ms_step,
        "launches_timed": sum(kt[n][1] for n in gemm_names),
        "flops_per_layer_fwd_bwd": work["gemm_flops_fwd_bwd"],
    }
    # second half of BASELINE.json's metric: "MoE dispatch HBM GB/s" (dispatch = permute, combine = unpermute)
    hbm_peak = peaks.get("hbm_gbs") or 6650.0
    roofline_dispatch = None
    perm_name = "xtb_moe_permute_prepared" if "xtb_moe_permute_prepared" in kt else "xtb_moe_permute"
    if perm_name in kt and "xtb_moe_combine" in kt:
        # per layer-step the timed calls are: gather fwd (1), combine fwd (1) and combine again as the dispatch
        # backward (1).  The bucket/scan index work of the dispatch runs inside the router kernel
        # (xtb_router_greedy_dispatch) — its whole duration is charged to the dispatch below.
        t_perm = kt[perm_name][0] / kt[perm_name][1]
        t_route = kt.get("xtb_router_greedy_dispatch", [0.0, 1])[0] / kt.get("xtb_router_greedy_dispatch", [0.0, 1])[1]
        gate_bytes = 0
        if "xtb_gate_route_dispatch" in kt:
            # one-launch gate+router+bucketing (the default): the whole kernel (it also reads x for the gate) is charged, with
            # the gate's bytes added to the numerator so the figure stays an honest bytes-over-time
            t_route = kt["xtb_gate_route_dispatch"][0] / kt["xtb_gate_route_dispatch"][1]
            gate_bytes = T * H * 2 + E * H * 4
        t_comb = kt["xtb_moe_combine"][0] / kt["xtb_moe_combine"][1]
        route_bytes = T * E * 4 + T * K * (8 + 4 + 4) + T * E * 4 + E * 8
        b_disp = work["dispatch_bytes_fwd"] + route_bytes + gate_bytes
        # combine calls also read the residual / gate-grad stream: +T*H*2 bytes
        b_comb = work["combine_bytes_fwd"] + T * H * 2
        gbs_disp = b_disp / ((t_perm + t_route) * 1e-3) / 1e9
        gbs_gather = work["dispatch_bytes_fwd"] / (t_perm * 1e-3) / 1e9
        gbs_comb = b_comb / (t_comb * 1e-3) / 1e9
        gbs = (b_disp + b_comb) / ((t_perm + t_route + t_comb) * 1e-3) / 1e9
        roofline_dispatch = {
            "kernel": ("gate+route+bucket (xtb_gate_route_dispatch, gate bytes included)" if gate_bytes else
                       "route+bucket (xtb_router_greedy_dispatch)") + " + gather (xtb_moe_permute_prepared) + combine (xtb_moe_combine)",
            "note": "combine also streams the residual; in path=block the dispatch backward is a separate fused kernel (xtb_moe_dispatch_bwd_rmsnorm)",
            "bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
            "route_plus_dispatch_GBs": gbs_disp, "gather_only_GBs": gbs_gather, "combine_GBs": gbs_comb,
            "route_us": t_route * 1e3, "gather_us": t_perm * 1e3, "combine_us": t_comb * 1e3,
            "bytes_route_plus_dispatch": b_disp, "bytes_combine": b_comb,
            "traffic": {"gather": traffic_of("permute_scatter_bulk_kernel"), "combine": traffic_of("unpermute_kernel<2>"),
                        "note": "DRAM bytes per launch (ncu); the gather's 67 MB of writes mostly stay in L2"},
            "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback",
        }
    kernel_us = {n: round(1e3 * v[0] / v[1], 2) for n, v in sorted(kt.items())}
    return roofline, roofline_dispatch, kernel_us


def kernel_table(prof_ms, cfg, hbm_peak=None, tf_peak=None):
    """Per-entry-point roofline table from the same (name, ms) event list: algorithmic bytes (HBM-bound kernels) or
    flops (grouped GEMMs) per LAYER for each C-ABI entry point, divided by the time that entry point took per layer.
    Names called more than once per layer (the two NN and two TN products) are aggregated."""
    T, H, I, E, K = (cfg[k] for k in "THIEK")
    M, s = T * K, 2
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = hbm_peak or peaks.get("hbm_gbs") or 6650.0
    tf_peak = tf_peak or peaks.get("bf16_tflops_sustained") or 1400.0
    route_bytes = T * E * 4 + T * K * (8 + 4 + 4) + T * E * 4 + E * 8
    byte_model = {  # bytes per layer (forward + backward calls of that name)
        "xtb_rmsnorm_gate": 2 * T * H * s + T * 4 + H * 4,
        "xtb_gate_logits": T * H * s + E * H * 4 + T * E * 4,
        "xtb_router_greedy_dispatch": route_bytes,
        "xtb_router_greedy": route_bytes,
        "xtb_gate_route_dispatch": route_bytes + T * H * s + E * H * 4,
        "xtb_moe_permute_prepared": T * H * s * (1 + K) + T * K * 8,
        "xtb_moe_permute": T * H * s * (1 + K) + T * K * 8,
        "xtb_moe_unpermute_bwd": T * H * s + 2 * M * H * s + T * K * 8,
        "xtb_swiglu_bwd": 5 * M * I * s,
        "xtb_router_greedy_bwd": 2 * T * E * 4 + T * K * (4 + 4 + 8),
        "xtb_gate_logits_bwd": T * E * 4 + 2 * T * H * s + 2 * E * H * 4,
        "xtb_router_gate_bwd": 2 * T * H * s + 2 * E * H * 4 + 2 * T * E * 4 + T * K * (4 + 4 + 8),
        "xtb_moe_dispatch_bwd_rmsnorm": (K + 4) * T * H * s + T * K * 4 + T * 4 + 2 * H * 4,
    }
    # xtb_moe_combine: forward call streams the residual; in path=fused it is also the dispatch backward
    flop_model = {
        "xtb_group_gemm_nt_swiglu": 2 * M * 2 * I * H,
        "xtb_group_gemm_nt": 2 * M * H * I,
        "xtb_group_gemm_nn": 2 * M * H * I + 2 * M * 2 * I * H,
        "xtb_group_gemm_tn": 2 * M * H * I + 2 * M * 2 * I * H,
        "xtb_group_gemm_tn_pair": 2 * M * H * I + 2 * M * 2 * I * H,  # both weight gradients in one launch
    }
    kt: dict = {}
    for name, ms_ in prof_ms:
        d = kt.setdefault(name, [0.0, 0])
        d[0] += ms_
        d[1] += 1
    if not kt:
        return []
    # layer-steps profiled = calls of a once-per-layer kernel
    once = next((n for n in ("xtb_group_gemm_nt_swiglu", "xtb_gate_logits", "xtb_moe_unpermute_bwd") if n in kt), None)
    n_ls = kt[once][1] if once else max(v[1] for v in kt.values())
    rows = []
    for name, (tot_ms, calls) in sorted(kt.items()):
        us_layer = 1e3 * tot_ms / n_ls
        row = {"entry": name, "calls_per_layer": round(calls / n_ls, 2), "us_per_layer": round(us_layer, 2)}
        if name == "xtb_moe_combine":
            per_call = T * H * s * (K + 1) + T * K * 8 + T * H * s
            row.update(bound="hbm", bytes_per_layer=per_call * calls // n_ls)
        elif name in byte_model:
            row.update(bound="hbm", bytes_per_layer=byte_model[name])
        elif name in flop_model:
            row.update(bound="tensor", flops_per_layer=flop_model[name])
        if us_layer <= 0:
            rows.append(row)
            continue
        if row.get("bound") == "hbm":
            gbs = row["bytes_per_layer"] / (us_layer * 1e-6) / 1e9
            row.update(achieved_GBs=round(gbs, 1), frac=round(gbs / hbm_peak, 3))
        elif row.get("bound") == "tensor":
            tf = row["flops_per_layer"] / (us_layer * 1e-6) / 1e12
            row.update(achieved_TFLOPs=round(tf, 1), frac=round(tf / tf_peak, 3))
        rows.append(row)
    return rows


def contract_config(layers, world, parallelism):
    """the `config` object of the contract line — identical keys and values in both arms (ours / --impl reference)"""
    return {"workload": "C2 Qwen3-MoE 8e top-2: MoE layer stack fwd+bwd (RMSNorm, gate, router, dispatch, grouped GEMMs, SwiGLU, "
                        "combine, residual)",
            **C2, "layers": layers, "global_tokens_per_step": world * C2["T"], "parallelism": parallelism}


def gpu_reference_record(kernel_us, ms_step, L):
    """The UNMODIFIED reference's kernels timed on a B200 of this pool by ``baseline/gpu_reference.py`` (Triton grouped GEMMs
    autotuned with XTUNER_DETERMINISTIC unset, torch-fallback permute / unpermute, the reference's MoE half of the decoder
    layer), read from the committed record and placed next to this run's entry points.  Not re-measured here: ~100 Triton
    autotune compilations take minutes, so it is its own command (BASELINE.md section 3a)."""
    path = os.path.join(ROOT, "profiles", "r02_gpu_reference.json")
    try:
        ref = json.load(open(path))["gpu_reference"]
    except Exception:
        return None
    g = ref.get("gemm_us", {})
    ours = kernel_us or {}
    us = lambda k: g.get(k, {}).get("us")  # noqa: E731
    both = lambda *ks: (sum(us(k) for k in ks) if all(us(k) for k in ks) else None)  # noqa: E731
    side = {
        "w13 forward (+SwiGLU in ours)": {"reference_us": (us("nt_w13") or 0) + ref.get("swiglu_us", 0), "ours_us": ours.get("xtb_group_gemm_nt_swiglu")},
        "w2 forward": {"reference_us": us("nt_w2"), "ours_us": ours.get("xtb_group_gemm_nt")},
        "dA + dX": {"reference_us": both("nn_w2", "nn_w13"), "ours_us": ours.get("xtb_group_gemm_nn") and 2 * ours["xtb_group_gemm_nn"]},
        "dW2 + dW13": {"reference_us": both("tn_w2", "tn_w13"),
                       "ours_us": ours.get("xtb_group_gemm_tn_pair") or (ours.get("xtb_group_gemm_tn") and 2 * ours["xtb_group_gemm_tn"])},
        "gate + router (+ bucketing in ours)": {"reference_us": ref.get("gate_us", 0) + ref.get("router_us", 0),
                                                "ours_us": ours.get("xtb_gate_route_dispatch")},
        "permute (dispatch gather)": {"reference_us": ref.get("permute_us"), "ours_us": ours.get("xtb_moe_permute_prepared")},
        "unpermute (combine, + residual in ours)": {"reference_us": ref.get("unpermute_us"), "ours_us": ours.get("xtb_moe_combine")},
        "MoE half of the layer, fwd+bwd (ms)": {"reference_ms": ref.get("layer_fwd_bwd_ms"), "ours_ms": ms_step / L},
    }
    return {"source": "profiles/r02_gpu_reference.json — baseline/gpu_reference.py on a B200 of this pool (gpurun call 41), not re-measured "
                      "in this run; ours_* = this run (kernel_avg_us, per call)",
            "box": ref.get("box"), "triton": ref.get("triton"), "reference_ops": ref.get("reference_ops_bound"),
            "gemm_us": {k: v.get("us") for k, v in g.items()}, "permute_us": ref.get("permute_us"), "unpermute_us": ref.get("unpermute_us"),
            "layer_fwd_bwd_ms": ref.get("layer_fwd_bwd_ms"), "tokens_per_s_48_layers": ref.get("layer_tokens_per_s_48_layers"),
            "side_by_side": side}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes ``arrays`` (name -> tensor) as ``out_dir/<name>.npy`` in float32, at most ``DUMP_BYTES`` in all: an array
    larger than its equal share keeps that many elements, at positions drawn by a generator seeded with the array's size, so
    two runs with the same arguments store the same elements."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // 4 // max(1, len(arrays))
    picks = {}  # numel -> sampled positions
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > share:
            if t.numel() not in picks:
                g = torch.Generator().manual_seed(t.numel())
                picks[t.numel()] = torch.randperm(t.numel(), generator=g)[:share].sort().values.to(t.device)
            t = t.reshape(-1)[picks[t.numel()]]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def default_parallelism(world, fsdp_flag):
    return f"fsdp={world} (ep=1)" if (world > 1 and fsdp_flag != 0) else f"dp{world} (ep=1)"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rate, cores, t_layer = cpu_oracle_rate(C2, args.layers, args.cpu_sample_tokens, max(1, args.steps), max(1, args.warmup))
    sample = (f"1 MoE layer fwd+bwd over {args.cpu_sample_tokens} tokens per step (median of {max(1, args.steps)}), "
              f"scaled linearly to {args.layers} layers; oracle/moe_oracle.py (reference eager algorithm, torch CPU); "
              f"{cores} threads chosen by a probe over {{8,16,32,64,{os.cpu_count()}}} of {os.cpu_count()} host cores")
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": "tokens/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_layer * args.layers * C2["T"] / args.cpu_sample_tokens,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": contract_config(args.layers, max(1, args.gpus), default_parallelism(max(1, args.gpus), args.fsdp)),
        "run": {"arm": "CPU port of the reference's eager algorithm on the host cores of rank 0; the GPU arm's parallelism does "
                       "not apply to it (one host, one layer sample per step)",
                "extrapolated": True, "timed_seconds_per_step": t_layer, "layers_timed_per_step": 1,
                "tokens_timed_per_step": args.cpu_sample_tokens,
                "note": "value = sample tokens / (seconds per sampled layer x layers): ms_per_step is the extrapolated full "
                        "step, NOT the wall time of this run"},
        "cpu_baseline": {"value": rate, "unit": "tokens/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------
# N>1: the exchange kernels and the sharded step are checked against NCCL BEFORE anything is timed
# ----------------------------------------------------------------------------------------------------
def fsdp_selfcheck(eng, small, x_dev, K, step):
    """Raises on mismatch.  (1) cast+push all-gather == bf16 cast + NCCL all_gather, bit for bit; (2) pull reduce-scatter ==
    NCCL reduce_scatter on integer-valued gradients (exact in any summation order), bit for bit, and within fp32 rounding on
    random gradients; (3) one step of the sharded stack == the same stack on NCCL-gathered parameters with NCCL
    reduce-scattered gradients (loss and every shard gradient)."""
    import torch
    import torch.distributed as dist

    from xtuner_b200 import fused

    dev, world, rank = x_dev.device, eng.world, eng.rank
    bf = torch.bfloat16
    out = {}
    # (1) ------------------------------------------------------------------------------------------------
    eng.begin_step()
    eng.end_step()
    torch.cuda.synchronize()
    for name, master, view in (("w13", eng.master13[0], eng._p[0]["w13"]), ("w2", eng.master2[0], eng._p[0]["w2"])):
        ref = torch.empty(master.numel() * world, dtype=bf, device=dev)
        dist.all_gather_into_tensor(ref, master.detach().to(bf))
        if not torch.equal(ref, view.reshape(-1)):
            raise RuntimeError(f"fsdp selfcheck: cast+push all-gather of {name} differs from cast + NCCL all_gather")
    out["all_gather_vs_nccl"] = "bit-exact"
    # (2) ------------------------------------------------------------------------------------------------
    slot = eng._g[0]
    for kind in ("integers", "random"):
        g = torch.Generator(device=dev).manual_seed(77 + rank)
        for v in (slot["w13"], slot["w2"]):
            if kind == "integers":
                v.copy_(torch.randint(-8, 9, v.shape, generator=g, device=dev).to(bf))
            else:
                v.copy_((torch.randn(v.shape, generator=g, device=dev) * 0.01).to(bf))
        eng.be.record(slot["free"], False)
        eng._reduce_scatter(0, slot["w13"], slot["w2"])
        eng.be.wait(slot["free"], False)
        torch.cuda.synchronize()
        for name, v, got in (("w13", slot["w13"], eng.grad13[0]), ("w2", slot["w2"], eng.grad2[0])):
            ref = torch.empty_like(got)
            dist.reduce_scatter_tensor(ref, v.reshape(-1).float(), op=dist.ReduceOp.SUM)
            ref /= world
            if kind == "integers":
                if not torch.equal(ref, got):
                    raise RuntimeError(f"fsdp selfcheck: reduce-scatter of {name} (integer-valued) differs from NCCL")
            else:
                err = (ref - got).abs().max().item()
                if err > 2e-6 * ref.abs().max().item() + 1e-12:
                    raise RuntimeError(f"fsdp selfcheck: reduce-scatter of {name} off by {err:.3e} vs NCCL fp32")
    out["reduce_scatter_vs_nccl"] = "bit-exact on integer-valued gradients; <= 2e-6 rel on random ones (fp32 summation order)"
    # (3) ------------------------------------------------------------------------------------------------
    for p in eng.parameters():
        p.grad = None
    loss_e = step(x_dev).detach().clone()
    torch.cuda.synchronize()
    got13 = [g.clone() for g in eng.grad13]
    got2 = [g.clone() for g in eng.grad2]
    small_g = [(a.grad.clone(), b.grad.clone()) for a, b in small]
    full = []
    for i in range(eng.L):
        pair = []
        for master, shape in ((eng.master13[i], (eng.E, 2 * eng.I, eng.H)), (eng.master2[i], (eng.E, eng.H, eng.I))):
            t = torch.empty(master.numel() * world, dtype=bf, device=dev)
            dist.all_gather_into_tensor(t, master.detach().to(bf))
            pair.append(t.view(shape).requires_grad_(True))
        full.append(pair)
    for a, b in small:
        a.grad = b.grad = None
    h = x_dev.detach().requires_grad_(True)
    for i in range(eng.L):
        h, _ = fused.fused_moe_block(h, small[i][0], 1e-6, small[i][1], full[i][0], full[i][1], top_k=K)
    loss_r = h.float().square().mean()
    loss_r.backward()
    torch.cuda.synchronize()
    rel = abs(loss_e.item() - loss_r.item()) / max(abs(loss_r.item()), 1e-30)
    if rel > 1e-6:
        raise RuntimeError(f"fsdp selfcheck: loss of the sharded step {loss_e.item()} vs NCCL-gathered reference {loss_r.item()}")
    worst = 0.0
    for i in range(eng.L):
        for got, t in ((got13[i], full[i][0]), (got2[i], full[i][1])):
            ref = torch.empty_like(got)
            dist.reduce_scatter_tensor(ref, t.grad.reshape(-1).float(), op=dist.ReduceOp.SUM)
            ref /= world
            err = (ref - got).abs().max().item() / max(ref.abs().max().item(), 1e-30)
            worst = max(worst, err)
            if err > 1e-5:
                raise RuntimeError(f"fsdp selfcheck: shard gradient of layer {i} off by {err:.3e} (relative to max) vs NCCL")
        for (ga, gb), (a, b) in ((small_g[i], small[i]),):
            for got, p in ((ga, a), (gb, b)):
                ref = p.grad.clone()
                dist.all_reduce(ref, op=dist.ReduceOp.SUM)  # NCCL average of the replicated gradients
                ref /= world
                err = (ref - got).abs().max().item() / max(ref.abs().max().item(), 1e-30)
                if err > 1e-5:
                    raise RuntimeError(f"fsdp selfcheck: averaged replicated gradient of layer {i} off by {err:.3e} vs NCCL")
    out["step_vs_nccl_reference"] = {"loss_rel_diff": rel, "worst_shard_grad_rel_to_max": worst, "layers": eng.L}
    del full
    torch.cuda.empty_cache()
    return out


def ulysses_selfcheck(dev, world, iters=10):
    """N>1: the Ulysses head<->sequence all-to-all (row a12) at config C4's per-rank Q shape, [1, 32, 8192, 128] bf16 =
    64 MiB with sp = N: bit-exact against the reference's algorithm on NCCL (ops/comm/all_to_all.py:30-51: movedim,
    all_to_all_single, split + cat), both directions, then both timed (CUDA events, max over ranks taken by the caller)."""
    import torch
    import torch.distributed as dist

    from xtuner_b200 import comm

    group = dist.group.WORLD

    def reference(x, scatter_dim, gather_dim):
        inp = x.contiguous().movedim(scatter_dim, 0).contiguous()
        out = torch.empty_like(inp)
        dist.all_to_all_single(out, inp, group=group)
        out = out.movedim(0, scatter_dim)
        return torch.cat(torch.tensor_split(out, world, scatter_dim), dim=gather_dim).contiguous()

    g = torch.Generator(device=dev).manual_seed(5 + dist.get_rank())
    q = torch.randn(1, 32, 8192, 128, generator=g, device=dev).to(torch.bfloat16)
    out = comm.ulysses_all_to_all(q, 1, 2, group)
    if not torch.equal(out, reference(q, 1, 2)):
        raise RuntimeError("ulysses selfcheck: heads->sequence all-to-all differs from the NCCL reference")
    back = comm.ulysses_all_to_all(out, 2, 1, group)
    if not (torch.equal(back, reference(out, 2, 1)) and torch.equal(back, q)):
        raise RuntimeError("ulysses selfcheck: sequence->heads all-to-all differs from the NCCL reference / is not the inverse")
    res = {"parity": "bit-exact vs NCCL all_to_all_single + the reference's copies, both directions; round trip == identity"}
    for name, fn in (("ours_us", lambda: comm.ulysses_all_to_all(q, 1, 2, group)), ("nccl_reference_us", lambda: reference(q, 1, 2))):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        res[name] = e0.elapsed_time(e1) * 1e3 / iters
    res["bytes_per_rank_per_direction"] = q.numel() * 2 * (world - 1) // world
    return res


def fsdp_exchange_bench(eng, iters=20):
    """the exchange kernels alone (nothing else on the GPU): microseconds per layer's all-gather (barrier, 2 cast+push
    kernels, barrier) and reduce-scatter (barrier, 2 pull kernels, barrier), timed on the exchange stream"""
    import torch

    st = eng.be.stream
    res = {}
    for name in ("all_gather", "reduce_scatter"):
        for s in eng._p + eng._g:
            eng.be.record(s["free"], False)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for it in range(iters + 3):
            if it == 3:
                e0.record(st)
            if name == "all_gather":
                eng._all_gather(it % 2)
            else:
                slot = eng._g[it % 2]
                eng._reduce_scatter(it % 2, slot["w13"], slot["w2"])
        e1.record(st)
        torch.cuda.synchronize()
        res[name + "_us"] = e0.elapsed_time(e1) * 1e3 / iters
    return res


# ----------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import __graft_entry__ as ge

    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    from xtuner_b200 import _capi, fused, ops
    from xtuner_b200.fused import FusedMoEBlock, FusedMoELayer
    from xtuner_b200.moe import MoELayer

    Layer = {"block": FusedMoEBlock, "fused": FusedMoELayer, "modules": MoELayer}[args.path]

    lib = _capi.ensure_init()
    cfg = dict(C2)
    T, H, I, E, K = (cfg[k] for k in "THIEK")
    L = args.layers

    if os.environ.get("XTB_BENCH_FSDP") == "0":  # A/B convenience for scripts that pass every variant through the environment
        args.fsdp = 0
    use_fsdp = world > 1 and args.fsdp != 0
    if use_fsdp and args.path != "block":
        raise SystemExit("--fsdp needs --path block")
    eng = None
    layers = []
    fsdp_error = None
    if use_fsdp:
        # data parallel replicas: identical parameters on every rank (same seed), rank-local tokens
        try:
            from xtuner_b200.fsdp_experts import ExpertShards

            torch.manual_seed(1234)
            eng = ExpertShards(dist.group.WORLD, dev, n_layers=L, n_experts=E, hidden=H, inter=I,
                               reshard_after_forward=bool(args.reshard or os.environ.get("XTB_BENCH_RESHARD") == "1"))
            small = []  # per layer (post_attention_layernorm.weight, gate.weight): 0.05 % of the parameter bytes, replicated
            for i in range(L):
                gate_w = torch.randn(E, H, device=dev) * 0.02
                if args.skew > 0:
                    pop = torch.log(1.0 / torch.arange(1, E + 1, device=dev).float() ** args.skew)
                    gate_w.add_(pop[:, None] * 0.05)
                w13_full = torch.randn(E * 2 * I, H, device=dev) * H**-0.5
                w2_full = torch.randn(E * H, I, device=dev) * (2 * I) ** -0.5
                eng.load_full(i, w13_full, w2_full)
                del w13_full, w2_full
                small.append((torch.nn.Parameter(torch.ones(H, device=dev)), torch.nn.Parameter(gate_w)))
            params = eng.parameters() + [p for pair in small for p in pair]
            eng.register_replicated([p for pair in small for p in pair])  # their gradients: one coalesced all-reduce per step
            torch.manual_seed(4321 + rank)
        except Exception as ex:  # noqa: BLE001 — infrastructure only (symmetric-memory set-up); parity failures raise later
            fsdp_error = f"{type(ex).__name__}: {ex}"[:300]
        ok = torch.tensor([0 if fsdp_error else 1], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            # every rank falls back together and SAYS so in the line (config.parallelism, fsdp_error): a number is still
            # produced, but it is the no-exchange one and is labelled as such
            fsdp_error = fsdp_error or "another rank could not set up the symmetric-memory exchange"
            sys.stderr.write(f"[bench] rank {rank}: FSDP expert sharding unavailable ({fsdp_error}); independent replicas\n")
            use_fsdp, eng = False, None
    def build_replicas():
        torch.manual_seed(1234 + rank)
        ls = []
        for _ in range(L):
            m = Layer(hidden_size=H, moe_intermediate_size=I, n_routed_experts=E, num_experts_per_tok=K).to(dev)
            m.experts.to(torch.bfloat16)
            with torch.no_grad():
                m.gate.weight.normal_(0, 0.02)
                if args.skew > 0:
                    pop = torch.log(1.0 / torch.arange(1, E + 1, device=dev).float() ** args.skew)
                    m.gate.weight.add_(pop[:, None] * 0.05)
                m.experts.fused_w1w3.weight.normal_(0, H**-0.5)
                m.experts.fused_w2.weight.normal_(0, (2 * I) ** -0.5)
            ls.append(m)
        return ls

    if not use_fsdp:
        layers = build_replicas()
        params = [p for m in layers for p in m.parameters()]

    x_host = torch.randn(T, H).to(torch.bfloat16).pin_memory()
    x_dev = x_host.to(dev)
    loss_host = torch.zeros(1, dtype=torch.float32).pin_memory()

    # per-kernel CUDA-event timing inside the timed region (fused path: every C-ABI kernel; modules path: GEMMs)
    prof: list = []
    orig_gg = ops._gg_call

    def timed_gg(fn_name, a, b, tpe, M, N, Kd, E_, out):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        orig_gg(fn_name, a, b, tpe, M, N, Kd, E_, out)
        e.record()
        prof.append((fn_name, s, e))

    last: dict = {}  # --dump-outputs: the tensors the most recent step() returned or wrote (in graph mode: the graph's own)

    def keep(loss, h, x_leaf):
        if args.dump_outputs:
            last.clear()
            last.update(loss=loss.detach(), output=h.detach(), input_grad=x_leaf.grad, grads=[p.grad for p in params])

    def step(x_in):
        for p in params:
            p.grad = None
        h = x_leaf = x_in.detach().requires_grad_(True)
        if use_fsdp:
            eng.begin_step()  # all-gather (cast + push) of layer 0 on the exchange stream
            for i in range(L):
                w13, w2 = eng.layer_params(i)  # waits for this layer's gather, prefetches the next layer's
                h, _ = fused.fused_moe_block(h, small[i][0], 1e-6, small[i][1], w13, w2, top_k=K)
                h = eng.mark_output(i, h)      # backward: re-gather + prefetch; dW lands in the reduce-scatter buffer
            loss = h.float().square().mean()
            loss.backward()
            eng.end_step()  # the compute stream joins the last reduce-scatter; .grad = averaged fp32 shard gradients
            keep(loss, h, x_leaf)
            return loss
        for m in layers:
            # MoE half of the decoder layer: residual = h; x = post_attention_layernorm(h); h = moe(x) + residual
            # ("block": the norm and the residual are inside the fused node; otherwise torch's RMSNorm)
            h, _ = m(h) if args.path == "block" else m(norm(h), h)
        loss = h.float().square().mean()
        loss.backward()
        keep(loss, h, x_leaf)
        return loss

    norm_w = torch.ones(H, dtype=torch.bfloat16, device=dev)

    def norm(t):
        return torch.nn.functional.rms_norm(t, (H,), norm_w, 1e-6)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up; N>1: parity of the exchange kernels and of the sharded step against NCCL, before anything is timed ----
    selfcheck = None
    if use_fsdp:
        try:
            for _ in range(max(args.warmup, 3)):
                step(x_dev)
            barrier()
            selfcheck = fsdp_selfcheck(eng, small, x_dev, K, step)
        except RuntimeError as ex:  # a parity failure (or a recoverable runtime error): no number is reported for that path
            fsdp_error = f"{type(ex).__name__}: {ex}"[:400]
            sys.stderr.write(f"[bench] rank {rank}: FSDP path rejected: {fsdp_error}\n")
        ok = torch.tensor([0 if fsdp_error else 1], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            # every rank drops to independent replicas TOGETHER and the line says so (run.parallelism_detail, fsdp_error,
            # config.parallelism = dp): the sharded path produced no number
            fsdp_error = fsdp_error or "another rank's selfcheck failed"
            from xtuner_b200 import fused as _f

            _f.GRAD_SINK = None
            use_fsdp, eng, small = False, None, None
            torch.cuda.empty_cache()
            layers = build_replicas()
            params = [p for m in layers for p in m.parameters()]
    if not use_fsdp:
        for _ in range(max(args.warmup, 3)):
            step(x_dev)
    barrier()

    # ---- optional CUDA-graph capture of the whole step (no host syncs on the path, so it is capturable) ----
    mode = "eager"
    graph = graph_outputs = None
    static_x = x_dev.clone()
    static_loss = None
    side = torch.cuda.Stream()

    def capture():
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            step(static_x)  # one more warm-up on the capture stream (workspaces are per stream)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            loss_ = step(static_x)
        torch.cuda.synchronize()
        g.replay()
        torch.cuda.synchronize()
        return g, loss_

    sampler = ClockSampler(local_rank)
    sampler.start()  # nvidia-smi takes a few hundred ms to its first line: started ahead of the capture, samples filtered by time
    if args.mode == "graph":
        try:
            graph, static_loss = capture()
            graph_outputs = dict(last)  # the captured step's tensors: every replay rewrites them in place
            mode = "cuda_graph"
        except Exception as ex:  # noqa: BLE001
            sys.stderr.write(f"[bench] CUDA graph capture failed ({type(ex).__name__}: {ex}); falling back to eager\n")
            graph = None
            torch.cuda.synchronize()
    if world > 1:
        # every rank must run the same mode (a rank replaying a graph and a rank launching eagerly still meet at the same
        # barriers, but the timing would mix two regimes)
        flag = torch.tensor([1 if graph is not None else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0 and graph is not None:
            graph, mode = None, "eager"

    def run_step(x_in):
        if graph is not None:
            if x_in is not static_x:
                static_x.copy_(x_in, non_blocking=True)
            graph.replay()
            return static_loss
        return step(x_in)

    sampler.load_begins()
    for _ in range(2):
        run_step(static_x)
    barrier()

    # ---- timed: device-resident inputs ----------------------------------------------------------------
    lib.xtb_reset_launch_count()
    barrier()
    sampler.begin()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        run_step(static_x)
    ev1.record()
    barrier()
    sampler.end()
    launches = int(lib.xtb_launch_count())
    ms_total = ev0.elapsed_time(ev1)
    final_loss = float(run_step(static_x).item())
    if not (final_loss == final_loss and abs(final_loss) < 1e30):
        raise RuntimeError(f"bench workload is not finite (loss={final_loss}); numbers would be meaningless")
    if graph is not None:
        # launches are replayed by the graph, not re-issued by the library: count them from one eager step
        lib.xtb_reset_launch_count()
        step(x_dev)
        torch.cuda.synchronize()
        launches = int(lib.xtb_launch_count()) * args.steps

    # ---- timed: end to end with host buffers (H2D of the step input, D2H of the loss, every step) ------
    barrier()
    sampler.begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        if graph is not None:
            static_x.copy_(x_host, non_blocking=True)
            graph.replay()
            loss = static_loss
        else:
            xin = x_host.to(dev, non_blocking=True)
            loss = step(xin)
        loss_host.copy_(loss.detach().reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()  # the caller reads the loss every step
    e1.record()
    barrier()
    sampler.end()
    clocks = sampler.stop()
    ms_e2e = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        out = graph_outputs if graph is not None else last
        if use_fsdp:
            names = ([f"layer{i:02d}.experts.fused_w1w3.weight_shard" for i in range(L)]
                     + [f"layer{i:02d}.experts.fused_w2.weight_shard" for i in range(L)]
                     + [f"layer{i:02d}.{n}" for i in range(L) for n in ("post_attention_layernorm.weight", "gate.weight")])
        else:
            names = [f"layer{i:02d}.{n}" for i, m in enumerate(layers) for n, _ in m.named_parameters()]
        arrays = {"loss": out["loss"], "output": out["output"], "input_grad": out["input_grad"]}
        arrays.update({n + ".grad": g for n, g in zip(names, out["grads"], strict=True) if g is not None})
        dump_outputs(args.dump_outputs, arrays)

    # ---- N>1: the same step with the exchange switched off (stream/event choreography kept, no barrier/push/pull) ->
    # exposed exchange time; then the exchange kernels alone -> NVLink roofline ---------------------------------
    ms_noexch = None
    exch = None
    a2a = None
    if use_fsdp:
        # XTB_BENCH_EXCHANGE_KEEP (diagnosis): parts of the exchange left ON in this second capture, e.g. "ag+bar" -> the
        # difference to the full step is what the reduce-scatter costs; default: everything off
        eng.exchange_enabled = os.environ.get("XTB_BENCH_EXCHANGE_KEEP") or False
        try:
            if graph is not None:
                g2, _ = capture()
                run2 = g2.replay
            else:
                run2 = lambda: step(static_x)  # noqa: E731
            for _ in range(2):
                run2()
            barrier()
            n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n0.record()
            for _ in range(args.steps):
                run2()
            n1.record()
            barrier()
            ms_noexch = n0.elapsed_time(n1)
        finally:
            eng.exchange_enabled = True
        barrier()
        exch = fsdp_exchange_bench(eng)
        barrier()
        try:
            a2a = ulysses_selfcheck(dev, world)
        except RuntimeError:
            raise
        barrier()

    # ---- per-kernel CUDA-event timing (eager, same step): the GPU is first parked on a spin kernel so the
    # host can enqueue ahead and the event intervals contain no launch gaps --------------------------------
    prof_layers = layers[: min(L, 6)]

    def prof_step(x_in):
        if use_fsdp:
            step(x_in)
            return
        h = x_in.detach().requires_grad_(True)
        for m in prof_layers:
            h, _ = m(h) if args.path == "block" else m(norm(h), h)
        h.float().square().mean().backward()

    prof_step(x_dev)
    torch.cuda.synchronize()
    n_prof_iters = 3
    for _ in range(n_prof_iters):
        # ~40 ms head start: the host enqueues the whole eager step (6 layers, ~450 launches and event records, well inside the
        # launch queue) while the GPU spins, so no interval waits for a launch — with 10 ms the first backward kernel of every
        # layer (unpermute_bwd: the host is busiest right before it) showed 45 us against 26 us under ncu
        torch.cuda._sleep(int(8.0e7))
        if args.path in ("block", "fused"):
            fused.PROFILE = prof
        else:
            ops._gg_call = timed_gg
        prof_step(x_dev)
        fused.PROFILE = None
        ops._gg_call = orig_gg
        torch.cuda.synchronize()
    n_prof_layer_steps = (L if use_fsdp else len(prof_layers)) * n_prof_iters

    t = torch.tensor([ms_total, ms_e2e, ms_noexch or 0.0, (exch or {}).get("all_gather_us", 0.0),
                      (exch or {}).get("reduce_scatter_us", 0.0), (a2a or {}).get("ours_us", 0.0),
                      (a2a or {}).get("nccl_reference_us", 0.0)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e, ms_noexch_max, ag_us, rs_us, a2a_us, a2a_nccl_us = t.tolist()
    ms_step = ms_total / args.steps
    value = world * T / (ms_step * 1e-3)
    e2e_value = world * T / (ms_e2e / args.steps * 1e-3)

    # ---- roofline of the dominant kernel (grouped GEMMs, tensor-core bound) ----------------------------
    prof_ms = [(n, s_.elapsed_time(e_)) for n, s_, e_ in prof]
    roofline, roofline_dispatch, kernel_us = summarize_profile(prof_ms, cfg, L, ms_step, n_prof_layer_steps)
    try:
        ktable = kernel_table(prof_ms, cfg)
    except Exception as e:  # reporting extra: never let it take the contract line down
        ktable = [{"error": repr(e)}]

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    cpu_baseline = None
    if not args.no_cpu_baseline:
        rate, cores, t_layer = cpu_oracle_rate(cfg, L, args.cpu_sample_tokens, 3, 1)
        cpu_baseline = {
            "value": rate, "unit": "tokens/s", "cores": cores, "kind": "port",
            "sample": f"1 MoE layer fwd+bwd over {args.cpu_sample_tokens} tokens (median of 3), scaled linearly to {L} layers "
                      f"({t_layer:.2f} s per sampled layer); oracle/moe_oracle.py on torch CPU; {cores} threads chosen by a "
                      f"probe, {os.cpu_count()} host cores",
        }
    line = {
        "metric": METRIC, "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic", "loss": final_loss,
        "config": contract_config(L, world, default_parallelism(world, args.fsdp if fsdp_error is None else 0)),
        "run": {"parallelism_detail": (
                    f"fsdp={world}: tokens sharded; expert parameters fp32-sharded over the ranks, per layer cast+push all-gather "
                    f"with prefetch, " + ("re-gather in backward (reshard_after_forward=True)" if use_fsdp and eng.reshard else
                                          "gathered bf16 parameters resident until backward (reshard_after_forward=False)")
                    + ", reduce-scatter of the gradients, all-reduce of the replicated ones"
                    if use_fsdp else f"dp{world}: tokens sharded, independent replicas"
                    + (f" — FSDP expert sharding was requested but unavailable: {fsdp_error}" if fsdp_error else "")),
                "path": args.path, "mode": mode, "skew": args.skew,
                "l2": "per-step working set (weights+activations, > 10 GB at 48 layers) >> 126 MB L2"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "tokens/s", "h2d_bytes_per_step": x_host.numel() * 2, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches,
        "roofline": roofline,
        "roofline_dispatch": roofline_dispatch,
        "kernel_avg_us": kernel_us,
        "kernel_table": ktable,
        "cpu_baseline": cpu_baseline,
    }
    try:
        gref = gpu_reference_record(kernel_us, ms_step, L)
    except Exception:  # noqa: BLE001 — a side-by-side annotation must never cost the line
        gref = None
    if gref is not None:
        line["gpu_reference"] = gref
    if use_fsdp:
        nvl_peak = 770.0  # GB/s per direction per GPU: measured peer copy on this pool (B200_PROFILING.md); 900 nominal
        bpl = eng.bytes_per_layer
        ag_per_step, rs_per_step = (2 * L - 1) if eng.reshard else L, L
        step_bytes = ag_per_step * bpl["all_gather"] + rs_per_step * bpl["reduce_scatter"]
        ms_on = ms_total / args.steps
        ms_off = ms_noexch_max / args.steps if ms_noexch_max else None
        line["selfcheck"] = selfcheck
        line["roofline_comm"] = {
            "bound": "nvlink", "peak": nvl_peak, "unit": "GB/s per direction per GPU",
            "peak_source": "measured peer copy 770 GB/s (B200_PROFILING.md); nominal 900",
            "all_gather": {"kernel": "barrier + 2x allgather_push_kernel<fp32->bf16> + barrier (one layer's expert parameters)",
                           "us": ag_us, "bytes_out_per_rank": bpl["all_gather"],
                           "achieved": bpl["all_gather"] / (ag_us * 1e-6) / 1e9 if ag_us else None,
                           "frac": bpl["all_gather"] / (ag_us * 1e-6) / 1e9 / nvl_peak if ag_us else None},
            "reduce_scatter": {"kernel": "barrier + 2x reduce_scatter_pull_kernel<fp32 out> + barrier (one layer's gradients)",
                               "us": rs_us, "bytes_in_per_rank": bpl["reduce_scatter"],
                               "achieved": bpl["reduce_scatter"] / (rs_us * 1e-6) / 1e9 if rs_us else None,
                               "frac": bpl["reduce_scatter"] / (rs_us * 1e-6) / 1e9 / nvl_peak if rs_us else None},
            "timed": "exchange kernels alone on the exchange stream (max over ranks), after the timed steps",
            "per_step": {"all_gathers": ag_per_step, "reduce_scatters": rs_per_step, "nvlink_bytes_per_rank_per_direction": step_bytes,
                         "ms_if_serial": (ag_per_step * ag_us + rs_per_step * rs_us) * 1e-3},
            "step_ms_with_exchange": ms_on, "step_ms_exchange_off": ms_off,
            "exposed_exchange_frac": (1.0 - ms_off / ms_on) if ms_off else None,
            "limiting_collective": ("all_gather" if ag_per_step * ag_us >= rs_per_step * rs_us else "reduce_scatter"),
        }
        if a2a:
            line["selfcheck"]["ulysses_a2a"] = a2a["parity"]
            line["roofline_comm"]["ulysses_a2a"] = {
                "kernel": "staging copy + barrier + a2a_pull_kernel (C4 per-rank Q, 64 MiB, sp = N); not part of the timed step",
                "us": a2a_us, "nccl_reference_us": a2a_nccl_us, "bytes_per_rank_per_direction": a2a["bytes_per_rank_per_direction"],
                "achieved": a2a["bytes_per_rank_per_direction"] / (a2a_us * 1e-6) / 1e9 if a2a_us else None,
                "frac": a2a["bytes_per_rank_per_direction"] / (a2a_us * 1e-6) / 1e9 / nvl_peak if a2a_us else None}
    if fsdp_error:
        line["fsdp_error"] = fsdp_error
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
