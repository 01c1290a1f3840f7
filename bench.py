#!/usr/bin/env python
"""bench.py — headline benchmark of the quantized-linear hot path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--bs 32] [--impl ours|reference] [--quick] [--dump-outputs DIR]

Metric (BASELINE.json): tok/s of the Llama-3-8B int4 weight-only (tile_packed_to_4d, group_size=32) linear stack.
One "step" = one pass of all 32 layers of quantized linears over a batch of `bs` tokens per GPU (decode: one token
per sequence).  `value` is the whole-job tok/s with inputs resident in HBM, timed with CUDA events over K CUDA-graph
replays; `e2e` is the same pass driven from pinned HOST buffers (H2D of the step's activations + D2H of its result
inside the timed region) through the public API (quantize_ -> fuse_parallel_linears -> nn.Linear.forward ->
tensor-subclass dispatch -> torch.ops.ao_b200).  The same JSON line carries
  * the bs=1 half of the metric (`config.bs1`),
  * `gpu_reference`: the kernel the reference itself calls on a GPU for this path, aten._weight_int4pack_mm
    (int4_tile_packed_to_4d_tensor.py:287), on the same weights, same chain, same CUDA-graph protocol, same box,
  * `configs`: the other BASELINE configs (int8-dynamic, fp8-rowwise, mxfp8, nvfp4, 70B nvfp4-weight x fp8-act), each with
    its roofline fraction and the library kernel the reference calls (`torch._int_mm` / `torch._scaled_mm`) timed on
    the same shapes,
  * the roofline of the dominant kernel and a CPU baseline.

Weights are synthetic random-init of the real shapes (no checkpoints offline); 4.36 GB of packed weights per step
>> the 126 MB L2, so no L2 flush is needed between iterations.  Multi-GPU (torchrun): batch sharding, one NCCL
broadcast of the packed weights at setup, no collective in the forward; value = N*bs / max-over-ranks time.

--impl reference: the reference's own CPU implementation of the path (torchao's CPU int4 route is the PyTorch-core op
aten._weight_int4pack_mm_for_cpu, int4_opaque_tensor.py:414), whole steps timed on the host cores, this repo's package
never imported.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from (which may be read-only)

GROUP = 32
# (hidden, intermediate, kv, layers): SURVEY §8 shape table.  Kept here (not imported from ao_b200) so that the
# reference arm never loads this repo's package or its native libraries.
SHAPES = {"llama-3-8b": (4096, 14336, 1024, 32), "llama-3-70b": (8192, 28672, 1024, 80)}
METRIC = "tok/s Llama-3-8B int4-wo (tile_packed_to_4d, g=32) linear stack, decode"


def linears_of(name):
    h, i, kv, _ = SHAPES[name]
    return [("q_proj", h, h), ("k_proj", kv, h), ("v_proj", kv, h), ("o_proj", h, h),
            ("gate_proj", i, h), ("up_proj", i, h), ("down_proj", h, i)]


def params_per_layer(name):
    return sum(n * k for _, n, k in linears_of(name))


def workload_config(bs, world, layers):
    """The `config` object: identical for both arms (the driver compares them)."""
    return {"workload": f"Llama-3-8B int4-wo tile_packed_to_4d g=32, {layers} layers x 7 linears, bs={bs}/GPU decode",
            "bs_per_gpu": bs, "layers": layers, "parallelism": f"batch-shard x{world} (replicated weights)",
            "l2": "inputs larger than L2 (4.36 GB packed weights per step)"}


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops", 1590.0)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


def _traffic_from_profiles(bs):
    """dram bytes per launch of the dominant kernel from the committed ncu capture (profiles/r02_int4_traffic.json,
    written by scripts/ncu_traffic.py from an `ncu --set full` report); None when no capture is committed."""
    p = os.path.join(ROOT, "profiles", "r02_int4_traffic.json")
    try:
        with open(p) as f:
            return float(json.load(f)[f"bs{bs}"]["dram_bytes_per_launch"])
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            time.sleep(0.25)   # first sample before the timed region starts
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


BYTES_PER_PARAM = {"int4": 0.5 + 4.0 / GROUP, "int8": 1.0, "fp8": 1.0, "mxfp8": 1.0 + 1.0 / 32, "nvfp4": 0.5 + 1.0 / 16,
                   "nvfp4w_fp8a": 0.5 + 1.0 / 16}


def algo_bytes(model_name, fmt, layers, bs):
    """SURVEY §8d: packed weight bytes (incl. scales) + activations in + out, per step."""
    w = params_per_layer(model_name) * layers * BYTES_PER_PARAM[fmt]
    act = sum(bs * k * 2 + bs * n * 2 for _, n, k in linears_of(model_name)) * layers
    return w + act


# ------------------------------------------------------------------------------------------------ our arm
def build_stack(model_name, config, layers, device, fuse=True, seed=0):
    """Random-init Llama linear stack, quantized through the public API layer by layer (a 70B bf16 stack would not
    fit next to its quantized copy), then q|k|v and gate|up fused into one launch each."""
    import torch
    import torch.nn as nn

    from ao_b200.fusion import fuse_parallel_linears
    from ao_b200.models import LlamaLinearLayer, LlamaLinearStack, LlamaShape
    from ao_b200.quantization import quantize_

    h, i, kv, _ = SHAPES[model_name]
    shape = LlamaShape(model_name, h, i, kv, layers)
    stack = LlamaLinearStack(shape, layers=0, device=device, seed=seed)
    gen = torch.Generator(device=device).manual_seed(seed)
    for _ in range(layers):
        layer = LlamaLinearLayer(shape, device)
        with torch.no_grad():
            for p in layer.parameters():
                # unit gain per linear (std = 1 / sqrt(fan_in)): the 32- / 80-layer chain of bare linears neither
                # overflows nor underflows bf16, so every GEMM of the step sees realistic magnitudes
                p.copy_((torch.randn(p.shape, device=device, generator=gen) * (p.shape[-1] ** -0.5)).to(p.dtype))
        quantize_(layer, config)
        if fuse:
            fuse_parallel_linears(layer)
        stack.layers.append(layer)
    torch.cuda.empty_cache()
    return stack


def graph_of(fn, x_static):
    """Capture fn(x_static) in a CUDA graph (after eager warm-up on a side stream); returns (graph, y_static, launches)."""
    import torch

    launch_count = torch.ops.ao_b200.launch_count
    with torch.no_grad():
        for _ in range(2):
            fn(x_static)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side), torch.no_grad():
        fn(x_static)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    c0 = launch_count()
    with torch.cuda.graph(graph), torch.no_grad():
        y_static = fn(x_static)
    return graph, y_static, int(launch_count() - c0)


def time_replays(graph, steps, warmup, barrier):
    import torch

    for _ in range(warmup):
        graph.replay()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        graph.replay()
    e1.record()
    barrier()
    return e0.elapsed_time(e1) / steps


def run_ours(args):
    import torch
    import torch.distributed as dist

    import ao_b200  # noqa: F401  (loads the native library; raises if missing)
    from ao_b200.quantization import Int4WeightOnlyConfig

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    model_name = "llama-3-8b"
    hidden = SHAPES[model_name][0]
    layers = args.layers or SHAPES[model_name][3]
    peak, peak_tf, peak_src = _peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(vals):
        t = torch.tensor(vals, device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    # ---- setup: build, quantize through the public API, fuse, replicate the packed weights ----------
    model = build_stack(model_name, Int4WeightOnlyConfig(group_size=GROUP, int4_packing_format="tile_packed_to_4d"),
                        layers, dev, fuse=not args.no_fuse)
    bcast_bytes = 0
    if world > 1:
        from ao_b200.parallel import broadcast_packed_weights

        bcast_bytes = broadcast_packed_weights(model, src=0)  # the one collective of the whole job
        torch.cuda.synchronize()

    dumps = {}

    def measure(bs, with_e2e=True, clocks=False):
        gen = torch.Generator(device=dev).manual_seed(1 + rank)
        x_static = (torch.randn(bs, hidden, device=dev, generator=gen)).to(torch.bfloat16)
        graph, y_static, launches = graph_of(model, x_static)
        sampler = ClockSampler(local) if (clocks and rank == 0) else None
        if sampler:
            sampler.start()
        ms = time_replays(graph, args.steps, args.warmup, barrier)
        clk = sampler.stop() if sampler else None
        if args.dump_outputs:
            dumps[f"int4_stack_bs{bs}"] = y_static.float().cpu().numpy()   # the last timed step's model output
        res = {"ms": ms, "launches": launches, "clocks": clk, "finite": bool(torch.isfinite(y_static.float()).all())}
        if with_e2e:
            # end-to-end: host buffers, H2D + D2H inside the timed region
            x_host = x_static.cpu().pin_memory()
            y_host = torch.empty(bs, hidden, dtype=torch.bfloat16).pin_memory()
            for _ in range(args.warmup):
                x_static.copy_(x_host, non_blocking=True)
                graph.replay()
                y_host.copy_(y_static, non_blocking=True)
            barrier()
            e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e2.record()
            for _ in range(args.steps):
                x_static.copy_(x_host, non_blocking=True)
                graph.replay()
                y_host.copy_(y_static, non_blocking=True)
            e3.record()
            barrier()
            res["ms_e2e"] = e2.elapsed_time(e3) / args.steps
            # eager (no graph) end-to-end, for reference
            e4, e5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e4.record()
            with torch.no_grad():
                for _ in range(args.steps):
                    y = model(x_host.to(dev, non_blocking=True))
                    y_host.copy_(y, non_blocking=True)
            e5.record()
            barrier()
            res["ms_eager"] = e4.elapsed_time(e5) / args.steps
            res["h2d"], res["d2h"] = x_host.numel() * 2, y_host.numel() * 2
            res["ms"], res["ms_e2e"], res["ms_eager"] = max_over_ranks([res["ms"], res["ms_e2e"], res["ms_eager"]])
        else:
            res["ms"] = max_over_ranks([res["ms"]])[0]
        return res

    main = measure(args.bs, clocks=True)
    bs1 = measure(1) if args.bs != 1 else main
    if args.dump_outputs and rank == 0:
        write_dumps(args.dump_outputs, dumps)

    # ---- the kernel the reference calls on a GPU, same weights / chain / protocol / box --------------------
    gpu_ref = None
    if world == 1 and not args.quick:
        try:
            gpu_ref = gpu_reference_int4(model, hidden, [args.bs, 1] if args.bs != 1 else [1], args, dev, barrier)
        except Exception as ex:  # pragma: no cover
            gpu_ref = {"error": f"{type(ex).__name__}: {ex}"[:300]}
    del model
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs -------------------------------------------------------------------------
    sub = None
    if not args.quick:
        try:
            sub = other_configs(args, dev, world, rank, barrier, max_over_ranks, peak)
        except Exception as ex:  # pragma: no cover
            sub = {"error": f"{type(ex).__name__}: {ex}"[:300]}

    # ---- per-GEMM tensor-core roofline at prefill token counts (one GPU) ------------------------------------
    prefill = None
    if world == 1 and not args.quick:
        try:
            prefill = prefill_gemms(args, dev, peak_tf)
        except Exception as ex:  # pragma: no cover
            prefill = {"error": f"{type(ex).__name__}: {ex}"[:300]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    toks = world * args.bs
    value = toks / (main["ms"] * 1e-3)
    ab = algo_bytes(model_name, "int4", layers, args.bs)
    achieved = ab / (main["ms"] * 1e-3) / 1e9
    ab1 = algo_bytes(model_name, "int4", layers, 1)
    cfg = workload_config(args.bs, world, layers)
    cfg.update({"timing": "CUDA events over CUDA-graph replays, max over ranks", "weight_broadcast_bytes": bcast_bytes,
                "launches_per_layer": main["launches"] // layers,
                "fused_parallel_linears": not args.no_fuse,
                "bs1": {"value": world / (bs1["ms"] * 1e-3), "unit": "tok/s", "ms_per_step": bs1["ms"],
                        "e2e_value": world / (bs1["ms_e2e"] * 1e-3), "roofline_frac": ab1 / (bs1["ms"] * 1e-3) / 1e9 / peak}})
    out = {
        "metric": METRIC, "value": value, "unit": "tok/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": main["ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int4 weights -> bf16 MMA (f32 accumulate)", "data": "synthetic (random-init weights of the real shapes)",
        "config": cfg,
        "e2e": {"value": toks / (main["ms_e2e"] * 1e-3), "unit": "tok/s", "h2d_bytes_per_step": main["h2d"],
                "d2h_bytes_per_step": main["d2h"], "mode": "pinned host -> H2D -> CUDA-graph replay of model.forward -> D2H",
                "eager_no_graph_tok_s": toks / (main["ms_eager"] * 1e-3), "bs1_value": world / (bs1["ms_e2e"] * 1e-3)},
        "gpu_launches": main["launches"] * args.steps,
        "clocks": main["clocks"],
        "roofline": {"bound": "hbm", "kernel": "ao::tsg::ts_gemm_kernel<ao::int4k::Int4Fmt, 32>", "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak, "traffic": _traffic_from_profiles(args.bs),
                     "algorithmic_bytes_per_launch": ab / max(1, main["launches"]), "peak_source": peak_src,
                     "algorithmic_bytes_per_step": ab, "launches_per_step": main["launches"]},
        "finite_outputs": main["finite"],
    }
    if gpu_ref is not None:
        out["gpu_reference"] = gpu_ref
        for key, ours_ms in ((f"bs{args.bs}", main["ms"]), ("bs1", bs1["ms"])):
            if isinstance(gpu_ref.get(key), dict) and gpu_ref[key].get("ms_per_step"):
                gpu_ref[key]["speedup"] = gpu_ref[key]["ms_per_step"] / ours_ms
    if sub is not None:
        out["configs"] = sub
    if prefill is not None:
        out["prefill"] = prefill
    if world == 1:
        out["cpu_baseline"] = cpu_baseline(args.bs)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


DUMP_LIMIT = 64 << 20


def write_dumps(out_dir, arrays):
    """Write each output as out_dir/<name>.npy in float32.  Above DUMP_LIMIT bytes in all, an array keeps a fixed,
    seeded sample of its rows (in order), so two runs with the same arguments write files that compare element for
    element."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    items = sorted(arrays.items(), key=lambda kv: kv[1].nbytes)
    budget = DUMP_LIMIT - 1024 * len(items)   # room for the .npy headers
    for i, (name, a) in enumerate(items):
        a = np.ascontiguousarray(a, dtype=np.float32)
        share = budget // (len(items) - i)
        if a.nbytes > share:
            keep = share // (a.nbytes // a.shape[0])
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        budget -= a.nbytes
        np.save(os.path.join(out_dir, name + ".npy"), a)


def gpu_reference_int4(model, hidden, batch_sizes, args, dev, barrier):
    """aten._weight_int4pack_mm (PyTorch-core tinygemm kernel; what Int4TilePackedTo4dTensor's handler calls at
    int4_tile_packed_to_4d_tensor.py:287) on OUR packed weights (the layouts are bit-identical, tests/test_int4_gpu.py),
    the same dependent chain, CUDA-graph replays, CUDA events.  This is the kernel-level ceiling of the reference's
    eager or torch.compile'd forward for this path (compile removes Python and pointwise overhead around the extern
    GEMM call, not the GEMM).  Timed as the reference would launch it (7 GEMMs / layer) and, for completeness, on
    the fused q|k|v / gate|up weights (4 / layer) where the model holds them."""
    import torch

    mm = torch.ops.aten._weight_int4pack_mm

    def weights_of(layer, names):
        return [(getattr(layer, n).weight.qdata.contiguous(), getattr(layer, n).weight.scale_and_zero.contiguous()) for n in names]

    per_layer = [weights_of(L, ["q_proj", "k_proj", "v_proj", "o_proj", "gate_proj", "up_proj", "down_proj"]) for L in model.layers]
    fused_layers = None
    if hasattr(model.layers[0].q_proj, "_group"):
        fused_layers = []
        for L in model.layers:
            gq, gg = L.q_proj._group.weight, L.gate_proj._group.weight
            fused_layers.append([(gq.qdata, gq.scale_and_zero), per_layer[len(fused_layers)][3], (gg.qdata, gg.scale_and_zero),
                                 per_layer[len(fused_layers)][6]])
    h = hidden
    inter = per_layer[0][4][0].shape[0] * 8

    def unfused(x):
        for q, k, v, o, g, u, d in per_layer:
            qo = mm(x, q[0], GROUP, q[1])
            mm(x, k[0], GROUP, k[1])
            mm(x, v[0], GROUP, v[1])
            oo = mm(qo, o[0], GROUP, o[1])
            go = mm(oo, g[0], GROUP, g[1])
            mm(oo, u[0], GROUP, u[1])
            x = mm(go, d[0], GROUP, d[1])
        return x

    def fused(x):
        for qkv, o, gu, d in fused_layers:
            a = mm(x, qkv[0], GROUP, qkv[1])
            oo = mm(a[:, :h].contiguous(), o[0], GROUP, o[1])
            b = mm(oo, gu[0], GROUP, gu[1])
            x = mm(b[:, :inter].contiguous(), d[0], GROUP, d[1])
        return x

    out = {"kernel": "aten._weight_int4pack_mm (torch " + torch.__version__ + ")",
           "protocol": "same packed weights, same dependent chain, CUDA-graph replays, CUDA events"}
    steps = args.steps
    for bs in batch_sizes:
        x = torch.randn(bs, hidden, device=dev).to(torch.bfloat16)
        rec = {}
        for name, fn in (("unfused_7_per_layer", unfused), ("fused_4_per_layer", fused if fused_layers else None)):
            if fn is None:
                continue
            g, _, _ = graph_of(fn, x)
            rec[name + "_ms"] = time_replays(g, steps, 3, barrier)
            del g
        best = min(v for v in rec.values())
        rec["ms_per_step"] = best
        rec["value"] = bs / (best * 1e-3)
        rec["unit"] = "tok/s"
        out[f"bs{bs}"] = rec
    return out


def prefill_gemms(args, dev, peak_tf):
    """Per-GEMM tensor-core roofline at prefill token counts (SURVEY section 8d: the only place the north star's
    ">= 70 % of the tensor-core roofline" clause applies): the four fused Llama-3-8B projections at M = 512 and 4096,
    int4 weight-only (the prefill-shaped TS kernel, csrc/ts_prefill.cuh) with the kernel the reference calls
    (aten._weight_int4pack_mm, M = 512 only: it needs tens of milliseconds at 4096) and cuBLAS bf16 (F.linear on
    bf16 weights, what `peak_tf` was measured with) beside it; fp8-rowwise, int8-dynamic, mxfp8 and nvfp4 with their library kernels.
    TFLOP/s = 2 M N K / time, CUDA events over back-to-back launches on weights + activations larger than L2 for
    the big shapes; `frac` is against the measured bf16 peak (x2 for the 8-bit kinds)."""
    import torch

    ops = torch.ops.ao_b200
    h, inter, kv, _ = SHAPES["llama-3-8b"]
    shapes = [("qkv", h + 2 * kv, h), ("o", h, h), ("gate_up", 2 * inter, h), ("down", h, inter)]

    def t_us(fn, iters):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters * 1e3

    out = {"peak_bf16_tflops": peak_tf, "unit": "TFLOP/s", "note": "one GEMM per entry; frac = TFLOP/s over the measured bf16 "
           "tensor peak (x2 for fp8 / int8 / mxfp8, x4 for nvfp4); int4 runs ao::tsp::ts_prefill_kernel, the others lowp_linear_kernel in 128-token blocks"}
    for M in (512, 4096):
        for name, N, K in shapes:
            flops = 2.0 * M * N * K
            x = torch.randn(M, K, device=dev).to(torch.bfloat16)
            rec = {}
            qd = torch.randint(-2**31, 2**31 - 1, (N // 8, K // 128, 32, 4), device=dev, dtype=torch.int32)
            sz = ((torch.rand(K // GROUP, N, 2, device=dev) - 0.5) * 0.004).to(torch.bfloat16)
            us = t_us(lambda: ops.int4_tilepacked_linear(x, qd, GROUP, sz, None, N, 1), 5)
            rec["int4"] = {"us": us, "tflops": flops / us / 1e6, "frac": flops / us / 1e6 / peak_tf}
            if M == 512:
                lus = t_us(lambda: torch.ops.aten._weight_int4pack_mm(x, qd, GROUP, sz), 2)
                rec["int4"]["aten_int4pack_mm_us"] = lus
            del qd, sz
            w = torch.randn(N, K, device=dev).to(torch.bfloat16)
            rec["bf16_cublas_us"] = t_us(lambda: torch.nn.functional.linear(x, w), 5)
            for fmt in ("fp8", "int8", "mxfp8", "nvfp4"):
                if fmt == "mxfp8":
                    wq, ws = ops.mxfp8_quantize(w, True)
                    xq, xs = ops.mxfp8_quantize(x, True)
                    fn = lambda: ops.mxfp8_linear(xq, xs, wq, ws, None)
                    lib = lambda: torch._scaled_mm(xq, wq.t(), scale_a=xs.view(torch.float8_e8m0fnu), scale_b=ws.view(torch.float8_e8m0fnu),
                                                   out_dtype=torch.bfloat16)
                elif fmt == "nvfp4":
                    wq, ws = ops.nvfp4_quantize(w, None, True)
                    xq, xs = ops.nvfp4_quantize(x, None, True)
                    fn = lambda: ops.nvfp4_linear(xq, xs, None, wq, ws, None, None)
                    lib = lambda: torch._scaled_mm(xq.view(torch.float4_e2m1fn_x2), wq.view(torch.float4_e2m1fn_x2).t(),
                                                   scale_a=xs.view(torch.float8_e4m3fn), scale_b=ws.view(torch.float8_e4m3fn),
                                                   out_dtype=torch.bfloat16)
                elif fmt == "fp8":
                    wq, ws = ops.fp8_quantize_rowwise(w)
                    xq, xs = ops.fp8_quantize_rowwise(x)
                    fn = lambda: ops.fp8_rowwise_linear(xq, xs.reshape(-1), wq, ws.reshape(-1), None)
                    lib = lambda: torch._scaled_mm(xq, wq.t(), scale_a=xs.reshape(-1, 1), scale_b=ws.reshape(1, -1),
                                                   out_dtype=torch.bfloat16, use_fast_accum=True)
                else:
                    wq, ws = ops.int8_quantize_rowwise(w)
                    xq, xs = ops.int8_quantize_rowwise(x)
                    fn = lambda: ops.int8_dyn_linear(xq, xs.reshape(-1), wq, ws.reshape(-1), None)
                    lib = lambda: torch._int_mm(xq, wq.t())
                us = t_us(fn, 5)
                mul = 4 if fmt == "nvfp4" else 2   # dense peak of the kind relative to bf16
                rec[fmt] = {"us": us, "tflops": flops / us / 1e6, "frac": flops / us / 1e6 / (mul * peak_tf)}
                try:
                    rec[fmt]["library_us"] = t_us(lib, 5)
                except Exception as ex:  # pragma: no cover
                    rec[fmt]["library_error"] = f"{type(ex).__name__}: {ex}"[:120]
                del wq, ws, xq, xs
            out[f"M{M}_{name}"] = rec
            del x, w
            torch.cuda.empty_cache()
    return out


def other_configs(args, dev, world, rank, barrier, max_over_ranks, peak):
    """BASELINE configs 3-5 (+ mxfp8, nvfp4 x nvfp4): ms/step, algorithmic-bytes roofline fraction and the library
    kernel the reference calls for the same GEMMs (`torch._int_mm`, `torch._scaled_mm`), on the same box in the same
    run.  Under --gpus N only configs 4 and 5 run, at their BASELINE batch (global 32 resp. 256 sharded over N)."""
    import torch

    from ao_b200.prototype.mx_formats import (MXDynamicActivationMXWeightConfig, NVFP4DynamicActivationNVFP4WeightConfig)
    from ao_b200.prototype.mx_formats.inference_workflow import NVFP4WeightFloat8ActivationConfig
    from ao_b200.quantization import (Float8DynamicActivationFloat8WeightConfig, Int8DynamicActivationInt8WeightConfig, PerRow)

    steps = args.steps
    plans = []
    if world == 1:
        plans = [
            ("int8_dyn_8b", "llama-3-8b", "int8", Int8DynamicActivationInt8WeightConfig(), [32], "config 3"),
            ("fp8_rowwise_8b", "llama-3-8b", "fp8", Float8DynamicActivationFloat8WeightConfig(granularity=PerRow()), [32, 4], "config 4 (per-GPU share of bs=32 over 8 GPUs is M=4)"),
            ("mxfp8_8b", "llama-3-8b", "mxfp8", MXDynamicActivationMXWeightConfig(), [32], "mxfp8"),
            ("nvfp4_8b", "llama-3-8b", "nvfp4", NVFP4DynamicActivationNVFP4WeightConfig(use_dynamic_per_tensor_scale=False), [32], "nvfp4 x nvfp4"),
            ("nvfp4w_fp8a_70b", "llama-3-70b", "nvfp4w_fp8a", NVFP4WeightFloat8ActivationConfig(), [32], "config 5 (per-GPU share of bs=256 over 8 GPUs is M=32)"),
        ]
    else:
        plans = [
            ("fp8_rowwise_8b", "llama-3-8b", "fp8", Float8DynamicActivationFloat8WeightConfig(granularity=PerRow()), [max(1, 32 // world)], f"config 4: global bs=32 over {world} GPUs"),
            ("nvfp4w_fp8a_70b", "llama-3-70b", "nvfp4w_fp8a", NVFP4WeightFloat8ActivationConfig(), [max(1, 256 // world)], f"config 5: global bs=256 over {world} GPUs"),
        ]
    out = {}
    for key, model_name, fmt, cfg, batch_sizes, note in plans:
        rec = {"note": note, "model": model_name}
        try:
            layers = SHAPES[model_name][3]
            hidden = SHAPES[model_name][0]
            stack = build_stack(model_name, cfg, layers, dev, fuse=not args.no_fuse, seed=1)
            for bs in batch_sizes:
                x = torch.randn(bs, hidden, device=dev).to(torch.bfloat16)
                g, y, launches = graph_of(stack, x)
                ms = max_over_ranks([time_replays(g, steps, 3, barrier)])[0]
                ab = algo_bytes(model_name, fmt, layers, bs)
                r = {"ms_per_step": ms, "value": world * bs / (ms * 1e-3), "unit": "tok/s", "launches_per_step": launches,
                     "roofline_frac": ab / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_step": ab,
                     "finite": bool(torch.isfinite(y.float()).all())}
                del g
                if world == 1:
                    try:
                        r["library"] = library_chain(stack, fmt, x, steps, barrier)
                        if r["library"].get("ms_per_step"):
                            r["library"]["speedup"] = r["library"]["ms_per_step"] / ms
                    except Exception as ex:
                        r["library"] = {"error": f"{type(ex).__name__}: {ex}"[:240]}
                rec[f"bs{bs}"] = r
            del stack
        except Exception as ex:  # pragma: no cover
            rec["error"] = f"{type(ex).__name__}: {ex}"[:300]
        torch.cuda.empty_cache()
        out[key] = rec
    return out


def library_chain(stack, fmt, x, steps, barrier):
    """The GEMM library calls the reference makes for this format, on the same (fused) weights and the same chain:
    int8 -> torch._int_mm (int8/kernels.py:40,70); fp8 -> torch._scaled_mm rowwise (float8/inference.py:104-123);
    mxfp8 / nvfp4 -> torch._scaled_mm block-scaled (mx_tensor.py:803-810, nvfp4_tensor.py:561-578).  The activation
    quantization in front of each GEMM uses this engine's fused quantizer (the reference would run several eager
    kernels there), and the library's separate scale / bias epilogue kernels are NOT added: both favour the library."""
    import torch

    ops = torch.ops.ao_b200
    if fmt == "nvfp4w_fp8a":
        return {"note": "no library kernel exists for nvfp4-weight x fp8-activation (SURVEY §0-5)"}
    groups = []
    for L in stack.layers:
        gq = L.q_proj._group.weight if hasattr(L.q_proj, "_group") else None
        gg = L.gate_proj._group.weight if hasattr(L.gate_proj, "_group") else None
        if gq is None or gg is None:
            return {"note": "unfused stack: library chain not built"}
        groups.append((gq, L.o_proj.weight, gg, L.down_proj.weight))
    h = x.shape[1]
    inter = groups[0][3].shape[1]

    def gemm(a, w):
        K = a.shape[1]
        if fmt == "int8":
            q, s = ops.int8_quantize_rowwise(a)
            return torch._int_mm(q, w.qdata.t()).to(torch.bfloat16)   # the cast stands in for the scale epilogue
        if fmt == "fp8":
            q, s = ops.fp8_quantize_rowwise(a)
            return torch._scaled_mm(q, w.qdata.t(), scale_a=s.reshape(-1, 1), scale_b=w.scale.reshape(1, -1).float(),
                                    out_dtype=torch.bfloat16, use_fast_accum=True)
        if fmt == "mxfp8":
            q, s = ops.mxfp8_quantize(a, True)
            return torch._scaled_mm(q, w.qdata.t(), scale_a=s.view(torch.float8_e8m0fnu), scale_b=w.scale.view(torch.float8_e8m0fnu),
                                    out_dtype=torch.bfloat16)
        if fmt == "nvfp4":
            q, s = ops.nvfp4_quantize(a, None, True)
            return torch._scaled_mm(q.view(torch.float4_e2m1fn_x2), w.qdata.view(torch.float4_e2m1fn_x2).t(),
                                    scale_a=s.view(torch.float8_e4m3fn), scale_b=w.scale.view(torch.float8_e4m3fn),
                                    out_dtype=torch.bfloat16)
        raise ValueError(fmt)

    def chain(xx):
        for qkv, o, gu, d in groups:
            a = gemm(xx, qkv)
            oo = gemm(a[:, :h].contiguous(), o)
            b = gemm(oo, gu)
            xx = gemm(b[:, :inter].contiguous(), d)
        return xx

    if fmt == "int8" and x.shape[0] <= 16:
        return {"note": "torch._int_mm needs M > 16"}
    g, _, _ = graph_of(chain, x)
    ms = time_replays(g, steps, 3, barrier)
    name = "torch._int_mm" if fmt == "int8" else "torch._scaled_mm"
    return {"kernel": name + " (cuBLASLt, torch " + torch.__version__ + ")", "ms_per_step": ms,
            "chain": "fused q|k|v and gate|up weights, 4 GEMMs per layer, this engine's activation quantizer in front"}


# ------------------------------------------------------------------------------------------------ CPU arm
def host_threads():
    """Threads the CPU arm may use, deterministically: the affinity mask, capped by the cgroup CPU quota (a
    container's os.cpu_count() can exceed what it may run; oversubscribed, the CPU int4 kernel is >10x slower)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:   # cgroup v2
            q, p = f.read().split()
            if q != "max":
                quota = float(q) / float(p)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f1, open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f2:
                q, p = float(f1.read()), float(f2.read())
                if q > 0:
                    quota = q / p
        except Exception:
            pass
    if quota is not None:
        n = max(1, min(n, int(math.floor(quota + 1e-6)) or 1))
    return n


class CpuInt4Stack:
    """The reference's own CPU implementation of the path: torchao's CPU int4 route (Int4OpaqueTensor,
    torchao/prototype/quantization/int4/int4_opaque_tensor.py:197,414; BASELINE config[0]) is two PyTorch-core ops,
    aten._convert_weight_to_int4pack_for_cpu + aten._weight_int4pack_mm_for_cpu.  `distinct` layers of packed weights
    (each 136 MB, together far beyond the last-level cache) are built once and cycled through the 32 layers of a
    step; every linear of every layer is executed in every step (nothing is extrapolated)."""

    def __init__(self, bs, threads, distinct=8):
        import torch

        self.torch = torch
        torch.set_num_threads(threads)
        self.threads = threads
        self.kind = "reference"
        self.what = ("aten._weight_int4pack_mm_for_cpu (the PyTorch-core kernel the reference's CPU int4 path calls, "
                     "int4_opaque_tensor.py:414)")
        gen = torch.Generator().manual_seed(0)
        self.layers = []
        for _ in range(distinct):
            mats = []
            for _, n, k in linears_of("llama-3-8b"):
                q = torch.randint(0, 16, (n, k), dtype=torch.int32, generator=gen)
                packed = torch.ops.aten._convert_weight_to_int4pack_for_cpu(q, 1)
                sz = (torch.rand(k // GROUP, n, 2, generator=gen) * 0.01).to(torch.bfloat16)
                mats.append((packed, sz))
            self.layers.append(mats)
        self.x = torch.randn(bs, SHAPES["llama-3-8b"][0], generator=gen).to(torch.bfloat16)
        self.distinct = distinct

    def step(self, n_layers=32):
        mm = self.torch.ops.aten._weight_int4pack_mm_for_cpu
        x = self.x
        for li in range(n_layers):
            q, k, v, o, g, u, d = self.layers[li % self.distinct]
            qo = mm(x, q[0], GROUP, q[1])
            mm(x, k[0], GROUP, k[1])
            mm(x, v[0], GROUP, v[1])
            oo = mm(qo, o[0], GROUP, o[1])
            go = mm(oo, g[0], GROUP, g[1])
            mm(oo, u[0], GROUP, u[1])
            x = mm(go, d[0], GROUP, d[1])
        return x


class OraclePortStack:
    """Fallback when the PyTorch build has no CPU int4 op: the oracle's C restatement (kind "port")."""

    def __init__(self, bs, threads, distinct=2):
        import numpy as np

        from oracle import oracle as o

        self.o = o
        os.environ["OMP_NUM_THREADS"] = str(threads)
        o.lib().ao_oracle_set_threads(int(threads))
        self.threads, self.kind, self.what, self.distinct = threads, "port", "oracle/ao_oracle.c int4_linear", distinct
        rng = np.random.default_rng(0)
        self.layers = []
        for _ in range(distinct):
            mats = []
            for _, n, k in linears_of("llama-3-8b"):
                qd = rng.integers(-2**31, 2**31 - 1, size=(n // 8, k // 128, 32, 4), dtype=np.int64).astype(np.int32)
                mats.append((qd, o.f32_to_bf16((rng.random((k // GROUP, n, 2), dtype=np.float32) * 0.01).astype(np.float32))))
            self.layers.append(mats)
        self.xs = {k: o.f32_to_bf16(rng.standard_normal((bs, k), dtype=np.float32)) for k in (4096, 14336)}

    def step(self, n_layers=32):
        for li in range(n_layers):
            for (qd, sz), (_, n, k) in zip(self.layers[li % self.distinct], linears_of("llama-3-8b")):
                self.o.int4_linear(self.xs[k], qd, sz, GROUP)


def cpu_stack(bs, threads, distinct=8):
    try:
        import torch

        torch.ops.aten._weight_int4pack_mm_for_cpu  # noqa: B018
        return CpuInt4Stack(bs, threads, distinct)
    except Exception:
        return OraclePortStack(bs, threads)


def cpu_baseline(bs):
    """Bounded sample on the host cores, at the headline batch size: one whole step (all 32 layers x 7 linears) after
    one warm-up step over 2 distinct layers' worth of weights."""
    threads = host_threads()
    try:
        st = cpu_stack(bs, threads, distinct=2)
        st.step(2)
        t0 = time.perf_counter()
        st.step(32)
        dt = time.perf_counter() - t0
        return {"value": bs / dt, "unit": "tok/s", "cores": st.threads, "kind": st.kind,
                "sample": f"one whole step (32 layers x 7 int4 g=32 linears, weights of {st.distinct} distinct layers cycled) at bs={bs}, {st.what}"}
    except Exception as ex:  # pragma: no cover
        return {"value": None, "unit": "tok/s", "cores": threads, "kind": "port", "sample": f"failed: {ex}"}


def run_reference(args):
    """The reference arm: this repo's package is never imported here."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    threads = host_threads()
    layers = args.layers or SHAPES["llama-3-8b"][3]
    st = cpu_stack(args.bs, threads, distinct=8)
    warm = max(1, min(args.warmup, 3))     # a CPU step is 0.2-1.5 s: three warm-up steps settle the caches / threads
    for _ in range(warm):
        st.step(layers)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        st.step(layers)
    dt = time.perf_counter() - t0
    ms_step = dt / args.steps * 1e3
    value = args.bs / (ms_step * 1e-3)
    sample = (f"every step = all {layers} layers x 7 int4 g=32 linears at bs={args.bs} (weights of {st.distinct} distinct layers, "
              f"{st.distinct * 136} MB packed, cycled), {st.what}, {st.threads} threads (affinity / cgroup quota)")
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": "tok/s", "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "warmup_steps_run": warm, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "int4 weights -> bf16 (CPU)", "data": "synthetic (random-init weights of the real shapes)",
           "config": workload_config(args.bs, world, layers),
           "cpu_baseline": {"value": value, "unit": "tok/s", "cores": st.threads, "kind": st.kind, "sample": sample},
           "e2e": {"value": value, "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "timed_region_s": dt}
    print(json.dumps(out))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--bs", type=int, default=32, help="tokens per GPU per step (decode batch)")
    ap.add_argument("--layers", type=int, default=0, help="override layer count (debug only; default = 32)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--quick", action="store_true", help="headline only: skip gpu_reference and the other configs")
    ap.add_argument("--no-fuse", action="store_true", help="7 launches per layer (q, k, v, gate, up not fused)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the headline stack's output of the last timed step at --bs and at "
                         "bs=1 as DIR/int4_stack_bs<N>.npy (float32, seeded inputs, at most 64 MB in all)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if a.warmup < 3:
        a.warmup = 3
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
