#!/usr/bin/env python
"""bench.py -- PTQ hot-path throughput on the BASELINE workload (Llama-3-8B NVFP4 PTQ).

A "step" is one calibration batch (8 x 512 = 4096 tokens of synthetic bf16 activations) through the
quantizer hot path of the whole model: for each of the 32 x 7 input quantizers a calibration collect
(per-tensor |x| max folded into the amax arena) and, after the arena all-reduce + export, the NVFP4
block-16 two-level-scale fake-quant forward of the same activation.  GEMMs / attention are not part of
the path.  With N GPUs the decoder layers are sharded contiguously over ranks (strong scaling of the
fixed model): the ranks form a pipeline -- every step a rank receives the hidden state of the next micro-batch
from rank - 1 and sends its own to rank + 1 (NCCL point-to-point over NVLink, overlapped with the kernels) -- and
the only collective is ONE all-reduce(MAX) of the amax arena per calibration job (the timed K steps are one job).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Prints one JSON line (rank 0).  See DESIGN.md "Measurement" for every key.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ptq_calib_tokens_per_sec"
UNIT = "tokens/s"
BATCH, SEQ = 8, 512
TOKENS = BATCH * SEQ


def measured_traffic():
    """dram bytes per launch of the dominant kernel from the newest committed ncu capture (or None)."""
    import glob

    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))
    if not files:
        return None, None
    try:
        t = json.load(open(files[-1]))
        return int(t["bytes_per_launch_step_average"]), os.path.relpath(files[-1], ROOT) + ": " + t["note"]
    except Exception:  # noqa: BLE001
        return None, None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for ts, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                smax = float(f[2])
                if t0 - 0.05 <= ts <= t1 + 0.15:
                    sm.append(float(f[1]))
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                        if v.lower().startswith("active"):
                            reasons.add(name)
            except ValueError:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's path on the host cores
# ------------------------------------------------------------------------------------------------
class CpuOracleSample:
    """A bounded sample of the step for the CPU arms: ``tokens`` tokens through the 7 input quantizers of
    ONE decoder layer -- calibration collect + NVFP4 fake quant -- with the C/OpenMP oracle
    (oracle/oracle_c.c, bit-identical to the NumPy oracle that is pinned to the reference), all host cores."""

    def __init__(self, tokens: int):
        import numpy as np

        from model_optimizer_b200.engine import LLAMA3_8B

        os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")  # no spinning if the cgroup grants fewer CPUs than it shows
        os.environ.setdefault("OMP_PROC_BIND", "false")
        from oracle import oracle_c

        self.oc = oracle_c
        self.tokens = tokens
        rng = np.random.default_rng(0)
        self.inputs = []
        for _, cin, _ in LLAMA3_8B.linears():
            f = rng.standard_normal((tokens, cin), dtype=np.float32)
            self.inputs.append((f.view(np.uint32) >> 16).astype(np.uint16))  # bf16 bit patterns (truncated)
        self.cores = self._pick_threads()

    def _usable_cpus(self) -> int:
        n = os.cpu_count() or 1
        try:
            n = min(n, len(os.sched_getaffinity(0)))
        except AttributeError:
            pass
        try:  # cgroup v2 CPU quota
            quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
            if quota != "max":
                n = min(n, max(1, int(float(quota) / float(period) + 0.5)))
        except Exception:  # noqa: BLE001
            pass
        return max(1, n)

    def _pick_threads(self) -> int:
        """All the host threads that actually help: time one tensor at a few thread counts (containers often
        expose more CPUs than they may use) and keep the fastest."""
        limit = self._usable_cpus()
        cands = sorted({c for c in (limit, limit // 2, limit // 4, 64, 32, 16, 8) if 1 <= c <= limit})
        bits = self.inputs[0]
        best, best_t = cands[-1], float("inf")
        for c in cands:
            self.oc.set_threads(c)
            self.oc.amax_bf16(bits)
            t0 = time.perf_counter()
            self.oc.fake_quant_nvfp4_bf16(bits, 4.5)
            t = time.perf_counter() - t0
            if t < best_t:
                best, best_t = c, t
        return self.oc.set_threads(best)

    def step(self) -> float:
        t0 = time.perf_counter()
        for bits in self.inputs:
            amax = self.oc.amax_bf16(bits)                  # calibration collect
            self.oc.fake_quant_nvfp4_bf16(bits, amax)       # fake-quant forward
        return time.perf_counter() - t0

    def describe(self, n: int) -> str:
        return (f"{n} x ({self.tokens} tokens through the 7 input quantizers of 1 of 32 decoder layers: collect + "
                f"NVFP4 fake quant, C/OpenMP oracle port of the reference, {self.cores} threads); "
                "tokens/s = tokens / (32 * seconds)")


def cpu_tokens_per_sec(sample_tokens: int, seconds: float, n_layers: int = 32) -> float:
    """sample_tokens through ONE layer took `seconds` -> the 32-layer model needs 32x that per token."""
    return sample_tokens / (seconds * n_layers)


class CpuReferenceSample:
    """The REAL reference on the host cores (BASELINE.md section 3): for the 7 input quantizers of ONE decoder
    layer, ``reduce_amax`` (quantization/utils/core_utils.py:147) + ``NVFP4QTensor.quantize -> dequantize``
    (qtensor/nvfp4_tensor.py:253-408; the reference has no CPU NVFP4 fake quant, tensor_quant.py:172) from the
    unmodified install in ``baseline/_ref``.  torch threads = the CPUs this process may use."""

    def __init__(self, tokens: int):
        import torch

        from baseline import ref_env
        from model_optimizer_b200.engine import LLAMA3_8B

        ref_env.activate()
        from modelopt.torch.quantization.qtensor import NVFP4QTensor
        from modelopt.torch.quantization.utils import reduce_amax

        self.torch, self.q, self.reduce_amax = torch, NVFP4QTensor, reduce_amax
        self.tokens = tokens
        self.cores = CpuOracleSample._usable_cpus(self)
        torch.set_num_threads(self.cores)
        g = torch.Generator().manual_seed(0)
        self.inputs = [torch.randn(tokens, cin, generator=g).to(torch.bfloat16) for _, cin, _ in LLAMA3_8B.linears()]

    def step(self) -> float:
        t0 = time.perf_counter()
        with self.torch.no_grad():
            for x in self.inputs:
                amax = self.reduce_amax(x)                                   # calibration collect
                wsf2 = amax.float() / (6.0 * 448.0)
                qt, sf, sf2 = self.q.quantize(x, 16, weights_scaling_factor_2=wsf2)
                qt.dequantize(dtype=x.dtype, scale=sf, double_scale=sf2, block_sizes={-1: 16})   # fake-quant forward
        return time.perf_counter() - t0

    def describe(self, n: int) -> str:
        return (f"{n} x ({self.tokens} tokens through the 7 input quantizers of 1 of 32 decoder layers: the reference's "
                f"own reduce_amax + NVFP4QTensor.quantize->dequantize from baseline/_ref, torch CPU, "
                f"torch.get_num_threads()={self.torch.get_num_threads()}, os.cpu_count()={os.cpu_count()}); "
                "tokens/s = tokens / (32 * seconds)")


def _reference_available() -> bool:
    try:
        from baseline import ref_env

        return ref_env.available()
    except Exception:  # noqa: BLE001
        return False


def cpu_arm(steps: int, warmup: int, budget_s: float | None = None):
    """-> (tokens/s, seconds per sample step, cpu_baseline dict).  ``kind: "reference"`` (the real reference
    functions) when baseline/_ref travelled with the snapshot, with the C/OpenMP oracle port as a second figure;
    else the port alone."""
    port = CpuOracleSample(TOKENS)
    port.step()
    tp = min(port.step() for _ in range(2))
    port_v = cpu_tokens_per_sec(port.tokens, tp)
    if _reference_available():
        ref = CpuReferenceSample(TOKENS)
        for _ in range(max(1, min(warmup, 1))):
            ref.step()
        times = []
        t0 = time.perf_counter()
        while len(times) < steps and (budget_s is None or time.perf_counter() - t0 < budget_s or len(times) < 2):
            times.append(ref.step())
        t = sum(times) / len(times)
        v = cpu_tokens_per_sec(ref.tokens, t)
        return v, t, {"value": round(v, 2), "unit": UNIT, "cores": ref.cores, "kind": "reference",
                      "os_cpu_count": os.cpu_count(), "torch_threads": ref.torch.get_num_threads(),
                      "sample": ref.describe(len(times)),
                      "port": {"value": round(port_v, 2), "cores": port.cores,
                               "what": "C/OpenMP oracle port of the same sample (oracle/oracle_c.c)"}}
    times = [port.step() for _ in range(max(steps, 1))]
    t = sum(times) / len(times)
    v = cpu_tokens_per_sec(port.tokens, t)
    return v, t, {"value": round(v, 2), "unit": UNIT, "cores": port.cores, "kind": "port",
                  "os_cpu_count": os.cpu_count(), "sample": port.describe(len(times))}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from model_optimizer_b200.engine import PLANS

    v, t, base = cpu_arm(args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(args.gpus, PLANS[args.model]),
        "cpu_baseline": base,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(n_gpus, plan):
    gb = plan.act_elems_per_token() * TOKENS * 2 * plan.n_layers / 1e9
    return {
        "workload": f"{plan.name} NVFP4 PTQ hot path: per step one calibration batch (8x512 tokens, bf16) "
                    f"through all {plan.n_layers}x7 input quantizers = amax collect + export + NVFP4 "
                    "block-16 two-level fake-quant forward (GEMMs/attention not on the path)",
        "global_batch": BATCH, "seq_len": SEQ, "tokens_per_step": TOKENS, "layers": plan.n_layers,
        "quantizers": plan.n_layers * 7,
        "parallelism": f"layer-sharded x{n_gpus} (pipeline: hidden-state hand-off rank g -> g+1 over NVLink every step, "
                       "overlapped; ONE NCCL all-reduce(MAX) of the amax arena per calibration job = per timed "
                       "region)",
        "l2_policy": "inputs larger than L2: one distinct activation buffer per quantizer "
                     f"({gb:.1f} GB of activations read per step over all ranks)",
    }


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def _event_ms(fn, reps, dev):
    import torch

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / reps


def north_star_4096(dev, peak):
    """The north-star tensor alone: per-tensor amax collect and NVFP4 fake quant of ONE 4096 x 4096 bf16 tensor per
    launch, CUDA-event timed over a rotation of 16 distinct inputs (512 MiB >> 126 MB L2) replayed from a CUDA
    graph (launch-latency free, like the step); plus the grouped (pointer-array) launch over the same 16."""
    import torch

    from model_optimizer_b200 import ops

    n = 16
    g = torch.Generator(device=dev).manual_seed(4096)
    xs = [torch.randn(4096, 4096, device=dev, generator=g, dtype=torch.float32).to(torch.bfloat16) for _ in range(n)]
    ys = [torch.empty_like(xs[0]) for _ in range(4)]
    slots = torch.zeros(n, dtype=torch.float32, device=dev)
    amax = xs[0].abs().max().float().reshape(1)
    side = torch.cuda.Stream(dev)
    out = {}

    def graph_of(fn):
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            fn()
        torch.cuda.synchronize(dev)
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, stream=side):
            fn()
        return gr

    cases = {
        "amax_per_tensor": (lambda: [ops.amax_per_tensor_(slots[i:i + 1], xs[i]) for i in range(n)], 2),
        "fake_quant_nvfp4": (lambda: [ops.fake_quant_nvfp4(xs[i], amax, out=ys[i % 4]) for i in range(n)], 4),
    }
    outs16 = [torch.empty_like(xs[0]) for _ in range(n)]
    t_amax = ops.TensorTable(xs, unit="vec32")
    t_fq = ops.TensorTable(xs, ys=outs16, unit="block16")
    amax16 = amax.repeat(n).contiguous()
    cases["amax_per_tensor_grouped16"] = (lambda: ops.amax_per_tensor_multi_(slots, t_amax), 2)
    cases["fake_quant_nvfp4_grouped16"] = (lambda: ops.fake_quant_nvfp4_multi(t_fq, amax16), 4)
    for name, (fn, bpe) in cases.items():
        gr = graph_of(fn)
        for _ in range(3):
            gr.replay()
        ms = _event_ms(gr.replay, 20, dev)
        us = ms * 1e3 / n
        gbs = 4096 * 4096 * bpe / (us * 1e-6) / 1e9
        out[name] = {"us_per_tensor": round(us, 3), "GBps": round(gbs, 1), "frac": round(gbs / peak, 4),
                     "algorithmic_bytes": 4096 * 4096 * bpe}
    out["how"] = ("4096x4096 bf16, 16 distinct inputs (512 MiB) per CUDA-graph replay, 20 replays, CUDA events; "
                  "frac of the measured HBM copy peak; north-star target 0.70")
    return out


def config_extras(dev, peak):
    """BASELINE configs 2 (FP8 per-tensor) and 4 (INT4-AWQ weight-only): the kernels those configs add, at the
    Llama-3-8B shapes, CUDA-graph replays over rotating buffers."""
    import torch

    from model_optimizer_b200 import ops

    out = {}
    g = torch.Generator(device=dev).manual_seed(7)
    side = torch.cuda.Stream(dev)

    def timed(fn, reps=10):
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            fn()
        torch.cuda.synchronize(dev)
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, stream=side):
            fn()
        gr.replay()
        return _event_ms(gr.replay, reps, dev)

    # config 2: FP8 per-tensor collect + fake quant of [4096 tokens, 4096] activations (8 distinct buffers)
    xs = [torch.randn(4096, 4096, device=dev, generator=g, dtype=torch.float32).to(torch.bfloat16) for _ in range(8)]
    ys = [torch.empty_like(xs[0]) for _ in range(4)]
    slot = torch.zeros(8, dtype=torch.float32, device=dev)
    amax = xs[0].abs().max().reshape(())
    ms = timed(lambda: [ops.amax_per_tensor_(slot[i:i + 1], xs[i]) for i in range(8)]) / 8
    ms2 = timed(lambda: [ops.fake_quant_fp8(xs[i], amax, out=ys[i % 4]) for i in range(8)]) / 8
    e = 4096 * 4096
    out["config2_fp8"] = {"collect_us": round(ms * 1e3, 2), "collect_GBps": round(e * 2 / ms / 1e6, 1),
                          "fake_quant_us": round(ms2 * 1e3, 2), "fake_quant_GBps": round(e * 4 / ms2 / 1e6, 1),
                          "fake_quant_frac": round(e * 4 / ms2 / 1e6 / peak, 4),
                          "tokens_per_sec_hot_path": round(TOKENS / ((ms + ms2) * 1e-3 * (6 + 3.5) * 32), 1),
                          "what": "FP8 per-tensor: amax collect + fake_e4m3fy forward, 4096x4096 bf16; tokens/s = the "
                                  "32x7 quantizers' collect + fake quant at these rates (down_proj input = 3.5 units)"}
    # config 4: INT4-AWQ weight-only: AWQ search step (W * s -> block-128 amax -> INT4 fake quant) + blockwise pack
    ws = [torch.randn(4096, 4096, device=dev, generator=g, dtype=torch.float32).to(torch.bfloat16) for _ in range(4)]
    wl = [torch.randn(14336, 4096, device=dev, generator=g, dtype=torch.float32).to(torch.bfloat16) for _ in range(2)]
    sc = (torch.rand(4096, device=dev, generator=g) + 0.5).to(torch.bfloat16)
    o1, o2 = torch.empty_like(ws[0]), torch.empty_like(wl[0])
    ms_a = timed(lambda: [ops.awq_scale_fake_quant(w, sc, 128, 4, False, out=o1) for w in ws]) / 4
    ms_al = timed(lambda: [ops.awq_scale_fake_quant(w, sc, 128, 4, False, out=o2) for w in wl]) / 2
    ms_p = timed(lambda: [ops.pack_int4_blockwise(w, 128) for w in ws]) / 4
    el = 14336 * 4096
    per_layer = (2 * 4096 * 4096 + 2 * 1024 * 4096 + 3 * el)            # weight elements of one decoder layer
    out["config4_int4_awq"] = {
        "awq_step_4096x4096_us": round(ms_a * 1e3, 2), "awq_step_GBps": round(e * 4 / ms_a / 1e6, 1),
        "awq_step_14336x4096_GBps": round(el * 4 / ms_al / 1e6, 1),
        "awq_step_frac": round(el * 4 / ms_al / 1e6 / peak, 4),
        "pack_int4_4096x4096_us": round(ms_p * 1e3, 2), "pack_GBps": round(e * (2 + 0.5 + 2 / 128) / ms_p / 1e6, 1),
        "pack_elements_per_sec": round(e / (ms_p * 1e-3), 1),
        "search_11_alphas_whole_model_ms": round(11 * 32 * per_layer * (ms_al / el), 2),
        "what": "awq_lite inner step in ONE kernel per alpha (reference: ~6 ATen passes) and the INT4 block-128 "
                "compress pack; whole-model figure = 11 alphas x 32 layers of weight elements at the 14336x4096 rate"}
    return out


def run_gpu(args):
    import torch
    import torch.distributed as dist

    from model_optimizer_b200 import _lib
    from model_optimizer_b200.engine import PLANS, ShardedPTQEngine

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the b200 engine has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version banner on stdout when the first communicator comes up: point fd 1 at
        # stderr until then so that stdout carries exactly one JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    _lib.load()

    plan = PLANS[args.model]
    peak, peak_kind = peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed_job(eng, steps, warmup, sampler=None):
        """W untimed steps, then EXACTLY `steps` steps = one calibration job (one arena all-reduce, joined inside
        the timed region), CUDA events on the launching stream, max over ranks."""
        eng.allreduce_every = 1 << 30
        for _ in range(warmup):
            eng.step_graph()
        eng.join_comm()
        barrier()
        eng._step = 0
        eng.allreduce_every = steps
        eng.comm_log = {k: 0 for k in eng.comm_log}
        if sampler is not None:
            sampler.start()
            time.sleep(0.25)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        barrier()
        e0.record()
        for _ in range(steps):
            eng.step_graph()
        eng.join_comm()
        e1.record()
        barrier()
        t1 = time.time()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps, (t0, t1)

    eng = ShardedPTQEngine(plan, TOKENS, "nvfp4", torch.bfloat16, dev, rank, world, allreduce_every=args.steps)
    acts = eng.alloc_activations(seed=0)
    # fake-quant outputs: a ring of four buffers (quantizer i writes slot i % 4), except the last four quantizers,
    # which get buffers of their own.  In the ring, several quantizers of one grouped launch write the same slot, so
    # what a slot holds afterwards depends on the order in which CTAs run; the own buffers hold exactly those four
    # quantizers' outputs after a step (--dump-outputs reads them).  Same bytes written either way.
    ring = eng.alloc_outputs(4)
    nq = len(eng.quantizers)
    outs = [ring[i % 4] for i in range(nq - 4)] + [torch.empty(x.numel(), dtype=x.dtype, device=dev) for x in acts[nq - 4:]]
    eng.capture(acts, outs)

    # ---- device-resident timing (value) -------------------------------------------------------------
    sampler = ClockSampler(local) if rank == 0 else None
    ms_step, (t_wall0, t_wall1) = timed_job(eng, args.steps, max(args.warmup, 3), sampler)
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(eng, acts, outs, args.dump_outputs, rank, world)
    value = TOKENS / (ms_step * 1e-3)
    comm_counts = dict(eng.comm_log)

    # ---- per-phase kernel timing for the roofline (events on the launching stream) ---------------------
    g = eng._graphs
    reps = max(3, args.steps)
    barrier()
    ms_collect = _event_ms(g["collect"].replay, reps, dev)
    ms_export = _event_ms(g["export"].replay, reps, dev)
    ms_fq = _event_ms(g["fake_quant"].replay, reps, dev)
    b_collect, b_fq = eng.act_bytes_per_step()
    nq = len(eng.quantizers)
    fq_gbs = b_fq / (ms_fq * 1e-3) / 1e9
    collect_gbs = b_collect / (ms_collect * 1e-3) / 1e9
    roofline = {
        "kernel": ("b200q::nvfp4_dyn_multi_kernel<BF16,32,2> (NVFP4 dynamic fake quant, ONE grid over this rank's "
                   f"{nq} activations)") if eng.grouped else "b200q::nvfp4_dyn_kernel<BF16,32,2> (NVFP4 dynamic fake quant)",
        "bound": "hbm", "achieved": round(fq_gbs, 1), "peak": peak, "unit": "GB/s",
        "frac": round(fq_gbs / peak, 4), "peak_kind": peak_kind,
        "bytes_per_launch": b_fq if eng.grouped else b_fq // nq,
        "us_per_launch": round(ms_fq * 1e3 / (1 if eng.grouped else nq), 3),
        "launches_timed": (1 if eng.grouped else nq) * reps, "tensors_per_launch": nq if eng.grouped else 1,
        "traffic": measured_traffic()[0], "traffic_source": measured_traffic()[1],
        "second_kernel": {"kernel": "b200q::amax_tensor_multi_kernel<BF16,32,4> (calibration collect, one grid)"
                          if eng.grouped else "b200q::amax_tensor_kernel<BF16,32,4> (calibration collect)",
                          "achieved": round(collect_gbs, 1), "frac": round(collect_gbs / peak, 4),
                          "bytes_per_launch": b_collect if eng.grouped else b_collect // nq,
                          "us_per_launch": round(ms_collect * 1e3 / (1 if eng.grouped else nq), 3),
                          "note": "a read-only kernel can exceed the COPY peak (read + write) it is normalised by"},
    }
    # ---- per-step breakdown: where a step's time goes on this rank (max over ranks for the comm figures) ------
    breakdown = {"collect_ms": round(ms_collect, 4), "export_ms": round(ms_export, 4), "fake_quant_ms": round(ms_fq, 4),
                 "kernels_ms": round(ms_collect + ms_export + ms_fq, 4), "step_ms": round(ms_step, 4),
                 "join_idle_us": round((ms_step - ms_collect - ms_export - ms_fq) * 1e3, 1),
                 "what": "graph replays timed alone on this rank vs the pipelined step; join_idle = step - kernels "
                         "(launch gaps, stream joins, bandwidth shared with the hand-off)"}
    if world > 1:
        barrier()
        ms_ar = _event_ms(lambda: dist.all_reduce(eng.global_arena, op=dist.ReduceOp.MAX), 20, dev)
        eng._step = 0
        eng.allreduce_every = 1 << 30

        def xchg():
            q = eng._step & 1
            eng._ev_step_done[q].record(torch.cuda.current_stream(dev))
            eng._exchange(q)
            torch.cuda.current_stream(dev).wait_event(eng._ev_comm[q])
            eng._step += 1

        barrier()
        ms_x = _event_ms(xchg, 20, dev)
        t = torch.tensor([ms_ar, ms_x], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        hb = TOKENS * plan.hidden * 2
        breakdown.update({"allreduce_us": round(float(t[0]) * 1e3, 1), "allreduce_bytes": eng.global_arena.numel() * 4,
                          "allreduce_per_job": comm_counts["allreduce_calls"],
                          "handoff_us": round(float(t[1]) * 1e3, 1), "handoff_bytes_per_step": hb,
                          "handoff_GBps": round(hb / (float(t[1]) * 1e-3) / 1e9, 1),
                          "p2p_calls_per_job": comm_counts["p2p_calls"],
                          "handoff_transport": eng.handoff_transport,
                          "comm": "hand-off and all-reduce run on the communication stream; allreduce_us / handoff_us are "
                                  "each timed ALONE (serialised, max over ranks) -- inside the step they overlap the kernels"})
        barrier()

    # ---- end to end: host (pinned) activations -> H2D -> collect + fake quant -> D2H of the amax arena ---
    e2e = run_e2e(eng, acts, outs, dev, world, args, barrier)

    # ---- weight pass (one-off per model): amax + NVFP4 quant-and-pack of the owned weights ------------
    wshapes = [(cout, cin) for _, cin, cout in plan.linears()]
    ws = [torch.randn(s, device=dev, dtype=torch.float32).to(torch.bfloat16) for s in wshapes]
    eng.weight_pass(ws)
    ms_weights = _event_ms(lambda: eng.weight_pass(ws), len(eng.layers), dev) * len(eng.layers)
    w_elems = plan.weight_elems_per_layer() * len(eng.layers)
    job_s = ms_weights * 1e-3 + 64 * ms_step * 1e-3
    extras = {
        "fake_quant_GBps": round(fq_gbs, 1), "collect_GBps": round(collect_gbs, 1), "breakdown": breakdown,
        "weight_pass": {"ms": round(ms_weights, 3), "what": "amax + NVFP4 pack of this rank's weights "
                        "(one layer's random bf16 weights reused per layer)",
                        "GBps": round(w_elems * (2 + 2 + 0.5 + 1 / 16) / (ms_weights * 1e-3) / 1e9, 1)},
        "job_512_samples": {"tokens": 64 * TOKENS, "seconds": round(job_s, 4),
                            "tokens_per_sec": round(64 * TOKENS / job_s, 1),
                            "what": "weight pass + 64 calibration batches (512 samples x 512 tokens)"},
    }
    del ws

    if world == 1:
        try:
            roofline["north_star_4096"] = north_star_4096(dev, peak)
        except Exception as e:  # noqa: BLE001  (context numbers only: never break the JSON line)
            roofline["north_star_4096"] = {"error": repr(e)[:300]}
        try:
            extras.update(config_extras(dev, peak))
        except Exception as e:  # noqa: BLE001
            extras["config_extras_error"] = repr(e)[:300]

    # ---- BASELINE config 5 (Llama-3-70B layer-sharded over 8 GPUs) in the same invocation ------------------
    if world == 8 and args.model == "llama-3-8b" and not args.no_config5:
        try:
            del acts, outs
            acts = outs = None
            eng._graph_sets = eng._graphs = None
            torch.cuda.empty_cache()
            e70 = ShardedPTQEngine(PLANS["llama-3-70b"], TOKENS, "nvfp4", torch.bfloat16, dev, rank, world,
                                   allreduce_every=args.steps)
            a70, o70 = e70.alloc_activations(seed=1), e70.alloc_outputs(4)
            e70.capture(a70, o70)
            ms70, _ = timed_job(e70, args.steps, 3)
            b70 = sum(e70.act_bytes_per_step())
            extras["config5_llama70b_x8"] = {"tokens_per_sec": round(TOKENS / (ms70 * 1e-3), 1), "ms_per_step": round(ms70, 4),
                                             "per_gpu_GBps": round(b70 / (ms70 * 1e-3) / 1e9, 1),
                                             "per_gpu_frac": round(b70 / (ms70 * 1e-3) / 1e9 / peak, 4),
                                             "layers_per_gpu": len(e70.layers),
                                             "what": "same step on the Llama-3-70B shape plan, 10 layers per GPU"}
            del e70, a70, o70
        except Exception as e:  # noqa: BLE001
            extras["config5_llama70b_x8"] = {"error": repr(e)[:300]}

    if rank == 0 and world == 1 and args.llama_ptq > 0:
        try:
            from tools.ptq_twin import run_llama_ptq_all

            del acts, outs
            eng._graph_sets = eng._graphs = None
            torch.cuda.empty_cache()
            extras["mtq_quantize_llama"] = run_llama_ptq_all("NVFP4_DEFAULT_CFG", 512, SEQ, BATCH, layers=args.llama_ptq)
        except Exception as e:  # noqa: BLE001  (context number only: never break the JSON line)
            extras["mtq_quantize_llama"] = {"error": repr(e)[:300]}

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_base = cpu_arm(3, 1, budget_s=20.0)[2]

    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": round(ms_step, 4), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": workload_config(world, plan), "clocks": clocks, "e2e": e2e,
            "gpu_launches": eng.launches_per_step() * args.steps, "launches_per_step": eng.launches_per_step(),
            "step_submission": "CUDA graphs (collect / export / fake quant)" + (
                f" + per step one hidden-state hand-off ({getattr(eng, 'handoff_transport', 'nccl send/recv')}) and per job one "
                "NCCL all-reduce of the amax arena, both on a communication stream overlapped with the kernels"
                if world > 1 else ""),
            "roofline": roofline, "cpu_baseline": cpu_base, **extras,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


DUMP_ROWS = 256           # token rows of each dumped activation, shared out over the ranks
DUMP_BUDGET = 64 << 20    # bytes --dump-outputs may write over all ranks


def dump_outputs(eng, acts, outs, out_dir, rank, world):
    """Write what the last timed step left on the device as ``out_dir/<name>.npy`` (float32): the fp32 amax arena
    (``amax``), the amax exported to the quantizers (``amax_export``) and the fake-quantized activations of the last
    four quantizers, which have output buffers of their own (``fake_quant.<quantizer>``), on DUMP_ROWS // world token
    rows drawn with a fixed seed.  With several GPUs every name is prefixed by ``rank<r>.``.  The rows are split over
    the ranks so that the total stays bounded: at most 256 x (3 x 8192 + 28672) x 4 B = 54.5 MB of activations over all
    ranks (Llama-3-70B; 27.3 MB for Llama-3-8B), plus 8 B per quantizer of amax per rank."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    prefix = f"rank{rank}." if world > 1 else ""
    n_rows = max(1, DUMP_ROWS // world)
    rows = torch.randperm(TOKENS, generator=torch.Generator().manual_seed(0))[:n_rows].sort().values
    arrays = {"amax": eng.global_arena, "amax_export": eng.amax_arena}
    parity = (eng._step - 1) & 1 if eng.handoff else 0
    last_hidden = len(eng.quantizers) - 4 if (eng.handoff and eng.hand_out is not None) else -1
    for i in range(len(eng.quantizers) - 4, len(eng.quantizers)):
        x = acts[i]
        y = eng.hand_out[parity] if i == last_hidden else outs[i % len(outs)][: x.numel()].view_as(x)
        arrays[f"fake_quant.{eng.quantizers[i][0]}"] = y[rows.to(y.device)]
    nbytes = sum(t.numel() * 4 for t in arrays.values())
    assert nbytes * world <= DUMP_BUDGET, f"--dump-outputs would write {nbytes * world} bytes over {world} ranks"
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), t.float().cpu().numpy())


def run_e2e(eng, acts, outs, dev, world, args, barrier):
    """Same step through the engine API with HOST buffers: every step copies each quantizer's
    activation from pinned host memory into its device buffer (copy stream, overlapped with the collect
    kernels of earlier quantizers), runs collect -> finish -> fake quant, and reads back the amax arena AND the
    fake-quantized activation of the last quantizer (what a consumer of the step would fetch)."""
    import torch

    steps = max(1, min(args.steps, 3))
    shapes = sorted({tuple(x.shape) for x in acts})
    host = {s: torch.randn(s, dtype=torch.float32).to(torch.bfloat16).pin_memory() for s in shapes}
    copy_stream = torch.cuda.Stream(dev)
    main = torch.cuda.current_stream(dev)
    ready = [torch.cuda.Event() for _ in acts]
    arena_host = torch.empty(len(eng.arena), dtype=torch.float32).pin_memory()
    out_host = torch.empty(acts[-1].shape, dtype=acts[-1].dtype).pin_memory()
    h2d = sum(x.numel() * x.element_size() for x in acts)
    d2h = arena_host.numel() * 4 + out_host.numel() * out_host.element_size()

    def one_step():
        eng.reset()
        copy_stream.wait_stream(main)            # previous step's kernels are done with the buffers
        with torch.cuda.stream(copy_stream):
            for i, x in enumerate(acts):
                x.copy_(host[tuple(x.shape)], non_blocking=True)
                ready[i].record(copy_stream)
        for i, ((_, q, _), x) in enumerate(zip(eng.quantizers, acts)):
            main.wait_event(ready[i])
            q._calibrator.collect(x)             # collect of quantizer i overlaps the copy of i+1
        eng.export_amax()
        res = eng.fake_quant(acts, outs)
        arena_host.copy_(eng.arena.freeze(), non_blocking=True)
        out_host.copy_(res[-1], non_blocking=True)
        main.synchronize()
        return float(arena_host[0]) + float(out_host[0, 0])

    one_step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        one_step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / steps
    if world > 1:
        import torch.distributed as dist

        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return {"value": round(TOKENS / (ms * 1e-3), 1), "unit": UNIT, "ms_per_step": round(ms, 3),
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": steps,
            "what": "pinned host activations -> H2D into per-quantizer device buffers -> collect -> export -> "
                    "fake quant through the engine API -> D2H of the amax arena and of the last quantizer's "
                    "fake-quantized activation; per-rank bytes (PCIe-bound by construction: the step streams "
                    "every activation once)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config5", action="store_true", help="skip the Llama-3-70B extra of an 8-GPU run")
    ap.add_argument("--llama-ptq", type=int, default=32, metavar="LAYERS",
                    help="also time quantize() on a random-init HF Llama-3-8B-shaped model with this many layers "
                         "(32 = full model, 0 = skip; N=1 only; a context number, not the headline)")
    ap.add_argument("--model", default="llama-3-8b", choices=["llama-3-8b", "llama-3-70b"],
                    help="shape plan; the default is the BASELINE metric's model (70b = BASELINE config 5)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float32, same seeded inputs on "
                         "every run) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs; it does not apply to --impl reference")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
