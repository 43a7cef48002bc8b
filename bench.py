"""Headline benchmark: forward images/sec of a tfimm classifier on N B200 GPUs (one node).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--model vit_base_patch16_224]
                    [--batch 256] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one forward pass of the model over one synthetic batch (``--batch`` images per GPU,
224x224x3 unless the model's native size differs; weak scaling: per-GPU batch fixed).  Rank 0
prints ONE JSON line (see the task contract): whole-job images/sec with inputs resident in HBM
(``value``), the same through the public API from pinned host memory (``e2e``), the roofline of
the dominant kernel family measured live with CUDA events, the CPU oracle timed beside it, and the
SM clocks sampled during the timed region.

``--impl reference`` times the CPU stand-in for the reference (the torch-CPU oracle restatement;
TensorFlow is not installed in this image, see BASELINE.md section 3) on the same config.

``--dump-outputs DIR`` writes, after the timed steps, the logits of the last timed step of every model as
``DIR/<model>.npy`` (and of the end-to-end path as ``DIR/<model>_e2e.npy``), float32.  Inputs and weights are seeded,
so two builds run with the same arguments can be compared output for output.  Compare with a bf16 tolerance: the
depthwise kernels sum the squeeze-excite pooling with atomics, so EfficientNet logits can differ from run to run by a
bf16 rounding step (measured on one B200, 1000 W power limit: 2 of 256 rows, up to 6e-4 of max|logit|).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT / "tensorflow-image-models_b200"))
sys.path.insert(0, str(ROOT))

METRIC = "images/sec fwd bs=256 224px"
# the other BASELINE.json configs, timed after the headline model and reported under "extra"
EXTRA_MODELS = ["convnext_base", "swin_base_patch4_window7_224", "efficientnet_b4"]
# Algorithmic work per image (SURVEY.md 8d): GFLOP and op-level HBM MB in bf16
WORK = {
    "vit_base_patch16_224": {"gflop": 35.13, "mb": 80.5, "bound": "tensor"},
    "vit_tiny_patch16_224": {"gflop": 2.51, "mb": 20.3, "bound": "tensor"},
    "convnext_base": {"gflop": 30.71, "mb": 124.6, "bound": "hbm"},
    "swin_base_patch4_window7_224": {"gflop": 30.86, "mb": 140.2, "bound": "hbm"},
    "efficientnet_b4": {"gflop": 8.79, "mb": 322.5, "bound": "hbm"},
}


# --dump-outputs writes at most this much; an output over its share keeps a fixed, seeded sample of its rows
DUMP_BYTES = 64 << 20


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        """Index of the next sample: window(mark) summarises what was sampled after this call."""
        return len(self.lines)

    def stop(self):
        if self.proc is None:
            return
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()

    def window(self, mark):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if len(self.lines) - mark < 2:
            time.sleep(0.25)  # a 20-step region can be shorter than two 100 ms samples
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lines = self.lines[mark:] or self.lines[-3:]
        for line in lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def _input_hw(cfg):
    return tuple(cfg.input_size)


def _oracle_forward(model_name):
    import importlib

    import tfimm

    cfg = tfimm.models.model_config(model_name)
    fam = {"ViT": "vit", "SwinTransformer": "swin", "ConvNeXt": "convnext", "EfficientNet": "efficientnet",
           "ResNet": "resnet"}[tfimm.models.model_class(model_name).__name__]
    mod = importlib.import_module(f"oracle.{fam}")
    return cfg, mod


def host_cores():
    """CPU threads this process may actually use: the scheduler affinity mask capped by the cgroup CPU quota
    (os.cpu_count() reports the whole host and oversubscribes a quota-limited container 10x)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                quota = int(txt[0])
                period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if quota > 0:
                    n = min(n, max(1, quota // period))
            break
        except Exception:
            continue
    return max(1, n)


def cpu_oracle_throughput(model_name, batch, iters, warmup=1):
    """images/sec of the torch-CPU oracle (the reference's CPU stand-in) on the host cores we may use."""
    import torch

    from oracle import params

    cores = host_cores()
    torch.set_num_threads(cores)
    cfg, mod = _oracle_forward(model_name)
    w = params.random_params(mod.param_shapes(cfg), seed=0)
    h, wd = _input_hw(cfg)
    x = params.test_images(batch, h, wd, cfg.in_channels)
    times = []
    with torch.no_grad():
        for i in range(warmup + iters):
            t0 = time.perf_counter()
            y = mod.forward(cfg, w, x)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    med = statistics.median(times)
    return {"value": batch / med, "unit": "images/sec", "cores": cores, "kind": "port",
            "sample": f"{model_name} fp32 forward, batch {batch}, median of {iters} after {warmup} warm-up "
                      f"(torch-CPU oracle restatement; TensorFlow is not installed)",
            "ms_per_step": med * 1e3, "last_output": y}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    batch = args.ref_batch
    res = cpu_oracle_throughput(args.model, batch, max(1, args.steps), max(1, min(args.warmup, 1)))
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": "images/sec",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.model} forward, per-GPU batch {args.batch}, 224px NHWC synthetic; "
                               f"CPU sample batch {batch}"},
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": res["value"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {args.model: res["last_output"]})
    print(json.dumps(line))


def dump_outputs(directory, arrays):
    """Writes {name: tensor} as ``<directory>/<name>.npy`` (float32), DUMP_BYTES in all at most."""
    import numpy as np

    out = Path(directory)
    out.mkdir(parents=True, exist_ok=True)
    share = DUMP_BYTES // max(1, len(arrays))
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        if a.nbytes > share:
            keep = max(1, share // a[0].nbytes)
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        np.save(out / f"{name}.npy", np.ascontiguousarray(a))


def _random_weights(model, torch, np):
    """Random-init every weight (the reference's zeros/ones initialisers would make whole branches inert)."""
    g = torch.Generator().manual_seed(1234)
    rnd = {}
    for k, v in model.params.items():
        leaf = k.rsplit("/", 1)[-1]
        if leaf in ("kernel", "depthwise_kernel"):
            fan_in = int(np.prod(v.shape[:-1]))
            rnd[k] = torch.randn(v.shape, generator=g) / fan_in ** 0.5
        elif leaf in ("gamma", "moving_variance"):
            rnd[k] = 1.0 + 0.1 * torch.rand(v.shape, generator=g)
        else:
            rnd[k] = 0.1 * torch.randn(v.shape, generator=g)
    model.load_weights_dict(rnd, strict=True)


def measure_model(model_name, args, ctx, sampler, with_roofline=True):
    """Times one model on this rank's GPU (weak scaling: ``args.batch`` images per GPU): device-resident throughput,
    end-to-end throughput from pinned host memory, per-kernel-family roofline.  Returns the fields of the JSON line."""
    import numpy as np
    import torch
    import torch.distributed as dist

    import tfimm
    from tfimm.backend import ops
    from tfimm.serving import InferencePipeline

    world, rank, local_rank, dev = ctx["world"], ctx["rank"], ctx["local_rank"], ctx["dev"]
    model = tfimm.create_model(model_name, precision="bf16", device=dev, seed=0)
    _random_weights(model, torch, np)
    B = args.batch
    h, w = _input_hw(model.cfg)
    rng = np.random.default_rng(2021 + rank)
    host = torch.from_numpy(rng.random((B, h, w, model.cfg.in_channels), dtype=np.float32)).pin_memory()
    x_dev = host.to(dev)
    nb_classes = model.cfg.nb_classes
    # The user-facing call: model(x) eagerly, or the same forward captured once into a CUDA graph
    # (model.cuda_graph) so that a step is one graph launch instead of ~100-400 kernel launches.
    forward = model.cuda_graph(B) if args.graph else model

    # Multi-GPU step = forward + ONE all-gather of the logits (SURVEY.md 8e).  The gather is issued asynchronously on
    # NCCL's stream from a double-buffered staging copy of the logits, so that the forward of step i+1 does not wait
    # for the slowest rank's step i (ranks may drift by up to two steps; a lock-step loop runs at the pace of the most
    # power-starved GPU every single step).
    send = [torch.empty((B, nb_classes), device=dev, dtype=torch.float32) for _ in range(2)] if world > 1 else None
    recv = [torch.empty((world * B, nb_classes), device=dev, dtype=torch.float32) for _ in range(2)] if world > 1 else None
    pending = [None, None]
    counter = {"i": 0}

    def step(x):
        logits = forward(x)
        if world == 1:
            return logits
        k = counter["i"] % 2
        counter["i"] += 1
        if pending[k] is not None:
            pending[k].wait()          # slot k's previous gather (two steps ago) has finished reading send[k]
        send[k].copy_(logits)
        pending[k] = dist.all_gather_into_tensor(recv[k], send[k], async_op=True)
        return recv[k]

    def drain():
        for k in (0, 1):
            if pending[k] is not None:
                pending[k].wait()
                pending[k] = None

    def barrier():
        drain()
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    # ---------------- device-resident timing ----------------
    for _ in range(max(args.warmup, 3)):
        step(x_dev)
    barrier()
    mark = sampler.mark() if sampler is not None else None
    launches0 = ops.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        logits = step(x_dev)
    drain()
    e1.record()
    barrier()
    ms_local = e0.elapsed_time(e1)
    outputs = {model_name: logits.float().cpu()} if (args.dump_outputs and rank == 0) else {}
    launches = ops.launch_count - launches0
    clocks = sampler.window(mark) if sampler is not None else None
    per_rank_ms = [ms_local / args.steps]
    if world > 1:
        t = torch.tensor([ms_local / args.steps, float((clocks or {}).get("sm_mhz") or 0.0)], device=dev,
                         dtype=torch.float64)
        allt = torch.empty(2 * world, device=dev, dtype=torch.float64)
        dist.all_gather_into_tensor(allt, t)
        vals = allt.view(world, 2).tolist()
        per_rank_ms = [float(v[0]) for v in vals]
        if clocks is not None:
            clocks["per_rank_sm_mhz"] = [float(v[1]) for v in vals]
    ms_per_step = max(per_rank_ms)
    value = world * B / (ms_per_step / 1e3)

    # ---------------- end to end through the public API from pinned host memory ----------------
    # tfimm.serving.InferencePipeline: every step uploads its own batch from pinned host memory (H2D on a copy
    # stream, overlapping the previous step's forward), runs the forward (+ all-gather) and downloads its logits.
    # Host images are raw uint8 pixels when the family fuses create_preprocessing into its first kernel, else
    # preprocessed fp32.
    e2e_dtype = torch.uint8 if (model.accepts_uint8 and args.e2e_input == "uint8") else torch.float32
    if e2e_dtype == torch.uint8:
        host_e2e = [torch.from_numpy(rng.integers(0, 256, (B, h, w, model.cfg.in_channels), dtype=np.uint8)).pin_memory()
                    for _ in range(2)]
    else:
        host_e2e = [host, host.clone().pin_memory()]
    gathered = torch.empty((world * B, nb_classes), device=dev, dtype=torch.float32) if world > 1 else None

    def _gather(logits):
        dist.all_gather_into_tensor(gathered, logits.contiguous())
        return gathered

    pipe = InferencePipeline(model, B, depth=2, input_dtype=e2e_dtype, gather=_gather if world > 1 else None)
    for i in range(3):
        out_host = pipe.submit(host_e2e[i % 2])
    pipe.synchronize()
    barrier()
    e0.record()
    for i in range(args.steps):
        out_host = pipe.submit(host_e2e[i % 2])
    e1.record()
    pipe.synchronize()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    if outputs:
        outputs[f"{model_name}_e2e"] = out_host.clone()
    if world > 1:
        t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e_value = world * B * args.steps / (e2e_ms / 1e3)
    h2d_bytes = host_e2e[0].numel() * host_e2e[0].element_size()

    roof = kernel_roofline(model, x_dev, model_name, ops) if (rank == 0 and with_roofline) else None
    res = {
        "value": value, "ms_per_step": ms_per_step, "per_rank_ms_per_step": [round(v, 4) for v in per_rank_ms],
        "workload": f"{model_name} forward, per-GPU batch {B}, {h}x{w}x{model.cfg.in_channels} NHWC fp32 synthetic "
                    f"images, random-init weights, bf16 operands / fp32 accumulate",
        "graph_level": ("ViT last block: attention/proj/MLP evaluated for the class-token rows only (the other rows "
                        "cannot reach the logits); model.prune_last_block = False disables"
                        if getattr(model, "prune_last_block", False) else "none"),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "images/sec", "h2d_bytes_per_step": h2d_bytes,
                "input": str(e2e_dtype).replace("torch.", ""),
                "pipeline": "tfimm.serving.InferencePipeline depth 2 (H2D of step i+1 overlaps forward of step i)",
                "d2h_bytes_per_step": out_host.numel() * 4, "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": launches, "roofline": roof, "outputs": outputs,
    }
    del pipe, forward, model, x_dev, host, host_e2e
    torch.cuda.empty_cache()
    return res


def run_b200(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"  # the version banner goes to stdout and would precede the JSON line
        dist.init_process_group("nccl", device_id=dev)
    ctx = {"world": world, "rank": rank, "local_rank": local_rank, "dev": dev}
    sampler = ClockSampler(local_rank)
    sampler.start()  # started before the warm-up: nvidia-smi needs ~1 s before its first sample

    head = measure_model(args.model, args, ctx, sampler)
    outputs = dict(head["outputs"])
    # The other BASELINE.json configs, in the same run and the same JSON line ("extra"): the metric is quoted on
    # ViT-B/16 AND ConvNeXt-B; Swin-B and EfficientNet-B4 (native 380 px, 256 per GPU = 2048 over 8 GPUs) are
    # configs[3] and configs[4].  Every rank runs them (weak scaling + logits all-gather), rank 0 reports.
    extra = {}
    if not args.no_extra:
        for name in EXTRA_MODELS:
            if name == args.model:
                continue
            r = measure_model(name, args, ctx, sampler)
            outputs.update(r["outputs"])
            extra[name] = {"value": r["value"], "unit": "images/sec", "ms_per_step": r["ms_per_step"],
                           "per_rank_ms_per_step": r["per_rank_ms_per_step"], "global_batch": world * args.batch,
                           "workload": r["workload"], "e2e": r["e2e"], "gpu_launches": r["gpu_launches"],
                           "roofline": r["roofline"], "clocks": r["clocks"]}
    sampler.stop()

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline:
            cpu = cpu_oracle_throughput(args.model, args.ref_batch, 3, 1)
            cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
        line = {
            "metric": METRIC, "value": head["value"], "unit": "images/sec", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": head["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": head["workload"], "global_batch": world * args.batch, "parallelism": f"dp{world}",
                       "cuda_graph": bool(args.graph),
                       "l2": "per-step working set (154 MB input + >1 GB activations) exceeds the 126 MB L2",
                       "graph_level": head["graph_level"],
                       "collective": ("one NCCL all-gather of the fp32 logits per step, issued asynchronously "
                                      "(double-buffered): ranks are not lock-stepped" if world > 1 else "none"),
                       "extra_models": list(extra)},
            "per_rank_ms_per_step": head["per_rank_ms_per_step"],
            "clocks": head["clocks"], "e2e": head["e2e"], "gpu_launches": head["gpu_launches"],
            "roofline": head["roofline"], "cpu_baseline": cpu, "extra": extra,
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def _traffic_table():
    """Measured DRAM bytes per kernel family per forward (ncu dram__bytes_read.sum + dram__bytes_write.sum, one pass
    per model, tools/ncu_traffic.py): profiles/dram_traffic.json = {model: {"batch": B, "families": {name: bytes}}}."""
    p = ROOT / "profiles" / "dram_traffic.json"
    try:
        return json.loads(p.read_text())
    except Exception:
        return {}


def kernel_roofline(model, x_dev, model_name, ops):
    """Per-kernel-family device time of one forward, measured with CUDA events around every launch
    (instrumented pass, after the timed region).  Reports the dominant family against its roof."""
    import torch

    peaks = _peaks()
    model(x_dev)  # warm the eager path (the timed region replays a graph)
    torch.cuda.synchronize()
    ops.trace = []
    model(x_dev)
    torch.cuda.synchronize()
    trace, ops.trace = ops.trace, None
    fam = {}
    for name, e0, e1, flops, nbytes in trace:
        d = fam.setdefault(name, {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "launches": 0})
        d["ms"] += e0.elapsed_time(e1)
        d["flops"] += flops
        d["bytes"] += nbytes
        d["launches"] += 1
    total_ms = sum(d["ms"] for d in fam.values())
    total_flops = sum(d["flops"] for d in fam.values())
    total_bytes = sum(d["bytes"] for d in fam.values())
    top = max(fam, key=lambda k: fam[k]["ms"])
    d = fam[top]
    work = WORK.get(model_name)
    B = x_dev.shape[0]
    table = _traffic_table().get(model_name, {})
    traffic = None
    if table.get("batch") == B and top in table.get("families", {}):
        traffic = table["families"][top] / d["launches"]  # measured DRAM bytes per launch of the dominant family
    if d["flops"] > 0 and (d["flops"] / max(d["bytes"], 1)) > 100:
        achieved = d["flops"] / (d["ms"] * 1e-3) / 1e12
        peak = peaks["bf16_tflops_sustained"]
        roof = {"bound": "tensor", "kernel": top, "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                "frac": achieved / peak, "frac_of_burst": achieved / peaks["bf16_tflops"], "traffic": traffic,
                "peak_source": f"{peaks['source']} bf16_tflops_sustained (kernel timed inside a long step); "
                               f"burst {peaks['bf16_tflops']}"}
    else:
        achieved = d["bytes"] / (d["ms"] * 1e-3) / 1e9
        peak = peaks["hbm_gbs"]
        roof = {"bound": "hbm", "kernel": top, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": f"{peaks['source']} hbm_gbs"}
    roof["algorithmic_bytes_per_launch"] = d["bytes"] / d["launches"]
    roof["traffic_source"] = ("profiles/dram_traffic.json (ncu dram__bytes_read.sum + dram__bytes_write.sum per launch)"
                              if traffic is not None else None)
    roof["share_of_step"] = d["ms"] / total_ms
    roof["launches_per_step"] = d["launches"]
    roof["avg_launch_ms"] = d["ms"] / d["launches"]
    roof["families_ms"] = {k: round(v["ms"], 4) for k, v in sorted(fam.items(), key=lambda kv: -kv[1]["ms"])}
    # whole-model view, instrumented pass: EXECUTED work (what the launches actually did, after graph-level pruning)
    # and the nominal SURVEY.md 8(d) per-image figures, each against both bf16 denominators / the HBM peak
    secs = total_ms * 1e-3
    roof["model"] = {
        "instrumented_ms": round(total_ms, 4),
        "executed_gflop_per_image": total_flops / B / 1e9,
        "executed_mb_per_image": total_bytes / B / 1e6,
        "tensor_frac_executed_sustained": total_flops / secs / 1e12 / peaks["bf16_tflops_sustained"],
        "tensor_frac_executed_burst": total_flops / secs / 1e12 / peaks["bf16_tflops"],
        "hbm_frac_executed": total_bytes / secs / 1e9 / peaks["hbm_gbs"],
    }
    if work:
        roof["model"].update({
            "nominal_gflop_per_image": work["gflop"], "nominal_mb_per_image": work["mb"],
            "tensor_frac_nominal_sustained": B * work["gflop"] * 1e9 / secs / 1e12 / peaks["bf16_tflops_sustained"],
            "tensor_frac_nominal_burst": B * work["gflop"] * 1e9 / secs / 1e12 / peaks["bf16_tflops"],
            "hbm_frac_nominal": B * work["mb"] * 1e6 / secs / 1e9 / peaks["hbm_gbs"],
        })
    return roof


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--model", default="vit_base_patch16_224")
    ap.add_argument("--batch", type=int, default=256, help="per-GPU batch")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ref-batch", type=int, default=8, help="CPU sample batch for the oracle timing")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="time only --model, not the other BASELINE configs")
    ap.add_argument("--e2e-input", default="uint8", choices=["uint8", "fp32"],
                    help="host image dtype of the end-to-end path (uint8 = raw pixels, preprocessing fused on device)")
    ap.add_argument("--no-graph", dest="graph", action="store_false",
                    help="launch kernels eagerly instead of replaying a captured CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the logits of the last timed step of every model to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
