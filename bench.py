#!/usr/bin/env python
"""Headline benchmark: RepVGG-A0 224x224 bf16 TRAINING throughput (images/s) on N B200s of one node.

    python bench.py --gpus 1 --steps 20 --warmup 5                       # this repo's CUDA path (default arm)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps 2 --warmup 1                # reference algorithm on the host CPU cores

One "step" = forward + cross-entropy (label smoothing 0.1, references/classification/train.py:194 of the reference) +
backward + gradient all-reduce (N > 1) + AdaBelief(lr=1e-3, betas=(0.95, 0.99), eps=1e-6) update on a synthetic
ImageNet-shaped batch of 256 images per GPU (weak scaling). Prints ONE JSON line on rank 0 (see DESIGN.md §Measurement).
"""
import argparse
import datetime
import json
import os
import subprocess
import sys
import threading
import time

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "images/sec RepVGG-A0 224^2 bf16 train"
BATCH_PER_GPU = 256
NUM_CLASSES = 1000
IMAGENET_MEAN = (0.485, 0.456, 0.406)
IMAGENET_STD = (0.229, 0.224, 0.225)


def measured_peaks():
    """Roofline denominators: MEASURED_PEAKS.json (driver-written) or the profiling guide's fallback."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1400.0, "src": "fallback"}


class ClockSampler:
    """Samples SM clocks / throttle reasons while the timed region runs: NVML from a background thread (4 Hz; a
    100 ms `nvidia-smi -lms` poller was measured to slow kernel launches of the process under test by 2x), falling
    back to a 500 ms `nvidia-smi` loop when the NVML binding is unavailable."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index: int) -> None:
        self.index, self.proc, self.lines = index, None, []
        self.samples, self.max_mhz, self.reasons = [], None, set()
        self.stop_flag = threading.Event()
        self.thread = None
        self.mode = None

    def _nvml_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.index])
            except (ValueError, IndexError):
                return self.index
        return self.index

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self._nvml_index())
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.mode = "nvml"
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return
        except Exception:  # noqa: BLE001
            self.mode = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "500",
                                          "-i", str(self._nvml_index())], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                                         text=True)
            self.mode = "smi"
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _poll_nvml(self):
        nv = self.nvml
        masks = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self.stop_flag.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                for name, m in masks.items():
                    if r & m:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            self.stop_flag.wait(0.25)

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.mode == "nvml":
            self.stop_flag.set()
            self.thread.join(timeout=2)
            clocks = sorted(self.samples)
            med = clocks[len(clocks) // 2] if clocks else None
            return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(clocks),
                    "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        clocks, maxes, reasons = [], [], set()
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                clocks.append(float(parts[0])); maxes.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(self.NAMES, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        clocks.sort()
        med = clocks[len(clocks) // 2] if clocks else None
        return {"sm_mhz": med, "sm_max_mhz": max(maxes) if maxes else None, "reasons": sorted(reasons), "samples": len(clocks),
                "source": "nvidia-smi"}


def synthetic_batch(batch: int, seed: int, device, size: int = 224):
    """ImageNet-like synthetic batch: U[0,1) pixels normalised with the ImageNet mean/std, uniform random labels."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = torch.rand(batch, 3, size, size, generator=g)
    mean = torch.tensor(IMAGENET_MEAN).view(1, 3, 1, 1)
    std = torch.tensor(IMAGENET_STD).view(1, 3, 1, 1)
    x = (x - mean) / std
    t = torch.randint(0, NUM_CLASSES, (batch,), generator=g)
    return x.to(device), t.to(device)


# ------------------------------------------------------------------------------------------------ workloads
# classification workloads: (images, labels) + CE
CLS_KEYS = ("repvgg_a0", "rexnet1_0x", "repvgg_a1", "resnet50", "resnet18", "mobileone_s0", "res2net50_26w_4s", "sknet50",
            "convnext_tiny", "tridentnet50", "pyconv_resnet50")


class Workload:
    """One BASELINE.json configuration: model factory, synthetic batch (SURVEY.md §8d) and loss."""

    def __init__(self, key: str):
        self.key = key
        table = {
            # key: (model factory, kwargs, default batch / GPU, image size, CUDA-graph capturable, description)
            "repvgg_a0": ("repvgg_a0", {"num_classes": NUM_CLASSES}, 256, 224, True,
                          "repvgg_a0 (train form, 1000 classes) 224x224 bf16 train step: fwd + CE(label_smoothing=0.1) + bwd + "
                          "AdaBelief(lr=1e-3, betas=(0.95,0.99), eps=1e-6)"),
            "rexnet1_0x": ("rexnet1_0x", {"num_classes": NUM_CLASSES}, 256, 224, True,
                           "rexnet1_0x 224x224 bf16 train step (BASELINE configs[1]): fwd + CE(label_smoothing=0.1) + bwd + AdaBelief"),
            "repvgg_a1": ("repvgg_a1", {"num_classes": NUM_CLASSES}, 512, 224, True,
                          "repvgg_a1 224x224 bf16 train step (BASELINE configs[2]): fwd + CE(label_smoothing=0.1) + bwd + AdaBelief, "
                          "batch 512/GPU"),
            "yolov4": ("yolov4", {"num_classes": 80}, 16, 512, True,
                       "yolov4 (CSP-Darknet53) 512x512 detection train step (BASELINE configs[3]): fwd + CIoU/objectness/class "
                       "losses (sync-free per-box formulation) + bwd + AdaBelief; synthetic COCO-like boxes (1-19 per image)"),
            # SURVEY §8 f3 (widening, not a BASELINE.json configuration): the ResNet family on the same fused units
            "resnet50": ("resnet50", {"num_classes": NUM_CLASSES}, 256, 224, True,
                         "resnet50 224x224 bf16 train step (SURVEY 8-f3): fwd + CE(label_smoothing=0.1) + bwd + AdaBelief"),
            "mobileone_s0": ("mobileone_s0", {"num_classes": NUM_CLASSES}, 256, 224, True,
                             "mobileone_s0 (train form, over-parametrisation 4) 224x224 bf16 train step (SURVEY 8-f3): fwd + "
                             "CE(label_smoothing=0.1) + bwd + AdaBelief"),
            "resnet18": ("resnet18", {"num_classes": NUM_CLASSES}, 256, 224, True,
                         "resnet18 224x224 bf16 train step (SURVEY 8-f3): fwd + CE(label_smoothing=0.1) + bwd + AdaBelief"),
            **{k: (k, {"num_classes": NUM_CLASSES}, 128, 224, True,
                   f"{k} 224x224 bf16 train step (SURVEY 8-f3): fwd + CE(label_smoothing=0.1) + bwd + AdaBelief, batch 128/GPU")
               for k in ("res2net50_26w_4s", "sknet50", "convnext_tiny", "tridentnet50", "pyconv_resnet50")},
            "unet3p": ("unet3p", {"num_classes": 21}, 16, 256, True,
                       "unet3p 256x256 segmentation train step (BASELINE configs[4]): fwd + DiceLoss(softmax, one-hot) + bwd + "
                       "AdaBelief; synthetic masks"),
        }
        self.factory, self.kwargs, self.batch, self.size, self.graphable, self.desc = table[key]
        self.metric = METRIC if key == "repvgg_a0" else f"images/sec {key} {self.size}^2 bf16 train"

    def model(self, hb, dev):
        torch.manual_seed(0)
        m = getattr(hb.models, self.factory)(**self.kwargs)
        return m.to(dev).to(memory_format=torch.channels_last).train()

    def host_batch(self, batch: int, seed: int):
        """Synthetic batch on the HOST (pinned); structure depends on the task."""
        g = torch.Generator(device="cpu").manual_seed(seed)
        if self.key in CLS_KEYS:
            x, t = synthetic_batch(batch, seed, "cpu", self.size)
            return [x.pin_memory(), t.pin_memory()]
        x = torch.rand(batch, 3, self.size, self.size, generator=g)
        if self.key == "unet3p":
            mask = torch.randint(0, 21, (batch, self.size, self.size), generator=g)
            return [x.pin_memory(), mask.pin_memory()]
        # yolov4: n ~ U{1..19} boxes per image, xy1 ~ U[0,0.8), wh ~ U[0.05,0.2), clipped to [0,1] (SURVEY §8d);
        # padded to 20 rows per image, the row counts stay on the host (they define tensor shapes)
        counts = torch.randint(1, 20, (batch,), generator=g)
        xy = torch.rand(batch, 20, 2, generator=g) * 0.8
        wh = torch.rand(batch, 20, 2, generator=g) * 0.15 + 0.05
        boxes = torch.cat([xy, (xy + wh).clamp(max=1.0)], -1)
        labels = torch.randint(0, 80, (batch, 20), generator=g)
        self.counts = counts.tolist()
        return [x.pin_memory(), boxes.pin_memory(), labels.pin_memory()]

    def loss(self, model, hbF, *batch):
        if self.key in CLS_KEYS:
            x, t = batch
            return F.cross_entropy(model(x), t, label_smoothing=0.1)
        if self.key == "unet3p":
            x, mask = batch
            out = model(x)
            onehot = F.one_hot(mask, 21).movedim(-1, 1).float()
            return hbF.dice_loss(torch.softmax(out.float(), 1), onehot)
        x, boxes, labels = batch
        target = [{"boxes": boxes[i, :c], "labels": labels[i, :c]} for i, c in enumerate(self.counts)]
        losses = model(x, target)
        return sum(losses.values())


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference(args, rank):
    """The reference algorithm for the same step (oracle = CPU restatement of Holocron's RepVGG + AdaBelief on stock
    torch CPU kernels, pinned to the reference by tests/golden) timed on the host cores. Each step is a bounded
    sample of the workload (an 8-image batch instead of 256)."""
    if rank != 0:
        return
    from oracle.models import RepVGGOracle
    from oracle.optim import adabelief_step
    threads = cpu_threads()
    torch.set_num_threads(threads)
    sample = 8
    torch.manual_seed(0)
    model = RepVGGOracle("repvgg_a0", num_classes=NUM_CLASSES).train()
    params = [p for p in model.parameters()]
    state = [(torch.zeros_like(p), torch.zeros_like(p)) for p in params]
    x, t = synthetic_batch(sample, 0, "cpu")

    def step(i):
        loss = F.cross_entropy(model(x), t, label_smoothing=0.1)
        loss.backward()
        for p, (m, s) in zip(params, state):
            adabelief_step(p.data, p.grad, m, s, i, 1e-3, 0.95, 0.99, 1e-6)
            p.grad = None
        return loss

    for i in range(args.warmup):
        step(i + 1)
    t0 = time.perf_counter()
    for i in range(args.steps):
        loss = step(args.warmup + i + 1)
    dt = (time.perf_counter() - t0) / max(args.steps, 1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, loss, model)
    value = sample / dt
    print(json.dumps({
        "metric": METRIC, "value": value, "unit": "images/s", "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "repvgg_a0 224x224 train step (fwd + CE(ls=0.1) + bwd + AdaBelief), CPU reference path",
                   "batch_per_step": sample},
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": threads, "kind": "port",
                         "sample": f"{sample}-image batches, {args.steps} steps (full workload: 256/GPU)"},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def cpu_threads() -> int:
    """Threads for the CPU legs. Measured on the 128-thread GPU host (tools/cpu_thread_probe.py, fwd+bwd of an 8-image
    batch): 8 threads 0.26 s, 16 threads 0.21 s, 32 threads 0.30 s, 64 threads 0.70 s - torch's CPU convolutions stop
    scaling at ~16 threads for this workload, so the CPU legs use min(16, cpu_count). Override: HB_CPU_THREADS."""
    env = os.environ.get("HB_CPU_THREADS")
    if env:
        return max(1, int(env))
    return max(1, min(os.cpu_count() or 1, 16))


def cpu_baseline(budget_s: float = 20.0):
    """Bounded CPU sample of the same train step (oracle), for the `cpu_baseline` object of the main arm."""
    from oracle.models import RepVGGOracle
    from oracle.optim import adabelief_step
    threads = cpu_threads()
    torch.set_num_threads(threads)
    sample = 8
    torch.manual_seed(0)
    model = RepVGGOracle("repvgg_a0", num_classes=NUM_CLASSES).train()
    params = list(model.parameters())
    state = [(torch.zeros_like(p), torch.zeros_like(p)) for p in params]
    x, t = synthetic_batch(sample, 0, "cpu")
    n, t_total = 0, 0.0
    for i in range(1, 8):
        t0 = time.perf_counter()
        F.cross_entropy(model(x), t, label_smoothing=0.1).backward()
        for p, (m, s) in zip(params, state):
            adabelief_step(p.data, p.grad, m, s, i, 1e-3, 0.95, 0.99, 1e-6)
            p.grad = None
        dt = time.perf_counter() - t0
        if i > 1:  # first step = warm-up
            n += 1
            t_total += dt
        if t_total > budget_s or (i > 2 and t_total + dt > budget_s):
            break
    value = sample * n / t_total if n else sample / dt
    return {"value": value, "unit": "images/s", "cores": threads, "kind": "port",
            "sample": f"{max(n, 1)} steps of an {sample}-image batch (oracle: RepVGG-A0 train step, fp32, torch CPU)"}


def gpu_eager_baseline(batch: int, dev, steps: int = 5):
    """The reference's own execution model on the SAME B200 (SURVEY §8d, BASELINE.md §3.4): stock torch eager modules
    (cuDNN / ATen kernels), bf16 autocast, channels_last, per-tensor AdaBelief update written as the reference writes it
    (~9 ATen launches per parameter tensor). Uses the oracle's module tree (reference algorithm, stock torch layers); it
    is a reported baseline measured beside the product, never part of it."""
    from oracle.models import RepVGGOracle
    from oracle.optim import adabelief_step
    torch.manual_seed(0)
    model = RepVGGOracle("repvgg_a0", num_classes=NUM_CLASSES).to(dev).to(memory_format=torch.channels_last).train()
    params = list(model.parameters())
    state = [(torch.zeros_like(p), torch.zeros_like(p)) for p in params]
    x, t = synthetic_batch(batch, 7, dev)
    x = x.contiguous(memory_format=torch.channels_last)

    def step(i):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss = F.cross_entropy(model(x).float(), t, label_smoothing=0.1)
        loss.backward()
        for p, (m, s) in zip(params, state):
            adabelief_step(p.data, p.grad, m, s, i, 1e-3, 0.95, 0.99, 1e-6)
            p.grad = None

    for i in range(1, 4):
        step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(4 + i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"images_per_s": batch / ms * 1e3, "ms_per_step": ms, "steps": steps,
            "what": "torch eager (cuDNN), bf16 autocast, channels_last, reference-style per-tensor AdaBelief; same step, same GPU"}


# ------------------------------------------------------------------------------------------------ roofline leg
FAMILIES = {
    # timer kind -> (family label = the kernels it covers, bound)
    "fprop": "conv_fprop_kernel+conv_rows_kernel",
    "dgrad": "conv_fprop_kernel+conv_rows_kernel",
    "wgrad": "conv_wgrad_kernel+conv_wgrad_rows_kernel+wgrad_reduce_kernel",
    "bn_stats": "bn_act_fwd_kernel+bn_act_bwd_reduce_kernel+bn_act_bwd_apply_kernel",
    "bn_fwd": "bn_act_fwd_kernel+bn_act_bwd_reduce_kernel+bn_act_bwd_apply_kernel",
    "bn_bwd": "bn_act_fwd_kernel+bn_act_bwd_reduce_kernel+bn_act_bwd_apply_kernel",
    "optimizer": "adabelief_kernel",
}


def roofline_leg(K, run_step, opt_step, n_params: int, step_ms: float, images: int, train_macs_per_image: float):
    """Per-launch CUDA-event timing of ONE extra eager step (stream parked behind a spin kernel so that host gaps are not
    counted) -> per-family {ms, algorithmic GFLOP / GB, achieved TFLOP/s / GB/s, fraction of the measured peak}."""
    K.KERNEL_TIMER = []
    torch.cuda._sleep(int(2.5e8))
    run_step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    opt_step()
    e1.record()
    torch.cuda.synchronize()
    recs = K.KERNEL_TIMER
    K.KERNEL_TIMER = None
    # AdaBelief: read p, g, m, s + write p, m, s = 28 B / parameter (SURVEY §8d)
    recs.append(("optimizer", {"flops": 0.0, "bytes": 28.0 * n_params, "launches": 1, "shape": ("adabelief", n_params)}, e0, e1))
    peaks = measured_peaks()
    fam, by_shape = {}, {}
    for kind, info, a, b in recs:
        ms = a.elapsed_time(b)
        d = fam.setdefault(FAMILIES[kind], {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "launches": 0})
        d["ms"] += ms; d["flops"] += info["flops"]; d["bytes"] += info["bytes"]; d["launches"] += info.get("launches", 1)
        e = by_shape.setdefault((kind,) + tuple(info.get("shape", ())), [0, 0.0, 0.0])
        e[0] += 1; e[1] += ms; e[2] += info["flops"]
    if os.environ.get("HB_BENCH_DETAIL"):
        for key, (cnt, t, fl) in sorted(by_shape.items(), key=lambda kv: -kv[1][1]):
            print(f"DETAIL {key}: n={cnt} total {t:.3f} ms  {fl / max(t, 1e-9) / 1e9:.0f} TFLOP/s", file=sys.stderr)
    per = {}
    for name, d in fam.items():
        t_fl = d["flops"] / (peaks["bf16_tflops"] * 1e12) * 1e3
        t_by = d["bytes"] / (peaks["hbm_gbs"] * 1e9) * 1e3
        tf, gb = d["flops"] / d["ms"] / 1e9, d["bytes"] / d["ms"] / 1e6
        bound = "tensor" if t_fl > t_by else "hbm"
        per[name] = {"ms": round(d["ms"], 3), "launches": d["launches"], "GFLOP": round(d["flops"] / 1e9, 1),
                     "GB": round(d["bytes"] / 1e9, 3), "TFLOP/s": round(tf, 1), "GB/s": round(gb, 1), "bound": bound,
                     "frac": round(tf / peaks["bf16_tflops"] if bound == "tensor" else gb / peaks["hbm_gbs"], 4)}
    conv_fams = [k for k in per if k.startswith("conv_")]
    dom = max(conv_fams or per, key=lambda k: fam[k]["ms"])
    d = fam[dom]
    if per[dom]["bound"] == "tensor":
        roof = {"bound": "tensor", "achieved": d["flops"] / d["ms"] / 1e9, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s"}
    else:
        roof = {"bound": "hbm", "achieved": d["bytes"] / d["ms"] / 1e6, "peak": peaks["hbm_gbs"], "unit": "GB/s"}
    roof["frac"] = roof["achieved"] / roof["peak"]
    roof["traffic"] = None
    roof["algorithmic_bytes"] = d["bytes"] / d["launches"]
    roof["algorithmic_flops"] = d["flops"] / d["launches"]
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            tk = json.load(f)["kernels"]
        names = dom.split("+")      # ncu prints template arguments: conv_fprop_kernel<0>, bn_act_fwd_kernel<3, 1>, ...
        famk = [v for k, v in tk.items() if any(k == n or k.startswith(n + "<") for n in names)]
        if famk:
            roof["traffic"] = sum(k["dram_read_bytes"] + k["dram_write_bytes"] for k in famk) / max(sum(k["launches"] for k in famk), 1)
            roof["traffic_source"] = "ncu dram__bytes_read.sum + dram__bytes_write.sum (profiles/r02_traffic.json), per launch"
    except (OSError, KeyError, ValueError):
        pass
    roof["kernel"] = dom
    roof["peak_source"] = peaks["src"]
    roof["peaks"] = {"bf16_tflops_sustained": peaks["bf16_tflops"], "hbm_gbs": peaks["hbm_gbs"]}
    roof["per_family"] = per
    # whole step: all convolution FLOPs of fwd + dgrad + wgrad (6 x MACs, SURVEY §8d) over the measured step time
    if train_macs_per_image:
        roof["whole_step_tflops"] = round(6.0 * train_macs_per_image * images / (step_ms * 1e-3) / 1e12, 1)
    roof["timed_ms_sum"] = round(sum(v["ms"] for v in per.values()), 3)
    return roof


DUMP_BUDGET_BYTES = 60_000_000     # under 64 MB (10^6 bytes) in all, .npy headers included


def dump_outputs(out_dir: str, loss, model) -> None:
    """Writes what the last timed step computed, as float32 .npy files in `out_dir`: ``loss`` and ``state.<key>`` for every
    floating-point entry of the model's state_dict (parameters after the update, normalisation statistics). When the state
    exceeds the budget, every tensor is cut to the same fraction by a fixed, seeded sample of its flattened elements, so
    that two runs with the same arguments write the same elements."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    state = {f"state.{k}": v.detach() for k, v in model.state_dict().items() if v.is_floating_point()}
    frac = min(1.0, DUMP_BUDGET_BYTES / (4 * sum(v.numel() for v in state.values())))
    g = torch.Generator().manual_seed(0)
    arrays = {"loss": loss.detach().float().reshape(())}
    for k, v in state.items():
        if frac < 1.0:
            idx = torch.randperm(v.numel(), generator=g)[:max(1, int(v.numel() * frac))].sort().values
            v = v.reshape(-1)[idx.to(v.device)]
        arrays[k] = v.float()
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), v.cpu().numpy())
    print(f"[bench] wrote {len(arrays)} arrays to {out_dir} (state sampled at {frac:.3f})", file=sys.stderr)


TRAIN_MACS = {"repvgg_a0": 2.821e9, "repvgg_a1": 4.329e9, "rexnet1_0x": 0.398e9, "yolov4": 45.52e9, "unet3p": 195.49e9,
              "resnet50": 4.09e9, "resnet18": 1.81e9, "mobileone_s0": 1.07e9}


# ------------------------------------------------------------------------------------------------ main arm
def measure(args, wl: Workload, rank: int, local_rank: int, world: int, full: bool):
    """Times `wl` on this process' GPU (all ranks); rank 0 returns the result dict. `full`: roofline / baselines legs."""
    import torch.distributed as dist
    import holocron_b200 as hb
    from holocron_b200.nn import _fused as K
    from holocron_b200.nn import functional as hbF
    from holocron_b200.distributed import GradBucket, OverlappedReducer, broadcast_parameters
    from holocron_b200._lib import lib
    from holocron_b200.graphs import GraphedTrainStep

    dev = torch.device("cuda", local_rank)
    warmup = max(args.warmup, 3)
    model = wl.model(hb, dev)
    broadcast_parameters(model)
    bucket = GradBucket(model.parameters(), direct=not args.no_direct_grads)
    use_graph = wl.graphable and not args.no_graph
    opt = hb.optim.AdaBelief(model.parameters(), lr=1e-3, betas=(0.95, 0.99), eps=1e-6, capturable=use_graph)
    batch = args.batch or wl.batch
    host = wl.host_batch(batch, 1000 + rank)
    devb = [t.to(dev) for t in host]
    if devb[0].ndim == 4:
        devb[0] = devb[0].contiguous()

    # N > 1: the gradient all-reduce leaves in chunks on a side stream while backward is still running (stage boundaries of
    # model.features); the un-overlapped tail is the first stages' few MB
    reducer = None
    if world > 1 and not args.no_overlap and not args.no_direct_grads:
        bounds = OverlappedReducer.stage_boundaries(model)
        if bounds:
            reducer = OverlappedReducer(bucket, bounds)

    def eager_step(*b, collective=True, optimizer=True):
        if reducer is not None:
            reducer.enabled = collective
        loss = wl.loss(model, hbF, *b)
        loss.backward()
        if collective and reducer is not None:
            reducer.finish()
        elif collective:
            bucket.all_reduce_mean()
        if optimizer:
            opt.step()
            bucket.zero_()
        return loss

    train_step, graphed = eager_step, None
    if use_graph:
        try:
            graphed = GraphedTrainStep(eager_step, devb, warmup=3)
            train_step = graphed
        except Exception as e:  # noqa: BLE001 - capture is an optimisation: report and run the same CUDA path eagerly
            import traceback
            traceback.print_exc(file=sys.stderr)
            print(f"[bench] CUDA-graph capture failed ({e!r}); running the step eagerly", file=sys.stderr)
            torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(2 + warmup):
        train_step(*devb)
    barrier()

    # ---- timed region 1: inputs resident in HBM ----------------------------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    lib().hb_launch_count_reset()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    h0 = time.perf_counter()
    for _ in range(args.steps):
        loss = train_step(*devb)
    host_ms = (time.perf_counter() - h0) * 1e3 / args.steps   # host time to ENQUEUE a step (no sync inside the loop)
    e1.record()
    barrier()
    launches = lib().hb_launch_count() + (graphed.launches_per_replay * args.steps if graphed is not None else 0)
    ms = e0.elapsed_time(e1) / args.steps
    clocks = sampler.stop() if rank == 0 else None

    # ---- timed region 2: end to end through the public API with host buffers -----------------------
    copy_stream = torch.cuda.Stream()
    bufs = [[torch.empty_like(t) for t in devb] for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]

    def prefetch(i):
        with torch.cuda.stream(copy_stream):
            for dst, src in zip(bufs[i], host):
                dst.copy_(src, non_blocking=True)
            ready[i].record(copy_stream)

    loss_host = 0.0
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    prefetch(0)
    for i in range(args.steps):
        cur = i & 1
        torch.cuda.current_stream().wait_event(ready[cur])
        if i + 1 < args.steps:
            copy_stream.wait_stream(torch.cuda.current_stream())   # the other buffer is free once step i-1 is queued behind
            prefetch(cur ^ 1)
        loss = train_step(*bufs[cur])
        loss_host = loss.item()                                     # device -> host read of the step's result
    e3.record()
    barrier()
    ms_e2e = e2.elapsed_time(e3) / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, model)

    if world > 1:
        tt = torch.tensor([ms, ms_e2e], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms, ms_e2e = tt.tolist()
    if rank != 0:
        return None

    images = batch * world
    n_params = sum(p.numel() for p in model.parameters())
    roof = roofline_leg(K, lambda: eager_step(*devb, collective=False, optimizer=False),
                        lambda: (opt.step(), bucket.zero_()), n_params, ms, batch, TRAIN_MACS.get(wl.key, 0.0))
    result = {
        "metric": wl.metric, "value": images / ms * 1e3, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": wl.desc, "batch_per_gpu": batch, "global_batch": images, "parallelism": f"dp{world}",
                   "allreduce": ("none" if world == 1 else ("overlapped chunks on a side stream" if reducer is not None
                                                            else "single all-reduce after backward")),
                   "l2": "per-step working set (GBs of activations) exceeds the 126 MB L2; no explicit flush",
                   "launch": "cuda_graph" if graphed is not None else "eager"},
        "e2e": {"value": images / ms_e2e * 1e3, "unit": "images/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(sum(t.numel() * t.element_size() for t in host)), "d2h_bytes_per_step": 4,
                "last_loss": loss_host},
        "gpu_launches": int(launches), "host_enqueue_ms_per_step": round(host_ms, 3),
        "clocks": clocks,
        "roofline": roof,
    }
    if full and world == 1:
        if not args.no_cpu_baseline:
            result["cpu_baseline"] = cpu_baseline()
        if wl.key == "repvgg_a0" and not args.no_eager_baseline:
            try:
                del graphed, train_step
                torch.cuda.empty_cache()
                g = gpu_eager_baseline(batch, dev)
                g["speedup_of_this_repo"] = round(g["ms_per_step"] / ms, 2)
                result["gpu_eager_baseline"] = g
            except Exception as e:  # noqa: BLE001
                result["gpu_eager_baseline"] = {"error": repr(e)[:200]}
    return result


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the configuration's own)")
    ap.add_argument("--model", "--workload", dest="model", default="repvgg_a0",
                    choices=["repvgg_a0", "rexnet1_0x", "repvgg_a1", "yolov4", "unet3p", "resnet50", "resnet18", "mobileone_s0",
                             "res2net50_26w_4s", "sknet50", "convnext_tiny", "tridentnet50", "pyconv_resnet50"],
                    help="repvgg_a0 = the contract metric (default); the others are BASELINE.json configs[1..4]")
    ap.add_argument("--config", type=int, default=0, help="BASELINE.json configs index 1..4 (alias of --model)")
    ap.add_argument("--micro", action="store_true", help="leaf-kernel micro rows (GB/s vs the measured HBM peak) instead of a model")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true", help="skip the torch-eager (cuDNN) baseline leg on the GPU")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel of the step eagerly (no CUDA graph)")
    ap.add_argument("--no-direct-grads", action="store_true", help="let autograd accumulate parameter gradients (A/B switch)")
    ap.add_argument("--no-overlap", action="store_true", help="N > 1: one all-reduce after backward instead of overlapped chunks")
    ap.add_argument("--no-secondary", action="store_true", help="skip the ReXNet-1.0x leg (BASELINE configs[1]) at N=1")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's loss and the model state it left as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.config:
        args.model = {1: "rexnet1_0x", 2: "repvgg_a1", 3: "yolov4", 4: "unet3p"}[args.config]

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl b200) needs a CUDA device: there is no CPU fallback")
    if args.micro:
        if args.dump_outputs:
            raise SystemExit("--dump-outputs: --micro runs no training step")
        from tools.micro_bench import run_micro
        if rank == 0:
            print(json.dumps(run_micro(measured_peaks())), flush=True)
        return

    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=240))

    result = measure(args, Workload(args.model), rank, local_rank, world, full=True)
    if rank == 0 and world == 1 and args.model == "repvgg_a0" and not args.no_secondary:
        # BASELINE.json configs[1] (north_star's second target) measured with the same harness, reported beside the
        # contract metric; never allowed to disturb it
        try:
            import gc
            gc.collect()
            torch.cuda.empty_cache()
            sargs = argparse.Namespace(**vars(args))
            sargs.steps, sargs.warmup, sargs.batch, sargs.dump_outputs = 10, 3, 0, None
            sec = measure(sargs, Workload("rexnet1_0x"), 0, local_rank, 1, full=False)
            result["secondary"] = {"workload": sec["config"]["workload"] + ", batch 256, CUDA-graph replay, inputs resident in HBM",
                                   "images_per_s": sec["value"], "ms_per_step": sec["ms_per_step"], "steps": sec["steps"],
                                   "last_loss": sec["e2e"]["last_loss"], "e2e_images_per_s": sec["e2e"]["value"],
                                   "roofline": sec["roofline"]}
        except Exception as e:  # noqa: BLE001
            result["secondary"] = {"workload": "rexnet1_0x 224x224 bf16 train step, batch 256", "error": repr(e)[:200]}
    if rank == 0:
        print(json.dumps(result), flush=True)
    if world > 1:
        _exit_watchdog()
        # orderly teardown: every captured graph (it holds NCCL kernels) is released before the communicator goes away
        import gc
        torch.cuda.synchronize()
        gc.collect()
        try:
            dist.barrier()
            torch.cuda.synchronize()
            dist.destroy_process_group()
        except Exception as e:  # noqa: BLE001
            print(f"[bench] process-group teardown: {e!r}", file=sys.stderr)
        sys.stdout.flush()
        sys.stderr.flush()


def _exit_watchdog(seconds: float = 25.0):
    """Orderly teardown first; if the NCCL communicator teardown blocks (seen once with captured collectives, NCCL 2.28)
    the process still ends: a daemon timer leaves through os._exit after the result line has been flushed."""
    def _kill():
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    t = threading.Timer(seconds, _kill)
    t.daemon = True
    t.start()


if __name__ == "__main__":
    main()
