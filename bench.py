"""Benchmark of the Gram + attention classifier on B200 (contract: one JSON line on stdout from rank 0).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload (BASELINE.json configs[1]): truncated ResNet50 (truncate_layer 7) + Gram + attention, random-init weights,
synthetic batch of 256 images per GPU at 224x224, 4 classes, inference (eval mode, no_grad). A step is one forward of
the whole model on one batch: cuDNN encoder (left to the reference's path, timed separately in `breakdown`) followed by
the sm_100a head (3 pooled-Gram launches + attention/classifier). Multi-GPU: the batch is sharded, 256 images per rank
(weak scaling); the only collective is the all-gather of logits and embeddings, inside the timed region.

  value      images/s with the batch resident in HBM (154 MB of fp32 images per rank: larger than the 126 MB L2)
  e2e        same through the public call model(x_host): pinned host batch -> H2D -> forward -> logits+embeddings D2H;
             the median of three passes of the K-step loop (all three under `passes_ms_per_step`)
  e2e_uint8  the same loop fed uint8 pixels (opt-in loader path: a quarter of the upload, ToTensor + Normalize on the GPU,
             bit-identical batch); reported beside e2e, never as it
  roofline   the HEAD kernel (Gram / attention, SURVEY 8(a)) that takes the most time inside the timed steps, measured
             live with CUDA events; backbone-side kernels of the library (max pool, stem staging) are listed under
             `breakdown.kernels` only
  cpu_baseline  the UNMODIFIED reference module (staged under baseline/_ref by tools/stage_reference.py and loaded by
             file path; the oracle port when it is absent) on this box's host cores, bounded sample; next to it
             `cpu_extra`: the reference head alone on captured stage activations and its training step at batch 8 with
             anomaly detection as shipped (on) and off (BASELINE.md section 4, items 3b / 3c)
  reference_gpu  the same unmodified reference module on this B200 in fp32 (its own cuBLAS / cuDNN path): configs[1]
             forward and configs[2] training step, backbone and head separated (BASELINE.md section 4, item 4)
  train      BASELINE.json configs[2]: full training step (forward + Gram backward + AdamW), global batch 512 sharded
             over the N ranks with DDP/NCCL (strong scaling); reported as an extra object, not as `value`; its headline
             scalars are repeated as the LAST keys of the line (train_strong_img_s, head_fwd_bwd_frac_of_bf16_peak, ...)

--dump-outputs DIR writes what the last timed step returned (embeddings, logits) as DIR/<name>.npy; the weights and the
batch come from fixed seeds, so two builds run with the same arguments can be compared output for output.

--impl reference times the reference's own CPU implementation of the same forward (the unmodified reference class,
kind "reference"; the oracle port, kind "port", only when baseline/_ref was not staged) with every host thread.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# The training leg replays its step from a CUDA graph that contains DDP's NCCL all-reduce (functions.GraphedTrainStep):
# torch requires NCCL's asynchronous error handling to be off for that, set before init_process_group.
os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")
os.environ.setdefault("NCCL_ASYNC_ERROR_HANDLING", "0")

import torch  # noqa: E402

TRUNC, NUM_CLASSES, GRAM_SIZE, IMAGE = 7, 4, 32, 224
WORKLOAD = ("configs[1]: truncated ResNet50 (7 children) + Gram + attention, random init, synthetic batch 256/GPU at "
            "224x224, 4 classes, inference")


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p["hbm_gbs"], tensor_tflops=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                    tensor_tflops_burst=p["bf16_tflops"], source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tensor_tflops=1400.0, tensor_tflops_burst=1590.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """SM clock and throttle reasons of GPU `index`, sampled through NVML every 10 ms from a thread while the timed
    region runs (an nvidia-smi subprocess needs longer to start than a 0.1 s region lasts, which left the multi-rank
    runs of round 1 without samples)."""
    REASONS = (("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40), ("sw_power_cap", 0x4))

    def __init__(self, device):
        self.rows, self.stop, self.thread, self.handle, self.nv = [], threading.Event(), None, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            p = torch.cuda.get_device_properties(device)
            bus_id = f"{p.pci_domain_id:08x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
            self.handle = pynvml.nvmlDeviceGetHandleByPciBusId(bus_id.encode())
            self.nv = pynvml
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.handle = None

    def _pump(self):
        nv = self.nv
        while not self.stop.is_set():
            try:
                self.rows.append((nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM),
                                  nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)))
            except Exception:
                pass
            self.stop.wait(0.01)

    def __enter__(self):
        if self.handle is not None:
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        return self

    def __exit__(self, *exc):
        self.stop.set()
        if self.thread is not None:
            self.thread.join(timeout=2)
        return False

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = [r[0] for r in self.rows]
        reasons = sorted({name for _, mask in self.rows for name, bit in self.REASONS if mask & bit})
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(sm),
                "how": "NVML, 10 ms period, during the timed region"}


def guarded(name, fn, *a, **kw):
    """Side legs (everything beside the headline numbers) must not cost the run its JSON line: a failure is reported in
    the leg's place and on stderr. Only for legs without collectives -- a rank that skips one would hang the others."""
    try:
        return fn(*a, **kw)
    except Exception as exc:                                           # noqa: BLE001 - reported, not hidden
        import traceback
        traceback.print_exc()
        return {"error": f"{name}: {type(exc).__name__}: {exc}"[:400]}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory, arrays):
    """Writes `arrays` (name -> tensor, one row per image) as <directory>/<name>.npy in float32, so that two builds can be
    compared output for output on the same inputs. Above DUMP_LIMIT_BYTES in all, the same fixed, seeded sample of rows
    is kept from every array."""
    import numpy as np
    rows = next(iter(arrays.values())).shape[0]
    row_bytes = sum(t[0].numel() * 4 for t in arrays.values())
    keep = min(rows, DUMP_LIMIT_BYTES // row_bytes)
    if keep == 0:
        raise ValueError(f"dump_outputs: one row takes {row_bytes} bytes, more than the {DUMP_LIMIT_BYTES}-byte limit")
    index = None
    if keep < rows:
        index = torch.from_numpy(np.sort(np.random.default_rng(0).choice(rows, keep, replace=False)))
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float().cpu()
        np.save(os.path.join(directory, name + ".npy"), (t if index is None else t[index]).numpy())


def timed_region(fn, steps, device, dist_mod):
    """barrier + synchronize, CUDA events on the current stream around exactly `steps` calls, max over ranks (ms)."""
    dist_mod.barrier(device)
    torch.cuda.synchronize(device)
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(steps):
        fn()
    end.record()
    torch.cuda.synchronize(device)
    dist_mod.barrier(device)
    return dist_mod.max_over_ranks(start.elapsed_time(end), device)


HEAD_KINDS = ("gram_fwd", "gram_bwd", "attn")      # SURVEY 8(a) rows a2-a7, a9: what the roofline object may name
HEAD_TIME_KINDS = HEAD_KINDS + ("split",)          # + the per-step split of the attention weights into bf16 planes (training)


def head_totals(records, steps, peaks):
    """Per-step time and algorithmic FLOPs of the head kernels (Gram forward: symmetric count C(C+1)HW; Gram backward:
    dense 2 C^2 HW; attention: its GEMMs; the weight-plane splits a training step needs count as attention-forward time,
    with no FLOPs) and the fraction of the measured bf16 tensor peak they amount to."""
    t = {"gram_fwd": 0.0, "gram_bwd": 0.0, "attn_fwd": 0.0, "attn_bwd": 0.0}
    flops = 0.0
    for name, work, s, e in records:
        kind = work.get("kind")
        if kind not in HEAD_TIME_KINDS:
            continue
        key = kind if kind in ("gram_fwd", "gram_bwd") else ("attn_bwd" if name.startswith("attn_head_bwd") else "attn_fwd")
        t[key] += s.elapsed_time(e) * 1e3
        flops += work["flops"]
    total_us = sum(t.values()) / steps
    if total_us <= 0:
        return None
    tf = flops / steps / total_us / 1e6
    return {"gram_fwd_us": round(t["gram_fwd"] / steps, 1), "gram_bwd_us": round(t["gram_bwd"] / steps, 1),
            "attn_fwd_us": round(t["attn_fwd"] / steps, 1), "attn_bwd_us": round(t["attn_bwd"] / steps, 1),
            "head_us": round(total_us, 1), "algorithmic_gflop_per_step": round(flops / steps / 1e9, 1),
            "TFLOPs": round(tf, 1), "frac_of_bf16_peak_burst": round(tf / peaks["tensor_tflops_burst"], 4),
            "frac_of_bf16_peak_sustained": round(tf / peaks["tensor_tflops"], 4)}


def summarise_profile(records, peaks):
    """records: ops.PROFILE entries -> per-kernel averages and the roofline object of the dominant one."""
    agg = {}
    for name, work, s, e in records:
        a = agg.setdefault(name, dict(ms=0.0, n=0, work=work))
        a["ms"] += s.elapsed_time(e)
        a["n"] += 1
    kernels = {}
    for name, a in agg.items():
        ms = a["ms"] / a["n"]
        kernels[name] = dict(avg_us=round(ms * 1e3, 2), launches=a["n"], total_ms=round(a["ms"], 3),
                             GBps=round(a["work"]["bytes"] / ms / 1e6, 1), TFLOPs=round(a["work"]["flops"] / ms / 1e9, 1))
    head = {k: v for k, v in agg.items() if v["work"].get("kind") in HEAD_KINDS}
    if not head:
        return kernels, None
    top = max(head, key=lambda k: head[k]["ms"])
    a = agg[top]
    ms = a["ms"] / a["n"]
    t_hbm = a["work"]["bytes"] / (peaks["hbm_gbs"] * 1e9)
    t_tc = a["work"]["flops"] / (peaks["tensor_tflops"] * 1e12)
    if t_hbm >= t_tc:
        ach, peak, unit, bound = a["work"]["bytes"] / ms / 1e6, peaks["hbm_gbs"], "GB/s", "hbm"
    else:
        ach, peak, unit, bound = a["work"]["flops"] / ms / 1e9, peaks["tensor_tflops"], "TFLOP/s", "tensor"
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.isfile(tpath):
        table = json.load(open(tpath))
        traffic = table.get(top)
        captured = table.get("_algorithmic_bytes_of_captured_launch", {}).get(top)
        if traffic is not None and captured:          # ncu capture was taken at batch 256: scale to this launch's size
            traffic = int(round(traffic * a["work"]["bytes"] / captured))
    roof = dict(kernel=top, bound=bound, achieved=round(ach, 1), peak=peak, unit=unit, frac=round(ach / peak, 4),
                traffic=traffic, avg_launch_us=round(ms * 1e3, 2), algorithmic_bytes=a["work"]["bytes"],
                algorithmic_flops=a["work"]["flops"], peak_source=peaks["source"],
                share_of_library_time=round(a["ms"] / sum(v["ms"] for v in agg.values()), 3))
    return kernels, roof


def patchgan_leg(device, peaks, steps, batch=256):
    """MultiScaleDiscriminator_test (ndf 64, gram_matrix_dim 64, batch norm, patches 10/70/150) on `batch` 224x224 images,
    eval + no_grad: cuDNN extractor + the library's head kernels. The head's dominant launch is the pooling pass
    (HBM-bound). Parity against the reference's op sequence is checked in tests/test_gpu_patchgan.py and smoke(); its
    timing on the same GPU is in profiles/r01x_patchgan_head_summary.md (tests/tools/bench_patchgan.py)."""
    from heuristique_style_transfer_code_b200 import ops
    from heuristique_style_transfer_code_b200.patchgan import MultiScaleDiscriminator_test
    torch.manual_seed(0)
    m = MultiScaleDiscriminator_test(ndf=64, norm='batch', num_classes=NUM_CLASSES, gram_matrix_dim=64).to(device).eval()
    x = torch.randn(batch, 3, IMAGE, IMAGE, device=device)
    with torch.no_grad():
        for _ in range(3):
            m(x)
        torch.cuda.synchronize(device)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        saved, ops.PROFILE = ops.PROFILE, []
        s.record()
        for _ in range(steps):
            emb, out = m(x)
        e.record()
        torch.cuda.synchronize(device)
        rec, ops.PROFILE = ops.PROFILE, saved
    ours = s.elapsed_time(e) / steps
    kernels, roof = summarise_profile(rec, peaks)
    head_ms = sum(k["total_ms"] for k in kernels.values()) / steps
    return {"workload": f"MultiScaleDiscriminator_test ndf 64, gram_matrix_dim 64, 3 scales, batch {batch} at {IMAGE}x{IMAGE}, "
                        "eval/no_grad", "images_per_s": round(batch / ours * 1e3, 1), "ms_per_step": round(ours, 3),
            "head_kernels_ms": round(head_ms, 3), "finite": bool(torch.isfinite(emb).all() and torch.isfinite(out).all()),
            "kernels": kernels, "roofline": roof}


def reference_classes():
    """-> (train class, test class, kind): the UNMODIFIED reference classes, loaded by file path from the staged copy of
    the reference tree (baseline/_ref travels to the GPU box; /root/reference does not); the oracle port only when no
    copy of the reference is available."""
    try:
        from heuristique_style_transfer_code_b200._reference import load_reference_file
        m = load_reference_file(os.path.join("Models", "Models_RESNET50_TRUNCATE_GRAM_with_Attention.py"))
        return m.TruncatedResNet50, m.TruncatedResNet50_for_test, "reference"
    except NotImplementedError:
        from oracle.torch_port import PortModel

        def train_cls(base, trunc, nc, g, device="cpu"):
            return PortModel(base, trunc, nc, g, device=device, return_embeddings=False)

        def test_cls(base, trunc, nc, g, device="cpu"):
            return PortModel(base, trunc, nc, g, device=device, return_embeddings=True)
        return train_cls, test_cls, "port"


def reference_head(model, stages):
    """The reference's head on given stage activations: its own op sequence (Models/...Attention.py:50-61) issued through
    the reference module's gram_matrix / attention / classifier."""
    F = torch.nn.functional
    g = model.gram_matrix_size
    grams = [F.adaptive_avg_pool2d(model.gram_matrix(a), (g, g)) for a in stages]
    tokens = torch.stack(grams, dim=1).flatten(2).permute(1, 0, 2)
    out, _ = model.attention(tokens, tokens, tokens)
    emb = out.mean(dim=0)
    return emb, model.classifier(emb)


def capture_stages(model, x):
    got = []
    hooks = [blk.register_forward_hook(lambda m, i, o: got.append(o.detach()))
             for blk in list(model.truncated_encoder.children())[4:]]
    with torch.no_grad():
        model(x)
    for h in hooks:
        h.remove()
    return got


def wall_time(fn, warmup, steps, sync=None):
    times = []
    for i in range(warmup + steps):
        if sync:
            sync()
        t0 = time.perf_counter()
        fn()
        if sync:
            sync()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return statistics.median(times)


def cpu_reference_forward(sample, steps, warmup, threads):
    """The reference's CPU path, eval + no_grad, on `sample` images of the synthetic batch -> (images/s, s/step, kind)."""
    from torchvision import models
    _, test_cls, kind = reference_classes()
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    model = test_cls(models.resnet50(weights=None), TRUNC, NUM_CLASSES, GRAM_SIZE, device="cpu")
    model.eval()
    torch.manual_seed(1)
    x = torch.randn(sample, 3, IMAGE, IMAGE)
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            model(x)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    return sample * len(times) / sum(times), sum(times) / len(times), kind


def cpu_extra_legs(threads):
    """BASELINE.md section 4, items 3b / 3c on this box's host cores: the reference head alone on captured stage
    activations (batch 8), and its training step at batch 8 (SGD momentum 0.9, the reference's optimizer) with
    torch.autograd anomaly detection as the reference ships it (on, Models/...Attention.py:9) and off."""
    from torchvision import models
    train_cls, test_cls, kind = reference_classes()
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    model = test_cls(models.resnet50(weights=None), TRUNC, NUM_CLASSES, GRAM_SIZE, device="cpu").eval()
    torch.manual_seed(1)
    x = torch.randn(8, 3, IMAGE, IMAGE)
    stages = capture_stages(model, x)
    with torch.no_grad():
        head_s = wall_time(lambda: reference_head(model, stages), 2, 8)
        fwd_s = wall_time(lambda: model(x), 2, 6)
    tm = train_cls(models.resnet50(weights=None), TRUNC, NUM_CLASSES, GRAM_SIZE, device="cpu").train()
    opt = torch.optim.SGD(tm.parameters(), lr=1e-3, momentum=0.9)
    y = torch.randint(0, NUM_CLASSES, (8,))

    def step():
        opt.zero_grad()
        torch.nn.functional.cross_entropy(tm(x), y).backward()
        opt.step()
    out = {"kind": kind, "cores": threads, "batch": 8, "forward_images_per_s": round(8 / fwd_s, 2),
           "head_only_ms": round(head_s * 1e3, 2), "head_only_images_per_s": round(8 / head_s, 1)}
    prev = torch.is_anomaly_enabled()
    try:
        for flag, key in ((True, "train_step_anomaly_on_s"), (False, "train_step_anomaly_off_s")):
            torch.autograd.set_detect_anomaly(flag)
            out[key] = round(wall_time(step, 1, 4), 3)
    finally:
        torch.autograd.set_detect_anomaly(prev)
    out["train_images_per_s_as_shipped"] = round(8 / out["train_step_anomaly_on_s"], 2)
    return out


def reference_gpu_legs(device, steps):
    """BASELINE.md section 4, item 4: the unmodified reference module on this B200 in fp32, its own cuBLAS / cuDNN path
    (torch defaults: fp32 matmul without TF32, cuDNN convolutions with TF32 allowed): configs[1] forward at batch 256 and
    configs[2] training step at batch 512 (AdamW), the cuDNN backbone and the reference's head timed separately."""
    from torchvision import models
    train_cls, test_cls, kind = reference_classes()
    sync = lambda: torch.cuda.synchronize(device)
    torch.manual_seed(0)
    model = test_cls(models.resnet50(weights=None), TRUNC, NUM_CLASSES, GRAM_SIZE, device=device).to(device).eval()
    torch.manual_seed(1)
    x = torch.randn(256, 3, IMAGE, IMAGE, device=device)
    stages = capture_stages(model, x)
    enc = model.truncated_encoder
    with torch.no_grad():
        fwd = wall_time(lambda: model(x), 3, steps, sync)
        backbone = wall_time(lambda: enc(x), 3, steps, sync)
        head = wall_time(lambda: reference_head(model, stages), 3, steps, sync)
    out = {"kind": kind, "dtype": "fp32 (torch defaults)",
           "infer_batch256": {"images_per_s": round(256 / fwd, 1), "ms_per_step": round(fwd * 1e3, 3),
                              "backbone_ms": round(backbone * 1e3, 3), "head_ms": round(head * 1e3, 3)}}
    del model, stages, x
    torch.cuda.empty_cache()
    torch.manual_seed(0)
    tm = train_cls(models.resnet50(weights=None), TRUNC, NUM_CLASSES, GRAM_SIZE, device=device).to(device).train()
    opt = torch.optim.AdamW(tm.parameters(), lr=1e-3)
    xt = torch.randn(512, 3, IMAGE, IMAGE, device=device)
    yt = torch.randint(0, NUM_CLASSES, (512,), device=device)

    def step():
        opt.zero_grad(set_to_none=True)
        torch.nn.functional.cross_entropy(tm(xt), yt).backward()
        opt.step()

    def backbone_step():
        tm.truncated_encoder(xt).sum().backward()
    tstep = wall_time(step, 2, max(3, steps // 2), sync)
    bstep = wall_time(backbone_step, 2, max(3, steps // 2), sync)
    tm.zero_grad(set_to_none=True)
    out["train_batch512"] = {"images_per_s": round(512 / tstep, 1), "ms_per_step": round(tstep * 1e3, 2),
                             "backbone_fwd_bwd_ms": round(bstep * 1e3, 2),
                             "head_fwd_bwd_and_optimizer_ms": round((tstep - bstep) * 1e3, 2),
                             "anomaly_detection": "off (the reference switches it on at import; see cpu_extra)"}
    del tm, opt, xt, yt
    torch.cuda.empty_cache()
    return out


def reference_sample_size(steps, warmup, threads, budget_s=150.0):
    """Images per CPU step: the largest of 256 (the whole batch) / 128 / 64 / 32 with which `warmup + steps` forwards stay
    inside `budget_s`, from the rate of one probe forward of 32 images (the per-image cost grows with the batch on a CPU:
    the (B, C, C) Gram intermediates leave the caches)."""
    ips, _, _ = cpu_reference_forward(32, 1, 1, threads)
    for sample in (256, 128, 64):
        if (steps + warmup) * sample / (0.6 * ips) <= budget_s:
            return sample
    return 32


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    sample = reference_sample_size(args.steps, max(args.warmup, 1), cores)
    ips, sec, kind = cpu_reference_forward(sample, args.steps, max(args.warmup, 1), cores)
    what = ("the UNMODIFIED reference class TruncatedResNet50_for_test, loaded by file path from baseline/_ref "
            "(tools/stage_reference.py)") if kind == "reference" else \
        "oracle/torch_port.py: the reference's op sequence (no staged copy of the reference on this box)"
    line = {"impl": "reference", "metric": "images/sec", "value": round(ips, 2), "unit": "images/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(sec * 1e3, 2), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "global_batch": sample, "per_gpu_batch": sample, "image": IMAGE,
                       "truncate_layer": TRUNC, "gram_matrix_size": GRAM_SIZE, "num_classes": NUM_CLASSES,
                       "note": f"each step is one eval/no_grad forward of {sample} images of the batch on the host cores"},
            "cpu_baseline": {"value": round(ips, 2), "unit": "images/s", "cores": cores, "kind": kind,
                             "sample": f"{sample} images per step, {args.steps} steps after {max(args.warmup, 1)} warm-ups, "
                                       f"torch {torch.__version__} CPU fp32, {cores} threads; {what}"},
            "e2e": {"value": round(ips, 2), "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(json.dumps(line))


def run_ours(args):
    from torchvision import models
    from heuristique_style_transfer_code_b200 import TruncatedResNet50, TruncatedResNet50_for_test, ops, _lib
    from heuristique_style_transfer_code_b200 import distributed as D

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the head has no CPU path (use --impl reference for the CPU arm)")
    _lib.lib()
    rank, world, local, device = D.init_from_env()
    if world != args.gpus and rank == 0:
        print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; launch with torch.distributed.run", file=sys.stderr)
    peaks = load_peaks()
    B = args.batch_per_gpu

    torch.manual_seed(0)
    model = TruncatedResNet50_for_test(models.resnet50(weights=None), TRUNC, NUM_CLASSES, GRAM_SIZE, device=device)
    model.eval()
    torch.manual_seed(1 + rank)
    x_host = torch.randn(B, 3, IMAGE, IMAGE).pin_memory()
    x = x_host.to(device)
    total = B * world

    last = {}

    def infer_step():
        with torch.no_grad():
            emb, logits = model(x)
            if world > 1:
                logits = D.gather_rows(logits, total, world)
                emb = D.gather_rows(emb, total, world)
        last["embeddings"], last["logits"] = emb, logits
        return emb, logits

    for _ in range(args.warmup):
        infer_step()
    ops.PROFILE = []
    ops.LAUNCHES = 0
    with ClockSampler(device) as clocks:
        ms = timed_region(infer_step, args.steps, device, D)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)          # the last timed step's results, before any other leg runs
    records, ops.PROFILE = ops.PROFILE, None
    launches = ops.LAUNCHES
    kernels, roof = summarise_profile(records, peaks)
    value = total * args.steps / (ms / 1e3)

    # ---- breakdown: encoder alone, head alone (device resident, same batch) ----
    with torch.no_grad():
        _, stages = model._stage_activations(x)

        def enc_only():
            with torch.no_grad():
                model._stage_activations(x)

        def head_only():
            with torch.no_grad():
                d = ops.style_descriptor(stages, GRAM_SIZE)
                ops.attention_head(d, model.attention.in_proj_weight, model.attention.in_proj_bias,
                                   model.attention.out_proj.weight, model.attention.out_proj.bias,
                                   model.classifier.weight, model.classifier.bias)
        for _ in range(3):
            enc_only(); head_only()
        enc_ms = timed_region(enc_only, args.steps, device, D) / args.steps
        head_ms = timed_region(head_only, args.steps, device, D) / args.steps
    del stages

    # ---- end to end through the public API: pinned host batches in, logits + embeddings back on the host ----
    # The loop is the package's evaluation loop shape (functions.evaluate_model_test): cuda_prefetch uploads batch i+1
    # on a side stream while batch i is in the model and HostCollector brings every step's embeddings + logits back
    # into pinned host memory without a per-step synchronisation; every step's H2D copy and D2H read are inside the
    # timed region, which ends only when the last step's results are on the host.
    from heuristique_style_transfer_code_b200.functions import HostCollector, cuda_prefetch

    def e2e_loop(n):
        results = HostCollector()
        with torch.no_grad():
            for (xb,) in cuda_prefetch(((x_host,) for _ in range(n)), device, reuse_buffers=True):
                emb, logits = model(xb)
                if world > 1:
                    logits = D.gather_rows(logits, total, world)
                    emb = D.gather_rows(emb, total, world)
                results.push(emb, logits)             # D2H of this step's results into pinned host memory
        out = results.finish()                        # every step's results are on the host when the region ends
        assert len(out) == n and out[-1][1].shape == (total, NUM_CLASSES)

    # warm-up: more steps than HostCollector has ring slots (4), so that every pinned buffer a pass needs exists before the
    # timed passes (a cudaHostAlloc inside a 0.13 s timed region costs it whole per cent, on some hosts far more)
    e2e_loop(6)
    # the copy alone, for reading the end-to-end number: a step cannot be faster than its 154 MB upload
    cp0, cp1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(device)
    cp0.record()
    t_issue = time.perf_counter()
    for _ in range(3):
        x.copy_(x_host, non_blocking=True)
    h2d_issue_ms = (time.perf_counter() - t_issue) / 3 * 1e3   # host time of the copy CALL: ~0.01 ms when it is asynchronous;
    cp1.record()                                               # close to h2d_alone_ms on a box whose driver blocks in it
    torch.cuda.synchronize(device)
    h2d_alone_ms = cp0.elapsed_time(cp1) / 3
    # Does this box overlap a host->device copy with kernels at all? The same 154 MB copy on a side stream, issued together
    # with one forward on resident data, no dependency between them: ~max(forward, copy) on a box that overlaps them (then
    # e2e ~ value), ~forward + copy on one that does not. (Earlier runs read e2e 8.8-9.7 ms per step on part of the pool;
    # DESIGN section 5 traces that to a pinned allocation inside the timed pass, not to missing overlap.
    # tools/diag_copy_overlap.py is the longer version of this probe.)
    probe_stream = torch.cuda.Stream(device)
    x_probe = torch.empty_like(x)
    torch.cuda.synchronize(device)
    t_probe = time.perf_counter()
    for _ in range(5):
        with torch.cuda.stream(probe_stream):
            x_probe.copy_(x_host, non_blocking=True)
        infer_step()
    torch.cuda.synchronize(device)
    overlap_probe_ms = (time.perf_counter() - t_probe) / 5 * 1e3
    del x_probe
    # three passes of the K-step loop, each timed on its own; the MEDIAN pass is the e2e number and all three are kept in the
    # record (a pass is 0.13 s: one host hiccup moves it by several per cent, a box that does not overlap moves all three)
    e2e_passes = [timed_region(lambda: e2e_loop(args.steps), 1, device, D) for _ in range(3)]     # in the order they ran
    e2e_ms = sorted(e2e_passes)[1]
    # what one fresh pinned allocation costs on this host (cudaHostAlloc maps the pages for every GPU of the box: sub-ms on
    # some hosts, tens of ms on others) -- the reason the warm-up above has to create every ring slot before the timed passes
    t_pin = time.perf_counter()
    fresh_pinned = torch.empty(3 << 20, dtype=torch.uint8, pin_memory=True)
    pinned_alloc_ms = (time.perf_counter() - t_pin) * 1e3
    del fresh_pinned
    e2e_value = total * args.steps / (e2e_ms / 1e3)
    h2d = B * 3 * IMAGE * IMAGE * 4
    d2h = total * (GRAM_SIZE * GRAM_SIZE + NUM_CLASSES) * 4

    # ---- the same loop fed uint8 pixels (opt-in loader path, functions.uint8_transform): a quarter of the upload, ToTensor's
    # /255 and Normalize applied on the GPU by gh_normalize_u8, the model sees bit for bit the fp32 batch the host transforms
    # would have produced. Reported beside `e2e` (which keeps the reference loader's fp32 batches), never as it.
    def e2e_uint8_setup():
        """Everything of the leg that is local to a rank, including one dry step of the uint8 path without collectives."""
        from heuristique_style_transfer_code_b200.functions import IMAGENET_MEAN, IMAGENET_STD, _normalize_host
        u8_host = torch.randint(0, 256, (B, 3, IMAGE, IMAGE), dtype=torch.uint8,
                                generator=torch.Generator().manual_seed(7 + rank)).pin_memory()
        same = torch.equal(ops.normalize_u8(u8_host[:8].to(device), IMAGENET_MEAN, IMAGENET_STD).cpu(),
                           _normalize_host(u8_host[:8], IMAGENET_MEAN, IMAGENET_STD))
        with torch.no_grad():
            for (xb,) in cuda_prefetch(iter([(u8_host,)]), device, reuse_buffers=True):
                assert xb.dtype == torch.float32 and xb.shape == (B, 3, IMAGE, IMAGE)
                model(xb)
        torch.cuda.synchronize(device)
        return u8_host, bool(same)

    def e2e_uint8_run(u8_host, same):
        def loop(n):
            results = HostCollector()
            with torch.no_grad():
                for (xb,) in cuda_prefetch(((u8_host,) for _ in range(n)), device, reuse_buffers=True):
                    emb, logits = model(xb)
                    if world > 1:
                        logits = D.gather_rows(logits, total, world)
                        emb = D.gather_rows(emb, total, world)
                    results.push(emb, logits)
            assert len(results.finish()) == n

        loop(6)
        passes = [timed_region(lambda: loop(args.steps), 1, device, D) for _ in range(3)]
        med = sorted(passes)[1]
        return {"value": round(total * args.steps / (med / 1e3), 1), "unit": "images/s",
                "ms_per_step": round(med / args.steps, 3), "passes_ms_per_step": [round(p / args.steps, 3) for p in passes],
                "h2d_bytes_per_step": B * 3 * IMAGE * IMAGE, "d2h_bytes_per_step": d2h,
                "device_batch_bit_identical_to_host_transforms": same,
                "input": "uint8 pixels in pinned host memory; /255 and Normalize on the GPU (gh_normalize_u8) on the upload stream"}

    e2e_u8 = None
    if not args.skip_uint8:
        # a side leg must not cost the run its line: the rank-local part runs guarded, the ranks then agree on whether all of
        # them got through it, and only then enter the loops that contain collectives
        state = guarded("e2e_uint8", e2e_uint8_setup)
        failed = isinstance(state, dict)
        if D.max_over_ranks(1.0 if failed else 0.0, device) > 0:
            e2e_u8 = state if failed else {"error": "e2e_uint8: set-up failed on another rank"}
        elif world > 1:
            e2e_u8 = e2e_uint8_run(*state)
        else:
            e2e_u8 = guarded("e2e_uint8", e2e_uint8_run, *state)
        del state

    # ---- opt-in backbone hand-off (SURVEY 8(f) n1): encoder under bf16 autocast, channels_last; same batch, device resident.
    # Reported beside the headline, never as it: it changes the numerics of the cuDNN backbone (not of the head).
    handoff = None
    if not args.skip_handoff:
        model.set_backbone_mode("bf16_channels_last")
        for _ in range(3):
            infer_step()
        hms = timed_region(infer_step, args.steps, device, D)
        default_mode = "channels_last"
        with torch.no_grad():
            _, lg_fast = model(x)
            model.set_backbone_mode("reference")
            for _ in range(2):
                infer_step()
            rms = timed_region(infer_step, max(3, args.steps // 4), device, D) / max(3, args.steps // 4)
            _, lg_ref = model(x)
            model.set_backbone_mode(default_mode)
            _, lg_def = model(x)
            model.fold_batchnorm = False                 # children executed one by one, as the reference does
            for _ in range(2):
                infer_step()
            nsteps = max(3, args.steps // 4)
            ums = timed_region(infer_step, nsteps, device, D) / nsteps
            _, lg_unf = model(x)
            model.fold_batchnorm = True
        handoff = {"default_mode": default_mode + (" + folded eval-mode batch norm (cuDNN conv+bias+ReLU epilogues)"
                                                   if model._plan is not None else ""),
                   "default_vs_unfolded_logits_rel_diff": float((lg_def - lg_unf).norm() / lg_unf.norm()),
                   "default_vs_unfolded_argmax_equal": bool((lg_def.argmax(1) == lg_unf.argmax(1)).all()),
                   "unfolded_channels_last_ms_per_step": round(ums, 3),
                   "unfolded_channels_last_images_per_s": round(total / (ums / 1e3), 1),
                   "default_vs_nchw_logits_rel_diff": float((lg_def - lg_ref).norm() / lg_ref.norm()),
                   "nchw_reference_mode_ms_per_step": round(rms, 3),
                   "nchw_reference_mode_images_per_s": round(total / (rms / 1e3), 1),
                   "mode": "bf16_channels_last", "value": round(total * args.steps / (hms / 1e3), 1), "unit": "images/s",
                   "ms_per_step": round(hms / args.steps, 3),
                   "logits_rel_diff_vs_fp32_backbone": float((lg_fast.float() - lg_ref).norm() / lg_ref.norm()),
                   "argmax_equal": bool((lg_fast.argmax(1) == lg_ref.argmax(1)).all())}

    # ---- SURVEY 8(f) n4: Multi-PatchGAN discriminators (MultiScaleDiscriminator_test) with the Gram head on this library,
    # against the fp32 torch port of the reference forward on the same GPU and weights; reported beside the headline.
    patchgan = None
    if not args.skip_patchgan and rank == 0:
        patchgan = guarded("patchgan_head", patchgan_leg, device, peaks, max(3, args.steps // 4))

    # ---- configs[2]: training step, global batch 512 over the ranks (strong scaling), AdamW ----
    train = None
    if not args.skip_train:
        del x
        torch.cuda.empty_cache()
        gb = args.train_global_batch
        lo, hi = D.shard_bounds(gb, rank, world)
        torch.manual_seed(0)
        tmodel = TruncatedResNet50(models.resnet50(weights=None), TRUNC, NUM_CLASSES, GRAM_SIZE, device=device)
        tmodel.train()
        # DDP settings from tools/sweep_ddp.py (profiles/r2_ddp_sweep_*.json): 16 MB buckets start the all-reduce of the
        # head's gradients (ready first) under the encoder's backward; fused AdamW is one launch (capturable: the step is
        # also replayed from a CUDA graph below); DDP is constructed on a side stream, as graph capture requires
        ddp = D.wrap_ddp(tmodel, device, bucket_cap_mb=16, for_graph_capture=True)
        opt = torch.optim.AdamW(tmodel.parameters(), lr=1e-3, fused=True, capturable=True)
        crit = torch.nn.CrossEntropyLoss()
        torch.manual_seed(100 + rank)
        xt = torch.randn(hi - lo, 3, IMAGE, IMAGE, device=device)
        yt = torch.randint(0, NUM_CLASSES, (hi - lo,), device=device)

        def train_step():
            opt.zero_grad(set_to_none=True)
            loss = crit(ddp(xt), yt)
            loss.backward()
            opt.step()
            return loss

        tsteps = max(3, min(args.steps, args.train_steps))
        for _ in range(3):
            train_step()
        ops.PROFILE = []
        tms = timed_region(train_step, tsteps, device, D)
        trec, ops.PROFILE = ops.PROFILE, None
        tk, troof = summarise_profile(trec, peaks)
        thead = head_totals(trec, tsteps, peaks)
        train = {"metric": "images/sec", "value": round(gb * tsteps / (tms / 1e3), 1), "unit": "images/s",
                 "ms_per_step": round(tms / tsteps, 2), "steps": tsteps, "scaling": "strong",
                 "config": {"workload": "configs[2]: full training step (forward + Gram/attention backward + cuDNN "
                                        "backward + AdamW), train-mode BN, CE loss", "global_batch": gb,
                            "per_gpu_batch": hi - lo, "optimizer": "AdamW(lr=1e-3, fused=True)",
                            "ddp": "bucket_cap_mb=16, gradient_as_bucket_view=True, fp32 all-reduce" if world > 1 else None,
                            "parallelism": f"ddp{world}" if world > 1 else "single"},
                 "kernels": tk, "roofline": troof, "head": thead}
        if world == 1 and not args.skip_handoff:
            # The same step with the opt-in bf16 channels_last backbone (SURVEY 8(f) n1): the head then reads bf16 features
            # (kind::f16 operands), half the HBM bytes of the default fp32 hand-off. Reported beside, never as, the default.
            tmodel.set_backbone_mode("bf16_channels_last")
            for _ in range(2):
                train_step()
            ops.PROFILE = []
            bms = timed_region(train_step, tsteps, device, D)
            brec, ops.PROFILE = ops.PROFILE, None
            bk, _ = summarise_profile(brec, peaks)
            train["bf16_handoff"] = {"value": round(gb * tsteps / (bms / 1e3), 1), "unit": "images/s",
                                     "ms_per_step": round(bms / tsteps, 2), "head": head_totals(brec, tsteps, peaks),
                                     "kernel_us": {k: v["avg_us"] for k, v in bk.items()}}
            tmodel.set_backbone_mode("channels_last")
        if world > 1:
            # The same step with the per-GPU batch held at the single-GPU size (weak scaling, global batch gb * world):
            # at 512 / world images per GPU the cuDNN encoder's train-mode kernels stop shrinking with the shard
            # (DESIGN section 6), which bounds the strong-scaling number above whatever the all-reduce costs.
            del xt, yt
            torch.manual_seed(200 + rank)
            xt = torch.randn(gb, 3, IMAGE, IMAGE, device=device)
            yt = torch.randint(0, NUM_CLASSES, (gb,), device=device)
            for _ in range(2):
                train_step()
            wms = timed_region(train_step, tsteps, device, D)
            train["weak_scaling"] = {"value": round(gb * world * tsteps / (wms / 1e3), 1), "unit": "images/s",
                                     "ms_per_step": round(wms / tsteps, 2), "global_batch": gb * world,
                                     "per_gpu_batch": gb, "steps": tsteps, "scaling": "weak"}
        # ---- the same step replayed from ONE CUDA graph (functions.GraphedTrainStep, the package's public API for fixed-shape
        # training loops): forward, loss, backward, DDP's all-reduce and the fused AdamW update without a single host launch.
        # At 64 images per GPU the eager step leaves the GPU idle ~15 % of the time (profiles/r2_ddp_sweep_timeline_8gpu.json).
        # `value` of this leg is the replayed step; the eager measurement above stays beside it as `eager`.
        if not args.no_graph_train:
            from heuristique_style_transfer_code_b200.functions import GraphedTrainStep
            if world > 1:
                del xt, yt
                torch.manual_seed(100 + rank)
                xt = torch.randn(hi - lo, 3, IMAGE, IMAGE, device=device)
                yt = torch.randint(0, NUM_CLASSES, (hi - lo,), device=device)
            gstep = GraphedTrainStep(ddp, crit, opt, xt, yt, warmup=11)
            for _ in range(3):
                gstep()
            gms = timed_region(lambda: gstep(), tsteps, device, D)
            train["eager"] = {"value": train["value"], "ms_per_step": train["ms_per_step"]}
            train["value"] = round(gb * tsteps / (gms / 1e3), 1)
            train["ms_per_step"] = round(gms / tsteps, 2)
            train["config"]["step"] = "replayed from one CUDA graph (GraphedTrainStep); `eager` = the same step launched kernel by kernel"
            train["loss_after"] = float(gstep().item())
            gstep.release()                         # before destroy_process_group: the graph holds NCCL work
            del gstep
        del xt, yt, tmodel, ddp, opt
        torch.cuda.empty_cache()

    if rank != 0:
        return

    ref_gpu = None
    if world == 1 and not args.skip_reference_gpu:
        ref_gpu = guarded("reference_gpu", reference_gpu_legs, device, max(3, args.steps // 4))

    cpu_base, cpu_extra = None, None
    if world == 1 and not args.skip_cpu:
        D.restore_cpu_affinity()                  # the CPU baseline gets every host core, not only the GPU-local ones
        cores = os.cpu_count() or 1
        sample = 64
        ips, sec, kind = cpu_reference_forward(sample, 5, 2, cores)
        cpu_base = {"value": round(ips, 2), "unit": "images/s", "cores": cores, "kind": kind,
                    "sample": f"{sample} images of the batch per step, 5 steps after 2 warm-ups ({sec:.2f} s/step), torch "
                              f"{torch.__version__} CPU fp32 eval/no_grad, {cores} threads, "
                              + ("unmodified reference class loaded from baseline/_ref" if kind == "reference"
                                 else "oracle/torch_port.py")}
        cpu_extra = guarded("cpu_extra", cpu_extra_legs, cores)

    line = {"metric": "images/sec", "value": round(value, 1), "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "tf32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "global_batch": total, "per_gpu_batch": B, "image": IMAGE,
                       "truncate_layer": TRUNC, "gram_matrix_size": GRAM_SIZE, "num_classes": NUM_CLASSES,
                       "precision": "encoder: cuDNN fp32 convolutions in channels_last (TF32 conv allowed, torch default), eval-mode "
                                    "batch norm folded into them and ReLU / residual add as cuDNN epilogues (same function; "
                                    "backbone_handoff reports the difference to the unfolded and NCHW executions); Gram forward and backward (tcgen05, "
                                    "fp32 accumulate): tf32 operands, rounded to nearest by the TMA unit (TFLOAT32 tensor "
                                    "maps); attention/classifier: split-bf16 x3 (fp32-accurate)",
                       "l2_policy": "inputs larger than L2 (154 MB images, 210/105/51 MB stage activations per step)",
                       "parallelism": f"batch-sharded x{world}, all_gather of logits+embeddings" if world > 1 else "single GPU"},
            "e2e": {"value": round(e2e_value, 1), "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": round(e2e_ms / args.steps, 3), "passes_ms_per_step": [round(p / args.steps, 3) for p in e2e_passes],
                    "h2d_alone_ms": round(h2d_alone_ms, 3), "h2d_call_host_ms": round(h2d_issue_ms, 3),
                    "forward_with_concurrent_copy_ms": round(overlap_probe_ms, 3), "fresh_pinned_alloc_ms": round(pinned_alloc_ms, 3),
                    "h2d_alone_GBps": round(h2d / h2d_alone_ms / 1e6, 1)},
            "e2e_uint8": e2e_u8,
            "gpu_launches": launches,
            "roofline": roof,
            "cpu_baseline": cpu_base,
            "clocks": clocks.summary(),
            "breakdown": {"encoder_cudnn_ms": round(enc_ms, 3), "head_ms": round(head_ms, 3),
                          "head_images_per_s": round(B / (head_ms / 1e3), 1), "kernels": kernels},
            "backbone_handoff": handoff,
            "patchgan_head": patchgan,
            "cpu_extra": cpu_extra,
            "reference_gpu": ref_gpu,
            "train": train}
    # headline scalars repeated as the LAST keys, so that they survive a truncated tail of this (long) line
    ihead = head_totals(records, args.steps, peaks)
    line["infer_head_us"] = ihead["head_us"] if ihead else None
    line["infer_attn_fwd_us"] = ihead["attn_fwd_us"] if ihead else None
    if train is not None:
        th = train.get("head") or {}
        key = "train_strong_img_s" if world > 1 else "train_img_s"
        line[key] = train["value"]
        line["train_ms_per_step"] = train["ms_per_step"]
        if "eager" in train:
            line[key.replace("img_s", "eager_img_s")] = train["eager"]["value"]
        if "weak_scaling" in train:
            line["train_weak_img_s"] = train["weak_scaling"]["value"]
        line["train_attn_fwd_us"] = th.get("attn_fwd_us")
        line["train_attn_bwd_us"] = th.get("attn_bwd_us")
        line["train_head_fwd_bwd_us"] = th.get("head_us")
        line["head_fwd_bwd_frac_of_bf16_peak"] = th.get("frac_of_bf16_peak_burst")
        bh = (train.get("bf16_handoff") or {}).get("head") or {}
        line["head_fwd_bwd_frac_of_bf16_peak_bf16_handoff"] = bh.get("frac_of_bf16_peak_burst")
    if ref_gpu is not None and "error" not in ref_gpu:
        line["reference_gpu_infer_img_s"] = ref_gpu["infer_batch256"]["images_per_s"]
        line["reference_gpu_train_img_s"] = ref_gpu["train_batch512"]["images_per_s"]
    if e2e_u8 and "value" in e2e_u8:
        line["e2e_uint8_img_s"] = e2e_u8["value"]
    line["e2e_img_s"] = round(e2e_value, 1)
    emit(json.dumps(line))


_RESULT_FD = None


def claim_stdout():
    """Keep stdout for the one JSON line: libraries that write to fd 1 (NCCL prints its version there) go to stderr."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(text):
    sys.stdout.flush()
    if _RESULT_FD is None:
        print(text, flush=True)
    else:
        os.write(_RESULT_FD, (text + "\n").encode())


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--batch-per-gpu", type=int, default=256)
    ap.add_argument("--train-global-batch", type=int, default=512)
    ap.add_argument("--train-steps", type=int, default=10)
    ap.add_argument("--skip-train", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-handoff", action="store_true")
    ap.add_argument("--skip-patchgan", action="store_true")
    ap.add_argument("--skip-reference-gpu", action="store_true")
    ap.add_argument("--skip-uint8", action="store_true", help="no e2e_uint8 leg (opt-in uint8 upload)")
    ap.add_argument("--no-graph-train", action="store_true", help="training leg: eager step only")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the embeddings and logits of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours (the reference arm's sample size depends on the host's speed)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
