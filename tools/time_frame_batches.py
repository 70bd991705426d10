"""Several camera frames per forward: streaming.FrameBatchPipeline at N frames against CameraPipeline called N times on
the same frames, and the batched preprocessing kernel alone against N launches of the one-frame kernel.

    python tools/time_frame_batches.py [--frames 1,4,16,64] [--reps 5] [--out FILE]

Synthetic 1080p BGR frames (seeded), the camera model of tools/bench_camera.py (ResNet-50 truncated after layer3,
g = 32, 4 classes), two transforms: Resize((448, 448)) (the camera benchmark's) and Resize(256) + CenterCrop(224).
End to end, one call = host copy of the frames into the pinned arena, graph replay, probabilities on the host: each
repetition times `calls` calls of the batched pipeline, then N * `calls` CameraPipeline calls on the same frames,
alternating; ms per call is the median repetition. Kernels: CUDA events around 200 launches of gh_preprocess_frames
(N frames, the pipeline's band height) and around 200 rounds of N gh_preprocess_frame launches (one per frame). The
GPU's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
from torchvision import models  # noqa: E402
from heuristique_style_transfer_code_b200 import TruncatedResNet50_for_test  # noqa: E402
from heuristique_style_transfer_code_b200.streaming import CameraPipeline, FrameBatchPipeline  # noqa: E402

MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
TRANSFORMS = {"resize448": ((448, 448), None), "resize256_crop224": (256, 224)}
SHAPE = (1080, 1920, 3)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def wall_ms(fn, calls):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(calls):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / calls


def event_ms(fn, launches=200):
    for _ in range(5):
        fn()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(launches):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", default="1,4,16,64")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = [json.dumps({"gpu": gpu_info()})]
    print(lines[0], flush=True)
    torch.manual_seed(0)
    model = TruncatedResNet50_for_test(models.resnet50(weights=None), 7, 4, 32, device="cuda:0").eval()
    rng = np.random.default_rng(0)
    for name, (resize, crop) in TRANSFORMS.items():
        cam = CameraPipeline(model, SHAPE, resize, crop, MEAN, STD)
        for n in [int(v) for v in args.frames.split(",")]:
            frames = [rng.integers(0, 256, SHAPE, dtype=np.uint8) for _ in range(n)]
            pipe = FrameBatchPipeline(model, [SHAPE] * n, resize, crop, MEAN, STD)
            batch_probs = pipe(frames)
            cam_probs = np.stack([cam(f) for f in frames])
            calls = max(3, 64 // n)
            batched, single = [], []
            for _ in range(args.reps):
                batched.append(wall_ms(lambda: pipe(frames), calls))
                single.append(wall_ms(lambda: [cam(f) for f in frames], calls))
            b, s = float(np.median(batched)), float(np.median(single))
            # the kernels alone, on the frames already uploaded by the calls above
            k_batch = event_ms(pipe.preprocess_)
            k_single = event_ms(lambda: [cam.preprocess_() for _ in range(n)])
            rec = {"transform": name, "frames": n, "band_rows": pipe.band_rows, "max_band_rows": pipe.max_band_rows,
                   "calls_per_rep": calls,
                   "batch_ms_per_call": round(b, 4), "batch_ms_per_frame": round(b / n, 4),
                   "camera_ms_per_frame": round(s / n, 4), "speedup_per_frame": round(s / b, 2),
                   "batch_ms_per_call_min_max": [round(min(batched), 4), round(max(batched), 4)],
                   "camera_ms_per_frame_min_max": [round(min(single) / n, 4), round(max(single) / n, 4)],
                   "kernel_batched_ms": round(k_batch, 4), "kernel_one_frame_x_n_ms": round(k_single, 4),
                   "kernel_speedup": round(k_single / k_batch, 2),
                   "max_abs_prob_diff_vs_camera": float(np.abs(batch_probs - cam_probs).max())}
            lines.append(json.dumps(rec))
            print(lines[-1], flush=True)
            del pipe
    lines.append(json.dumps({"gpu_after": gpu_info()}))
    print(lines[-1], flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
