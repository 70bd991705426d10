"""Style transfer with N images per step: time of the CUDA-graph-replayed step (encoder forward + backward, dense Gram
forward + backward, per-image loss, Adam, the N losses copied to the host) at N images and the first `layers` encoder
children, as style_transfer(images_per_step=N) runs it.

    python tools/time_style_batch.py [--images 1,8,32,64] [--layers 4,5,7] [--reps 3] [--out FILE]
    python tools/time_style_batch.py --profile 32 --layers 7 [--out FILE]    # torch.profiler table of one config

Each configuration: 10 warm-up steps, then `--reps` windows of at least 0.3 s each between CUDA events; ms per step is
the median window (min and max reported too), ms per image-step that over N. Peak memory is torch's peak allocation
while that configuration ran (the model's weights included). The GPU's name and power limit are read in the same run.
"""
import argparse
import gc
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from torchvision import models  # noqa: E402
from heuristique_style_transfer_code_b200 import TruncatedResNet50_for_test  # noqa: E402
from heuristique_style_transfer_code_b200.functions import _StyleIteration  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def runner_for(model, encoder, n, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    images = torch.randn(n, 3, 224, 224, generator=g).cuda()
    with torch.no_grad():
        target = model.gram_matrix(encoder(images))
    it = _StyleIteration(model, encoder, "cuda:0", 0.01, use_graph=True, images=n)
    it.start(target, torch.randn(n, 3, 224, 224, generator=g).cuda())
    return it


def time_config(model, encoder, n, reps):
    torch.cuda.synchronize()
    gc.collect()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    it = runner_for(model, encoder, n, seed=n)
    for _ in range(10):
        it.step_losses()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(5):
        it.step_losses()
    end.record()
    end.synchronize()
    steps = max(20, int(300.0 / (start.elapsed_time(end) / 5)))
    windows = []
    for _ in range(reps):
        start.record()
        for _ in range(steps):
            losses = it.step_losses()
        end.record()
        end.synchronize()
        windows.append(start.elapsed_time(end) / steps)
    windows.sort()
    ms = windows[len(windows) // 2]
    res = {"images": n, "gram": list(it.target.shape[1:]), "steps_per_window": steps,
           "ms_per_step": round(ms, 4), "ms_per_step_min_max": [round(windows[0], 4), round(windows[-1], 4)],
           "ms_per_image_step": round(ms / n, 4), "peak_mem_gib": round(torch.cuda.max_memory_allocated() / 2**30, 3),
           "mean_loss_last": sum(losses) / n}
    del it
    return res


def profile_config(model, encoder, n, out):
    from torch.profiler import ProfilerActivity, profile
    it = runner_for(model, encoder, n, seed=n)
    for _ in range(10):
        it.step_losses()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(20):
            it.step_losses()
        torch.cuda.synchronize()
    table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=30, max_name_column_width=90)
    print(table, file=out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", default="1,8,32,64")
    ap.add_argument("--layers", default="4,5,7")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--profile", type=int, default=0, help="N: print a torch.profiler table of 20 steps instead")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_style_batch.py needs a CUDA device")
    out = open(args.out, "a") if args.out else sys.stdout
    torch.manual_seed(0)
    model = TruncatedResNet50_for_test(models.resnet50(weights=None), 7, 4, 32, device="cuda:0").eval()
    print(json.dumps({"gpu": gpu_info(), "torch": torch.__version__, "cudnn_allow_tf32": torch.backends.cudnn.allow_tf32,
                      "workload": "style-transfer step, graph replay, N 224x224 images"}), file=out, flush=True)
    for layers in [int(v) for v in args.layers.split(",")]:
        encoder = torch.nn.Sequential(*list(model.truncated_encoder.children())[:layers]).to("cuda:0")
        if args.profile:
            print(f"# torch.profiler, layers={layers}, N={args.profile}, 20 steps", file=out)
            profile_config(model, encoder, args.profile, out)
            continue
        for n in [int(v) for v in args.images.split(",")]:
            print(json.dumps({"layers": layers, **time_config(model, encoder, n, args.reps)}), file=out, flush=True)
    if out is not sys.stdout:
        out.close()


if __name__ == "__main__":
    main()
