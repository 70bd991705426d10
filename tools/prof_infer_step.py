"""Where does bench.py's inference step spend its GPU time? torch.profiler (CUDA activities) over the seeded workload
bench.py times: eval + no_grad forward of TruncatedResNet50_for_test (trunc 7, 4 classes, Gram 32) on 256 images of
224 x 224 resident on the device.
    python tools/prof_infer_step.py [--chain] [batch]
Prints the card, the event-timed step, the per-step kernel table and the launches of the stem (the fused stem kernel,
or with --chain the three launches it replaces: space-to-depth staging, cuDNN convolution, max pool), found by
profiling the stem alone."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402
from torchvision import models  # noqa: E402

from heuristique_style_transfer_code_b200 import TruncatedResNet50_for_test  # noqa: E402

CHAIN = "--chain" in sys.argv
ARGS = [a for a in sys.argv[1:] if a != "--chain"]
B = int(ARGS[0]) if ARGS else 256
STEPS = 10
dev = torch.device("cuda:0")


def card() -> str:
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def kernel_table(fn, steps):
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
    ev = [k for k in prof.key_averages() if k.device_time_total > 0 and k.device_type == torch.autograd.DeviceType.CUDA]
    return sorted(ev, key=lambda k: -k.device_time_total)


def main():
    print(f"card: {card()}")
    torch.manual_seed(0)
    model = TruncatedResNet50_for_test(models.resnet50(weights=None), 7, 4, 32, device=dev).eval()
    torch.manual_seed(1)
    x = torch.randn(B, 3, 224, 224).pin_memory().to(dev)
    print(f"batch {B}, allow_tf32={torch.backends.cudnn.allow_tf32}, stem: {'chain' if CHAIN else 'fused'}")
    with torch.no_grad():
        plan = model._inference_plan(x)
    if plan is not None:
        plan._stem_fused = not CHAIN

    def step():
        with torch.no_grad():
            model(x)

    for _ in range(5):
        step()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(20):
        step()
    e.record()
    torch.cuda.synchronize()
    print(f"step: {s.elapsed_time(e) / 20:.3f} ms (events, 20 steps, profiler off)")

    ev = kernel_table(step, STEPS)
    busy = sum(k.device_time_total for k in ev) / STEPS / 1e3
    print(f"GPU busy {busy:.3f} ms/step over {sum(k.count for k in ev) / STEPS:.0f} kernels+copies per step")
    for k in ev[:30]:
        print(f"{k.device_time_total / STEPS:9.1f} us/step {k.count / STEPS:5.0f}x {k.device_time_total / k.count:8.1f} us  "
              f"{k.key[:120]}")

    if plan is None:
        print("no inference plan for this model / mode")
        return

    def stem():
        with torch.no_grad():
            plan.stem_forward(x)

    for _ in range(3):
        stem()
    stem_ev = kernel_table(stem, STEPS)
    print("stem launches (profiled alone):")
    tot = 0.0
    for k in stem_ev:
        us = k.device_time_total / STEPS
        tot += us
        print(f"{us:9.1f} us/step {k.count / STEPS:5.0f}x  {k.key[:120]}")
    print(f"stem total {tot:.1f} us/step")


if __name__ == "__main__":
    main()
