"""The uint8 fused stem (gh_stem_conv_pool_u8_nhwc: ToTensor + Normalize in the stem kernel's producers) against
normalize_u8 followed by the fp32 fused stem, on one box, in one process:
    python tools/time_stem_u8.py [batch]
Input: bench.py's seeded uint8 batch (256 x 3 x 224 x 224, torch.Generator seed 7), ImageNet constants.
(a) the stem alone: CUDA events, warm-up, 5 alternating rounds of 20 launches per arm; us per call and GB/s on the
    algorithmic bytes of each arm (normalize_u8: uint8 in + fp32 out; stem: image in + pooled result out). Arms:
    normalize_u8 + fp32 fused stem, the uint8 fused stem, and the fp32 fused stem alone on the normalised batch;
(b) the whole eval + no_grad forward of bench.py's model configuration, 5 alternating passes of 20 steps per arm:
    (b1) batch resident on the device: model(normalize_u8(x)) vs model(x) with set_input_normalization;
    (b2) through cuda_prefetch from pinned host memory (reuse_buffers=True, as the loops run it): the default uint8
         path (normalize_u8 on the upload stream) vs normalize=None with set_input_normalization;
    ms per step of every pass, peak device memory of one pass, and whether the arms' outputs are bitwise equal.
Card name and power limit come from an NVML query (nvidia-smi) in the same run."""
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from torchvision import models  # noqa: E402

from heuristique_style_transfer_code_b200 import TruncatedResNet50_for_test, ops  # noqa: E402
from heuristique_style_transfer_code_b200.functions import IMAGENET_MEAN, IMAGENET_STD, cuda_prefetch  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 256
H = W = 224
ROUNDS, LAUNCHES, STEPS = 5, 20, 20
NORM = (IMAGENET_MEAN, IMAGENET_STD)
dev = torch.device("cuda:0")


def card() -> str:
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def timed(fn, n):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(n):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / n


def alternate(arms, n, warm=3):
    """arms: name -> callable. Warm-up, then ROUNDS rounds of n calls per arm in turn -> name -> [ms per call]."""
    for fn in arms.values():
        for _ in range(warm):
            fn()
    t = {k: [] for k in arms}
    for _ in range(ROUNDS):
        for k, fn in arms.items():
            t[k].append(timed(fn, n))
    return t


def peak_mb(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    fn()
    torch.cuda.synchronize()
    return (torch.cuda.max_memory_allocated(dev) - base) / 1e6


def main():
    print(f"card: {card()}")
    print(f"batch {B} x 3 x {H} x {W} uint8 (bench.py's e2e_uint8 batch), allow_tf32={torch.backends.cudnn.allow_tf32}")
    torch.manual_seed(0)
    model = TruncatedResNet50_for_test(models.resnet50(weights=None), 7, 4, 32, device=dev).eval()
    u8_host = torch.randint(0, 256, (B, 3, H, W), dtype=torch.uint8, generator=torch.Generator().manual_seed(7)).pin_memory()
    x8 = u8_host.to(dev)
    with torch.no_grad():
        plan = model._inference_plan(x8)
    assert plan is not None and plan.stem_packed is not None, "no fused stem for this configuration"
    wp, bias = plan.stem_packed, plan.stem_s2d[1]
    xf = ops.normalize_u8(x8, *NORM)

    # ---- (a) the stem alone ----
    same = torch.equal(ops.stem_conv_pool_u8(x8, *NORM, wp, bias), ops.stem_conv_pool(ops.normalize_u8(x8, *NORM), wp, bias))
    print(f"(a) u8 stem output bitwise equal to normalize_u8 + fp32 stem: {same}")
    arms = {"normalize_u8 + fp32 stem": lambda: ops.stem_conv_pool(ops.normalize_u8(x8, *NORM), wp, bias),
            "u8 stem": lambda: ops.stem_conv_pool_u8(x8, *NORM, wp, bias),
            "fp32 stem alone": lambda: ops.stem_conv_pool(xf, wp, bias)}
    t = alternate(arms, LAUNCHES)
    ph, pw = (H // 2 - 1) // 2 + 1, (W // 2 - 1) // 2 + 1
    n_px, n_out = B * 3 * H * W, B * 64 * ph * pw
    nbytes = {"normalize_u8 + fp32 stem": n_px * 5 + n_px * 4 + n_out * 4, "u8 stem": n_px + n_out * 4,
              "fp32 stem alone": n_px * 4 + n_out * 4}
    for k in arms:
        med = statistics.median(t[k]) * 1e3
        print(f"    {k}: median {med:.1f} us per call; rounds " + ", ".join(f"{v * 1e3:.1f}" for v in t[k]) +
              f"; algorithmic bytes {nbytes[k] / 1e6:.1f} MB, {nbytes[k] / med / 1e3:.0f} GB/s")
    gain = (statistics.median(t["normalize_u8 + fp32 stem"]) - statistics.median(t["u8 stem"])) * 1e3
    print(f"    u8 stem faster than normalize_u8 + fp32 stem by {gain:.1f} us median; every u8 round faster than every "
          f"two-launch round: {max(t['u8 stem']) < min(t['normalize_u8 + fp32 stem'])}")
    del xf

    # ---- (b1) the whole eval forward, batch resident on the device ----
    def fwd_outside():
        model.set_input_normalization(None)
        with torch.no_grad():
            return model(ops.normalize_u8(x8, *NORM))

    def fwd_inside():
        model.set_input_normalization(*NORM)
        with torch.no_grad():
            return model(x8)

    outs = {k: tuple(o.clone() for o in f()) for k, f in (("outside", fwd_outside), ("inside", fwd_inside))}
    eq = all(torch.equal(a, b) for a, b in zip(outs["outside"], outs["inside"]))
    arms = {"normalize_u8 then model": fwd_outside, "model with input normalisation": fwd_inside}
    mem = {k: peak_mb(f) for k, f in arms.items()}
    t = alternate(arms, STEPS)
    for k in arms:
        print(f"(b1) {k}: median {statistics.median(t[k]):.3f} ms/step; passes " + ", ".join(f"{v:.3f}" for v in t[k]) +
              f"; peak memory of one step above the resident set {mem[k]:.0f} MB")
    gain = statistics.median(t["normalize_u8 then model"]) - statistics.median(t["model with input normalisation"])
    print(f"     in-model faster by {gain:.3f} ms/step median; embeddings and logits bitwise equal: {eq}")

    # ---- (b2) the loop through cuda_prefetch from pinned host memory ----
    def loop(inside, n):
        if inside:
            model.set_input_normalization(*NORM)
        else:
            model.set_input_normalization(None)
        last = None
        with torch.no_grad():
            for (xb,) in cuda_prefetch(((u8_host,) for _ in range(n)), dev, reuse_buffers=True,
                                       normalize=None if inside else "default"):
                last = model(xb)
        return last

    outs = {k: tuple(o.clone() for o in loop(k, 2)) for k in (False, True)}
    eq = all(torch.equal(a, b) for a, b in zip(outs[False], outs[True]))
    arms = {"cuda_prefetch normalises": lambda: loop(False, STEPS),
            "model normalises (normalize=None)": lambda: loop(True, STEPS)}
    mem = {k: peak_mb(lambda: loop(k.startswith("model"), 3)) for k in arms}
    t = alternate(arms, 1, warm=1)
    for k in arms:
        per = [v / STEPS for v in t[k]]
        print(f"(b2) {k}: median {statistics.median(per):.3f} ms/step; passes " + ", ".join(f"{v:.3f}" for v in per) +
              f" ({B * 1e3 / statistics.median(per):.0f} images/s); peak memory of a 3-step loop above the resident set "
              f"{mem[k]:.0f} MB")
    gain = (statistics.median(t["cuda_prefetch normalises"]) - statistics.median(t["model normalises (normalize=None)"])) / STEPS
    print(f"     in-model faster by {gain:.3f} ms/step median; embeddings and logits bitwise equal: {eq}")
    model.set_input_normalization(None)


if __name__ == "__main__":
    main()
