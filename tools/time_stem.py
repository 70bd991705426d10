"""The fused stem kernel (gh_stem_conv_pool_nhwc) against the three-launch chain it replaces in the inference plan
(gh_stem_space_to_depth -> cuDNN 4x4 convolution + bias + ReLU -> gh_maxpool2d_nhwc), on one box, in one process:
    python tools/time_stem.py [batch]
(a) the stem alone on bench.py's seeded batch (256 x 3 x 224 x 224 fp32, 154 MB: larger than L2): CUDA events,
    warm-up, 5 alternating rounds of 20 launches per arm; us per call, GB/s on the algorithmic bytes (image in, pooled
    result out), TFLOP/s on the useful FLOPs of the 7x7 convolution and on the FLOPs the tensor cores execute;
(b) the whole eval + no_grad forward of bench.py's model configuration, fused vs chain in alternating passes of 20
    steps: ms per step of every pass, and how far the two arms' embeddings and logits are apart.
Card name and power limit come from an NVML query (nvidia-smi) in the same run."""
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from torchvision import models  # noqa: E402

from heuristique_style_transfer_code_b200 import TruncatedResNet50_for_test, _lib, ops  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 256
H = W = 224
ROUNDS, LAUNCHES, STEPS = 5, 20, 20
TILE_COLS = 63                                  # csrc/stem.cuh: kScTileCols
MMA_FLOPS_PER_CONV_ROW = 24 * 2 * 128 * 64 * 8  # 4 tap rows x 6 MMAs of 128 x 64 x 8 per conv row and tile
dev = torch.device("cuda:0")


def card() -> str:
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def executed_conv_rows(b, h, w, ctas):
    """Conv rows (of one tile each) the kernel computes, halo included: the split of gh_stem_conv_pool_nhwc."""
    oh, ow = h // 2, w // 2
    ph, pw = (oh - 1) // 2 + 1, (ow - 1) // 2 + 1
    tiles = (pw + TILE_COLS - 1) // TILE_COLS
    units = b * tiles * ph
    grid = min(ctas, units)
    rows = 0
    for c in range(grid):
        u, u1 = units * c // grid, units * (c + 1) // grid
        while u < u1:
            bj = u // ph
            end = min((bj + 1) * ph, u1)
            py0, py1 = u - bj * ph, end - bj * ph
            rows += min(2 * py1 - 1, oh - 1) - max(2 * py0 - 1, 0) + 1
            u = end
    return rows


def timed(fn, n):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(n):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / n


def main():
    print(f"card: {card()}")
    print(f"batch {B} x 3 x {H} x {W} fp32, allow_tf32={torch.backends.cudnn.allow_tf32}")
    torch.manual_seed(0)
    model = TruncatedResNet50_for_test(models.resnet50(weights=None), 7, 4, 32, device=dev).eval()
    torch.manual_seed(1)
    x = torch.randn(B, 3, H, W).pin_memory().to(dev)
    with torch.no_grad():
        plan = model._inference_plan(x)
    assert plan is not None and plan.stem_packed is not None, "no fused stem for this configuration"

    def stem(fused):
        plan._stem_fused = fused
        with torch.no_grad():
            return plan.stem_forward(x)

    # ---- (a) the stem alone ----
    with torch.no_grad():
        a, b = stem(True), stem(False)
    print(f"(a) fused vs chain stem output: rel. diff {float((a - b).norm() / b.norm()):.3g}")
    del a, b
    for f in (True, False):
        for _ in range(3):
            stem(f)
    t = {True: [], False: []}
    for _ in range(ROUNDS):
        for f in (True, False):
            t[f].append(timed(lambda: stem(f), LAUNCHES) * 1e3)
    oh, ow = H // 2, W // 2
    ph, pw = (oh - 1) // 2 + 1, (ow - 1) // 2 + 1
    nbytes = B * 3 * H * W * 4 + B * 64 * ph * pw * 4
    useful = 2.0 * B * oh * ow * 64 * 147
    executed = executed_conv_rows(B, H, W, _lib.lib().gh_sm_count()) * MMA_FLOPS_PER_CONV_ROW
    print(f"    algorithmic bytes {nbytes / 1e6:.1f} MB, useful {useful / 1e9:.1f} GFLOP, executed (tensor) "
          f"{executed / 1e9:.1f} GFLOP")
    for f, name in ((True, "fused"), (False, "chain")):
        med = statistics.median(t[f])
        print(f"    {name}: median {med:.1f} us per call; rounds " + ", ".join(f"{v:.1f}" for v in t[f]) +
              f"; {nbytes / med / 1e3:.0f} GB/s; {useful / med / 1e6:.1f} TFLOP/s useful" +
              (f", {executed / med / 1e6:.1f} TFLOP/s executed" if f else ""))

    # ---- (b) the whole eval forward ----
    def step():
        with torch.no_grad():
            return model(x)

    out = {}
    for f in (True, False):
        plan._stem_fused = f
        for _ in range(3):
            step()
        emb, lg = step()
        out[f] = (emb.float().clone(), lg.float().clone())
    passes = {True: [], False: []}
    for _ in range(ROUNDS):
        for f in (True, False):
            plan._stem_fused = f
            step()
            passes[f].append(timed(step, STEPS))
    plan._stem_fused = True
    for f, name in ((True, "fused"), (False, "chain")):
        print(f"(b) {name}: median {statistics.median(passes[f]):.3f} ms/step; passes " +
              ", ".join(f"{v:.3f}" for v in passes[f]) + f" ({B * 1e3 / statistics.median(passes[f]):.0f} images/s)")
    gain = statistics.median(passes[False]) - statistics.median(passes[True])
    print(f"    fused faster by {gain:.3f} ms/step median; every fused pass faster than every chain pass: "
          f"{max(passes[True]) < min(passes[False])}")
    (e1, l1), (e0, l0) = out[True], out[False]
    print(f"    embeddings rel. diff {float((e1 - e0).norm() / e0.norm()):.3g}, logits rel. diff "
          f"{float((l1 - l0).norm() / l0.norm()):.3g}, argmax equal on {int((l1.argmax(1) == l0.argmax(1)).sum())}/{B}")


if __name__ == "__main__":
    main()
