"""Backward of the Multi-PatchGAN Gram head on one B200 (lives under tests/tools/ because it runs the fp32 torch port of
the reference forward from oracle/).

    python tests/tools/time_patchgan_backward.py [--batches 64,256] [--reps 5] [--launches 50] [--out FILE]

1. Forward + backward of MultiScaleDiscriminator_test (ndf 64, gram_matrix_dim 64, batch norm, patches 10/70/150, train
   mode) at 224x224: the library route (set_library_backward(True)) against the port's op sequence under autograd on the
   same module and input (oracle/torch_port.patchgan_multiscale_forward: what the reference's own forward runs),
   alternating, --reps passes each after two warm-up passes, with torch's default TF32 settings; loss = cross entropy of
   the output + 1e-3 * the sum of the Gram norms; host clock around each pass, which ends in a device synchronise. Peak memory of one pass of each route
   (torch.cuda.max_memory_allocated over the pass, minus what was allocated before it).
2. gh_patch_pool_bwd alone on the six maps a patch-70 discriminator collects at 224x224 (D 64, batch 256: 112..12 px),
   with and without ln_input: CUDA events over --launches launches after 5 warm-up launches; bytes the pass must move
   (maps read with ln_input + gradients written) over its time, against a 4 GiB device-to-device copy timed the same way
   in the same run. The working set (2.2 GB) is far larger than the 126 MB L2.
The GPU's name, power limit and max SM clock are read in the same run.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from heuristique_style_transfer_code_b200 import _lib, ops  # noqa: E402
from heuristique_style_transfer_code_b200.patchgan import MultiScaleDiscriminator_test  # noqa: E402
from oracle.torch_port import patchgan_forward  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def event_ms(fn, launches):
    for _ in range(5):
        fn()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(launches):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / launches


def copy_gbs():
    src = torch.empty(4 << 30, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    ms = event_ms(lambda: dst.copy_(src), 20)
    del src, dst
    return 2 * (4 << 30) / (ms * 1e-3) / 1e9


def library_loss(m, x, target):
    emb, out = m(x)
    return torch.nn.functional.cross_entropy(out, target) + 1e-3 * sum(n.sum() for n in m.get_gram_norms())


def port_loss(m, x, target):
    outs, norms = [], []
    for d in m.scale_discriminators.values():
        _, o, n = patchgan_forward(d, x)
        outs.append(o)
        norms.extend(n)
    out = torch.stack(outs, 0).mean(0)
    return torch.nn.functional.cross_entropy(out, target) + 1e-3 * sum(n.sum() for n in norms)


def one_pass(loss_fn, m, x, target):
    m.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    loss_fn(m, x, target).backward()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, (torch.cuda.max_memory_allocated() - base) / 2 ** 30


def module_timing(batch, reps):
    torch.manual_seed(0)
    m = MultiScaleDiscriminator_test(ndf=64, norm='batch', num_classes=4, gram_matrix_dim=64).cuda()
    m.set_library_backward(True)
    x = torch.randn(batch, 3, 224, 224, device="cuda").requires_grad_(True)
    target = torch.randint(0, 4, (batch,), device="cuda")
    routes = {"library": library_loss, "port": port_loss}
    for fn in routes.values():
        for _ in range(2):
            one_pass(fn, m, x, target)
    times = {k: [] for k in routes}
    peaks = {k: 0.0 for k in routes}
    for _ in range(reps):
        for k, fn in routes.items():
            ms, gib = one_pass(fn, m, x, target)
            times[k].append(round(ms, 2))
            peaks[k] = max(peaks[k], gib)
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    return {"batch": batch, "ms_per_pass": times, "median_ms": med, "speedup": round(med["port"] / med["library"], 2),
            "peak_gib_above_inputs": {k: round(v, 2) for k, v in peaks.items()}}


def pool_bwd_timing(launches, copy_rate):
    torch.manual_seed(1)
    b, d = 256, 64
    shapes = [(112, 112), (56, 56), (28, 28), (14, 14), (13, 13), (12, 12)]
    maps = [torch.randn(b, d, h, w, device="cuda") for h, w in shapes]
    grads = [torch.empty_like(m) for m in maps]
    L = len(maps)
    gram, norm, scratch = ops._patch_gram_fwd(maps, True)
    lib = _lib.lib()
    ws = torch.empty(lib.gh_patch_bwd_workspace(L, b, d), device="cuda")
    _, hs, wsz, st = ops._patch_map_arrays(maps)
    stream = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.gh_patch_gram_bwd(hs, wsz, L, b, d, 1, torch.randn_like(gram).data_ptr(),
                                     torch.randn_like(norm).data_ptr(), norm.data_ptr(), scratch.data_ptr(),
                                     ws.data_ptr(), stream), "gh_patch_gram_bwd")
    ptrs = (ctypes.c_void_p * L)(*[m.data_ptr() for m in maps])
    gptrs = (ctypes.c_void_p * L)(*[g.data_ptr() for g in grads])
    elems = sum(m.numel() for m in maps)
    out = {}
    for ln in (1, 0):
        ms = event_ms(lambda: lib.gh_patch_pool_bwd(ptrs, gptrs, hs, wsz, st, st, L, b, d, ln, ws.data_ptr(), stream),
                      launches)
        nbytes = elems * 4 * (2 if ln else 1)
        rate = nbytes / (ms * 1e-3) / 1e9
        out[f"ln_input={ln}"] = {"us": round(ms * 1e3, 1), "bytes": nbytes, "GB_s": round(rate, 1),
                                 "of_copy_rate": round(rate / copy_rate, 3)}
    torch.cuda.synchronize()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="64,256")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    rec = {"gpu": gpu_info()}
    rate = copy_gbs()
    rec["device_copy_GB_s"] = round(rate, 1)
    rec["pool_bwd_patch70_b256"] = pool_bwd_timing(args.launches, rate)
    rec["multiscale_fwd_bwd"] = [module_timing(int(b), args.reps) for b in args.batches.split(",")]
    text = json.dumps(rec, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
