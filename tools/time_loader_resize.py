"""Resize + CenterCrop of loader batches on the GPU (functions.gpu_resize_transform) against the host transforms.

    python tools/time_loader_resize.py [--images 3000] [--batch 64] [--reps 2] [--workers 4,0] [--out FILE]

Kernels: 256 seeded RGB images with sides drawn from 300-2000 px, Resize(256) + CenterCrop(224). CUDA events around 200
launches (after 5 warm-up launches) of gh_frame_tables and of gh_preprocess_frames, with the band height that
streaming.resample_images picks. Beside them, the host's streaming.pack_frame_tables for the same batch (best of 3), the
bytes each kernel must move, and the HBM bandwidth a 4 GiB device-to-device copy reaches in the same run. The device
tables are checked against pack_frame_tables bit for bit.

End to end: evaluate_model_test images/s over a seeded synthetic JPEG ImageFolder written to a temporary directory
(--images images, sides 300-2000 px, smooth content with noise, quality 90), batch --batch, pin_memory=True, with the
host-transform loader (Resize + CenterCrop + ToTensor + Normalize in the workers) and the gpu_resize_transform loader,
alternating, --reps times each, at each --workers count (0 stands for the CPU count). The model is the camera model of
tools/bench_camera.py, with ops.KSPLIT = 1 so that both loaders' arrays can be compared bit for bit. The host-to-device
bytes per batch, the CPU count and the GPU's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from multiprocessing import Pool

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
from PIL import Image  # noqa: E402

from heuristique_style_transfer_code_b200 import _lib, ops, streaming as S, functions as F  # noqa: E402

MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
RESIZE, CROP = 256, 224


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


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


def hbm_peak_gbs():
    src = torch.empty(4 << 30, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    ms = event_ms(lambda: dst.copy_(src), launches=20)
    del src, dst
    return 2 * (4 << 30) / ms / 1e6


def kernels(lines):
    rng = np.random.default_rng(0)
    shapes = [(int(rng.integers(300, 2001)), int(rng.integers(300, 2001)), 3) for _ in range(256)]
    images = [torch.from_numpy(rng.integers(0, 256, s, dtype=np.uint8)) for s in shapes]
    t = F.gpu_resize_transform(RESIZE, CROP)
    packed = t.collate([(x, 0) for x in images])
    host_ms = []
    for _ in range(3):
        t0 = time.perf_counter()
        ref = S.pack_frame_tables(shapes, RESIZE, CROP)
        host_ms.append((time.perf_counter() - t0) * 1e3)
    n, (oh, ow), (hk, vk) = len(shapes), packed.out_hw, packed.kmax
    lib = _lib.lib()
    stride = lib.gh_frame_tables_stride(oh, ow, hk, vk)
    pixels, geom = packed.pixels.cuda(), packed.geometry.cuda()
    tables = torch.empty(n * stride, dtype=torch.int32, device="cuda")
    frames = torch.empty(n * 80, dtype=torch.uint8, device="cuda")
    out = torch.empty((n, 3, oh, ow), dtype=torch.uint8, device="cuda")
    g = packed.geometry.numpy()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    band, span = S.images_band_rows(g[:, 0], g[:, 3], oh, ow, vk, sms)

    def run_tables():
        _lib.check(lib.gh_frame_tables(geom.data_ptr(), n, pixels.data_ptr(), oh, ow, hk, vk, tables.data_ptr(),
                                       frames.data_ptr(), None), "gh_frame_tables")

    def run_resample():
        _lib.check(lib.gh_preprocess_frames(frames.data_ptr(), n, oh, ow, band, span, tables.data_ptr(), hk, vk,
                                            out.data_ptr(), None), "gh_preprocess_frames")
    t_tables, t_resample = event_ms(run_tables), event_ms(run_resample)
    torch.cuda.synchronize()
    equal = bool(hk == ref["hkmax"] and vk == ref["vkmax"] and np.array_equal(tables.cpu().numpy(), ref["tables"]))
    # bytes: the tables kernel reads the geometry and writes tables + descriptors; the resample kernel reads at least the
    # input pixels of each image's crop window (once) and the tables, and writes the uint8 batch
    tables_bytes = n * 7 * 8 + n * stride * 4 + n * 80
    window = 0
    for i in range(n):
        o = ref["offsets"][i]
        x0, xn = ref["tables"][o[0]:o[0] + ow], ref["tables"][o[1]:o[1] + ow]
        y0, yn = ref["tables"][o[3]:o[3] + oh], ref["tables"][o[4]:o[4] + oh]
        window += int((y0 + yn).max() - y0.min()) * int((x0 + xn).max() - x0.min()) * 3
    resample_bytes = window + n * stride * 4 + n * 3 * oh * ow
    peak = hbm_peak_gbs()
    rec = {"kernels": {"images": n, "sides_px": [300, 2000], "transform": f"Resize({RESIZE}) + CenterCrop({CROP})",
                       "hkmax": hk, "vkmax": vk, "band_rows": band, "span_rows": span,
                       "gh_frame_tables_us": round(t_tables * 1e3, 2), "gh_frame_tables_bytes": tables_bytes,
                       "gh_frame_tables_hbm_share": round(tables_bytes / (t_tables * 1e-3) / (peak * 1e9), 4),
                       "gh_preprocess_frames_us": round(t_resample * 1e3, 2), "gh_preprocess_frames_bytes": resample_bytes,
                       "gh_preprocess_frames_hbm_share": round(resample_bytes / (t_resample * 1e-3) / (peak * 1e9), 4),
                       "measured_hbm_peak_GBs_d2d_copy_4GiB": round(peak, 1),
                       "host_pack_frame_tables_ms": round(min(host_ms), 1), "table_bytes": n * stride * 4,
                       "device_tables_equal_pack_frame_tables": equal}}
    lines.append(json.dumps(rec))
    print(lines[-1], flush=True)


def _write_jpeg(args):
    path, seed = args
    rng = np.random.default_rng(seed)
    h, w = int(rng.integers(300, 2001)), int(rng.integers(300, 2001))
    base = Image.fromarray(rng.integers(0, 256, (12, 12, 3), dtype=np.uint8), "RGB").resize((w, h), Image.BILINEAR)
    px = np.asarray(base, dtype=np.int16) + rng.integers(-12, 13, (h, w, 3), dtype=np.int16)
    Image.fromarray(np.clip(px, 0, 255).astype(np.uint8), "RGB").save(path, quality=90)
    return h, w


def make_folder(root, count):
    jobs = []
    for i in range(count):
        d = os.path.join(root, f"class_{i % 4}")
        os.makedirs(d, exist_ok=True)
        jobs.append((os.path.join(d, f"img_{i:05d}.jpg"), 1000 + i))
    with Pool(os.cpu_count()) as pool:
        sizes = pool.map(_write_jpeg, jobs, chunksize=16)
    return dict(zip([j[0] for j in jobs], sizes))


def end_to_end(lines, args):
    from torch.utils.data import DataLoader
    from torchvision import models, transforms
    from torchvision.datasets import ImageFolder
    from heuristique_style_transfer_code_b200 import TruncatedResNet50_for_test
    torch.manual_seed(0)
    model = TruncatedResNet50_for_test(models.resnet50(weights=None), 7, 4, 32, device="cuda:0").eval()
    ops.KSPLIT = 1
    host_tf = transforms.Compose([transforms.Resize(RESIZE), transforms.CenterCrop(CROP), transforms.ToTensor(),
                                  transforms.Normalize(MEAN, STD)])
    gpu_tf = F.gpu_resize_transform(RESIZE, CROP)
    cpus = len(os.sched_getaffinity(0))
    with tempfile.TemporaryDirectory() as root:
        t0 = time.perf_counter()
        sizes = make_folder(root, args.images)
        print(json.dumps({"generated": args.images, "s": round(time.perf_counter() - t0, 1)}), flush=True)
        ds_host, ds_gpu = ImageFolder(root, transform=host_tf), ImageFolder(root, transform=gpu_tf)
        order = [sizes[p] for p, _ in ds_gpu.samples]
        per_batch = [order[i:i + args.batch] for i in range(0, len(order), args.batch)]
        h2d_gpu = float(np.mean([sum(h * w * 3 for h, w in b) + len(b) * 7 * 8 for b in per_batch]))
        h2d_host = float(np.mean([len(b) * 3 * CROP * CROP * 4 for b in per_batch]))
        file_mb = sum(os.path.getsize(p) for p, _ in ds_host.samples) / 1e6
        for workers in [int(v) or cpus for v in args.workers.split(",")]:
            loaders = {
                "host": DataLoader(ds_host, batch_size=args.batch, shuffle=False, num_workers=workers, pin_memory=True),
                "gpu": DataLoader(ds_gpu, batch_size=args.batch, shuffle=False, num_workers=workers, pin_memory=True,
                                  collate_fn=gpu_tf.collate)}
            times, outs = {k: [] for k in loaders}, {}
            for _ in range(args.reps):
                for name, loader in loaders.items():
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    outs[name] = F.evaluate_model_test(model, loader, "cuda")
                    torch.cuda.synchronize()
                    times[name].append(time.perf_counter() - t0)
            identical = all(np.array_equal(a, b) for a, b in zip(outs["host"][:4], outs["gpu"][:4])) and \
                outs["host"][4] == outs["gpu"][4]
            ips = {k: len(ds_host) / min(v) for k, v in times.items()}
            rec = {"end_to_end": {"workers": workers, "cpu_count": cpus, "images": len(ds_host), "batch": args.batch,
                                  "jpeg_MB": round(file_mb, 1), "reps": args.reps,
                                  "host_images_per_s": round(ips["host"], 1), "gpu_images_per_s": round(ips["gpu"], 1),
                                  "gpu_over_host": round(ips["gpu"] / ips["host"], 3),
                                  "host_s_per_rep": [round(v, 2) for v in times["host"]],
                                  "gpu_s_per_rep": [round(v, 2) for v in times["gpu"]],
                                  "h2d_MB_per_batch_host": round(h2d_host / 1e6, 2),
                                  "h2d_MB_per_batch_gpu": round(h2d_gpu / 1e6, 2),
                                  "identical_arrays": bool(identical)}}
            lines.append(json.dumps(rec))
            print(lines[-1], flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=3000)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--workers", default="4,0")
    ap.add_argument("--skip-end-to-end", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_loader_resize.py measures on a GPU; none is visible")
    lines = [json.dumps({"gpu": gpu_info()})]
    print(lines[0], flush=True)
    kernels(lines)
    if not args.skip_end_to_end:
        end_to_end(lines, args)
    lines.append(json.dumps({"gpu_after": gpu_info()}))
    print(lines[-1], flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
