"""Baseline JPEG decoding on the GPU (functions.gpu_resize_transform(decode="gpu")) against the host loaders.

    python tools/time_loader_decode.py [--images 3000] [--batch 64] [--reps 2] [--workers 4,16] [--subseq 256,8192]
                                       [--out FILE]

Two seeded JPEG folders, written to a temporary directory: the one of tools/time_loader_resize.py (sides 300-2000 px,
smooth content with noise, quality 90, 4:2:0) and the same images at Pillow's default quality 75 / 4:2:0.

Kernels: the first 64 files of each folder as one batch; CUDA events around 20 launches (after 3 warm-up launches) of
each phase of gh_jpeg_decode alone (Huffman, IDCT, upsampling + colour), with the compressed bytes per second of the
Huffman phase and the bytes each phase writes. The decoded arena is checked against Pillow for those 64 files.

End to end: evaluate_model_test images/s over each folder with three loaders, alternating, --reps times each, at each
--workers count: the host transforms (Resize + CenterCrop + ToTensor + Normalize in the workers),
gpu_resize_transform() and gpu_resize_transform(decode="gpu"). The model is the one of tools/time_loader_resize.py with
ops.KSPLIT = 1, so that the three loaders' arrays are compared bit for bit. The host-to-device bytes per batch and the
GPU's name and power limit are read in the same run.
"""
import argparse
import io
import json
import os
import sys
import tempfile
import time
from multiprocessing import Pool

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from PIL import Image  # noqa: E402

from heuristique_style_transfer_code_b200 import ops, functions as F, jpeg  # noqa: E402
from time_loader_resize import gpu_info, make_folder, MEAN, STD, RESIZE, CROP  # noqa: E402


def _requality(args):
    src, dst = args
    Image.open(src).convert("RGB").save(dst, quality=75)


def event_ms(fn, launches=20):
    for _ in range(3):
        fn()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(launches):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / launches


def kernels(lines, root, label, subseqs=()):
    paths = sorted(os.path.join(d, f) for d, _, fs in os.walk(root) for f in fs)[:64]
    datas = [open(p, "rb").read() for p in paths]
    files = [jpeg.parse(d) for d in datas]
    sizes = [f.H * f.W * 3 for f in files]
    offsets = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
    t0 = time.perf_counter()
    files = [jpeg.parse(d) for d in datas]
    parse_ms = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter()
    for d in datas:
        Image.open(io.BytesIO(d)).convert("RGB")
    pillow_ms = (time.perf_counter() - t0) * 1e3
    scan, segs, imgs, tables = jpeg.pack(files, offsets, list(range(len(files))))
    scan_d, segs_d, imgs_d, tables_d = (t.cuda() for t in (scan, segs, imgs, tables))
    total = int(sum(sizes))
    arena = torch.empty(total, dtype=torch.uint8, device="cuda")
    n_coef, n_plane, n_rec = jpeg.workspace(imgs.numpy(), scan.numel(), len(segs))
    work = dict(coef=torch.empty(n_coef, dtype=torch.int16, device="cuda"),
                planes=torch.empty(n_plane, dtype=torch.uint8, device="cuda"),
                records=torch.empty(n_rec // 4, dtype=torch.int32, device="cuda"),
                status=torch.empty(len(files), dtype=torch.int32, device="cuda"))

    def run(phases, subseq=jpeg.SUBSEQ_BYTES):
        return jpeg.decode_batch(scan_d, segs_d, imgs_d, tables_d, imgs.numpy(), segs.numpy(), arena, total,
                                 phases=phases, subseq=subseq, **work)
    status = run(7)
    torch.cuda.synchronize()
    host = arena.cpu().numpy()
    equal = not status.cpu().numpy().any() and all(
        np.array_equal(host[o:o + s], np.asarray(Image.open(io.BytesIO(d)).convert("RGB")).reshape(-1))
        for d, o, s in zip(datas, offsets, sizes))
    t_huff, t_idct, t_color = (event_ms(lambda ph=ph: run(ph)) for ph in (1, 2, 4))
    t_all = event_ms(lambda: run(7))
    sweep = {}
    for sub in subseqs:
        n_rec = jpeg.workspace(imgs.numpy(), scan.numel(), len(segs), sub)[2]
        if work["records"].numel() * 4 < n_rec:
            work["records"] = torch.empty(n_rec // 4, dtype=torch.int32, device="cuda")
        sweep[sub] = round(event_ms(lambda: run(1, sub), launches=5), 3)
    rec = {"kernels": {"folder": label, "images": len(files), "compressed_MB": round(scan.numel() / 1e6, 2),
                       "decoded_MB": round(total / 1e6, 2), "coef_MB": round(n_coef * 2 / 1e6, 2),
                       "planes_MB": round(n_plane / 1e6, 2), "segments": len(segs),
                       "subseq_bytes": jpeg.SUBSEQ_BYTES,
                       "huffman_ms": round(t_huff, 3), "idct_ms": round(t_idct, 3), "color_ms": round(t_color, 3),
                       "all_phases_ms": round(t_all, 3),
                       "huffman_compressed_GBs": round(scan.numel() / (t_huff * 1e-3) / 1e9, 2),
                       "host_parse_ms_64_files": round(parse_ms, 1), "host_pillow_decode_ms_64_files": round(pillow_ms, 1),
                       "host_parse_over_pillow": round(parse_ms / pillow_ms, 3),
                       "arena_equal_pillow": bool(equal), "huffman_ms_by_subseq_bytes": sweep}}
    lines.append(json.dumps(rec))
    print(lines[-1], flush=True)


def end_to_end(lines, root, label, args):
    from torch.utils.data import DataLoader
    from torchvision import models, transforms
    from torchvision.datasets import ImageFolder
    from heuristique_style_transfer_code_b200 import TruncatedResNet50_for_test
    torch.manual_seed(0)
    model = TruncatedResNet50_for_test(models.resnet50(weights=None), 7, 4, 32, device="cuda:0").eval()
    ops.KSPLIT = 1
    host_tf = transforms.Compose([transforms.Resize(RESIZE), transforms.CenterCrop(CROP), transforms.ToTensor(),
                                  transforms.Normalize(MEAN, STD)])
    resize_tf = F.gpu_resize_transform(RESIZE, CROP)
    decode_tf = F.gpu_resize_transform(RESIZE, CROP, decode="gpu")
    sets = {"host": ImageFolder(root, transform=host_tf), "gpu_resize": ImageFolder(root, transform=resize_tf),
            "gpu_decode": ImageFolder(root, loader=decode_tf.loader, transform=decode_tf)}
    n = len(sets["host"])
    probe = DataLoader(sets["gpu_decode"], batch_size=args.batch, num_workers=8, collate_fn=decode_tf.collate)
    up = [b.pixels.numel() + sum(t.numel() * t.element_size() for t in b.jpeg) + b.geometry.numel() * 8 for b in probe]
    h2d = {"host": args.batch * 3 * CROP * CROP * 4, "gpu_decode": float(np.mean(up))}
    for workers in [int(v) for v in args.workers.split(",")]:
        loaders = {"host": DataLoader(sets["host"], batch_size=args.batch, num_workers=workers, pin_memory=True),
                   "gpu_resize": DataLoader(sets["gpu_resize"], batch_size=args.batch, num_workers=workers,
                                            pin_memory=True, collate_fn=resize_tf.collate),
                   "gpu_decode": DataLoader(sets["gpu_decode"], batch_size=args.batch, num_workers=workers,
                                            pin_memory=True, collate_fn=decode_tf.collate)}
        times, outs = {k: [] for k in loaders}, {}
        for _ in range(args.reps):
            for name, loader in loaders.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                outs[name] = F.evaluate_model_test(model, loader, "cuda")
                torch.cuda.synchronize()
                times[name].append(time.perf_counter() - t0)
        identical = all(all(np.array_equal(a, b) for a, b in zip(outs["host"][:4], outs[k][:4]))
                        and outs["host"][4] == outs[k][4] for k in ("gpu_resize", "gpu_decode"))
        rec = {"end_to_end": {"folder": label, "workers": workers, "cpu_count": len(os.sched_getaffinity(0)),
                              "images": n, "batch": args.batch, "reps": args.reps,
                              **{f"{k}_images_per_s": round(n / min(v), 1) for k, v in times.items()},
                              **{f"{k}_s_per_rep": [round(x, 2) for x in v] for k, v in times.items()},
                              "h2d_MB_per_batch_host": round(h2d["host"] / 1e6, 2),
                              "h2d_MB_per_batch_gpu_decode": round(h2d["gpu_decode"] / 1e6, 2),
                              "identical_arrays": bool(identical)}}
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=3000)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--workers", default="4,16")
    ap.add_argument("--skip-end-to-end", action="store_true")
    ap.add_argument("--subseq", default="", help="also time the Huffman phase at these subsequence sizes (bytes)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_loader_decode.py measures on a GPU; none is visible")
    lines = [json.dumps({"gpu": gpu_info()})]
    print(lines[0], flush=True)
    with tempfile.TemporaryDirectory() as tmp:
        q90, q75 = os.path.join(tmp, "q90"), os.path.join(tmp, "q75")
        t0 = time.perf_counter()
        sizes = make_folder(q90, args.images)
        jobs = [(p, p.replace(q90, q75, 1)) for p in sizes]
        for _, dst in jobs:
            os.makedirs(os.path.dirname(dst), exist_ok=True)
        with Pool(os.cpu_count()) as pool:
            pool.map(_requality, jobs, chunksize=16)
        lines.append(json.dumps({"generated": args.images, "s": round(time.perf_counter() - t0, 1)}))
        print(lines[-1], flush=True)
        for root, label in ((q90, "q90_420"), (q75, "q75_420")):
            kernels(lines, root, label, [int(v) for v in args.subseq.split(",") if v])
        if not args.skip_end_to_end:
            for root, label in ((q90, "q90_420"), (q75, "q75_420")):
                end_to_end(lines, root, label, args)
    lines.append(json.dumps({"gpu_after": gpu_info()}))
    print(lines[-1], flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
