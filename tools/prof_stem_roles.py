"""Where each warp role of stem_conv_pool_kernel spends its cycles (a -DGH_SC_PROFILE build of the library: clock64
around every mbarrier wait, the TMEM loads, the epilogue's bar.sync and the store phase of one thread per role, summed
over the CTAs, csrc/stem.cuh).
    python tools/prof_stem_roles.py [--build] [batch]
Build the instrumented library first (here, without a GPU):  python tools/prof_stem_roles.py --build
GRAMHEAD_LIB=<another -DGH_SC_PROFILE build> profiles that one instead."""
from __future__ import annotations

import ctypes
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "heuristique_style_transfer_code_b200", "csrc")
PROF_LIB = os.path.join(CSRC, "libgramhead_sc_prof.so")


def build() -> None:
    cmd = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
           "-shared", "-DGH_SC_PROFILE", "gramhead.cu", "-o", PROF_LIB]
    subprocess.run(cmd, cwd=CSRC, check=True)
    print("built", PROF_LIB)


def card() -> str:
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def main() -> None:
    if "--build" in sys.argv:
        build()
        return
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    B = int(args[0]) if args else 256
    os.environ.setdefault("GRAMHEAD_LIB", PROF_LIB)
    sys.path.insert(0, ROOT)
    import torch
    from heuristique_style_transfer_code_b200 import _lib, ops
    from heuristique_style_transfer_code_b200.frozen_encoder import pack_stem_weight
    lib = _lib.lib()
    lib.gh_sc_profile_read.restype = ctypes.c_int
    lib.gh_sc_profile_read.argtypes = [ctypes.POINTER(ctypes.c_ulonglong)]
    buf = (ctypes.c_ulonglong * 16)()
    print(f"card: {card() or torch.cuda.get_device_name(0)}")
    print(f"library: {os.path.relpath(_lib.library_path(), ROOT)}")
    print("per conv row (one tile of 128 conv columns, halo rows included) in SM cycles of one thread per role, "
          "averaged over the CTAs; the waits are part of each role's loop")
    torch.manual_seed(0)
    w16 = torch.randn(64, 16, 4, 4, device="cuda") * 0.05
    w16.view(64, 4, 4, 4, 4)[:, 3] = 0.0
    packed, bias = pack_stem_weight(w16), torch.randn(64, device="cuda") * 0.1
    reps = 20
    for H in (224, 448):
        x = torch.randn(B if H == 224 else B // 4, 3, H, H, device="cuda")
        for u8 in (False, True):
            xin = (x * 40 + 128).clamp(0, 255).to(torch.uint8) if u8 else x
            run = ((lambda: ops.stem_conv_pool_u8(xin, (0.485, 0.456, 0.406), (0.229, 0.224, 0.225), packed, bias))
                   if u8 else (lambda: ops.stem_conv_pool(xin, packed, bias)))
            for _ in range(3):
                run()
            assert lib.gh_sc_profile_read(buf) == 0
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                run()
            b.record()
            torch.cuda.synchronize()
            assert lib.gh_sc_profile_read(buf) == 0
            v = [float(t) for t in buf]
            us = a.elapsed_time(b) / reps * 1e3
            rows, ctas = max(v[3], 1.0), max(v[14], 1.0)
            per = lambda i: v[i] / rows                 # noqa: E731  (one thread per CTA: that CTA's cycles per conv row)
            rows_cta = rows / ctas
            mhz = v[15] / ctas / us if us else 0.0
            print(f"{'uint8' if u8 else 'fp32'} {x.shape[0]}x3x{H}x{H}: {us:.1f} us, {ctas:.0f} CTAs, "
                  f"{rows_cta:.1f} conv rows per CTA, CTA lifetime {v[15] / ctas:.0f} cycles = "
                  f"{v[15] / rows:.0f} per conv row (~{mhz:.0f} MHz effective)")
            print(f"    issuer   loop {per(0):6.0f}  wait aempty {per(1):6.0f}  wait full {per(2):6.0f}  "
                  f"busy {per(0) - per(1) - per(2):6.0f}")
            print(f"    producer loop {per(4):6.0f}  wait empty {per(5):6.0f}  store phase {per(6):6.0f}  "
                  f"load phase + skips {per(4) - per(5) - per(6):6.0f}  (warp 0 staged {v[7] / ctas:.1f} rows per CTA)")
            print(f"    epilogue loop {per(8):6.0f}  wait afull {per(9):6.0f}  TMEM loads + row max {per(10):6.0f}  "
                  f"bar.sync {per(11):6.0f}  column max + store {per(12):6.0f}  ({v[13] / ctas:.1f} pooled rows per CTA)",
                  flush=True)
        del x


if __name__ == "__main__":
    main()
