#!/usr/bin/env python
"""Measures the release-tarball step on one B200 and writes profiles/r03_tarball.json (or argv[1]);
further arguments select trees by name prefix (config2, config3).

For the stripped config-2 and config-3 stand-in trees (tools/measure_configs.py) it records the reference's
`tarfile` "w:gz" leg as shipped, `tar cf - | gzip -6` for context, the GPU end-to-end call (cold once, then
best of 3 warm, with its phase split and size relative to zlib -6 / -9 of the same tar bytes) and
lb2_deflate_device on the HBM-resident tar (warm-up, then >= 10 CUDA-event-timed runs).  Fails without a GPU.
"""
import ctypes as C
import glob
import io
import json
import os
import subprocess
import sys
import tarfile
import tempfile
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import measure_configs as MC  # noqa: E402
from lambdipy_b200 import _native as N  # noqa: E402
from lambdipy_b200 import strip as S  # noqa: E402
from lambdipy_b200 import tarball as T  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def tar_bytes(d):
    bio = io.BytesIO()
    with tarfile.open(fileobj=bio, mode="w") as tar:
        for p in glob.glob(f"{d}/*"):
            tar.add(p, arcname=os.path.basename(p))
    return bio.getvalue()


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r03_tarball.json")
    ctx = N.Context(0)   # raises without a B200: no CPU fallback
    res = {"card (name, power limit, max SM clock)": card(), "trees": {}}
    names = [n for n in MC.TREES if n.startswith(tuple(sys.argv[2:]))] if len(sys.argv) > 2 else \
        ["config2_numpy+scipy+sklearn+PIL", "config3_torch (stand-in for tensorflow 1.13.1)"]
    for name in names:
        with tempfile.TemporaryDirectory() as tmp:
            d = os.path.join(tmp, "build")
            os.makedirs(d)
            MC.copy_tree(MC.TREES[name], d)
            S.strip_tree(d, ctx=ctx)
            tb = tar_bytes(d)
            r = {"tar_bytes": len(tb)}
            ref = os.path.join(tmp, "ref.tar.gz")
            t0 = time.perf_counter()
            with tarfile.open(ref, "w:gz") as tar:
                for p in glob.glob(f"{d}/*"):
                    tar.add(p, arcname=os.path.basename(p))
            r["reference_tarfile_w_gz_s"] = time.perf_counter() - t0
            r["reference_bytes"] = os.path.getsize(ref)
            t0 = time.perf_counter()
            subprocess.run("cd %s && tar cf - $(ls) | gzip -6 > %s/g6.tar.gz" % (d, tmp), shell=True, check=True)
            r["tar_gzip6_s"] = time.perf_counter() - t0
            z6, z9 = len(zlib.compress(tb, 6)), len(zlib.compress(tb, 9))
            gpu = os.path.join(tmp, "gpu.tar.gz")
            t0 = time.perf_counter()
            cold = T.create_tarball(d, gpu, ctx)
            r["gpu_e2e_cold_s"] = time.perf_counter() - t0
            r["gpu_e2e_cold_setup_s"] = cold["setup_s"]
            warm = []
            for _ in range(3):
                t0 = time.perf_counter()
                st = T.create_tarball(d, gpu, ctx)
                warm.append((time.perf_counter() - t0, st))
            best_s, st = min(warm, key=lambda x: x[0])
            r["gpu_e2e_warm_best_s"] = best_s
            r["gpu_e2e_phases"] = st
            r["gpu_out_bytes"] = st["out_bytes"]
            r["gpu_size_vs_zlib6"] = st["out_bytes"] / z6
            r["gpu_size_vs_zlib9"] = st["out_bytes"] / z9
            r["speedup_vs_reference"] = r["reference_tarfile_w_gz_s"] / best_s
            # device-resident: the tar in HBM, deflate kernel + concatenation timed with CUDA events
            n = len(tb)
            d_in = ctx.dev_alloc(n)
            ctx.h2d(d_in, C.c_char_p(tb), n)
            T.deflate_device(ctx, d_in, n)   # warm-up
            ms = []
            for _ in range(10):
                _, crc, s2 = T.deflate_device(ctx, d_in, n)
                ms.append(s2["kernel_ms"])
            assert crc == zlib.crc32(tb)
            ctx.dev_free(d_in)
            r["device_kernel_ms"] = ms
            r["device_GBps_best"] = n / (min(ms) * 1e-3) / 1e9
            r["device_GBps_median"] = n / (sorted(ms)[len(ms) // 2] * 1e-3) / 1e9
            pc = s2["phase_cycles"]
            r["kernel_phase_share"] = {k: v / max(1, sum(pc.values())) for k, v in pc.items()}
            r["gpu_beats_reference"] = best_s < r["reference_tarfile_w_gz_s"]
            res["trees"][name] = r
            print(json.dumps({name: r}), flush=True)
    os.makedirs(os.path.dirname(out_path), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
