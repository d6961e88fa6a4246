#!/usr/bin/env python
"""bench.py -- ELF-strip throughput of the B200 path vs the reference's host `strip` pipeline.

  python bench.py [--gpus N] [--steps K] [--warmup W]              # this repo (CUDA kernels)
  python bench.py --impl reference [--gpus N] [--steps K] ...      # the reference's CPU pipeline
  python bench.py ... --dump-outputs DIR                           # + what the last timed step returned, as DIR/*.npy

Metric (BASELINE.json): ELF-strip GB/s of build-tree `.so` INPUT bytes.

Workload (default, `--scaling strong`) = BASELINE config 4 as stated: the synthetic corpus of 10 000 `.so`
files, sizes log-uniform 1 KB..128 MB (seed 0xB200, dropped fraction U(0.05,0.8); 115 GB in, 67 GB out),
dealt size-sorted round-robin over the N ranks -- the SAME 10 000 files at every N (at N=8 this is also
config 5, "100 GB over 8 B200").  One "step" = one pass of the hot path over the rank's whole shard.  A
shard whose input + output does not fit in HBM side by side (N=1: 115 + 67 GB) keeps the input resident
and streams the output through a two-slot ring (lb2_strip_device_chunked), one batch per ~14 GB chunk.
`--scaling weak` is round 1's workload (1250 files per GPU).  No payload crosses GPUs; the one collective
is a single NCCL allgather of the per-rank byte counts after the last step, inside the timed region.

  value      device-resident: inputs already in HBM; timed = upload of offsets + plan kernel + offset scan +
             compaction kernel + fetch of sizes/status per batch, + the allgather.  CUDA events, max over ranks.
  e2e        the same hot path through the C ABI with HOST buffers (lb2_strip_host on pinned arenas placed on
             the GPU's NUMA node): headers and kept extents cross PCIe up, stripped files come down, inside the
             timed region.  Host memory bounds it to the first <= 15 GB of each rank's shard.
  tree       (N=1) lb2_strip_tree -- the call that replaces project_build.py:260 -- on a /dev/shm tree holding
             the same files the reference arm strips: file reads and in-place writes included.
  roofline   compaction kernel: algorithmic bytes (copied extents read + output written) over its CUDA-event
             duration against MEASURED_PEAKS.json hbm_gbs; every rank's figure is in `per_rank`.
  cpu_baseline / --impl reference: the reference's own line `find DIR/ -name "*.so" | xargs strip`
             (/root/reference/lambdipy/project_build.py:260) on /dev/shm over the first <= 15 GB of the
             corpus (1/8: ~1250 files): serial as the reference runs it, and `xargs -P nproc -n 1`.
  parity     after the timed region every rank strips 8 size-stratified files of ITS shard with the real
             `strip --strip-unneeded` and compares them byte for byte with what the GPU produced.
  real_trees (N=1) BASELINE configs 2 and 3 (stand-ins from this image's site-packages): kernels, tree call,
             reference line, fallback count.
"""
import argparse
import ctypes as C
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ELF-strip GB/s (build-tree .so bytes)"
TOTAL_FILES = 10000
FILES_PER_GPU = 1250
SEED = 0xB200
SAMPLE_SPAN = 15 << 30        # host-side legs (e2e, tree, CPU baseline) work on the first <= 15 GiB of a shard
LAUNCHES_PER_BATCH = 3        # plan, scan (+ tile expansion of the very big extents), compaction
# --dump-outputs: the stripped bytes of a whole shard are tens of GB, so a fixed, seeded sample of them is written:
# DUMP_FILES outputs, each by its two ends (ELF and program headers; section table and .shstrtab) and DUMP_WINDOWS
# windows of its body.  At most 64 x 64 KiB bytes = 16 MiB as float32.
DUMP_SEED = 0xD0B
DUMP_FILES = 64
DUMP_EDGE = 16 << 10
DUMP_WINDOWS, DUMP_WINDOW = 8, 4 << 10


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured)"
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md; MEASURED_PEAKS.json absent)"


# ---------------------------------------------------------------- clocks during the timed region
class ClockSampler:
    """SM clocks and throttle reasons DURING the timed regions.  NVML from a thread (a few microseconds
    per sample); `nvidia-smi -lms` as fallback -- polling nvidia-smi at 100 ms measurably slowed the
    sampled GPU's kernels in the 8-GPU runs, NVML queries do not."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.thread = None
        self.stop_flag = False
        self.sm, self.mx, self.reasons = [], [], set()

    def _nvml_loop(self):
        import pynvml as nv
        h = nv.nvmlDeviceGetHandleByIndex(self.idx)
        names = {getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                 getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                 getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                 getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap"}
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                self.mx.append(float(mx))
                r = get_reasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.02)

    def start(self):
        try:
            import pynvml as nv
            import threading
            nv.nvmlInit()
            nv.nvmlDeviceGetHandleByIndex(self.idx)
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.path = tempfile.mktemp(prefix="lb2_clocks_", suffix=".csv")
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "500"],
                                         stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": None}
        if self.thread:
            self.stop_flag = True
            self.thread.join(timeout=2)
            out["source"] = "nvml"
        elif self.proc:
            out["source"] = "nvidia-smi"
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
            self.f.close()
            try:
                with open(self.path) as f:
                    for line in f:
                        p = [x.strip() for x in line.split(",")]
                        if len(p) < 9:
                            continue
                        try:
                            self.sm.append(float(p[1])); self.mx.append(float(p[2]))
                        except ValueError:
                            continue
                        for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                            if v.lower().startswith("active"):
                                self.reasons.add(name)
                os.unlink(self.path)
            except Exception:
                pass
        if self.sm:
            out.update(sm_mhz=statistics.median(self.sm), sm_max_mhz=max(self.mx), reasons=sorted(self.reasons), samples=len(self.sm))
        return out


# ---------------------------------------------------------------- the reference pipeline on host cores
REF_LINE = 'find {d}/ -name "*.so" | xargs strip'              # project_build.py:260, verbatim
PAR_LINE = 'find {d}/ -name "*.so" | xargs -P {p} -n 1 strip'  # same tool, all host cores


def shm_dir():
    return "/dev/shm" if os.path.isdir("/dev/shm") else None


def copy_tree_parallel(src, dst, threads=32):
    """cp -r with many threads (the trees are tens of GB of tmpfs; strip rewrites files in place, so every
    timed run needs a fresh copy).  Keeps symlinks and modes."""
    jobs = []
    for d, dirs, fs in os.walk(src):
        rel = os.path.relpath(d, src)
        os.makedirs(os.path.join(dst, rel), exist_ok=True)
        for f in fs:
            jobs.append((os.path.join(d, f), os.path.join(dst, rel, f)))
        for x in list(dirs):
            if os.path.islink(os.path.join(d, x)):
                jobs.append((os.path.join(d, x), os.path.join(dst, rel, x)))

    def cp(j):
        s, t = j
        if os.path.islink(s):
            os.symlink(os.readlink(s), t)
        else:
            shutil.copyfile(s, t)
            shutil.copymode(s, t)

    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(cp, jobs))


def run_line(line, d, nproc):
    t0 = time.perf_counter()
    rc = subprocess.run(["bash", "-c", "set -e; set -o pipefail; " + line.format(d=d, p=nproc)], capture_output=True)
    dt = time.perf_counter() - t0
    if rc.returncode != 0:
        raise RuntimeError("reference strip pipeline failed: %s" % rc.stderr.decode()[:300])
    return dt


def cpu_lines_on_master(base, master, n_bytes, par_reps, par_warm, serial_reps):
    """Times the reference's line on fresh copies of `master`.  Returns the result dict and leaves the
    last parallel run's stripped tree in base/run_ref for comparisons."""
    nproc = os.cpu_count() or 1
    par, ser = [], []
    run = os.path.join(base, "run_ref")
    for r in range(par_warm + par_reps):
        shutil.rmtree(run, ignore_errors=True)
        copy_tree_parallel(master, run)
        dt = run_line(PAR_LINE, run, nproc)
        if r >= par_warm:
            par.append(dt)
    run2 = os.path.join(base, "run_ser")
    for r in range(serial_reps):
        shutil.rmtree(run2, ignore_errors=True)
        copy_tree_parallel(master, run2)
        ser.append(run_line(REF_LINE, run2, nproc))
    shutil.rmtree(run2, ignore_errors=True)
    return {"bytes": n_bytes, "nproc": nproc, "parallel_s": par, "parallel_gbs": n_bytes / 1e9 / (sum(par) / len(par)),
            "serial_s": ser, "serial_gbs": (n_bytes / 1e9 / (sum(ser) / len(ser))) if ser else None}


def strip_version():
    try:
        return subprocess.run(["strip", "--version"], capture_output=True, text=True).stdout.splitlines()[0]
    except Exception:
        return "unknown"


def gnu_strip(data, workdir, tag):
    """`strip --strip-unneeded -o OUT IN` of the real binary (the parity oracle of last resort)."""
    pi, po = os.path.join(workdir, "p%s.in.so" % tag), os.path.join(workdir, "p%s.out.so" % tag)
    with open(pi, "wb") as f:
        f.write(data)
    r = subprocess.run(["strip", "--strip-unneeded", "-o", po, pi], capture_output=True)
    out = None
    if r.returncode == 0:
        with open(po, "rb") as f:
            out = f.read()
    for p in (pi, po):
        if os.path.exists(p):
            os.unlink(p)
    return out


def trees_identical(a, b, threads=32):
    la, lb = [], []
    for root, acc in ((a, la), (b, lb)):
        for d, _, fs in os.walk(root):
            for f in fs:
                acc.append(os.path.relpath(os.path.join(d, f), root))
    if sorted(la) != sorted(lb):
        return False

    def same(rel):
        pa, pb = os.path.join(a, rel), os.path.join(b, rel)
        if os.path.islink(pa) or os.path.islink(pb):
            return os.path.islink(pa) and os.path.islink(pb) and os.readlink(pa) == os.readlink(pb)
        if os.path.getsize(pa) != os.path.getsize(pb):
            return False
        with open(pa, "rb") as fa, open(pb, "rb") as fb:
            while True:
                x, y = fa.read(1 << 24), fb.read(1 << 24)
                if x != y:
                    return False
                if not x:
                    return True

    with ThreadPoolExecutor(threads) as ex:
        return all(ex.map(same, la))


# ---------------------------------------------------------------- workload
def make_corpus(a, rank, world):
    from lambdipy_b200.corpus import Corpus
    if a.scaling == "strong":
        return Corpus(a.total_files, seed=SEED, rank=rank, world=world)
    return Corpus(a.files_per_gpu * world, seed=SEED, rank=rank, world=world)


def sample_count(corpus):
    """Number of leading files of the shard whose arena span is <= SAMPLE_SPAN."""
    import numpy as np
    return int(np.searchsorted(corpus.off[1:], SAMPLE_SPAN, side="right"))


def workload_config(a, world):
    if a.scaling == "strong":
        w = ("synthetic ELF corpus, BASELINE config 4 at full size (= config 5 at 8 GPUs): %d files, sizes log-uniform 1 KB-128 MB, "
             "seed 0x%X, dropped fraction U(0.05,0.8), ~115 GB in / ~67 GB out; the same files at every N, dealt size-sorted "
             "round-robin over %d rank(s)" % (a.total_files, SEED, world))
    else:
        w = ("synthetic ELF corpus (BASELINE config 4/5 generator): %d files per GPU (%d total), sizes log-uniform 1 KB-128 MB, "
             "seed 0x%X, dropped fraction U(0.05,0.8); files dealt size-sorted round-robin over ranks" %
             (a.files_per_gpu, a.files_per_gpu * world, SEED))
    return {"workload": w, "total_files": a.total_files if a.scaling == "strong" else a.files_per_gpu * world,
            "parallelism": "file-sharded x%d, no payload exchange, one allgather of byte counts" % world,
            "l2": "inputs (>10 GB per GPU) far larger than the 126 MB L2; no flush needed"}


def dump_files(n):
    """Indices of the outputs whose bytes --dump-outputs samples: the same for every run of a shard of n files."""
    import numpy as np
    return sorted(int(i) for i in np.random.default_rng(DUMP_SEED).choice(n, size=min(n, DUMP_FILES), replace=False))


def dump_sample(i, out):
    """Both ends of output i and DUMP_WINDOWS seeded windows of its body, concatenated."""
    import numpy as np
    b = np.frombuffer(out, dtype=np.uint8)
    parts = [b[:DUMP_EDGE], b[-DUMP_EDGE:]]
    if len(b) > DUMP_WINDOW:
        starts = np.random.default_rng([DUMP_SEED, i]).integers(0, len(b) - DUMP_WINDOW + 1, size=DUMP_WINDOWS)
        parts += [b[s:s + DUMP_WINDOW] for s in starts]
    return np.concatenate(parts)


def write_dump(d, out_sizes, status, files, outputs):
    """DIR/<name>.npy: per-file output sizes and status codes, the sampled file indices and their sampled bytes."""
    import numpy as np
    arrays = {"out_sizes": out_sizes.astype(np.float64), "status": status.astype(np.float64),
              "sample_files": np.array(files, dtype=np.float64),
              "sample_bytes": np.concatenate([dump_sample(i, outputs[i]) for i in files]).astype(np.float32)}
    assert sum(x.nbytes for x in arrays.values()) <= 64 << 20
    os.makedirs(d, exist_ok=True)
    for name, x in arrays.items():
        np.save(os.path.join(d, name + ".npy"), x)


def _materialize(args):
    corpus, i, path = args
    with open(path, "wb") as f:
        f.write(corpus.materialize(i))
    return os.path.getsize(path)


# ---------------------------------------------------------------- reference arm
def run_reference(a, rank, world):
    if rank != 0:
        return 0
    from multiprocessing import Pool
    corpus = make_corpus(a, 0, 1)          # the host-side legs always use the head of the whole corpus
    ns = sample_count(corpus)
    n_bytes = int(corpus.sizes[:ns].sum())
    base = tempfile.mkdtemp(prefix="lb2_ref_", dir=shm_dir())
    try:
        master = os.path.join(base, "master")
        os.makedirs(master)
        jobs = [(corpus, i, os.path.join(master, "f%05d.so" % i)) for i in range(ns)]
        with Pool(min(48, os.cpu_count() or 1)) as pool:
            pool.map(_materialize, jobs, chunksize=2)
        # bound the run: K timed + W warm-up parallel runs must end within a few minutes; the serial line once
        t_probe0 = time.perf_counter()
        res = cpu_lines_on_master(base, master, n_bytes, 1, 0, 1)
        per_run = (time.perf_counter() - t_probe0) / 2
        budget = 240.0
        steps = max(1, min(a.steps, int(budget / max(per_run, 1e-3)) - 1))
        warm = max(0, min(a.warmup, steps // 4))
        more = cpu_lines_on_master(base, master, n_bytes, steps, warm, 0) if steps > 1 else None
        if more:
            res["parallel_s"] = more["parallel_s"]; res["parallel_gbs"] = more["parallel_gbs"]
    finally:
        shutil.rmtree(base, ignore_errors=True)
    value = res["parallel_gbs"]
    sample = ("the first %d files (%.3f GB, 1 KB-128 MB each) of the corpus on /dev/shm, every timed run on a fresh copy; `%s` "
              "(GNU strip: %s) with all %d host cores; %d timed runs%s; serial as the reference runs it (1 process): %.3f GB/s"
              % (ns, n_bytes / 1e9, PAR_LINE.format(d="DIR", p=res["nproc"]), strip_version(), res["nproc"], len(res["parallel_s"]),
                 "" if len(res["parallel_s"]) == a.steps else " (of --steps %d: bounded to a few minutes)" % a.steps, res["serial_gbs"] or 0))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * sum(res["parallel_s"]) / len(res["parallel_s"]),
        "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(a, world),
        "cpu_baseline": {"value": value, "unit": "GB/s", "cores": res["nproc"], "kind": "reference", "sample": sample,
                         "serial_value": res["serial_gbs"], "timed_runs": len(res["parallel_s"])},
        "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------- real build trees (BASELINE configs 2, 3)
REAL_TREES = {
    "config2_numpy+scipy+sklearn+PIL": ["numpy", "scipy", "sklearn", "PIL", "numpy.libs", "scipy.libs", "pillow.libs", "scikit_learn.libs"],
    "config3_torch (stand-in for tensorflow 1.13.1)": ["torch"],
}


def real_trees_block(ctx, peak):
    """Kernels, tree call and the reference's line on copies of this image's real wheels (N=1, rank 0)."""
    import numpy as np
    import sysconfig
    from lambdipy_b200 import strip as S
    from lambdipy_b200.device import DeviceBatch
    sp = sysconfig.get_paths()["purelib"]
    out = {}
    nproc = os.cpu_count() or 1
    for name, roots in REAL_TREES.items():
        roots = [r for r in roots if os.path.isdir(os.path.join(sp, r))]
        if not roots:
            continue
        base = tempfile.mkdtemp(prefix="lb2_real_", dir=shm_dir())
        try:
            master = os.path.join(base, "master")
            for r in roots:
                shutil.copytree(os.path.join(sp, r), os.path.join(master, r), symlinks=True,
                                ignore=lambda d, names: [n for n in names if not (os.path.isdir(os.path.join(d, n)) or ".so" in n)])
            files = sorted(os.path.join(d, f) for d, _, fs in os.walk(master) for f in fs
                           if f.endswith(".so") and not os.path.islink(os.path.join(d, f)))
            in_bytes = sum(os.path.getsize(p) for p in files)
            ref = os.path.join(base, "ref")
            ser, par = [], []
            for _ in range(2):
                shutil.rmtree(ref, ignore_errors=True); copy_tree_parallel(master, ref)
                par.append(run_line(PAR_LINE, ref, nproc))
            for _ in range(2):
                shutil.rmtree(ref, ignore_errors=True); copy_tree_parallel(master, ref)
                ser.append(run_line(REF_LINE, ref, nproc))
            gpu = os.path.join(base, "gpu")
            tt = []
            for _ in range(3):
                shutil.rmtree(gpu, ignore_errors=True); copy_tree_parallel(master, gpu)
                t0 = time.perf_counter()
                st = S.strip_tree(gpu, ctx=ctx)
                tt.append(time.perf_counter() - t0)
            same = trees_identical(ref, gpu)
            blobs = [open(p, "rb").read() for p in files]
            b = DeviceBatch.from_blobs(ctx, blobs)
            plan, comp = [], []
            for k in range(15):
                b.strip_async(); d = b.results()
                if k >= 5:
                    plan.append(d["plan_ms"]); comp.append(d["compact_ms"])
            b.close()
            pm, cm = float(np.median(plan)), float(np.median(comp))
            alg = d["copy_bytes"] + d["out_bytes"]
            out[name] = {
                "files": len(files), "in_gb": in_bytes / 1e9, "out_gb": d["out_bytes"] / 1e9, "fallback_files": int(st["n_fallback"]),
                "unsupported_on_device": int(d["n_unsupported"]), "plan_ms": pm, "compact_ms": cm,
                "compact_frac": alg / 1e9 / (cm / 1e3) / peak, "whole_pass_frac": (alg + d["header_bytes"]) / 1e9 / ((pm + cm) / 1e3) / peak,
                "kernels_gbs_input": in_bytes / 1e9 / ((pm + cm) / 1e3),
                "tree_s": min(tt), "tree_first_call_s": tt[0], "tree_gbs": in_bytes / 1e9 / min(tt),
                "tree_phases_s": {k: st[k] for k in ("walk_read_s", "gpu_s", "write_s", "fallback_s", "read_cpu_s", "write_cpu_s", "dma_wait_s", "io_threads", "n_batches")},
                "tree_identical_to_reference": bool(same),
                "reference_serial_s": min(ser), "reference_serial_gbs": in_bytes / 1e9 / min(ser),
                "reference_parallel_s": min(par), "reference_parallel_gbs": in_bytes / 1e9 / min(par), "cores": nproc,
            }
        finally:
            shutil.rmtree(base, ignore_errors=True)
    return out


# ---------------------------------------------------------------- B200 arm
def run_b200(a, rank, local_rank, world):
    # NCCL's own INIT lines (communicator, nranks, transport) stay visible on its default sink (stdout; pointing
    # NCCL_DEBUG_FILE at /dev/stderr lost them on the GPU box).  The JSON line is the LAST line rank 0 prints.
    # (forced, not setdefault: the image exports NCCL_DEBUG=VERSION, which hides the communicator lines)
    os.environ["NCCL_DEBUG"] = os.environ.get("LB2_NCCL_DEBUG", "INFO")
    os.environ["NCCL_DEBUG_SUBSYS"] = os.environ.get("LB2_NCCL_DEBUG_SUBSYS", "INIT")
    import numpy as np
    import torch
    from lambdipy_b200 import _native as N
    from lambdipy_b200.device import DeviceBatch

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = N.Context(local_rank)
    peak, peak_src = peaks()
    corpus = make_corpus(a, rank, world)
    n = len(corpus)
    in_span = int(corpus.off[-1])
    free_b, total_b = torch.cuda.mem_get_info()
    # A shard whose input + output exceed HBM (N=1: 115 + 67 GB) keeps the input resident and streams the output through
    # the two-slot ring of lb2_strip_device_chunked; otherwise one batch per step (splitting a shard that fits into two
    # pipelined batches was measured: 2.84 vs 2.79 ms per step at N=8 -- the second plan/scan costs more than the hidden
    # host round trip).
    big = (2 * in_span + n * 4096 + (1 << 30)) > 0.85 * free_b
    chunked = big
    chunk_bytes = int(a.chunk_gb * (1 << 30)) if big else None
    batch = DeviceBatch.from_corpus(ctx, corpus, chunk_bytes=chunk_bytes)
    stream = torch.cuda.current_stream()
    sptr = C.c_void_p(stream.cuda_stream)
    counts_h = torch.zeros(4, dtype=torch.int64).pin_memory()
    counts = torch.zeros(4, dtype=torch.int64, device="cuda")
    gathered = torch.zeros(4 * world, dtype=torch.int64, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
            torch.cuda.synchronize()

    def run_steps(k):
        """k back-to-back passes over the shard; returns the stats of each.  A shard that fits is one batch per pass and the
        next pass is queued before the previous one's results are collected (two batches in flight, lb2_strip_device_async),
        so the GPU never waits for the host between passes; a chunked shard pipelines its batches the same way inside
        lb2_strip_device_chunked."""
        if chunked:
            return [batch.strip_chunked(stream=sptr) for _ in range(k)]
        out = []
        batch.strip_async(stream=sptr)
        for i in range(k):
            if i + 1 < k:
                batch.strip_async(stream=sptr)
            out.append(batch.results())
        return out

    def allgather_counts(st):
        # the ONE collective of the path: per-rank byte counts, 32 bytes per rank, pinned source
        counts_h[0], counts_h[1], counts_h[2], counts_h[3] = st["in_bytes"], st["out_bytes"], st["n_ok"], st["n_unsupported"]
        counts.copy_(counts_h, non_blocking=True)
        dist.all_gather_into_tensor(gathered, counts)

    warm = max(a.warmup, 3)
    st = run_steps(warm)[-1]
    if dist:
        allgather_counts(st)  # communicator + NVLS buffers come up outside the timed region
    assert st["n_unsupported"] == 0 and st["n_ok"] == n, st
    n_batches = 1 if not chunked else int(np.ceil(in_span / batch.chunk_bytes))  # reported; exact count below
    # ---- device-resident timed region
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    compact_ms, plan_ms = [], []
    e0.record(stream)
    for st in run_steps(a.steps):
        compact_ms.append(st["compact_ms"]); plan_ms.append(st["plan_ms"])
    if dist:
        allgather_counts(st)
    e1.record(stream)
    barrier()
    dev_ms = e0.elapsed_time(e1)
    if dist:
        g = gathered.cpu().numpy().reshape(world, 4)
        total_files = a.total_files if a.scaling == "strong" else a.files_per_gpu * world
        assert int(g[:, 2].sum()) == total_files and int(g[:, 3].sum()) == 0, g
    cms, pms = sum(compact_ms) / len(compact_ms), sum(plan_ms) / len(plan_ms)
    alg = st["copy_bytes"] + st["out_bytes"]
    if a.profile_mode:
        if rank == 0:
            print(json.dumps({"profile_mode": True, "ms_per_step": dev_ms / a.steps, "compact_ms": compact_ms, "plan_ms": plan_ms,
                              "alg_bytes": alg, "frac": alg / 1e9 / (cms / 1e3) / peak, "chunked": chunked, "note": "not a bench value"}))
        batch.close()
        if dist:
            dist.barrier()
            dist.destroy_process_group()
        return 0

    # ---- parity on the shard that was benchmarked: 8 size-stratified files per rank vs the real GNU strip
    last_sizes, last_status = batch.out_sizes[:n].copy(), batch.status[:n].copy()   # as the last timed step returned them
    order = np.argsort(batch.sizes[:n], kind="stable")
    picks = sorted(set(int(order[min(n - 1, (k * (n - 1)) // 7)]) for k in range(8)))
    dumped = dump_files(n) if a.dump_outputs and rank == 0 else []
    wanted = set(picks) | set(dumped)
    got = {}
    if chunked:
        # the ring keeps only the last two chunks of a pass: the outputs are taken from one more, identical pass
        def grab(chunk, f0, cnt, d_slot, ooff, osz, stat):
            for i in wanted:
                if f0 <= i < f0 + cnt:
                    buf = C.create_string_buffer(int(osz[i - f0]))
                    ctx.d2h(buf, d_slot + int(ooff[i - f0]), len(buf))
                    got[i] = buf.raw
        batch.strip_chunked(stream=sptr, on_chunk=grab)
        assert (batch.out_sizes[:n] == last_sizes).all() and (batch.status[:n] == last_status).all()
    else:
        for i in wanted:
            got[i] = batch.read_output(i)
    if dumped:
        write_dump(a.dump_outputs, last_sizes, last_status, dumped, got)
    pdir = tempfile.mkdtemp(prefix="lb2_par_%d_" % rank, dir=shm_dir())
    mismatches = 0
    for i in picks:
        want = gnu_strip(batch.read_input(i), pdir, str(i))
        mismatches += (want is None) or (want != got.get(i))
    shutil.rmtree(pdir, ignore_errors=True)

    # ---- end to end through host buffers (the first <= 15 GiB of the shard)
    ns = sample_count(corpus) if in_span > SAMPLE_SPAN else n
    s_span = int(corpus.off[ns])
    h_in = ctx.pinned_alloc(s_span + 256)
    out_cap = s_span + ns * 4096 + (16 << 20)
    h_out = ctx.pinned_alloc(out_cap)
    ctx.d2h(h_in, batch.d_in, s_span)
    out_off = np.zeros(ns + 1, dtype=np.uint64); out_sizes = np.zeros(ns, dtype=np.uint64); status = np.zeros(ns, dtype=np.int32)
    u64p = lambda x: x.ctypes.data_as(C.POINTER(C.c_uint64))
    hst = N.Stats()

    def e2e_step():
        ctx.check(ctx.lib.lb2_strip_host(ctx.h, h_in, u64p(batch.off), u64p(batch.sizes), ns, h_out, out_cap, u64p(out_off), u64p(out_sizes),
                                         status.ctypes.data_as(C.POINTER(C.c_int32)), 0, C.byref(hst)))

    e2e_steps = max(1, min(a.steps, a.e2e_steps))

    def time_e2e():
        e2e_step()  # warm-up (allocates workspaces / pipeline slots)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        if dist:
            allgather_counts({"in_bytes": hst.in_bytes, "out_bytes": hst.out_bytes, "n_ok": hst.n_ok, "n_unsupported": hst.n_unsupported})
        barrier()
        return (time.perf_counter() - t0) * 1e3

    # default path of lb2_strip_host for pinned, mapped arenas: zero-copy (kernels read and write the mapped arenas); then,
    # for comparison, the copy-engine variant (plan over the mapping, DMA of the kept ranges, compaction in HBM, DMA of the
    # output; 256 MB chunks, 3 slots) and the staged pipeline that uploads whole files
    e2e_ms = time_e2e()
    e2e_in, e2e_out, e2e_up = hst.in_bytes, hst.d2h_bytes, hst.h2d_bytes   # bytes the library moved over the bus in one step
    assert hst.n_ok == ns and int(status.max()) == 0
    probe = int(np.argsort(batch.sizes[:ns])[ns // 2])  # host result of one mid-sized file == what GNU strip / the device path gave
    e2e_probe = C.string_at(h_out + int(out_off[probe]), int(out_sizes[probe]))
    os.environ["LB2_HOST_DMA"] = "1"
    zc_ms = time_e2e()   # (variable name kept: the second variant's time)
    os.environ["LB2_HOST_DMA"] = "0"
    os.environ["LB2_HOST_ZEROCOPY"] = "0"
    staged_ms = time_e2e()
    os.environ.pop("LB2_HOST_ZEROCOPY"); os.environ.pop("LB2_HOST_DMA")
    clocks = sampler.stop() if rank == 0 else None  # sampled across the device-resident and the e2e timed regions
    pdir = tempfile.mkdtemp(prefix="lb2_par_%d_" % rank, dir=shm_dir())
    mismatches += gnu_strip(batch.read_input(probe), pdir, "e2e") != e2e_probe
    shutil.rmtree(pdir, ignore_errors=True)

    # ---- reduce over ranks: totals, max time, every rank's kernel figures
    local = torch.tensor([st["in_bytes"], st["out_bytes"], st["copy_bytes"], st["header_bytes"], st["n_ok"], st["n_unsupported"],
                          float(e2e_in), float(e2e_out), float(e2e_up), float(s_span), float(len(picks) + 1), float(mismatches)],
                         dtype=torch.float64, device="cuda")
    times = torch.tensor([dev_ms, e2e_ms, staged_ms, zc_ms], dtype=torch.float64, device="cuda")
    mine = torch.tensor([cms, pms, dev_ms / a.steps, float(alg), float(st["in_bytes"]), e2e_ms / e2e_steps], dtype=torch.float64, device="cuda")
    allr = torch.zeros(6 * world, dtype=torch.float64, device="cuda")
    if dist:
        dist.all_reduce(local, op=dist.ReduceOp.SUM)
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
        dist.all_gather_into_tensor(allr, mine)
    else:
        allr.copy_(mine)
    tot_in, tot_out, tot_copy, tot_hdr, n_ok, n_uns, te_in, te_out, te_up, te_span, n_par, n_bad = [float(x) for x in local.tolist()]
    dev_ms, e2e_ms, staged_ms, zc_ms = [float(x) for x in times.tolist()]
    per_rank = [{"rank": r, "compact_ms": v[0], "plan_ms": v[1], "step_ms": v[2], "frac": v[3] / 1e9 / (v[0] / 1e3) / peak,
                 "in_gb": v[4] / 1e9, "e2e_ms": v[5]} for r, v in enumerate(allr.cpu().numpy().reshape(world, 6).tolist())]

    if rank == 0:
        ms_per_step = dev_ms / a.steps
        value = tot_in / 1e9 / (ms_per_step / 1e3)
        e2e_value = te_in / 1e9 / (e2e_ms / e2e_steps / 1e3)
        achieved = alg / 1e9 / (cms / 1e3)
        batches_per_step = 1
        if chunked:
            b_, f_ = 0, 0
            while f_ < n:
                g_ = f_ + 1
                while g_ < n and int(corpus.off[g_ + 1] - corpus.off[f_]) <= batch.chunk_bytes:
                    g_ += 1
                b_ += 1; f_ = g_
            batches_per_step = b_
        wkey = "%s:%d:%d:%x" % (a.scaling, a.total_files if a.scaling == "strong" else a.files_per_gpu, world, SEED)
        traffic, tnote = None, "no ncu capture for this workload in profiles/traffic.json"
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                with open(tp) as f:
                    tj = json.load(f)
                if tj.get("workload_key") == wkey:  # a capture of another workload says nothing about this one
                    traffic = tj.get("compact_dram_bytes_per_launch")
                    tnote = tj.get("how")
            except Exception:
                pass
        line = {
            "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": a.steps, "warmup": warm,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
            "dtype": "u8", "data": "synthetic", "config": dict(workload_config(a, world), batches_per_step_rank0=batches_per_step,
                                                               output_ring=("two slots of %.1f GB (input + output exceed HBM)" % (batch.slot_cap / 1e9)) if chunked else None),
            "totals": {"files": int(n_ok), "unsupported_files": int(n_uns), "in_gb": tot_in / 1e9, "out_gb": tot_out / 1e9,
                       "copied_gb": tot_copy / 1e9, "header_gb": tot_hdr / 1e9},
            "roofline": {"bound": "hbm", "kernel": "lb2_compact_kernel" if os.environ.get("LB2_COMPACT_TMA") == "0" else "lb2_compact_tma_kernel",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_note": tnote, "traffic_workload_key": wkey, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg / batches_per_step, "kernel_ms": cms / batches_per_step,
                         "launches_per_step": batches_per_step, "plan_kernel_ms": pms / batches_per_step,
                         "whole_pass_frac": (alg + st["header_bytes"]) / 1e9 / ((cms + pms) / 1e3) / peak,
                         "rank": 0, "min_frac_over_ranks": min(r["frac"] for r in per_rank)},
            "per_rank": per_rank,
            "parity": {"against": "strip --strip-unneeded -o OUT IN (%s), byte for byte" % strip_version(), "files_checked": int(n_par),
                       "mismatches": int(n_bad), "what": "8 size-stratified outputs of every rank's own shard after the timed region + 1 output of the host-buffer path"},
            "e2e": {"value": e2e_value, "unit": "GB/s", "h2d_bytes_per_step": int(te_up), "d2h_bytes_per_step": int(te_out),
                    "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps, "in_bytes_per_step": int(te_in),
                    "workload": "the first %d files (%.2f GB) of each rank's shard -- host memory bounds it" % (ns, s_span / 1e9) if ns < n else "every rank's whole shard",
                    "api": "lb2_strip_host on pinned, device-mapped host arenas on the GPU's NUMA node: kernels pull headers + kept extents "
                           "over PCIe and push stripped files back (dropped sections never cross the bus)",
                    "dma": {"value": te_in / 1e9 / (zc_ms / e2e_steps / 1e3), "ms_per_step": zc_ms / e2e_steps,
                            "api": "LB2_HOST_DMA=1: plan over the mapping, copy-engine upload of the kept ranges only, compaction in HBM, "
                                   "DMA of the output; 256 MB chunks, 3 in flight"},
                    "staged": {"value": te_in / 1e9 / (staged_ms / e2e_steps / 1e3), "ms_per_step": staged_ms / e2e_steps,
                               "h2d_bytes_per_step": int(te_span), "d2h_bytes_per_step": int(te_out),
                               "api": "LB2_HOST_ZEROCOPY=0: cudaMemcpyAsync of whole files in 256 MB chunks on 3 streams"}},
            "gpu_launches": LAUNCHES_PER_BATCH * batches_per_step * a.steps,
            "clocks": clocks,
        }
        assert n_bad == 0, "parity sample failed: %d mismatches" % n_bad
        if world == 1 and not a.no_host_legs:
            line.update(host_legs(a, ctx, corpus, batch, ns, peak))
    ctx.pinned_free(h_in); ctx.pinned_free(h_out)
    batch.close()
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        if dist:
            time.sleep(1.5)  # let the other ranks' NCCL shutdown lines out first: the JSON line is the last thing on stdout
        sys.stdout.flush()
        print(json.dumps(line), flush=True)
        if dist:
            os._exit(0)      # NCCL logs another INFO line from a library destructor at interpreter exit; everything is released
    return 0


def host_legs(a, ctx, corpus, batch, ns, peak):
    """N=1 only: the reference's line and lb2_strip_tree on the SAME /dev/shm tree, and the real build trees."""
    from lambdipy_b200 import strip as S
    out = {}
    n_bytes = int(corpus.sizes[:ns].sum())
    base = tempfile.mkdtemp(prefix="lb2_cpu_", dir=shm_dir())
    try:
        free = shutil.disk_usage(base).free
        if free < 3.2 * n_bytes:
            out["cpu_baseline"] = {"value": None, "unit": "GB/s", "cores": os.cpu_count(), "kind": "reference",
                                   "sample": "skipped: /dev/shm has %.1f GB free, the sample tree needs %.1f GB" % (free / 1e9, 3.2 * n_bytes / 1e9)}
            return out
        master = os.path.join(base, "master")
        os.makedirs(master)

        def dump(i):
            with open(os.path.join(master, "f%05d.so" % i), "wb") as f:
                f.write(batch.read_input(i))

        with ThreadPoolExecutor(8) as ex:  # cudaMemcpy D2H + tmpfs write per file
            list(ex.map(dump, range(ns)))
        r = cpu_lines_on_master(base, master, n_bytes, 2, 1, 1)
        out["cpu_baseline"] = {
            "value": r["parallel_gbs"], "unit": "GB/s", "cores": r["nproc"], "kind": "reference",
            "sample": "the first %d files (%.3f GB) of the corpus as a /dev/shm tree, fresh copy per run, through the reference's line "
                      "`find DIR/ -name \"*.so\" | xargs strip` with -P %d -n 1 (%s), mean of 2 runs after 1 warm-up; serial (1 process, "
                      "as the reference runs it): %.3f GB/s" % (ns, n_bytes / 1e9, r["nproc"], strip_version(), r["serial_gbs"]),
            "serial_value": r["serial_gbs"]}
        # ---- the product call on the same tree: walk + read + H2D + kernels + D2H + in-place write
        gpu = os.path.join(base, "run_gpu")
        tt, sts = [], []
        for _ in range(3):
            shutil.rmtree(gpu, ignore_errors=True)
            copy_tree_parallel(master, gpu)
            t0 = time.perf_counter()
            st = S.strip_tree(gpu, ctx=ctx)
            tt.append(time.perf_counter() - t0); sts.append(st)
        same = trees_identical(os.path.join(base, "run_ref"), gpu)
        best = min(range(len(tt)), key=lambda k: tt[k])
        out["tree"] = {"value": n_bytes / 1e9 / tt[best], "unit": "GB/s", "s": tt[best], "first_call_s": tt[0], "runs_s": tt,
                       "files": ns, "in_gb": n_bytes / 1e9, "fallback_files": int(sts[best]["n_fallback"]), "failed_files": int(sts[best]["n_failed"]),
                       "phases_s": {k: sts[best][k] for k in ("walk_read_s", "gpu_s", "write_s", "fallback_s", "read_cpu_s", "write_cpu_s", "dma_wait_s", "io_threads", "n_batches")},
                       "identical_to_reference_tree": bool(same),
                       "vs_reference_parallel": (n_bytes / 1e9 / tt[best]) / r["parallel_gbs"], "vs_reference_serial": (n_bytes / 1e9 / tt[best]) / r["serial_gbs"],
                       "api": "lb2_strip_tree (the call that replaces project_build.py:260) on a fresh /dev/shm copy of the tree the reference line strips"}
        assert same and sts[best]["n_failed"] == 0, "tree leg: GPU-stripped tree differs from the reference-stripped tree"
    finally:
        shutil.rmtree(base, ignore_errors=True)
    if not a.no_real_trees:
        try:
            out["real_trees"] = real_trees_block(ctx, peak)
        except Exception as e:  # the stand-in wheels are an image detail; the synthetic line must survive their absence
            out["real_trees"] = {"error": repr(e)[:300]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--total-files", type=int, default=TOTAL_FILES, help="strong scaling: files in the whole corpus")
    ap.add_argument("--files-per-gpu", type=int, default=FILES_PER_GPU, help="weak scaling: files per GPU")
    ap.add_argument("--chunk-gb", type=float, default=14.0, help="output-ring chunk when input + output exceed HBM")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-host-legs", action="store_true", help="skip cpu_baseline / tree / real_trees (N=1)")
    ap.add_argument("--no-real-trees", action="store_true")
    ap.add_argument("--profile-mode", action="store_true", help="device-resident steps only (for runs under ncu; not a bench value)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write rank 0's results of the last step to DIR/*.npy: out_sizes and status "
                         "(float64, one per file) and a seeded sample of the stripped bytes (sample_files, sample_bytes as float32)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.impl == "reference":
        return run_reference(a, rank, world)
    if world != a.gpus and world == 1 and a.gpus > 1:
        sys.stderr.write("bench.py: --gpus %d needs torchrun (WORLD_SIZE=1 seen); running 1 GPU\n" % a.gpus)
    return run_b200(a, rank, local_rank, world)


if __name__ == "__main__":
    sys.exit(main())
