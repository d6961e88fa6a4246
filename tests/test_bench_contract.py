"""bench.py contract checks: the reference arm runs the reference's own pipeline on host cores and prints
ONE JSON line with the agreed keys; --steps is validated; --dump-outputs writes a fixed, bounded sample of
what the timed path returned (on the GPU: equal to the oracle's outputs and the same from run to run)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--total-files", "96", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-500:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "GB/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["metric"].startswith("ELF-strip GB/s") and d["dtype"] == "u8" and d["data"] == "synthetic"
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] == os.cpu_count()
    assert d["cpu_baseline"]["serial_value"] > 0 and "xargs" in d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--steps" in r.stderr


def test_dump_sample_is_fixed_and_bounded(tmp_path):
    import numpy as np
    import bench
    files = bench.dump_files(10000)
    assert files == bench.dump_files(10000) and len(set(files)) == len(files) == bench.DUMP_FILES
    assert bench.dump_files(5) == [0, 1, 2, 3, 4]
    rng = np.random.default_rng(3)
    sizes = [0, 1, 100, 5000, 40000, 300000] + [int(s) for s in rng.integers(1, 8 << 20, size=len(files) - 6)]
    outputs = {i: rng.integers(0, 256, size=s, dtype=np.uint8).tobytes() for i, s in zip(files, sizes)}
    bench.write_dump(str(tmp_path / "d"), np.array([7, 8], dtype=np.uint64), np.array([0, 6], dtype=np.int32), files, outputs)
    got = {f[:-4]: np.load(str(tmp_path / "d" / f)) for f in os.listdir(tmp_path / "d")}
    assert sorted(got) == ["out_sizes", "sample_bytes", "sample_files", "status"]
    assert got["out_sizes"].dtype == np.float64 and list(got["out_sizes"]) == [7, 8] and list(got["status"]) == [0, 6]
    assert got["sample_bytes"].dtype == np.float32 and list(got["sample_files"]) == files
    assert sum(x.nbytes for x in got.values()) <= 64 << 20
    want = np.concatenate([bench.dump_sample(i, outputs[i]) for i in files])
    assert (got["sample_bytes"] == want).all()
    big = outputs[files[-1]]
    s = bench.dump_sample(files[-1], big)
    assert len(s) == 2 * bench.DUMP_EDGE + bench.DUMP_WINDOWS * bench.DUMP_WINDOW
    assert s[:bench.DUMP_EDGE].tobytes() == big[:bench.DUMP_EDGE] and s[bench.DUMP_EDGE:2 * bench.DUMP_EDGE].tobytes() == big[-bench.DUMP_EDGE:]
    assert (bench.dump_sample(files[-1], big) == s).all()
    assert bench.dump_sample(0, b"").size == 0 and bench.dump_sample(0, b"\x05").tolist() == [5, 5]


@pytest.mark.gpu
def test_dump_outputs_are_what_the_timed_path_computed(tmp_path):
    """bench.py --dump-outputs on a small corpus: the dumped sizes, status and sampled bytes equal the oracle's
    stripped files, the JSON line reports the --steps it was given, and a second run dumps the same arrays."""
    import numpy as np
    import bench
    import oracle_lib
    from lambdipy_b200.corpus import Corpus
    dumps = []
    for run in range(2):
        d = str(tmp_path / ("d%d" % run))
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--total-files", "40", "--steps", "3", "--warmup", "1",
                            "--no-host-legs", "--dump-outputs", d], capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == 3 and line["gpu_launches"] == bench.LAUNCHES_PER_BATCH * 3
        dumps.append({f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)})
    assert sorted(dumps[0]) == sorted(dumps[1]) and all((dumps[0][k] == dumps[1][k]).all() for k in dumps[0])
    oracle = oracle_lib.load()
    corpus = Corpus(40, seed=bench.SEED)
    outs = []
    for i in range(len(corpus)):
        rc, out = oracle.strip(corpus.materialize(i))
        assert rc == 0
        outs.append(out)
    got = dumps[0]
    assert list(got["out_sizes"]) == [len(o) for o in outs] and not got["status"].any()
    files = [int(i) for i in got["sample_files"]]
    assert files == bench.dump_files(len(corpus))
    assert (got["sample_bytes"] == np.concatenate([bench.dump_sample(i, outs[i]) for i in files])).all()
