"""GPU gzip writer: lb2_deflate_device round trips, the release tarball of a stripped build tree, determinism,
windowing and short reads (lambdipy_b200/csrc/deflate.cu, lambdipy_b200/tarball.py)."""
import ctypes as C
import glob
import gzip
import io
import os
import random
import shutil
import subprocess
import sys
import tarfile
import zlib

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from lambdipy_b200 import _native as N  # noqa: E402
from lambdipy_b200 import tarball as T  # noqa: E402

pytestmark = pytest.mark.gpu
S = 65536


@pytest.fixture(scope="module")
def ctx():
    with N.Context(0) as c:
        yield c


def inflate(raw):
    d = zlib.decompressobj(-15)
    out = d.decompress(raw) + d.flush()
    assert d.eof and not d.unused_data
    return out


def _some_so():
    import numpy
    libs = sorted(glob.glob(os.path.join(os.path.dirname(numpy.__file__), "**", "*.so"), recursive=True),
                  key=os.path.getsize)
    with open(libs[-1], "rb") as f:
        return f.read()[:3 << 20]


def _cases():
    rnd = random.Random(5)
    cross = bytearray(rnd.randbytes(2 * S))
    cross[S:S + 400] = cross[S - 32768:S - 32768 + 400]   # a match exactly 32 768 bytes back, across the boundary
    text = b"".join(b"line %d: the quick brown fox jumps over the lazy dog %d\n" % (i, i * i % 97) for i in range(40000))
    return {
        "empty": b"", "one": b"x", "S-1": rnd.randbytes(S - 1), "S": bytes(S), "S+1": b"ab" * (S // 2) + b"c",
        "zeros_1M": bytes(1 << 20), "repeated": b"\x7f" * 777777, "cross_32k": bytes(cross), "text": text,
        "so_slice": _some_so(),
    }


@pytest.mark.parametrize("name", list(_cases()))
def test_deflate_roundtrip(ctx, name):
    data = _cases()[name]
    raw, crc, st = T.deflate_bytes(ctx, data)
    assert inflate(raw) == data
    assert crc == zlib.crc32(data)
    assert st["in_bytes"] == len(data) and st["out_bytes"] == len(raw)


def test_deflate_random_does_not_grow(ctx):
    data = random.Random(8).randbytes(8 << 20)
    raw, crc, _ = T.deflate_bytes(ctx, data)
    assert inflate(raw) == data and crc == zlib.crc32(data)
    assert len(raw) <= len(data) * 1.0005 + 64


def test_deflate_incompressible_80mb(ctx):
    """~1 250 stored chunks in one call: their concatenation needs more than 5 tiles per chunk."""
    data = random.Random(80).randbytes(80 << 20)
    raw, crc, st = T.deflate_bytes(ctx, data)
    assert inflate(raw) == data and crc == zlib.crc32(data)
    assert len(raw) <= len(data) * 1.0005 + 64


def test_deflate_uses_distance_32768(ctx):
    """4 000 bytes repeated exactly 32 768 bytes back, across a chunk boundary, in random data: only a match of
    distance 32 768 can remove them, and it must."""
    rnd = random.Random(6)
    base = bytearray(rnd.randbytes(2 * S))
    copied = bytearray(base)
    copied[S:S + 4000] = copied[S - 32768:S - 32768 + 4000]
    raw_copy, _, _ = T.deflate_bytes(ctx, bytes(copied))
    raw_base, _, _ = T.deflate_bytes(ctx, bytes(base))
    assert inflate(raw_copy) == bytes(copied)
    assert len(raw_copy) <= len(raw_base) - 3000, (len(raw_copy), len(raw_base))


def test_deflate_history_and_continuation(ctx):
    """A non-final call ends with a sync flush; the next call, primed with the last 32 KiB, continues the stream."""
    data = _cases()["so_slice"]
    cut = 5 * S + 123
    a, ca, _ = T.deflate_bytes(ctx, data[:cut], final=False)
    b, cb, _ = T.deflate_bytes(ctx, data[cut:], history=data[:cut], final=True)
    assert a.endswith(b"\x00\x00\xff\xff")
    assert inflate(a + b) == data
    assert (ca, cb) == (zlib.crc32(data[:cut]), zlib.crc32(data[cut:]))


def test_deflate_deterministic(ctx):
    data = _cases()["so_slice"]
    assert T.deflate_bytes(ctx, data)[0] == T.deflate_bytes(ctx, data)[0]


def test_gzip_bytes(ctx):
    data = _cases()["text"]
    gz = T.gzip_bytes(ctx, data)
    assert gzip.decompress(gz) == data


# ---------------------------------------------------------------- the release tarball of a stripped tree
@pytest.fixture(scope="module")
def config2(tmp_path_factory):
    import measure_configs as MC
    from lambdipy_b200 import strip as Sx
    d = str(tmp_path_factory.mktemp("config2"))
    MC.copy_tree(MC.TREES["config2_numpy+scipy+sklearn+PIL"], d)
    Sx.strip_tree(d)
    bio = io.BytesIO()
    with tarfile.open(fileobj=bio, mode="w") as tar:
        for p in glob.glob(f"{d}/*"):
            tar.add(p, arcname=os.path.basename(p))
    return d, bio.getvalue()


def test_tarball_config2(ctx, config2, tmp_path):
    d, tar_bytes = config2
    out = str(tmp_path / "pkg.tar.gz")
    st = T.create_tarball(d, out, ctx)
    with open(out, "rb") as f:
        gz = f.read()
    assert gzip.decompress(gz) == tar_bytes
    if shutil.which("gzip"):
        subprocess.run(["gzip", "-t", out], check=True)
    x = tmp_path / "x"
    with tarfile.open(out, "r:gz") as tar:
        tar.extractall(x)
    for p in glob.glob(f"{d}/**", recursive=True):
        q = x / os.path.relpath(p, d)
        assert q.exists() or q.is_symlink()
        if os.path.isfile(p) and not os.path.islink(p):
            with open(p, "rb") as a, open(q, "rb") as b:
                assert a.read() == b.read()
    z9 = len(zlib.compress(tar_bytes, 9))
    assert st["out_bytes"] <= 1.06 * z9, (st["out_bytes"], z9)


def test_tarball_window_independent(ctx, config2, tmp_path, monkeypatch):
    d, _ = config2
    (tmp_path / "a").mkdir()
    (tmp_path / "b").mkdir()
    a, b = str(tmp_path / "a" / "pkg.tar.gz"), str(tmp_path / "b" / "pkg.tar.gz")   # same FNAME in the header
    T.create_tarball(d, a, ctx)
    monkeypatch.setenv("LB2_GZ_WINDOW_MB", "1")
    st = T.create_tarball(d, b, ctx)
    assert st["n_windows"] > 1
    with open(a, "rb") as fa, open(b, "rb") as fb:
        ga, gb = fa.read(), fb.read()
    assert ga[:4] == gb[:4] and ga[8:] == gb[8:]     # all but MTIME


def test_device_corpus_arena_roundtrip(ctx):
    """An HBM-resident synthetic corpus arena compressed in place, as two windows: the second call reads its
    32 KiB history straight from the arena."""
    from lambdipy_b200.corpus import Corpus
    from lambdipy_b200.device import DeviceBatch
    batch = DeviceBatch.from_corpus(ctx, Corpus(8, seed=3, max_size=1 << 20))
    try:
        n = int(batch.off[-1])
        host = (C.c_char * batch.in_bytes)()
        batch.read_input_arena(host)
        data = host.raw[:n]
        half = (n // 2) // S * S
        a, ca, _ = T.deflate_device(ctx, batch.d_in, half, 0, final=False)
        b, cb, _ = T.deflate_device(ctx, batch.d_in + half, n - half, half, final=True)
        assert inflate(a + b) == data
        assert (ca, cb) == (zlib.crc32(data[:half]), zlib.crc32(data[half:]))
    finally:
        batch.close()


def test_strip_then_tarball_matches_python_backend(ctx, config2, tmp_path):
    d, tar_bytes = config2
    out = str(tmp_path / "g.tar.gz")
    T.create_tarball(d, out, ctx)
    ref = str(tmp_path / "r.tar.gz")
    with tarfile.open(ref, "w:gz") as tar:
        for p in glob.glob(f"{d}/*"):
            tar.add(p, arcname=os.path.basename(p))
    with open(out, "rb") as a, open(ref, "rb") as b:
        assert gzip.decompress(a.read()) == gzip.decompress(b.read())


def test_truncated_file_gives_io_error(ctx, tmp_path):
    d = tmp_path / "t"
    d.mkdir()
    (d / "big.bin").write_bytes(os.urandom(300000))
    segs = T.record_tar(str(d))
    (d / "big.bin").write_bytes(b"short")
    out = str(tmp_path / "o.tar.gz")
    arr = (N.GzSegment * len(segs))()
    keep = []
    for i, s in enumerate(segs):
        if isinstance(s, bytes):
            b = C.create_string_buffer(s, len(s))
            keep.append(b)
            arr[i] = N.GzSegment(C.cast(b, C.c_void_p), None, len(s))
        else:
            arr[i] = N.GzSegment(None, os.fsencode(s[0]), s[1])
    hdr = T.gzip_header(out)
    rc = ctx.lib.lb2_gzip_segments(ctx.h, arr, len(segs), os.fsencode(out), hdr, len(hdr), None)
    assert rc == N.LB2_E_IO
    assert not os.path.exists(out)
