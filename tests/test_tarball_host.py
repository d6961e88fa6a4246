"""Host side of the GPU tarball path: the recorded tar stream, the gzip header, the backend switch and
patch.apply() (no GPU needed)."""
import glob
import gzip
import io
import os
import subprocess
import sys
import tarfile
import types

import pytest

from lambdipy_b200 import _native as N
from lambdipy_b200 import package_build as PB
from lambdipy_b200 import tarball as T


@pytest.fixture
def tree(tmp_path):
    d = tmp_path / "build"
    (d / "pkg" / "sub").mkdir(parents=True)
    (d / "empty_dir").mkdir()
    for name, size in [("e", 0), ("one", 1), ("b511", 511), ("b512", 512), ("b513", 513)]:
        (d / "pkg" / name).write_bytes(os.urandom(size))
    (d / "pkg" / ("n" * 120)).write_bytes(b"long name")
    (d / "pkg" / "ünïcødé.txt").write_bytes(b"non-ascii")
    os.symlink("one", d / "pkg" / "file_link")
    os.symlink("sub", d / "pkg" / "dir_link")
    os.link(d / "pkg" / "b513", d / "pkg" / "hard")
    (d / ".hidden").write_bytes(b"dotfile")
    (d / "top.py").write_bytes(b"print(1)\n")
    return str(d)


def _tarfile_bytes(d):
    bio = io.BytesIO()
    with tarfile.open(fileobj=bio, mode="w") as tar:
        for p in glob.glob(f"{d}/*"):
            tar.add(p, arcname=os.path.basename(p))
    return bio.getvalue()


def test_recorded_segments_equal_tarfile(tree):
    segs = T.record_tar(tree)
    assert T.materialize(segs) == _tarfile_bytes(tree)
    assert any(isinstance(s, tuple) for s in segs)
    with tarfile.open(fileobj=io.BytesIO(T.materialize(segs))) as tar:
        names = tar.getnames()
    assert ".hidden" not in names and "pkg/" + "n" * 120 in names and "pkg/ünïcødé.txt" in names


def test_gzip_header_matches_tarfile(tmp_path):
    path = str(tmp_path / "pkg-1.0.tar.gz")
    with tarfile.open(path, "w:gz"):
        pass
    with open(path, "rb") as f:
        ref = f.read()
    mine = T.gzip_header(path)
    assert mine[:4] == ref[:4] and mine[9:] == ref[9:len(mine)]
    assert mine[8] == 0 and ref[8] == 2   # XFL: tarfile writes level 9


class _StandIn:
    def __init__(self, d, tag):
        self.d, self.tag = d, tag

    def build_directory(self):
        return self.d

    def git_tag(self):
        return self.tag

    def create_compressed_tarball(self):   # what the reference's method does (package_build.py:165-172)
        home = os.environ['HOME']
        tarball_path = f'{home}/.lambdipy/build/{self.git_tag()}.tar.gz'
        with tarfile.open(tarball_path, "w:gz") as tar:
            for path in glob.glob(f'{self.build_directory()}/*'):
                tar.add(path, arcname=os.path.basename(path))
        return tarball_path


def _install_standins(monkeypatch):
    ref_pb, ref_cli = types.ModuleType("lambdipy.project_build"), types.ModuleType("lambdipy.cli")
    ref_pkg, pkg = types.ModuleType("lambdipy.package_build"), types.ModuleType("lambdipy")
    cls = type("PackageBuild", (_StandIn,), {})
    ref_pkg.PackageBuild = cls
    ref_pb.install_non_resolved_requirements = ref_cli.install_non_resolved_requirements = lambda *a, **k: None
    pkg.project_build, pkg.cli, pkg.package_build = ref_pb, ref_cli, ref_pkg
    for m in (pkg, ref_pb, ref_cli, ref_pkg):
        monkeypatch.setitem(sys.modules, m.__name__, m)
    monkeypatch.setattr(PB, "reference_create_compressed_tarball", None)
    monkeypatch.setenv("LAMBDIPY_B200_EAGER_WARMUP", "0")
    return cls


def test_patch_rebinds_and_python_backend_matches_reference(tree, tmp_path, monkeypatch):
    cls = _install_standins(monkeypatch)
    original = cls.create_compressed_tarball
    from lambdipy_b200 import patch
    patch.apply()
    patch.apply()   # idempotent: the saved original stays the reference's
    assert cls.create_compressed_tarball is PB.create_compressed_tarball
    assert PB.reference_create_compressed_tarball is original
    monkeypatch.setenv("HOME", str(tmp_path))
    (tmp_path / ".lambdipy" / "build").mkdir(parents=True)
    monkeypatch.setenv("LAMBDIPY_TARBALL_BACKEND", "python")
    path = cls(tree, "pkg-1.0").create_compressed_tarball()
    assert path == f"{tmp_path}/.lambdipy/build/pkg-1.0.tar.gz"
    with open(path, "rb") as f:
        assert gzip.decompress(f.read()) == _tarfile_bytes(tree)


def test_patch_unchanged_without_package_build(monkeypatch):
    cls = _install_standins(monkeypatch)
    monkeypatch.delitem(sys.modules, "lambdipy.package_build")
    original = cls.create_compressed_tarball
    from lambdipy_b200 import patch
    patch.apply()
    assert cls.create_compressed_tarball is original
    assert PB.reference_create_compressed_tarball is None


@pytest.mark.skipif(os.path.exists("/dev/nvidia0"), reason="checks the behaviour without a GPU")
def test_b200_backend_raises_without_gpu(tree, tmp_path, monkeypatch):
    if not os.path.exists(N.LIB_PATH):
        pytest.skip("library not built")
    monkeypatch.setenv("HOME", str(tmp_path))
    monkeypatch.setenv("LAMBDIPY_TARBALL_BACKEND", "b200")
    with pytest.raises(N.NativeError):
        PB.create_compressed_tarball(_StandIn(tree, "x"))


def test_sass_lists_deflate_kernel():
    if not os.path.exists(N.LIB_PATH):
        pytest.skip("library not built")
    cuobjdump = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not installed")
    out = subprocess.run([cuobjdump, "-sass", N.LIB_PATH], capture_output=True, text=True, check=True).stdout
    assert "lb2_deflate_chunk_kernel" in out
