"""Mirror of PackageBuild.create_compressed_tarball (/root/reference/lambdipy/package_build.py:165-172),
called by `lambdipy release` / `prepare --release` (release.py:54) for every published package.

Backend switch:
    LAMBDIPY_TARBALL_BACKEND=b200     default: gzip on the B200 (lambdipy_b200.tarball); raises without one
    LAMBDIPY_TARBALL_BACKEND=python   the reference's own method (tarfile "w:gz"), as saved by patch.apply()
"""
import os

# the reference's PackageBuild.create_compressed_tarball, saved by patch.apply() before it rebinds the name
reference_create_compressed_tarball = None


def _backend():
    backend = os.environ.get("LAMBDIPY_TARBALL_BACKEND", "b200").lower()
    if backend not in ("b200", "python"):
        raise ValueError("LAMBDIPY_TARBALL_BACKEND must be b200 or python (got %r)" % backend)
    return backend


def create_compressed_tarball(self):
    """Same path (~/.lambdipy/build/<git_tag>.tar.gz) and return value as the reference's method."""
    if _backend() == "python":
        if reference_create_compressed_tarball is None:
            raise RuntimeError("LAMBDIPY_TARBALL_BACKEND=python needs the reference method: call lambdipy_b200.patch.apply()")
        return reference_create_compressed_tarball(self)
    from .tarball import create_tarball
    home = os.environ['HOME']
    tarball_path = f'{home}/.lambdipy/build/{self.git_tag()}.tar.gz'
    create_tarball(self.build_directory(), tarball_path)
    return tarball_path
