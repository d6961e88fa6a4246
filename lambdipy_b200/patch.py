"""Drop-in installation: make an installed `lambdipy` use the B200 strip path, CLI unchanged.

    import lambdipy_b200.patch; lambdipy_b200.patch.apply()      # or: python -m lambdipy_b200.patch build ...

`install_non_resolved_requirements` is replaced -- in lambdipy.project_build and in
lambdipy.cli, which imported the name (/root/reference/lambdipy/cli.py:11-16) -- and, when
lambdipy.package_build is loaded, PackageBuild.create_compressed_tarball (GPU gzip; package_build.py).  `lambdipy build`,
its options, PackageBuild and every other function keep running the reference's own code.
"""
import os
import sys


def apply():
    import lambdipy.cli as cli
    import lambdipy.project_build as ref
    from . import project_build as mine
    ref.install_non_resolved_requirements = mine.install_non_resolved_requirements
    cli.install_non_resolved_requirements = mine.install_non_resolved_requirements
    # release tarballs (package_build.py:165-172, called from release.py:54); the real CLI imports the module
    # (cli.py:11), stand-in packages may not have it
    ref_pkg = sys.modules.get("lambdipy.package_build")
    if ref_pkg is not None:
        from . import package_build as mine_pkg
        method = ref_pkg.PackageBuild.create_compressed_tarball
        if method is not mine_pkg.create_compressed_tarball:
            mine_pkg.reference_create_compressed_tarball = method
            ref_pkg.PackageBuild.create_compressed_tarball = mine_pkg.create_compressed_tarball
    # `lambdipy build` spends seconds resolving, downloading and copying packages before it reaches the
    # strip step (cli.py:52-67): create the CUDA context behind that, not in front of the strip
    if os.environ.get("LAMBDIPY_B200_EAGER_WARMUP", "1") != "0":
        try:
            mine.warmup()
        except ValueError:
            pass
    return cli


def main(argv=None):
    cli = apply()
    sys.argv = ["lambdipy"] + list(sys.argv[1:] if argv is None else argv)
    return cli.cli()


if __name__ == "__main__":
    main()
