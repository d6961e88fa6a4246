"""Drop-in check at the CLI level: with lambdipy_b200.patch applied, `lambdipy build --no-docker` reaches our
mirror of install_non_resolved_requirements, and the mirror, called the way the original CLI's `build` command
calls it, prints, exits and leaves ./build as the original CLI did.  The original's behaviour is a record of
running it (tests/golden/ref_cli.json, written by tests/golden/make_ref_cli_golden.py)."""
import contextlib
import io
import json
import os
import shutil
import sys
import types

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "ref_cli.json")


def _listing(bd):
    out = {}
    for d, dirs, fs in os.walk(bd):
        for f in fs + dirs:
            p = os.path.join(d, f)
            out[os.path.relpath(p, bd)] = "link" if os.path.islink(p) else ("dir" if os.path.isdir(p) else "file")
    return out


def test_reference_cli_build_runs_our_strip_step(tmp_path, monkeypatch, variants):
    with open(GOLDEN) as f:
        gold = json.load(f)
    # stand-ins for the installed package: the original CLI module imported the name from project_build, so
    # patch.apply() has to rebind it in both modules
    pkg = types.ModuleType("lambdipy")
    pkg.__path__ = []
    ref_pb, ref_cli = types.ModuleType("lambdipy.project_build"), types.ModuleType("lambdipy.cli")
    ref_pb.install_non_resolved_requirements = ref_cli.install_non_resolved_requirements = lambda *a, **k: None
    pkg.project_build, pkg.cli = ref_pb, ref_cli
    for m in (pkg, ref_pb, ref_cli):
        monkeypatch.setitem(sys.modules, m.__name__, m)
    monkeypatch.setenv("LAMBDIPY_STRIP_BACKEND", "gnu")       # the original's own strip line as backend: no GPU needed
    monkeypatch.setenv("PYTHON_VERSION", "3.7")
    import lambdipy_b200.patch as patch
    from lambdipy_b200 import project_build as mine
    assert patch.apply() is ref_cli
    assert ref_pb.install_non_resolved_requirements is mine.install_non_resolved_requirements
    assert ref_cli.install_non_resolved_requirements is mine.install_non_resolved_requirements

    call = gold["call"]
    assert call["n_args"] == 5 and call["kwargs"] == [] and call["keep_tests_type"] == "tuple"
    strip_line = 'find ./build/ -name "*.so" | xargs strip'
    # an empty tree makes the original's line fail (xargs runs `strip` without arguments, rc 123); with a shared
    # object in ./build it is stripped and the CLI goes on to print "Build done"
    for case, seed in (("empty_tree", None), ("one_shared_object", variants["c_g"])):
        want = gold["cases"][case]
        run = tmp_path / case
        (run / "build").mkdir(parents=True)
        if seed:
            shutil.copy(seed, run / "build" / "mod.so")
        monkeypatch.chdir(run)
        out, code = io.StringIO(), 0
        with contextlib.redirect_stdout(out):
            try:
                ref_cli.install_non_resolved_requirements({}, [], call["python_version"], tuple(call["keep_tests"]), call["no_docker"])
            except SystemExit as e:
                code = e.code
        assert code == want["exit_code"], out.getvalue()
        ref_lines = want["output"].splitlines()
        assert strip_line in ref_lines
        if code == 0:
            assert ref_lines[-1] == "Build done"                  # printed by the CLI after the step returns
            ref_lines = ref_lines[:-1]
        assert out.getvalue().splitlines() == [l for l in ref_lines if l != strip_line]  # same script minus the strip line
        assert _listing(str(run / "build")) == want["listing"]
        if seed:
            assert want["stripped"] and os.path.getsize(run / "build" / "mod.so") < os.path.getsize(seed)
