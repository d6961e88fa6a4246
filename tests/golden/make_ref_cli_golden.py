#!/usr/bin/env python
"""Runs the original project's `lambdipy build --no-docker` (its click CLI, imported from a lambdipy source
checkout given as the only argument, with its missing third-party imports stubbed) and records, as
tests/golden/ref_cli.json:

  call   the arguments its `build` command passes to install_non_resolved_requirements, the function
         lambdipy_b200.patch replaces (the positional/keyword shape and the values that are not data);
  cases  exit code, printed output and the ./build listing afterwards, for an empty build tree and for
         one holding a single shared object.

tests/test_patch_reference_cli.py checks the replacement against this record.

    python tests/golden/make_ref_cli_golden.py /path/to/lambdipy-source
"""
import json
import os
import shutil
import sys
import tempfile
import types

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import elf_fixtures as F  # noqa: E402


def stub_third_party():
    for name in ("docker", "docker.errors", "requirementslib", "github", "github.GithubException", "github.GitRelease"):
        m = types.ModuleType(name)
        m.Requirement = object
        m.Github = m.InputGitAuthor = m.GitRelease = object
        m.UnknownObjectException = Exception
        m.BuildError = type("BuildError", (Exception,), {})
        m.from_env = lambda *a, **k: None
        m.__path__ = []
        sys.modules[name] = m


def listing(bd):
    out = {}
    for d, dirs, fs in os.walk(bd):
        for f in fs + dirs:
            p = os.path.join(d, f)
            out[os.path.relpath(p, bd)] = "link" if os.path.islink(p) else ("dir" if os.path.isdir(p) else "file")
    return out


def main(src):
    stub_third_party()
    sys.path.insert(0, os.path.abspath(src))
    from click.testing import CliRunner
    import lambdipy.cli as cli

    calls = []
    original = cli.install_non_resolved_requirements

    def recording(*args, **kwargs):
        calls.append({"n_args": len(args), "kwargs": sorted(kwargs), "python_version": args[2],
                      "keep_tests": list(args[3]), "keep_tests_type": type(args[3]).__name__, "no_docker": args[4]})
        return original(*args, **kwargs)

    cli.install_non_resolved_requirements = recording
    tmp = tempfile.mkdtemp()
    fixture = F.build_variants(os.path.join(tmp, "fx"))["c_g"]
    orig_copy = cli.copy_prepared_releases_to_build_directory
    cwd = os.getcwd()
    os.environ["PYTHON_VERSION"] = "3.7"
    cases = {}
    try:
        for case in ("empty_tree", "one_shared_object"):
            run = os.path.join(tmp, case)
            os.makedirs(run)
            os.chdir(run)
            with open("requirements.txt", "w"):
                pass

            def seeded(paths, build_directory="./build"):
                orig_copy(paths, build_directory)
                if case == "one_shared_object":
                    shutil.copy(fixture, os.path.join(build_directory, "mod.so"))

            cli.copy_prepared_releases_to_build_directory = seeded
            r = CliRunner().invoke(cli.cli, ["build", "--no-docker"])
            after = listing("build")
            cases[case] = {"exit_code": r.exit_code, "output": r.output, "listing": after,
                           "stripped": case == "one_shared_object" and os.path.getsize("build/mod.so") < os.path.getsize(fixture)}
            os.chdir(cwd)
    finally:
        os.chdir(cwd)
        shutil.rmtree(tmp)
    assert len(calls) == 2 and calls[0] == calls[1], calls
    with open(os.path.join(HERE, "ref_cli.json"), "w") as f:
        json.dump({"call": calls[0], "cases": cases}, f, indent=1, sort_keys=True)
        f.write("\n")
    print(json.dumps({"call": calls[0], "cases": cases}, indent=1))


if __name__ == "__main__":
    main(sys.argv[1])
