"""SURVEY.md section 8(f) row 2 without docker: the runtime layout deploy/Dockerfile assembles
(WORKDIR holding `vectorAdd` + `libb200va.so`, found through $ORIGIN) is built in a scratch
directory and driven by the container command PARSED FROM THE REFERENCE'S DEPLOYMENT
(cuda-test-deployment.yaml:19) -- only its loop bound is rewritten (5000 -> 3)."""
import json
import os
import re
import shutil
import subprocess

import pytest

from conftest import ROOT, has_gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden", "reference_command.json")
PKG = os.path.join(ROOT, "k8s-gpu-hpa_b200")


def reference_command() -> dict:
    return json.load(open(GOLD))


def dockerfile_runtime_copies() -> tuple[str, list[str]]:
    """(WORKDIR, files) of the final stage of deploy/Dockerfile."""
    text = open(os.path.join(ROOT, "deploy", "Dockerfile")).read()
    final = text[text.rindex("\nFROM "):]
    workdir = re.search(r"^WORKDIR\s+(\S+)", final, flags=re.M).group(1)
    copy = re.search(r"^COPY --from=build (.+?) \./$", final, flags=re.M).group(1).split()
    return workdir, [os.path.basename(p) for p in copy]


def test_extractor_reads_the_fixture_back_from_a_deployment(tmp_path):
    """The script that wrote the fixture from the reference's Deployment recovers exactly the
    fixture from a Deployment whose container carries its values."""
    import importlib.util

    import yaml

    spec = importlib.util.spec_from_file_location("mk", os.path.join(os.path.dirname(GOLD), "make_reference_command.py"))
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    ref = reference_command()
    container = {"name": ref["container"], "image": ref["image"], "command": ref["command"],
                 "resources": {"limits": {"nvidia.com/gpu": ref["gpu_limit"]}}}
    path = tmp_path / "cuda-test-deployment.yaml"
    path.write_text(yaml.safe_dump({"apiVersion": "apps/v1", "kind": "Deployment", "metadata": {"name": "cuda-test"},
                                    "spec": {"template": {"spec": {"containers": [container]}}}}))
    assert mk.parse(str(path)) == ref


def test_reference_command_is_the_bash_loop_over_a_zero_argument_binary():
    ref = reference_command()
    assert ref["command"][:2] == ["bash", "-c"] and len(ref["command"]) == 3
    m = re.fullmatch(r"for \(\( c=1; c<=(\d+); c\+\+ \)\); do (\S+); done", ref["command"][2])
    assert m and m.group(1) == "5000" and m.group(2) == "./vectorAdd"       # no arguments, relative to WORKDIR
    assert ref["gpu_limit"] == 1
    workdir, files = dockerfile_runtime_copies()
    assert sorted(files) == ["libb200va.so", "vectorAdd"] and workdir.endswith("/vectorAdd")
    # the image recipe builds the same two artefacts the tests run
    assert "make -C k8s-gpu-hpa_b200" in open(os.path.join(ROOT, "deploy", "Dockerfile")).read()


def test_runtime_layout_resolves_the_library_through_origin(tmp_path):
    """The two files of the image's WORKDIR, copied somewhere else, still find each other."""
    _, files = dockerfile_runtime_copies()
    for f in files:
        shutil.copy2(os.path.join(PKG, f), tmp_path / f)
    out = subprocess.run(["readelf", "-d", str(tmp_path / "vectorAdd")], capture_output=True, text=True).stdout
    assert re.search(r"R(UN)?PATH.*\$ORIGIN", out), out
    env = {k: v for k, v in os.environ.items() if k != "LD_LIBRARY_PATH"}
    ldd = subprocess.run(["ldd", str(tmp_path / "vectorAdd")], capture_output=True, text=True, env=env, cwd=tmp_path).stdout
    line = [l for l in ldd.splitlines() if "libb200va.so" in l][0]
    assert str(tmp_path) in line and "not found" not in ldd, ldd
    assert "libb200va_tune" not in ldd and "oracle" not in ldd


@pytest.mark.gpu
def test_reference_command_drives_the_assembled_layout(tmp_path):
    if not has_gpu():
        pytest.skip("needs a GPU")
    ref = reference_command()
    _, files = dockerfile_runtime_copies()
    for f in files:
        shutil.copy2(os.path.join(PKG, f), tmp_path / f)
    cmd = list(ref["command"])
    cmd[2], n = re.subn(r"c<=5000;", "c<=3;", cmd[2])                     # the ONLY edit: 5000 processes -> 3
    assert n == 1
    env = {k: v for k, v in os.environ.items() if k != "LD_LIBRARY_PATH"}
    p = subprocess.run(cmd, cwd=tmp_path, capture_output=True, text=True, timeout=600, env=env)
    assert p.returncode == 0, p.stderr
    assert p.stdout.count("[Vector addition of 50000 elements]") == 3
    assert p.stdout.count("Test PASSED") == 3 and p.stdout.count("Done") == 3 and p.stderr == ""
