"""bench.py's reference arm runs on CPU (oracle port on the host cores) and must print
exactly one JSON line with the contract's keys; the GPU arm must refuse to run without a GPU."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT, has_gpu

BENCH = os.path.join(ROOT, "bench.py")


def test_reference_arm_prints_one_contract_line():
    p = subprocess.run([sys.executable, BENCH, "--impl", "reference", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("fp32 elements/sec") and d["unit"] == "elements/s"
    assert d["higher_is_better"] is True and d["value"] > 1e8 and d["steps"] == 2 and d["gpu_launches"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert cb["stores"].split(" ")[0] in ("regular", "non-temporal") and cb["stores"] in cb["sample"]   # the store kind is stated
    import bench
    assert d["config"]["workload"] == bench.WORKLOAD        # the same string the GPU arm prints (same_config)
    assert d["e2e"] == {"value": d["value"], "unit": "elements/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_nonzero_ranks_exit_silently():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, BENCH, "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


@pytest.mark.skipif(has_gpu(), reason="checks the no-GPU failure mode")
def test_gpu_arm_refuses_to_run_on_cpu():
    p = subprocess.run([sys.executable, BENCH, "--steps", "1"], capture_output=True, text=True, timeout=300)
    assert p.returncode != 0 and "no CPU fallback" in (p.stderr + p.stdout)


def test_steps_below_one_are_refused():
    p = subprocess.run([sys.executable, BENCH, "--impl", "reference", "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert p.returncode == 2 and "--steps" in p.stderr and p.stdout == ""


def test_dump_outputs_writes_a_seeded_sample_with_its_global_indices(tmp_path):
    import numpy as np
    import torch

    import bench

    n, first = 3 << 20, 5 << 20
    c = torch.arange(first, first + n, dtype=torch.float32)         # exact integers: value == global index
    bench.dump_outputs(str(tmp_path / "a"), c, first, 1, 2)
    bench.dump_outputs(str(tmp_path / "b"), c, first, 1, 2)
    vals, idx = np.load(tmp_path / "a" / "c_rank1.npy"), np.load(tmp_path / "a" / "index_rank1.npy")
    assert vals.dtype == np.float32 and idx.dtype == np.float64
    assert n // 4 < len(vals) == len(idx) <= bench.DUMP_SAMPLE // 2
    assert np.array_equal(vals, idx) and idx.min() >= first and idx.max() < first + n and (np.diff(idx) > 0).all()
    for f in ("c_rank1.npy", "index_rank1.npy"):                     # same arguments, same sample
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes()
    assert 2 * sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 64 << 20   # both ranks together


@pytest.mark.gpu
def test_gpu_arm_times_exactly_the_requested_steps_and_dumps_them(tmp_path):
    import numpy as np

    import oracle

    n = (1 << 20) + 3
    p = subprocess.run([sys.executable, BENCH, "--steps", "7", "--warmup", "3", "--n-per-gpu", str(n), "--no-e2e",
                        "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr
    d = json.loads(p.stdout)
    assert d["steps"] == 7 and d["gpu_launches"] == 7
    want = oracle.vadd(oracle.fill_ctr(n, 0x0A), oracle.fill_ctr(n, 0x0B))
    idx = np.load(tmp_path / "index_rank0.npy").astype(np.int64)
    assert oracle.first_mismatch(np.load(tmp_path / "c_rank0.npy"), want[idx]) == -1


def test_rank_to_device_mapping_spreads_ranks_over_the_sockets():
    """bench.py maps rank -> GPU round-robin over NUMA nodes when there are fewer ranks than GPUs
    (VERDICT r01: four ranks behind one socket got 0.63 e2e efficiency), identity otherwise."""
    import bench

    numa = [0, 0, 0, 0, 1, 1, 1, 1].__getitem__
    assert [bench.device_for_rank(r, 4, 8, numa)[0] for r in range(4)] == [0, 4, 1, 5]
    assert [bench.device_for_rank(r, 2, 8, numa)[0] for r in range(2)] == [0, 4]
    assert bench.device_for_rank(0, 1, 8, numa)[0] == 0
    assert [bench.device_for_rank(r, 8, 8, numa)[0] for r in range(8)] == list(range(8))
    assert [bench.device_for_rank(r, 2, 4, [0, 0, 1, 1].__getitem__)[0] for r in range(2)] == [0, 2]
    # one socket, unknown topology, or an odd split: every rank still gets its own GPU
    assert [bench.device_for_rank(r, 2, 4, lambda i: 0)[0] for r in range(2)] == [0, 1]
    assert [bench.device_for_rank(r, 2, 4, lambda i: -1)[0] for r in range(2)] == [0, 1]
    got = [bench.device_for_rank(r, 5, 6, [0, 0, 0, 0, 1, 1].__getitem__)[0] for r in range(5)]
    assert sorted(got) == sorted(set(got)) and got[:4] == [0, 4, 1, 5]


def test_digest_constants_are_the_oracles():
    import bench
    import oracle

    assert oracle.ctr_vadd_digest(1 << 24) == bench.DIGEST_2P24
    assert oracle.ctr_vadd_digest(1 << 30) == bench.DIGEST_2P30


def test_cli_strong_leg_shows_the_executable_exactly_the_ranks_gpus(tmp_path, monkeypatch):
    """bench.cli_strong: rank 0 runs `vectorAdd --gpus G --n 2^30` on the GPUs the ranks drove (rank order),
    composed with any CUDA_VISIBLE_DEVICES already in force; its JSON is parsed into the bench line."""
    import stat

    import bench

    fake = tmp_path / "vectorAdd"
    fake.write_text("""#!/usr/bin/env python3
import json, os, sys
out = sys.argv[sys.argv.index("--json") + 1]
json.dump({"elements_per_s": 4.7e12, "ms_per_pass": 0.2268, "mismatches": 0, "roofline_frac_of_8TBps_per_gpu": 0.9,
           "digest_sum": "0fd8e36879aed49f", "digest_xor": "0f23c595", "seen": os.environ.get("CUDA_VISIBLE_DEVICES"),
           "argv": sys.argv[1:]}, open(out, "w"))
""")
    fake.chmod(fake.stat().st_mode | stat.S_IEXEC)
    seen = {}
    real_load = json.load

    def spy(f):
        d = real_load(f)
        seen.update(d)
        return d

    monkeypatch.setattr(bench.json, "load", spy)
    monkeypatch.delenv("CUDA_VISIBLE_DEVICES", raising=False)
    r = bench.cli_strong(4, str(fake), [0, 4, 1, 5])
    assert r["digest_ok"] and r["exit_code"] == 0 and r["value"] == 4.7e12 and r["devices"] == [0, 4, 1, 5]
    assert seen["seen"] == "0,4,1,5" and seen["argv"][:6] == ["--mode", "resident", "--gpus", "4", "--n", "2^30"]
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "2,3,6,7,GPU-x,9")          # indices are relative to what is already visible
    bench.cli_strong(2, str(fake), [0, 4])
    assert seen["seen"] == "2,GPU-x"
    assert "error" in bench.cli_strong(1, str(tmp_path / "missing"), [0])     # reported, never fatal
