#!/usr/bin/env python
"""bench.py -- BASELINE.json's headline: fp32 elements/sec on 2^28-element vectorAdd.

    python bench.py --gpus N --steps K --warmup W            # one rank per GPU under torchrun for N>1
    python bench.py --impl reference --gpus N --steps K --warmup W

A "step" is one pass of the hot path: C = A + B over this rank's 2^28-element shard
(weak scaling: every GPU holds 2^28 elements, 3 GiB of operands, far above the 126 MB L2,
so no L2 flush is needed between steps).  One step == one launch of OUR kernel through the
C ABI (include/b200va.h: b200va_add_f32).

ONE JSON line.  Top-level keys are the contract (configs[1] of BASELINE.json):
value        whole-job elements/s with operands resident in HBM (CUDA events, max over ranks)
e2e          the same metric through the host-buffer C-ABI call (b200va_stager_add_f32) on
             pinned host arrays: every step copies A and B to the GPU, adds, copies C back;
             e2e.roofline = the same bytes as plain concurrent whole-array copies, measured
             live on this box at this N (the PCIe / host-DMA ceiling)
e2e_pageable the same call on plain malloc'd arrays -- what the reference's process has --
             first step (page-locks them once) and steady state
roofline     dominant (only) kernel vs the measured HBM copy peak (MEASURED_PEAKS.json)
cpu_baseline / --impl reference
             the oracle port (oracle/vadd_oracle.c: the reference ships no source, so kind =
             "port") timed on this box's host cores, regular AND non-temporal stores, the
             faster reported.  The oracle is never on the product path.
The other BASELINE.json configs that fit a bench run ride in the same line:
strong_2p30  configs[2]: global N = 2^30 sharded over the N ranks (2^30/N per GPU), fixed total
cli_strong_2p30  the same shape through the C++ executable's one-thread-per-GPU path (`vectorAdd --gpus N`),
             run by rank 0 on exactly the GPUs the ranks drove
loop_2p24    configs[4]: 5000 launches of N = 2^24 in 50-launch CUDA graphs on each GPU

--dump-outputs DIR writes what the last timed step returned -- a fixed, seeded sample of C --
so that two builds run with the same arguments (hence the same inputs) can be compared
element for element (see dump_outputs).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "fp32 elements/sec on 2^28-elem vectorAdd"
UNIT = "elements/s"
WORKLOAD = "vectorAdd N=2^28 fp32 per GPU (BASELINE.json configs[1])"     # identical in both arms
INPUTS = "ctr generator (splitmix64 of the global index), seeds 0x0A/0x0B, uniform [0,1)"
N_PER_GPU = 1 << 28
CLOCK_PERIOD_MS = 2.0
STAGE_MODE = 2       # host-path pipeline used for e2e (0 slot streams, 2 lanes: 42.25 vs 42.56 ms, profiles/r01/m_*)
BYTES_PER_ELEM = 12  # 4 read A + 4 read B + 4 write C (SURVEY.md section 8(d))
# oracle.ctr_vadd_digest(1 << 30) / (1 << 24): asserted against the oracle in tests/test_oracle.py
DIGEST_2P30 = (0x0FD8E36879AED49F, 0x0F23C595)
DIGEST_2P24 = (0x003F639456AC9687, 0x064A9499)
READ_ONLY_CEILING_GBPS = 7436.0   # pure read stream (A and B in, nothing out) with the production geometry: profiles/r02/a_channel_skew.jsonl
LINK_ALONE_MS_PER_2P28 = 40.8   # one GPU's PCIe Gen5 x16 link, 2 GiB in + 1 GiB out concurrently (profiles/r01/l_pcie_probe.jsonl)
DUMP_SAMPLE = 1 << 22   # elements of C drawn for --dump-outputs over all ranks: 16 MiB of values + 32 MiB of indices


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while a timed region runs."""

    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown",
               0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown"}

    def __init__(self, cuda_index: int, period_s: float = 0.002):
        self.period_s = period_s
        self.samples: list[int] = []
        self.reason_bits = 0
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        self._h = None
        try:
            import pynvml
            import torch

            pynvml.nvmlInit()
            self._nv = pynvml
            try:
                uuid = "GPU-" + str(torch.cuda.get_device_properties(cuda_index).uuid)
                self._h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                self._h = pynvml.nvmlDeviceGetHandleByIndex(cuda_index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # NVML missing: report clocks as unknown, do not fail the bench
            self._err = repr(e)

    def _loop(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                try:
                    self.reason_bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                except Exception:
                    self.reason_bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
            except Exception:
                pass
            time.sleep(self.period_s)

    def __enter__(self):
        if self._h is not None:
            self._stop.clear()
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        if self._thread is not None:
            self._stop.set()
            self._thread.join()
            self._thread = None

    def summary(self) -> dict:
        if self._h is None or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz,
                "reasons": [n for b, n in self.REASONS.items() if self.reason_bits & b], "samples": len(s)}


def measured_peak() -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, torch copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def ncu_traffic(kernel: str, n: int) -> tuple[float | None, str | None]:
    """dram read+write bytes per launch of THE KERNEL THIS RUN LAUNCHED, from the per-kernel table
    of committed ncu captures (profiles/ncu_summary.json, key "<kernel>@<n>").  None when this
    kernel/size has no capture -- never another kernel's bytes."""
    try:
        table = json.load(open(os.path.join(ROOT, "profiles", "ncu_summary.json")))["kernels"]
        row = table[f"{kernel}@{n}"]
        return float(row["dram_bytes_per_launch"]), row.get("source")
    except Exception:
        return None, None


# --------------------------------------------------------------------------- reference arm
def cpu_baseline_line(n: int, warmup: int, steps: int) -> dict:
    """The oracle port on all the host threads it can use, with the store kind that is faster
    on this host (regular write-allocate vs non-temporal); `value` over `steps` passes of n."""
    import oracle  # the checker/baseline; never imported by the product package

    cfg = oracle.best_cpu_config()
    secs = oracle.time_vadd_mt(n, cfg["threads"], warmup, steps, cfg["nt"])
    v = n * len(secs) / sum(secs)
    tried = {k: f"{d['elements_per_s']:.3e} @ {d['threads']} thr" for k, d in cfg["tried"].items()}
    sample = (f"{steps} passes of C=A+B over 2^{n.bit_length() - 1} fp32 elements (one GPU's shard of the workload), "
              f"{cfg['threads']} host threads ({oracle.num_cpus()} CPUs in the affinity mask, cgroup quota "
              f"{oracle.cpu_quota() or 'none'}), contiguous static partition, stores: {cfg['stores']} "
              f"(faster of {tried} on a 2^26 sample), oracle/vadd_oracle.c (reference ships no source: port of its arithmetic)")
    return {"value": v, "unit": UNIT, "cores": cfg["threads"], "kind": "port", "stores": cfg["stores"], "sample": sample,
            "algorithmic_GBps": v * BYTES_PER_ELEM / 1e9, "secs": secs}


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = args.steps, args.warmup
    cb = cpu_baseline_line(N_PER_GPU, warmup, steps)
    total = sum(cb.pop("secs"))
    value = cb["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": 1e3 * total / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "n_per_gpu": N_PER_GPU, "inputs": INPUTS, "where": "host cores (rank 0 times one GPU's shard)"},
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference ships no source for this path (image k8s.gcr.io/cuda-vector-add:v0.1); "
                "this is the oracle port of its arithmetic on all host threads",
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- our arm
def device_for_rank(local_rank: int, ws: int, ndev: int, numa_of) -> tuple[int, list[int]]:
    """Which GPU a rank drives.  With fewer ranks than GPUs the ranks are spread over the
    sockets (round-robin over NUMA nodes: 0,4,1,5,... on a 2 x 4 box) so that the host-buffer
    path's DMA traffic does not pile onto one socket's memory; identity otherwise."""
    nodes = [numa_of(i) for i in range(ndev)]
    order = list(range(ndev))
    if ws < ndev and len(set(nodes)) > 1 and min(nodes) >= 0:
        by_node: dict[int, list[int]] = {}
        for d, nd in enumerate(nodes):
            by_node.setdefault(nd, []).append(d)
        lists = [by_node[k] for k in sorted(by_node)]
        order = [lst[i] for i in range(max(map(len, lists))) for lst in lists if i < len(lst)]
    return order[local_rank], nodes


class bound_to_node:
    """Runs the calling thread on the CPUs of one NUMA node for the duration of the block, so that
    pages it first-touches land on that node (what `numactl --cpunodebind` gives a process whose
    GPU hangs off that socket).  No-op when the node or its CPU list is unknown."""

    def __init__(self, node: int):
        self.node, self.old = node, None

    def __enter__(self):
        try:
            text = open(f"/sys/devices/system/node/node{self.node}/cpulist").read().strip()
            cpus = set()
            for part in text.split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
            old = os.sched_getaffinity(0)
            if cpus & old:
                os.sched_setaffinity(0, cpus & old)
                self.old = old
        except Exception:
            self.old = None
        return self

    def __exit__(self, *exc):
        if self.old is not None:
            os.sched_setaffinity(0, self.old)


def time_steps(fn, steps: int, stream, sharding, sampler=None):
    """barrier + sync, `steps` calls of fn between two CUDA events on `stream`, sync + barrier;
    returns the MAX over ranks of the elapsed milliseconds."""
    import contextlib

    import torch

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    sharding.barrier()
    torch.cuda.synchronize()
    with (sampler if sampler is not None else contextlib.nullcontext()):
        ev0.record(stream)
        for _ in range(steps):
            fn()
        ev1.record(stream)
        torch.cuda.synchronize()
    sharding.barrier()
    return sharding.max_over_ranks(ev0.elapsed_time(ev1))


def pcie_probe(a, b, c, ha, hb, hc, sharding, reps: int = 3) -> float:
    """The ceiling of the host-buffer step on this box at this rank count: the step's bytes as
    PLAIN whole-array copies (H2D A, H2D B on one stream, D2H C on another, concurrently), every
    rank at once.  Returns the best-of-reps max-over-ranks milliseconds.  torch copies: none of
    our code is on this path."""
    import torch

    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    best = float("inf")
    for _ in range(reps + 1):
        ev0, e_in, e_out = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        torch.cuda.synchronize()
        sharding.barrier()
        cur = torch.cuda.current_stream()
        ev0.record(cur)
        s_in.wait_event(ev0)
        s_out.wait_event(ev0)
        with torch.cuda.stream(s_in):
            a.copy_(ha, non_blocking=True)
            b.copy_(hb, non_blocking=True)
            e_in.record(s_in)
        with torch.cuda.stream(s_out):
            hc.copy_(c, non_blocking=True)
            e_out.record(s_out)
        torch.cuda.synchronize()
        ms = sharding.max_over_ranks(max(ev0.elapsed_time(e_in), ev0.elapsed_time(e_out)))
        best = min(best, ms)
    return best


def cli_strong(gpus: int, cli: str, devices: list[int] | None = None) -> dict:
    """configs[2] once more through the OTHER host path: the C++ executable's one-thread-per-GPU
    sharding (`vectorAdd --gpus G --n 2^30`, host/vectorAdd.cpp), run by rank 0 after the
    torchrun-side measurements so that this path, too, is exercised wherever the bench runs."""
    import subprocess
    import tempfile

    env = dict(os.environ)
    if devices:     # the executable numbers its GPUs 0..G-1: show it exactly the GPUs the ranks drove, in rank order
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        base = [v.strip() for v in visible.split(",")] if visible else None
        env["CUDA_VISIBLE_DEVICES"] = ",".join(base[d] if base else str(d) for d in devices)
    with tempfile.TemporaryDirectory() as d:
        out = os.path.join(d, "cli.json")
        try:
            p = subprocess.run([cli, "--mode", "resident", "--gpus", str(gpus), "--n", "2^30", "--iters", "20", "--json", out],
                               capture_output=True, text=True, timeout=300, env=env)
            r = json.load(open(out))
        except Exception as e:          # reported, never fatal for the contract line
            return {"error": repr(e)[:200]}
    return {"command": f"vectorAdd --mode resident --gpus {gpus} --n 2^30 --iters 20", "devices": devices, "exit_code": p.returncode,
            "value": r["elements_per_s"], "unit": UNIT, "ms_per_step": r["ms_per_pass"], "mismatches": r["mismatches"],
            "frac_of_8TBps_nameplate_per_gpu": r["roofline_frac_of_8TBps_per_gpu"],
            "digest_ok": (int(r["digest_sum"], 16), int(r["digest_xor"], 16)) == DIGEST_2P30}


def dump_outputs(out_dir: str, c, first: int, rank: int, ws: int) -> None:
    """Writes a sample of this rank's C as <out_dir>/c_rank<r>.npy (float32) and the global element
    index of every sampled value as <out_dir>/index_rank<r>.npy (float64, exact below 2^53).  The
    indices are drawn from a generator seeded with the rank, so they only depend on the shard size."""
    import numpy as np
    import torch

    rng = np.random.default_rng(rank)
    idx = np.unique(rng.integers(0, c.numel(), min(c.numel(), DUMP_SAMPLE // ws)))
    vals = c[torch.from_numpy(idx).to(c.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"c_rank{rank}.npy"), vals.astype(np.float32))
    np.save(os.path.join(out_dir, f"index_rank{rank}.npy"), (idx + first).astype(np.float64))


def run_ours(args, emit=print) -> None:
    import torch

    import k8s_gpu_hpa_b200 as pkg
    from k8s_gpu_hpa_b200 import capi, sharding, vector_add as va

    rank, ws, local_rank = sharding.world()
    if ws != args.gpus:
        if ws == 1 and args.gpus > 1:
            raise SystemExit("--gpus N>1 must be launched with torchrun (one rank per GPU)")
        args.gpus = ws
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the vectorAdd hot path has no CPU fallback")
    ndev = torch.cuda.device_count()
    if ndev < ws:
        raise SystemExit(f"{ws} ranks but only {ndev} CUDA devices")
    dev_index, dev_nodes = device_for_rank(local_rank, ws, ndev, lambda i: int(capi.lib.b200va_device_numa_node_of(i)))
    if args.identity_mapping:
        dev_index = local_rank
    torch.cuda.set_device(dev_index)
    dev = torch.device("cuda", dev_index)
    sharding.init("nccl")

    n = args.n_per_gpu
    first = rank * n  # this rank's shard of the global index space [0, ws*n)
    variant = pkg.VARIANTS[args.kernel]
    a = torch.empty(n, dtype=torch.float32, device=dev)
    b = torch.empty(n, dtype=torch.float32, device=dev)
    c = torch.empty(n, dtype=torch.float32, device=dev)
    va.fill_ctr(a, 0x0A, first)
    va.fill_ctr(b, 0x0B, first)
    stream = torch.cuda.current_stream()
    tune = pkg.resolve(variant, n, capi.F_INPUTS_STABLE if args.chain else 0)
    peak, peak_src = measured_peak()
    warm = max(3, args.warmup)

    def step():
        va.add(a, b, c, variant=variant, inputs_stable=args.chain)      # one C-ABI call == one kernel launch

    # ---- device-resident timing: W warm-up, K timed steps, barrier + sync both sides
    for _ in range(warm):
        step()
    sampler = ClockSampler(dev_index, args.clock_period_ms * 1e-3)
    ms_total = time_steps(step, args.steps, stream, sharding, sampler)
    launches = int(sharding.sum_over_ranks(args.steps))

    # ---- correctness of what was timed (outside the timed region): bit-exact recompute in
    # HBM plus the order-independent digest, combined over shards
    bad, first_bad = va.verify(a, b, c)
    bad_total = int(sharding.sum_over_ranks(bad))
    dig = sharding.combine_digests(va.digest(c))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, c, first, rank, ws)      # before the loop leg below rewrites c[:2^24]

    # ---- the ceiling, live: the same launch geometry with the stores removed (a pure read stream of A and B)
    for _ in range(3):
        va.probe("read2", a, b, c)
    probe_steps = max(5, min(args.steps, 50))
    ms_read = time_steps(lambda: va.probe("read2", a, b, c), probe_steps, stream, sharding)
    read_ceiling = 8 * n / (ms_read / probe_steps * 1e-3) / 1e9          # GB/s per GPU (slowest rank)

    # ---- e2e: host buffers through the C ABI, H2D + add + D2H inside the timed region
    e2e = e2e_pageable = None
    if not args.no_e2e:
        # pinned host buffers from the C ABI (pages on the GPU's NUMA node), filled from the
        # device arrays outside the timed region
        pa, pb, pc = va.PinnedBuffer(n, args.wc_inputs), va.PinnedBuffer(n, args.wc_inputs), va.PinnedBuffer(n)
        # [device, gpu's NUMA node, node of A, B, C] for every rank: the pinned buffers should sit next to their GPU
        host_nodes = sharding.gather_ints([dev_index, int(capi.lib.b200va_device_numa_node())] + [p.numa_node for p in (pa, pb, pc)])
        ha, hb, hc = (torch.from_numpy(p.array) for p in (pa, pb, pc))
        ha.copy_(a); hb.copy_(b)
        torch.cuda.synchronize()
        e2e_steps = max(1, min(args.steps, args.e2e_steps))
        with va.Stager(dev_index, args.chunk_elems, args.depth) as stg:
            mode = 1 if args.zero_copy else args.stage_mode
            for _ in range(2):
                stg.add(ha, hb, hc, variant=variant, mode=mode)
            sharding.barrier()
            ms_e2e = 0.0
            for _ in range(e2e_steps):
                ms_e2e += stg.add(ha, hb, hc, variant=variant, mode=mode)
            sharding.barrier()
        ms_e2e = sharding.max_over_ranks(ms_e2e)
        # the step's result must be the right one
        c2 = torch.empty_like(c)
        c2.copy_(hc)
        bad2, _ = va.verify(a, b, c2)
        bad_total += int(sharding.sum_over_ranks(bad2))
        del c2
        # the platform's ceiling for these bytes, live, all ranks at once
        probe_ms = pcie_probe(a, b, c, ha, hb, hc, sharding)
        step_bytes = BYTES_PER_ELEM * n * ws
        link_ms = LINK_ALONE_MS_PER_2P28 * n / (1 << 28)
        e2e = {"value": ws * n * e2e_steps / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": 8 * n * ws,
               "d2h_bytes_per_step": 4 * n * ws, "steps": e2e_steps, "ms_per_step": ms_e2e / e2e_steps,
               "path": "b200va_stager_add_f32 " + {0: "copy-engine pipeline, one stream per slot: H2D(A,B) -> add -> D2H(C) per chunk",
                                                   1: "zero-copy kernel over PCIe",
                                                   2: "copy-engine pipeline, one stream per direction (lanes): H2D(A,B) | add | D2H(C)"}[mode],
               "host_memory": "pinned (b200va_host_alloc, GPU-local NUMA node)" + (", write-combined inputs" if args.wc_inputs else ""),
               "roofline": {"bound": "pcie" if probe_ms <= 1.15 * link_ms else "host-dma",
                            "achieved": step_bytes / (ms_e2e / e2e_steps) / 1e6, "peak": step_bytes / probe_ms / 1e6, "unit": "GB/s",
                            "frac": probe_ms / (ms_e2e / e2e_steps), "probe_ms": probe_ms,
                            "peak_source": "live probe in this run: the step's bytes as plain whole-array torch copies, H2D(A,B) and D2H(C) "
                                           f"concurrently, all {ws} ranks at once, best of 3 (one link alone: {link_ms:.1f} ms, profiles/r01/l_pcie_probe.jsonl)"},
               "device_numaGpu_numaA_B_C_per_rank": host_nodes}
        del ha, hb, hc
        for p in (pa, pb, pc):
            p.free()

        # ---- the same call on the memory the reference's process has: plain malloc'd arrays
        with bound_to_node(int(capi.lib.b200va_device_numa_node())):             # first touch next to the GPU, like a pod pinned to its socket
            qa, qb, qc = (torch.empty(n, dtype=torch.float32) for _ in range(3))     # pageable
            for q in (qa, qb, qc):
                q.numpy()[::1024] = 0.0          # first touch of every page by THIS (bound) thread, not by an OpenMP pool
        pageable_nodes = sharding.gather_ints([int(capi.lib.b200va_host_node_of(q.data_ptr())) for q in (qa, qb, qc)])
        qa.copy_(a); qb.copy_(b)
        torch.cuda.synchronize()
        with va.Stager(dev_index, args.chunk_elems, args.depth) as stg:
            sharding.barrier()
            t0 = time.perf_counter()
            stg.add(qa, qb, qc, variant=variant, mode=capi.STAGE_AUTO)          # first sight: page-locks the three arrays
            first_ms = sharding.max_over_ranks((time.perf_counter() - t0) * 1e3)
            stage_mode = stg.last_mode
            stg.add(qa, qb, qc, variant=variant, mode=capi.STAGE_AUTO)
            sharding.barrier()
            ms_pg = 0.0
            for _ in range(e2e_steps):
                ms_pg += stg.add(qa, qb, qc, variant=variant, mode=capi.STAGE_AUTO)
            sharding.barrier()
        ms_pg = sharding.max_over_ranks(ms_pg)
        c2 = torch.empty_like(c)
        c2.copy_(qc)
        bad3, _ = va.verify(a, b, c2)
        bad_total += int(sharding.sum_over_ranks(bad3))
        del c2, qa, qb, qc
        e2e_pageable = {"value": ws * n * e2e_steps / (ms_pg * 1e-3), "unit": UNIT, "steps": e2e_steps, "ms_per_step": ms_pg / e2e_steps,
                        "first_step_wall_ms": first_ms, "h2d_bytes_per_step": 8 * n * ws, "d2h_bytes_per_step": 4 * n * ws,
                        "host_memory": "pageable (plain malloc: torch.empty on the CPU), as in the reference's ./vectorAdd process",
                        "path": "b200va_stager_add_f32 mode AUTO -> " + {4: "register-once (cudaHostRegister cached by range) + lanes pipeline",
                                                                          3: "pinned bounce ring + copy threads (registration refused)",
                                                                          2: "lanes"}.get(stage_mode, str(stage_mode)),
                        "stage_mode": stage_mode, "numa_A_B_C_per_rank": pageable_nodes,
                        "roofline_frac": probe_ms / (ms_pg / e2e_steps)}

    # ---- BASELINE.json configs[4]: the sustained launch loop, N = 2^24, 5000 launches in 50-launch graphs
    loop = None
    if not args.no_extras:
        m = min(1 << 24, n)
        la, lb, lc = a[:m], b[:m], c[:m]          # views of the resident arrays: [first, first+2^24) of the ctr stream
        iters, batch = 5000, 50
        with va.Loop(la, lb, lc, graph_batch=batch, variant=variant) as lp:
            lp.run(2 * batch)
            torch.cuda.synchronize()
            sharding.barrier()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            ev0.record(stream)
            lp.run(iters)
            ev1.record(stream)
            torch.cuda.synchronize()
            wall_ms = (time.perf_counter() - t0) * 1e3
            ms_loop = ev0.elapsed_time(ev1)
        lbad, _ = va.verify(la, lb, lc)
        bad_total += int(sharding.sum_over_ranks(lbad))
        ms_loop_max = sharding.max_over_ranks(ms_loop)
        ltune = pkg.resolve(variant, m, capi.F_INPUTS_STABLE)      # launches 2..50 of every graph
        loop = {"config": "BASELINE.json configs[4]: sustained 5000-iter loop N=2^24 on each GPU (b200va_loop_*; launches 2..50 of a graph "
                          "run with early loads)",
                "n": m, "iters": iters, "graph_batch": batch, "ms_total": ms_loop_max, "ms_per_iter": ms_loop_max / iters,
                "us_per_iter": 1e3 * ms_loop_max / iters, "value": ws * m * iters / (ms_loop_max * 1e-3), "unit": UNIT,
                "algorithmic_GBps_per_gpu": BYTES_PER_ELEM * m * iters / (ms_loop_max * 1e-3) / 1e9,
                "busy_frac": ms_loop / wall_ms, "wall_ms": wall_ms,
                "note": "L2-assisted: the 192 MiB footprint is 1.5x the 126 MB L2 and the same buffers are re-read every launch, so part "
                        "of the traffic is served from L2 -- not an HBM figure (cold-buffer rate: profiles/r02 sweep_n)",
                "kernel": ltune.kernel_name(), "mismatches": lbad,
                "digest_ok": (va.digest(lc) == DIGEST_2P24) if (first == 0 and m == 1 << 24) else None}
        del la, lb, lc, lp

    # ---- BASELINE.json configs[2]: fixed global N = 2^30 sharded over the ranks (strong scaling)
    strong = None
    if not args.no_extras:
        del a, b, c
        torch.cuda.empty_cache()
        gn = 1 << 30
        lo, hi = pkg.shard_range(gn, ws, rank)
        m = hi - lo
        sa = torch.empty(m, dtype=torch.float32, device=dev)
        sb = torch.empty(m, dtype=torch.float32, device=dev)
        sc = torch.empty(m, dtype=torch.float32, device=dev)
        va.fill_ctr(sa, 0x0A, lo)
        va.fill_ctr(sb, 0x0B, lo)
        s_steps = max(5, min(args.steps, 50))

        def sstep():
            va.add(sa, sb, sc, variant=variant, inputs_stable=args.chain)

        for _ in range(3):
            sstep()
        ms_s = time_steps(sstep, s_steps, stream, sharding)
        sbad, _ = va.verify(sa, sb, sc)
        sbad = int(sharding.sum_over_ranks(sbad))
        bad_total += sbad
        sdig = sharding.combine_digests(va.digest(sc))
        s_ms_step = ms_s / s_steps
        s_ach = BYTES_PER_ELEM * m / (s_ms_step * 1e-3) / 1e9
        strong = {"config": "BASELINE.json configs[2]: vectorAdd N=2^30 fp32 sharded over the ranks (b200va_shard_range), no collective",
                  "global_n": gn, "n_per_gpu": m, "scaling": "strong", "steps": s_steps, "ms_per_step": s_ms_step,
                  "value": gn * s_steps / (ms_s * 1e-3), "unit": UNIT, "per_gpu_GBps": s_ach, "frac": s_ach / peak,
                  "frac_of_8TBps_nameplate_per_gpu": s_ach / 8000.0, "kernel": pkg.resolve(variant, m, capi.F_INPUTS_STABLE if args.chain else 0).kernel_name(),
                  "mismatches": sbad, "digest_sum": f"{sdig[0]:016x}", "digest_xor": f"{sdig[1]:08x}",
                  "digest_ok": sdig == DIGEST_2P30}
        del sa, sb, sc

    if rank != 0:
        return
    if bad_total:
        raise SystemExit(f"bit-exactness check failed: {bad_total} mismatching elements (first at {first_bad})")

    value = ws * n * args.steps / (ms_total * 1e-3)
    ms_per_step = ms_total / args.steps
    achieved = BYTES_PER_ELEM * n / (ms_per_step * 1e-3) / 1e9  # per GPU, GB/s
    kname = tune.kernel_name()
    traffic, traffic_src = ncu_traffic(kname, n)
    grid, block = capi.C.c_uint(), capi.C.c_uint()
    capi.lib.b200va_geometry(capi.C.byref(tune), n, dev_index, capi.C.byref(grid), capi.C.byref(block), None)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": ws, "steps": args.steps,
        "warmup": warm, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "n_per_gpu": n, "global_n": ws * n,
                   "sharding": f"weak scaling: global N = {ws} x 2^28, contiguous shards, no collective on the data path",
                   "rank_to_device": "round-robin over NUMA nodes when ranks < GPUs" if not args.identity_mapping else "identity",
                   "device_numa_nodes": dev_nodes, "kernel": tune.as_dict(), "inputs": INPUTS,
                   "l2": "operands 3 GiB per GPU >> 126 MB L2: inputs larger than L2, no flush between steps",
                   "verified": "bit-exact recompute in HBM after the timed region",
                   "digest_sum": f"{dig[0]:016x}", "digest_xor": f"{dig[1]:08x}"},
        "algorithmic_GBps": value * BYTES_PER_ELEM / 1e9,
        "frac_of_8TBps_nameplate_per_gpu": achieved / 8000.0,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": BYTES_PER_ELEM * n,
                     "read_only_ceiling_GBps": read_ceiling, "frac_of_read_only_ceiling": achieved / read_ceiling,
                     "read_only_ceiling": "measured in this run: b200va_probe_f32(READ2) -- the production launch geometry loading A and B and storing "
                                          f"nothing, {probe_steps} launches (committed reference: {READ_ONLY_CEILING_GBPS:.0f} GB/s = 91 % of the 8.18 TB/s pin "
                                          "rate, profiles/r02/a_channel_skew.jsonl); a harder denominator than the torch copy peak",
                     "kernel": f"b200va::{kname} grid {grid.value} x {block.value} threads (one launch per step)"},
        "clocks": sampler.summary(),
        "gpu_launches": launches,
    }
    if e2e is not None:
        line["e2e"] = e2e
        line["e2e_pageable"] = e2e_pageable
    if strong is not None:
        line["strong_2p30"] = strong
        line["loop_2p24"] = loop
    if strong is not None:
        numa_of = lambda i: int(capi.lib.b200va_device_numa_node_of(i))      # noqa: E731
        devs = list(range(ws)) if args.identity_mapping else [device_for_rank(r, ws, ndev, numa_of)[0] for r in range(ws)]
        line["cli_strong_2p30"] = cli_strong(ws, capi.CLI_PATH, devs)
    if ws == 1 and not args.no_cpu_baseline:
        cb = cpu_baseline_line(n, 1, 5)
        cb.pop("secs")
        line["cpu_baseline"] = cb
    emit(json.dumps(line))


class SingleLineStdout:
    """stdout carries exactly ONE JSON line: while the run is in progress fd 1 points at stderr,
    so library banners (NCCL prints its version on stdout) cannot get in front of it."""

    def __enter__(self):
        sys.stdout.flush()
        self._saved = os.dup(1)
        os.dup2(2, 1)
        return self.emit

    def emit(self, line: str) -> None:
        sys.stdout.flush()
        os.dup2(self._saved, 1)
        print(line, flush=True)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self._saved, 1)
        os.close(self._saved)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--kernel", choices=["auto", "k0", "k1", "k2", "k3"], default="auto")
    ap.add_argument("--n-per-gpu", type=int, default=N_PER_GPU)
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--chunk-elems", type=int, default=0)
    ap.add_argument("--depth", type=int, default=0)
    ap.add_argument("--zero-copy", action="store_true")
    ap.add_argument("--stage-mode", type=int, choices=[0, 2], default=STAGE_MODE)
    ap.add_argument("--wc-inputs", action="store_true", help="write-combined pinned memory for the H2D sources")
    ap.add_argument("--clock-period-ms", type=float, default=CLOCK_PERIOD_MS, help="NVML clock sampling period during the timed region")
    ap.add_argument("--chain", action="store_true", help="launch the timed steps with B200VA_F_INPUTS_STABLE (early loads)")
    ap.add_argument("--identity-mapping", action="store_true", help="rank i drives GPU i even when ranks < GPUs")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip strong_2p30 and loop_2p24")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's C to DIR as .npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to --impl ours")
        run_reference(args)
        return
    try:
        with SingleLineStdout() as emit:
            run_ours(args, emit)
    finally:
        try:
            import torch.distributed as dist

            if dist.is_initialized():
                dist.destroy_process_group()
        except Exception:
            pass


if __name__ == "__main__":
    main()
