#!/usr/bin/env python
"""Grouped streaming ops (b200va_stream_grouped) on one GPU against the per-item launches they
replace.  One JSON line per measurement on stdout, and into OUT/<workload>.jsonl with --out.

  W1  5000 items x 50,000 f32, add (the reference loop, distinct data per item)
      vs 5000 b200va_add_f32 calls, plain and captured once into a CUDA graph
  W2  items of 2^12 .. 2^22 f32, K = 2^28 / n of them, add
      vs the K single launches in a graph, and one b200va_stream over 2^28 elements
  W3  seeded log-uniform sizes 1 .. 2^22, total ~2^28, every 16th item mixed-phase, add
      vs per-item b200va_stream launches in a graph
  W4  every op x dtype, items of 2^16 elements, 1 GiB per array in total
      vs one b200va_stream over the same 1 GiB array (the tools/stream_bench.py shape)
  W5  host wall clock of the enqueue alone, count = 1, 100, 800, 5000 items of 64 f32

Timing: CUDA events around each call (W5: host clock, no synchronise inside the window),
warm-up first, >= 20 reps, median and best.  Item arrays are built once, outside the timed
region.  W1-W4 touch >= 4 x L2 per call, so every call runs cold.  Byte counts are those of
stream_bench.py: 2 (copy, scale) or 3 (add, triad) arrays x element size x elements.
B200VA_GROUPED_GEOMETRY="threads,unroll,capacity" with --lib tune selects a candidate geometry.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import oracle  # noqa: E402
from k8s_gpu_hpa_b200 import capi  # noqa: E402

TORCH = {"f32": torch.float32, "f64": torch.float64, "f16": torch.float16, "bf16": torch.bfloat16}
ES = {"f32": 4, "f64": 8, "f16": 2, "bf16": 2}
ARRAYS = {"copy": 2, "scale": 2, "add": 3, "triad": 3}
L2 = 126 * 10**6
REPS, WARM = 20, 3

LIB = capi.lib
OUT = None
TAG = {}


def emit(workload, **kw):
    rec = {"workload": workload, **TAG, **kw}
    line = json.dumps(rec)
    print(line, flush=True)
    if OUT:
        with open(os.path.join(OUT, f"{workload.split('_')[0]}.jsonl"), "a") as f:
            f.write(line + "\n")


def stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def time_events(fn, reps=REPS, warm=WARM):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    ms.sort()
    return ms[len(ms) // 2], ms[0]


def rates(ms_med, ms_best, count, elems, nbytes):
    return {"us_per_call_median": ms_med * 1e3, "us_per_call_best": ms_best * 1e3, "us_per_item": ms_med * 1e3 / max(count, 1),
            "elements_per_s": elems / (ms_med * 1e-3), "TBps": nbytes / (ms_med * 1e-3) / 1e12,
            "TBps_best": nbytes / (ms_best * 1e-3) / 1e12}


def items_of(op, a, b, c, spans):
    """ctypes item array for spans (a_off, b_off, c_off, n) of flat tensors a, b, c."""
    es = a.element_size()
    arr = (capi.Item * len(spans))()
    for i, (oa, ob, oc, n) in enumerate(spans):
        arr[i] = capi.Item(a.data_ptr() + oa * es, b.data_ptr() + ob * es if op in ("add", "triad") else None,
                           c.data_ptr() + oc * es, n)
    return arr


def grouped(op, dt, arr, s=0.0):
    rc = LIB.b200va_stream_grouped(capi.OPS[op], capi.DTYPES[dt], arr, len(arr), s, stream_ptr())
    if rc != capi.OK:
        raise capi.B200VAError(rc, "b200va_stream_grouped")


def graph_of(fn):
    """fn() captured once into a CUDA graph (the capture stream is the current stream inside)."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    torch.cuda.synchronize()
    return g


def host(t, dt, lo, n):
    x = t[lo:lo + n]
    return x.view(torch.int16).cpu().numpy().view(np.uint16) if dt in ("f16", "bf16") else x.cpu().numpy()


def spot_check(op, dt, a, b, c, spans, s=0.0, picks=(0, -1)):
    """First mismatch (-1 = none) over a few items against the oracle."""
    for k in picks:
        oa, ob, oc, n = spans[k]
        want = oracle.stream(op, dt, host(a, dt, oa, n), host(b, dt, ob, n) if op in ("add", "triad") else None, s)
        bad = oracle.first_mismatch_bits(host(c, dt, oc, n), want, dt)
        if bad >= 0:
            return {"item": k if k >= 0 else len(spans) + k, "index": bad}
    return -1


def ctr_arrays(total):
    a = torch.empty(total, dtype=torch.float32, device="cuda")
    b, c = torch.empty_like(a), torch.zeros_like(a)
    for t, seed in ((a, 0x0A), (b, 0x0B)):
        rc = LIB.b200va_fill_ctr_f32(t.data_ptr(), total, seed, 0, stream_ptr())
        assert rc == capi.OK
    return a, b, c


def per_item_add(a, b, c, spans):
    pa, pb, pc = a.data_ptr(), b.data_ptr(), c.data_ptr()
    args = [(pa + oa * 4, pb + ob * 4, pc + oc * 4, n) for oa, ob, oc, n in spans]

    def run():
        st = stream_ptr()
        for x, y, z, n in args:
            LIB.b200va_add_f32(x, y, z, n, 0, st)
    return run


def per_item_stream(a, b, c, spans):
    pa, pb, pc = a.data_ptr(), b.data_ptr(), c.data_ptr()
    args = [(pa + oa * 4, pb + ob * 4, pc + oc * 4, n) for oa, ob, oc, n in spans]

    def run():
        st = stream_ptr()
        for x, y, z, n in args:
            LIB.b200va_stream(2, 0, x, y, z, n, 0.0, st)
    return run


def w1():
    k, n = 5000, 50000
    spans = [(i * n, i * n, i * n, n) for i in range(k)]
    a, b, c = ctr_arrays(k * n)
    nbytes, cold = 12 * k * n, 12 * k * n >= 4 * L2
    arr = items_of("add", a, b, c, spans)
    med, best = time_events(lambda: grouped("add", "f32", arr))
    emit("W1_grouped", items=k, n=n, cold=cold, **rates(med, best, k, k * n, nbytes), first_mismatch=spot_check("add", "f32", a, b, c, spans, picks=(0, 799, 800, -1)))
    c.zero_()
    loop = per_item_add(a, b, c, spans)
    med, best = time_events(loop, reps=REPS, warm=1)
    emit("W1_single_plain", items=k, n=n, cold=cold, **rates(med, best, k, k * n, nbytes), first_mismatch=spot_check("add", "f32", a, b, c, spans))
    g = graph_of(loop)
    c.zero_()
    med, best = time_events(g.replay)
    emit("W1_single_graph", items=k, n=n, cold=cold, **rates(med, best, k, k * n, nbytes), first_mismatch=spot_check("add", "f32", a, b, c, spans))


def w2(logs):
    total = 1 << 28
    a, b, c = ctr_arrays(total)
    nbytes = 12 * total
    med, best = time_events(lambda: LIB.b200va_stream(2, 0, a.data_ptr(), b.data_ptr(), c.data_ptr(), total, 0.0, stream_ptr()))
    emit("W2_one_array", n=total, cold=True, **rates(med, best, 1, total, nbytes))
    for lg in logs:
        n = 1 << lg
        k = total // n
        spans = [(i * n, i * n, i * n, n) for i in range(k)]
        arr = items_of("add", a, b, c, spans)
        c.zero_()
        med, best = time_events(lambda: grouped("add", "f32", arr))
        emit("W2_grouped", items=k, n=n, cold=True, **rates(med, best, k, total, nbytes), first_mismatch=spot_check("add", "f32", a, b, c, spans))
        if os.environ.get("GROUPED_BENCH_SKIP_SINGLE"):
            continue
        g = graph_of(per_item_add(a, b, c, spans))
        c.zero_()
        med, best = time_events(g.replay)
        emit("W2_single_graph", items=k, n=n, cold=True, **rates(med, best, k, total, nbytes), first_mismatch=spot_check("add", "f32", a, b, c, spans))
        del g


def w3():
    rng = np.random.default_rng(2026)
    spans, pos, i = [], 0, 0
    while pos < (1 << 28):
        n = int(np.exp(rng.uniform(0, np.log(1 << 22))))
        oc = pos + (1 if i % 16 == 15 else 0)          # every 16th item: C one element off A and B's phase
        spans.append((pos, pos, oc, n))
        pos += n + 8 + int(rng.integers(0, 4))
        i += 1
    total = pos + 8
    a, b, c = ctr_arrays(total)
    elems = sum(s[3] for s in spans)
    nbytes = 12 * elems
    arr = items_of("add", a, b, c, spans)
    med, best = time_events(lambda: grouped("add", "f32", arr))
    mixed = [k for k in range(len(spans)) if k % 16 == 15]
    emit("W3_grouped", items=len(spans), elements=elems, cold=True, **rates(med, best, len(spans), elems, nbytes),
         first_mismatch=spot_check("add", "f32", a, b, c, spans, picks=(0, mixed[0], mixed[-1], -1)))
    if os.environ.get("GROUPED_BENCH_SKIP_SINGLE"):
        return
    g = graph_of(per_item_stream(a, b, c, spans))
    c.zero_()
    med, best = time_events(g.replay)
    emit("W3_single_graph", items=len(spans), elements=elems, cold=True, **rates(med, best, len(spans), elems, nbytes),
         first_mismatch=spot_check("add", "f32", a, b, c, spans, picks=(0, mixed[0], -1)))


def w4():
    nbytes = 1 << 30
    for dt, tdt in TORCH.items():
        total = nbytes // ES[dt]
        a = torch.rand(total, device="cuda", dtype=torch.float32 if dt != "f64" else tdt).to(tdt)
        b = torch.rand(total, device="cuda", dtype=torch.float32 if dt != "f64" else tdt).to(tdt)
        c = torch.empty_like(a)
        n = 1 << 16
        k = total // n
        for op in ("copy", "scale", "add", "triad"):
            s = 3.0 if op in ("scale", "triad") else 0.0
            spans = [(i * n, i * n, i * n, n) for i in range(k)]
            arr = items_of(op, a, b, c, spans)
            moved = ARRAYS[op] * nbytes
            med, best = time_events(lambda: grouped(op, dt, arr, s))
            emit("W4_grouped", dtype=dt, op=op, items=k, n=n, cold=True, **rates(med, best, k, total, moved),
                 first_mismatch=spot_check(op, dt, a, b, c, spans, s))
            bb = b.data_ptr() if op in ("add", "triad") else None
            med, best = time_events(lambda: LIB.b200va_stream(capi.OPS[op], capi.DTYPES[dt], a.data_ptr(), bb, c.data_ptr(), total, s, stream_ptr()))
            emit("W4_one_array", dtype=dt, op=op, n=total, cold=True, **rates(med, best, 1, total, moved))
        del a, b, c


def w5():
    n = 64
    big = 5000
    a = torch.ones(big * n, dtype=torch.float32, device="cuda")
    b, c = torch.ones_like(a), torch.empty_like(a)
    for count in (1, 100, 800, 5000):
        arr = items_of("add", a, b, c, [(i * n, i * n, i * n, n) for i in range(count)])
        for _ in range(WARM):
            grouped("add", "f32", arr)
        torch.cuda.synchronize()
        us = []
        for _ in range(200):
            t0 = time.perf_counter()
            grouped("add", "f32", arr)
            us.append((time.perf_counter() - t0) * 1e6)
            torch.cuda.synchronize()
        us.sort()
        geo = os.environ.get("B200VA_GROUPED_GEOMETRY", "")
        cap = int(geo.split(",")[2]) if LIB is not capi.lib and geo.count(",") == 2 else 800
        emit("W5_enqueue", items=count, n=n, us_per_call_median=us[len(us) // 2], us_per_call_best=us[0],
             us_per_item=us[len(us) // 2] / count, launches=-(-count // cap))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def main():
    global LIB, OUT
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--lib", choices=("prod", "tune"), default="prod")
    ap.add_argument("--workloads", default="W1,W2,W3,W4,W5")
    ap.add_argument("--w2-logs", default="12,14,16,18,20,22")
    args = ap.parse_args()
    LIB = capi.tune_lib() if args.lib == "tune" else capi.lib
    OUT = args.out
    if OUT:
        os.makedirs(OUT, exist_ok=True)
    TAG.update({"card": card(), "lib": args.lib, "geometry": os.environ.get("B200VA_GROUPED_GEOMETRY", "default")})
    todo = args.workloads.split(",")
    if "W1" in todo:
        w1()
    if "W2" in todo:
        w2([int(x) for x in args.w2_logs.split(",")])
    if "W3" in todo:
        w3()
    if "W4" in todo:
        w4()
    if "W5" in todo:
        w5()


if __name__ == "__main__":
    main()
