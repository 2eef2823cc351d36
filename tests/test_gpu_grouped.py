"""b200va_stream_grouped: one call over many independent (A, B, C, n) items, each item bit-exact
against the oracle of b200va_stream -- ragged sizes, pointer phases, aliasing, calls that span
several launches, stream ordering behind a writer, CUDA-graph replay and argument errors.  The
CPU tests check the ctypes mirror of b200va_item_t and the grouped kernels' SASS."""
import ctypes as C
import re
import subprocess

import numpy as np
import pytest

import oracle
from conftest import has_gpu
from k8s_gpu_hpa_b200 import capi
from test_gpu_stream import DTS, OPS, SIZES, host_inputs, to_dev, to_host

if has_gpu():
    import torch

    from k8s_gpu_hpa_b200 import vector_add as va

BINARY = ("add", "triad")
ES = {"f32": 4, "f64": 8, "f16": 2, "bf16": 2}


def scalar_of(op):
    return 0.7001953125 if op in ("scale", "triad") else 0.0


def zeros(n, dtype):
    return to_dev(np.zeros(n, dtype=np.uint16 if dtype in ("f16", "bf16") else (np.float64 if dtype == "f64" else np.float32)), dtype)


def packed(sizes, rng, max_gap=5):
    """Offsets of items laid one after another with random gaps (so their 16-byte phases vary)."""
    offs, pos = [], 0
    for n in sizes:
        pos += int(rng.integers(0, max_gap + 1))
        offs.append(pos)
        pos += n
    return offs, pos + max_gap


def check_packed(op, dtype, ha, hb, out, offs, sizes, s):
    """Every item's range of `out` equals the oracle, everything outside the items is still zero."""
    want = oracle.stream(op, dtype, ha, hb if op in BINARY else None, s)
    got = to_host(out, dtype)
    covered = np.zeros(got.size, bool)
    for i, (o, n) in enumerate(zip(offs, sizes)):
        bad = oracle.first_mismatch_bits(got[o:o + n], want[o:o + n], dtype)
        assert bad < 0, f"{op} {dtype} item {i} (offset {o}, n={n}): first mismatch at {bad}"
        covered[o:o + n] = True
    assert not got[~covered].any(), "a write outside the items"


# ------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTS)
@pytest.mark.parametrize("op", OPS)
def test_grouped_ragged_batch_all_ops_and_dtypes(op, dtype):
    """One call, items of every size of the single-call test plus one tile and one tile + 1 for each
    candidate tile width, at equal-phase (vector path) and mixed-phase (scalar path) offsets.
    Every output sits inside a larger zeroed buffer whose guard regions must stay zero."""
    epv = 16 // ES[dtype]
    cycle = [(0, 0, 0), (1, 1, 1), (3, 3, 3), (0, 1, 2), (5, 5, 0), (7, 7, 7), (2, 0, 2)]
    batch = [(n, cycle[i % len(cycle)]) for i, n in enumerate(SIZES)]
    batch += [(tv * epv + extra, (0, 0, 0)) for tv in (256, 512, 1024) for extra in (0, 1)]   # one tile, one tile + 1
    s = scalar_of(op)
    a_l, b_l, c_l, outs, want = [], [], [], [], []
    for i, (n, (oa, ob, oc)) in enumerate(batch):
        ha, hb = host_inputs(dtype, n + 8, 100 + i)
        a, b = to_dev(ha, dtype), to_dev(hb, dtype)
        out = zeros(n + 24, dtype)
        a_l.append(a[oa:oa + n])
        b_l.append(b[ob:ob + n] if op in BINARY else None)
        c_l.append(out[8 + oc:8 + oc + n])
        outs.append((out, 8 + oc, n))
        want.append(oracle.stream(op, dtype, ha[oa:oa + n].copy(), hb[ob:ob + n].copy() if op in BINARY else None, s))
    va.stream_grouped(op, a_l, b_l if op in BINARY else None, c_l, scalar=s)
    torch.cuda.synchronize()
    for i, ((out, o, n), w) in enumerate(zip(outs, want)):
        got = to_host(out, dtype)
        bad = oracle.first_mismatch_bits(got[o:o + n], w, dtype)
        assert bad < 0, f"{op} {dtype} item {i} n={n} offsets {batch[i][1]}: first mismatch at {bad}"
        assert not got[:o].any() and not got[o + n:].any(), f"item {i}: guard region written"


@pytest.mark.gpu
def test_grouped_matches_the_single_calls():
    """Bitwise equal to per-item b200va_add_f32 (f32 add on ctr inputs, with the digest of the largest
    item against the oracle's) and to per-item b200va_stream for the other ops and dtypes."""
    n_big = 3_000_017
    a = torch.empty(n_big + 64, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    va.fill_ctr(a, 0x0A)
    va.fill_ctr(b, 0x0B)
    spans = [(0, n_big), (1, 50000), (4, 4097), (7, 1), (3, 17), (0, 1 << 16)]
    got = va.stream_grouped("add", [a[o:o + n] for o, n in spans], [b[o:o + n] for o, n in spans])
    torch.cuda.synchronize()
    for (o, n), g in zip(spans, got):
        ref = va.add(a[o:o + n], b[o:o + n])
        assert bool((g.view(torch.int32) == ref.view(torch.int32)).all()), (o, n)
    assert va.digest(got[0]) == oracle.ctr_vadd_digest(n_big)
    for op, dtype in (("triad", "bf16"), ("scale", "f64"), ("copy", "f16"), ("add", "f64"), ("triad", "f32")):
        ha, hb = host_inputs(dtype, 300_000, 7)
        x, y = to_dev(ha, dtype), to_dev(hb, dtype)
        spans = [(0, 300_000 - 9), (1, 1000), (5, 77), (2, 65_536)]
        ys = [y[o:o + n] for o, n in spans] if op in BINARY else None
        grouped = va.stream_grouped(op, [x[o:o + n] for o, n in spans], ys, scalar=-1.25)
        for k, (o, n) in enumerate(spans):
            single = va.stream(op, x[o:o + n], ys[k] if ys else None, scalar=-1.25)
            torch.cuda.synchronize()
            assert np.array_equal(to_host(grouped[k], dtype).view(np.uint8), to_host(single, dtype).view(np.uint8)), (op, dtype, o, n)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTS)
def test_grouped_aliasing(dtype):
    """C == A, C == B and the in-place triad y = y + s*x (axpy), mixed within one call."""
    kinds = ["c=a", "c=b", "axpy", "fresh", "c=a", "axpy", "c=b"]
    sizes = [20_011, 1, 50_000, 4097, 3, (1 << 16) + 5, 129]
    a_l, b_l, c_l, want = [], [], [], []
    for i, (kind, n) in enumerate(zip(kinds, sizes)):
        ha, hb = host_inputs(dtype, n + 4, 40 + i)
        o = i % 4
        a, b = to_dev(ha, dtype)[o:o + n], to_dev(hb, dtype)[o:o + n]
        a_l.append(a)
        b_l.append(b)
        c_l.append({"c=a": a, "c=b": b, "axpy": a, "fresh": zeros(n, dtype)}[kind])
        want.append(oracle.stream("triad", dtype, ha[o:o + n].copy(), hb[o:o + n].copy(), 2.0))
    va.stream_grouped("triad", a_l, b_l, c_l, scalar=2.0)
    torch.cuda.synchronize()
    for i, (c, w) in enumerate(zip(c_l, want)):
        assert oracle.first_mismatch_bits(to_host(c, dtype), w, dtype) == -1, (dtype, kinds[i], sizes[i])


@pytest.mark.gpu
def test_grouped_many_items_span_several_launches():
    """5000 ragged items (several parameter blocks), then one 2^24-element item among 3000 tiny ones:
    tile-to-item mapping at every item boundary and across launch boundaries."""
    rng = np.random.default_rng(5)
    for sizes in ([int(x) for x in rng.integers(0, 3000, 5000)],
                  [int(x) for x in rng.integers(1, 65, 1500)] + [1 << 24] + [int(x) for x in rng.integers(1, 65, 1500)]):
        offs, total = packed(sizes, rng)
        ha, hb = host_inputs("f32", total, 9)
        a, b = to_dev(ha, "f32"), to_dev(hb, "f32")
        out = zeros(total, "f32")
        va.stream_grouped("add", [a[o:o + n] for o, n in zip(offs, sizes)], [b[o:o + n] for o, n in zip(offs, sizes)],
                          [out[o:o + n] for o, n in zip(offs, sizes)])
        torch.cuda.synchronize()
        check_packed("add", "f32", ha, hb, out, offs, sizes, 0.0)


@pytest.mark.gpu
def test_grouped_runs_after_a_kernel_that_writes_its_inputs():
    """fill_ctr writes A and B, and the grouped add follows on the same stream at once.  48 items of
    2^20 f32 are 192 MiB per array, so the launch takes the L2-prefetch form ahead of its dependency
    wait; a result from stale inputs would change the digest."""
    item, k = 1 << 20, 48
    a = torch.empty(item * k, dtype=torch.float32, device="cuda")
    b, out = torch.empty_like(a), torch.empty_like(a)
    for first in (0, 1 << 33):
        va.fill_ctr(a, 0x0A, first)
        va.fill_ctr(b, 0x0B, first)
        va.stream_grouped("add", list(a.split(item)), list(b.split(item)), list(out.split(item)))
        assert va.digest(out) == oracle.ctr_vadd_digest(item * k, first), first


@pytest.mark.gpu
def test_grouped_call_captured_into_a_cuda_graph():
    """A call filling one whole parameter block (800 items) is captured once and replayed twice with
    new input values."""
    rng = np.random.default_rng(6)
    sizes = [int(x) for x in rng.integers(1, 5000, 800)]
    offs, total = packed(sizes, rng)
    a = torch.zeros(total, dtype=torch.float32, device="cuda")
    b, out = torch.zeros_like(a), torch.zeros_like(a)
    args = ([a[o:o + n] for o, n in zip(offs, sizes)], [b[o:o + n] for o, n in zip(offs, sizes)],
            [out[o:o + n] for o, n in zip(offs, sizes)])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        va.stream_grouped("triad", *args, scalar=0.5)        # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        va.stream_grouped("triad", *args, scalar=0.5)
    for seed in (21, 22):
        ha, hb = host_inputs("f32", total, seed)
        a.copy_(torch.from_numpy(ha))
        b.copy_(torch.from_numpy(hb))
        out.zero_()
        g.replay()
        torch.cuda.synchronize()
        check_packed("triad", "f32", ha, hb, out, offs, sizes, 0.5)


@pytest.mark.gpu
def test_grouped_argument_errors_enqueue_nothing():
    a = torch.zeros(256, dtype=torch.float32, device="cuda")
    x = torch.ones(256, dtype=torch.float32, device="cuda")
    out = torch.full((256,), -7.0, dtype=torch.float32, device="cuda")
    p = lambda t, off=0: t.data_ptr() + off  # noqa: E731
    good = [capi.Item(p(a), p(x), p(out), 64), capi.Item(p(x), p(x), p(out, 256), 64)]

    def call(op, dtype, extra, count=None):
        items = (capi.Item * (len(good) + len(extra)))(*good, *extra)
        rc = capi.lib.b200va_stream_grouped(op, dtype, items, len(items) if count is None else count, 0.0, None)
        torch.cuda.synchronize()
        assert bool((out == -7.0).all()), "an output was written by a refused call"
        return rc

    assert call(9, 0, []) == capi.ERR_VARIANT
    assert call(2, 7, []) == capi.ERR_VARIANT
    assert capi.lib.b200va_stream_grouped(2, 0, None, 3, 0.0, None) == capi.ERR_INVALID
    assert call(2, 0, [capi.Item(p(a), None, p(out, 512), 16)]) == capi.ERR_INVALID                 # add needs b
    assert call(2, 1, [capi.Item(p(a, 4), p(x), p(out, 512), 4)]) == capi.ERR_ALIGN                  # f64 needs 8 B
    assert call(2, 0, [capi.Item(p(a), p(x), p(out, 768), 16), capi.Item(p(out, 904), p(x), p(out, 900), 16)]) == capi.ERR_OVERLAP
    assert call(2, 0, [], count=0) == capi.OK
    assert capi.lib.b200va_stream_grouped(2, 0, None, 0, 0.0, None) == capi.OK
    with pytest.raises(TypeError):
        va.stream_grouped("add", [a], [x.double()])
    with pytest.raises(TypeError):
        va.stream_grouped("add", [a, a[:3]], [x])
    with pytest.raises(TypeError):
        va.stream_grouped("add", [a[::2]], [x[::2]])


# ------------------------------------------------------------------------------------ CPU
def test_item_struct_mirrors_the_header():
    text = re.sub(r"/\*.*?\*/", "", open(capi.HEADER_PATH).read(), flags=re.S)
    body = re.search(r"typedef struct b200va_item \{(.*?)\} b200va_item_t;", text, flags=re.S).group(1)
    assert re.findall(r"\*?(\w+)\s*;", body) == [n for n, _ in capi.Item._fields_] == ["a", "b", "c", "n"]
    assert C.sizeof(capi.Item) == 32
    assert [getattr(capi.Item, n).offset for n in "abcn"] == [0, 8, 16, 24]


def test_grouped_kernels_in_the_production_library():
    """16 stream_grouped kernels (op x dtype), each with 128-bit loads and stores, the PDL pair, and
    the dependency wait ahead of every global load; the cold form bulk-prefetches into L2 first."""
    sass = subprocess.run(["cuobjdump", "-sass", capi.LIB_PATH], capture_output=True, text=True).stdout
    funcs = [f for f in sass.split("Function : ")[1:] if f.startswith("_ZN6b200va14stream_grouped")]
    assert len(funcs) == 16, len(funcs)
    assert len({f.split()[0] for f in funcs}) == 16
    for f in funcs:
        ops = re.findall(r"\b(LDG\.E\S*|STG\.E\S*|ACQBULK|PREEXIT|UBLKPF\.L2)\b", f)
        assert any(re.fullmatch(r"LDG\.E\S*\.128", o) for o in ops), f.split()[0]
        assert any(re.fullmatch(r"STG\.E\S*\.128", o) for o in ops), f.split()[0]
        assert "PREEXIT" in ops and "ACQBULK" in ops
        first_ldg = next(i for i, o in enumerate(ops) if o.startswith("LDG"))
        assert ops.index("ACQBULK") < first_ldg, f.split()[0]
    assert any("UBLKPF.L2" in f for f in funcs)


@pytest.mark.skipif(has_gpu(), reason="checks the no-GPU failure mode")
def test_grouped_fails_loudly_without_a_gpu():
    a = np.ones(16, np.float32)
    out = np.full(16, -7.0, np.float32)
    items = (capi.Item * 2)(capi.Item(a.ctypes.data, a.ctypes.data, out.ctypes.data, 16), capi.Item(None, None, None, 0))
    assert capi.lib.b200va_stream_grouped(2, 0, items, 2, 0.0, None) != capi.OK
    assert capi.lib.b200va_stream_grouped(2, 0, items, 0, 0.0, None) != capi.OK
    assert (out == -7.0).all()
