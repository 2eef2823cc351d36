"""The oracle pinned: known answers of SURVEY.md section 8(c), the committed golden
fixtures, and an independent integer-only IEEE-754 implementation.

The reference ships no tests or vectors for this path ("parity unpinned"), so these are
the strongest anchors available: the glibc seed-1 rand() stream, the IEEE-754 standard.
"""
import json
import os

import numpy as np
import pytest

import oracle

GOLD = os.path.join(os.path.dirname(__file__), "golden")

# SURVEY.md section 8(c), produced independently of oracle/vadd_oracle.c
SURVEY_KAT = {
    0: (0x3F57168B, 0x3EC9EC8F, 0x3F9E0669),
    1: (0x3F487931, 0x3F4C6691, 0x3FCA6FE1),
    2: (0x3F6961B9, 0x3E4A4AE8, 0x3F8DFA3A),
    3: (0x3EABA251, 0x3F44AAB2, 0x3F8D3DED),
    49999: (0x3F2A3986, 0x3E9D8362, 0x3F78FB37),
}


def test_sample_recipe_known_answers():
    a, b = oracle.fill_rand(50000)
    c = oracle.vadd(a, b)
    ua, ub, uc = (v.view(np.uint32) for v in (a, b, c))
    for i, (wa, wb, wc) in SURVEY_KAT.items():
        assert (int(ua[i]), int(ub[i]), int(uc[i])) == (wa, wb, wc), i
    assert oracle.fnv1a64(a) == 0x1CDB0A2BFB6AA671
    assert oracle.fnv1a64(b) == 0xA798316A39E5FF4E
    assert oracle.fnv1a64(c) == 0x000CC9DBE012E750
    assert oracle.bits_digest(c) == (53174197755249, 0x0118998B)
    assert float(c.astype(np.float64).sum()) == pytest.approx(49986.813340499066, abs=1e-9)
    # value range the survey observed: all normal floats in (0, 1)
    assert a.min() > 0 and a.max() < 1 and b.min() > 0 and b.max() < 1
    # the sample's own tolerance check passes on its own recipe
    assert oracle.verify_sample_tolerance(a, b, c) == -1


def test_sample_recipe_is_reseeded_every_call():
    a1, b1 = oracle.fill_rand(1000)
    a2, b2 = oracle.fill_rand(1000)
    assert np.array_equal(a1, a2) and np.array_equal(b1, b2)


def test_golden_rand_fixture():
    g = json.load(open(os.path.join(GOLD, "rand_50000.json")))
    a, b = oracle.fill_rand(g["n"])
    c = oracle.vadd(a, b)
    for name, v in (("A", a), ("B", b), ("C", c)):
        assert f"{oracle.fnv1a64(v):016x}" == g["fnv1a64"][name]
        for i, bits in g[f"{name}_bits"].items():
            assert f"{v.view(np.uint32)[int(i)]:08x}" == bits
    assert oracle.bits_digest(c) == (g["C_bits_sum"], int(g["C_bits_xor"], 16))


def test_golden_ctr_fixture():
    g = json.load(open(os.path.join(GOLD, "ctr_1m.json")))
    a = oracle.fill_ctr(g["n"], g["seed_a"], g["first"])
    b = oracle.fill_ctr(g["n"], g["seed_b"], g["first"])
    c = oracle.vadd(a, b)
    assert [f"{v:08x}" for v in c.view(np.uint32)[:8]] == g["C_head_bits"]
    assert f"{oracle.fnv1a64(c):016x}" == g["fnv1a64"]["C"]
    assert oracle.bits_digest(c) == (g["C_bits_sum"], int(g["C_bits_xor"], 16))


def test_golden_special_values_fixture():
    g = np.load(os.path.join(GOLD, "special_values.npz"))
    c = oracle.vadd(g["a_bits"].view(np.float32), g["b_bits"].view(np.float32))
    assert oracle.first_mismatch(c, g["c_bits"].view(np.float32)) == -1


def _numpy_ctr(n, seed, first):
    m = (1 << 64) - 1
    z = (np.arange(n, dtype=np.uint64) + np.uint64((seed * 0x9E3779B97F4A7C15 + first) & m))
    with np.errstate(over="ignore"):
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return ((z >> np.uint64(40)).astype(np.float32) * np.float32(2.0 ** -24)).astype(np.float32)


def test_ctr_generator_matches_its_definition_and_is_shard_invariant():
    n = 100_003
    x = oracle.fill_ctr(n, 0x0A, 0)
    assert np.array_equal(x, _numpy_ctr(n, 0x0A, 0))
    assert x.min() >= 0.0 and x.max() < 1.0
    # any shard generated from the global index equals the slice of the whole
    for lo, hi in ((0, 17), (17, 4099), (4099, n)):
        assert np.array_equal(oracle.fill_ctr(hi - lo, 0x0A, lo), x[lo:hi])
    assert not np.array_equal(oracle.fill_ctr(64, 0x0A, 0), oracle.fill_ctr(64, 0x0B, 0))


def test_hardware_add_equals_softfloat_on_random_bit_patterns():
    rng = np.random.default_rng(20260921)
    n = 400_000
    ua = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
    ub = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
    # a third of the pairs: near-cancellation (opposite sign, nearby magnitude)
    k = n // 3
    ub[:k] = (ua[:k] ^ np.uint32(0x80000000)) + rng.integers(-(1 << 24), 1 << 24, k).astype(np.int64).astype(np.uint32)
    # a third: same exponent neighbourhood, same sign (carry / rounding paths)
    ub[k:2 * k] = ua[k:2 * k] + rng.integers(-(1 << 25), 1 << 25, k).astype(np.int64).astype(np.uint32)
    hw = oracle.vadd(ua.view(np.float32), ub.view(np.float32))
    sf = oracle.softfloat_vadd_bits(ua, ub).view(np.float32)
    assert oracle.first_mismatch(hw, sf) == -1


def test_softfloat_special_cases():
    f = oracle.softfloat_add_bits
    assert f(0x00000000, 0x80000000) == 0x00000000          # +0 + -0 = +0 (RNE)
    assert f(0x80000000, 0x80000000) == 0x80000000          # -0 + -0 = -0
    assert f(0x3F800000, 0xBF800000) == 0x00000000          # exact cancel -> +0
    assert f(0x00000001, 0x00000001) == 0x00000002          # subnormals are exact, no FTZ
    assert f(0x007FFFFF, 0x00000001) == 0x00800000          # subnormal -> smallest normal
    assert f(0x7F7FFFFF, 0x7F7FFFFF) == 0x7F800000          # overflow -> +Inf
    assert f(0x7F800000, 0xFF800000) == 0x7FC00000          # Inf - Inf -> NaN
    assert f(0x3F800000, 0x33800000) == 0x3F800000          # 1 + 2^-24: tie -> even
    assert f(0x3F800001, 0x33800000) == 0x3F800002          # odd + half ulp: tie -> even (up)
    assert f(0x3F800000, 0x33800001) == 0x3F800001          # just above the tie -> up


def test_first_mismatch_treats_nans_as_a_class():
    x = np.array([1.0, np.nan, 2.0], np.float32)
    y = x.copy()
    y.view(np.uint32)[1] = 0x7FFFFFFF                        # PTX canonical NaN
    assert oracle.first_mismatch(x, y) == -1
    y[2] = 2.0000002
    assert oracle.first_mismatch(x, y) == 2


def test_threaded_oracle_and_digests_agree_with_scalar():
    n = 1_000_003
    a, b = oracle.fill_ctr(n, 0x0A), oracle.fill_ctr(n, 0x0B)
    c = oracle.vadd(a, b)
    assert np.array_equal(c, oracle.vadd_mt(a, b, 3))
    assert np.array_equal(c, a + b)                          # numpy's IEEE add, third opinion
    assert oracle.vadd_digest(a, b) == oracle.bits_digest(c) == oracle.vadd_digest(a, b, threads=4)
    assert oracle.ctr_vadd_digest(n, 0, threads=2, block=65536) == oracle.bits_digest(c)


def test_empty_inputs():
    e = np.empty(0, np.float32)
    assert oracle.vadd(e, e).size == 0
    assert oracle.bits_digest(e) == (0, 0)
    assert oracle.ctr_vadd_digest(0) == (0, 0)


@pytest.mark.parametrize("n", [0, 1, 15, 16, 17, 1000, 100_003])
def test_non_temporal_timing_variant_returns_the_same_bits(n):
    """The CPU baseline's non-temporal-store leg (vaddps + movntps, widest ISA of the host) is a
    timing variant only: bit-identical to the scalar restatement, specials included."""
    rng = np.random.default_rng(n)
    ua = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
    ub = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
    a, b = ua.view(np.float32), ub.view(np.float32)
    assert oracle.nt_width() in (128, 256, 512)
    for threads in (1, 3):
        got = oracle.vadd_mt_nt(a[1:], b[1:], threads) if n > 1 else oracle.vadd_mt_nt(a, b, threads)   # misaligned start too
        want = oracle.vadd(np.ascontiguousarray(a[1:]), np.ascontiguousarray(b[1:])) if n > 1 else oracle.vadd(a, b)
        assert oracle.first_mismatch_bits(got, want, "f32") == -1


def test_cpu_baseline_reports_both_store_kinds():
    cfg = oracle.best_cpu_config(1 << 20)
    assert set(k.split(" ")[0] for k in cfg["tried"]) == {"regular", "non-temporal"}
    assert cfg["rate"] == max(d["elements_per_s"] for d in cfg["tried"].values()) and cfg["threads"] >= 1


def test_on_disk_nvidia_derivative_carries_the_restated_float_recipe():
    """The toolkit ships an NVIDIA derivative of the vectorAdd sample with FLOAT operands
    (CUPTI samples, cuda_memory_trace/memory_trace.cu).  It is not the reference's image, but it
    corroborates what oracle/vadd_oracle.c restates from recollection: the kernel body, the
    interleaved never-seeded rand()/(float)RAND_MAX fill, 256-thread blocks.  Its cited lines are
    recorded in golden/cupti_memory_trace_recipe.json (tests/golden/make_cupti_recipe.py)."""
    import re

    g = json.load(open(os.path.join(GOLD, "cupti_memory_trace_recipe.json")))
    src = "\n".join(g["lines"][k] for k in sorted(g["lines"], key=int))
    flat = re.sub(r"\s+", " ", src)
    assert re.search(r"VectorAdd\( const float \*pA, const float \*pB, float \*pC, int N\)", flat)
    assert "int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < N) { pC[i] = pA[i] + pB[i]; }" in flat
    assert "pHostA[n] = rand() / (float)RAND_MAX; pHostB[n] = rand() / (float)RAND_MAX;" in flat      # A then B, per index
    assert not g["calls_srand"] and "srand" not in src                                                  # glibc default seed 1
    assert "dim3 block(256);" in src
    # ... and that recipe, run through the oracle, is the one whose known answers are pinned above
    a, b = oracle.fill_rand(4)
    assert [int(v) for v in a.view(np.uint32)] == [k[0] for k in (SURVEY_KAT[i] for i in range(4))]
    assert [int(v) for v in b.view(np.uint32)] == [k[1] for k in (SURVEY_KAT[i] for i in range(4))]
