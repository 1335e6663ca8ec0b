"""Pins the CPU oracle to the reference's own weight-free golden vectors.

Every expected value below is a known answer held by the reference's tests or docs
(cited per test); tolerances are the reference's own (src/common/utils.go:13-17:
THRESHOLD_F32 = 1e-3, THRESHOLD_EXACT = 0).
"""
import math

import numpy as np
import pytest

from oracle import oracle as O
from tests.helpers import reference_vectors

GOLD = reference_vectors()                     # tests/golden/reference_vectors.json (the reference's own literals)
THRESHOLD_F32 = GOLD["threshold_f32"]["value"]


def bf(x):
    return O.bf16_bits(np.asarray(x, np.float32))


def f(b):
    return O.bf16_to_f32(b)


# ---- src/dtype/bfloat16_test.go:8-66 -------------------------------------------------

@pytest.mark.parametrize("inp,exp", [(c["input"], c["expected"]) for c in GOLD["bf16_from_f32"]])
def test_bf16_truncation(inp, exp):
    b = O.lib().orc_f32_to_bf16(inp)
    assert O.lib().orc_bf16_to_f32(b) == np.float32(exp)
    assert f(bf([inp]))[0] == np.float32(exp)


# src/dtype/bfloat16_test.go:68-106 (little-endian storage)
@pytest.mark.parametrize("raw,bits,val", [(bytes(c["bytes"]), c["bits"], c["f32"]) for c in GOLD["bf16_little_endian"]["cases"]])
def test_bf16_little_endian(raw, bits, val):
    b = np.frombuffer(raw, dtype="<u2")
    assert int(b[0]) == bits
    assert f(b)[0] == np.float32(val)


# ---- src/ml/operations_test.go:782-829 ------------------------------------------------

def test_linear_f32_golden():
    g = GOLD["linear_f32"]
    w, x, exp = (np.array(g[k], np.float32) for k in ("weightVals", "inputVals", "expected"))
    assert w.shape == (4, 3) and x.shape == (2, 3) and exp.shape == (2, 4)
    assert np.abs(O.linear_f32(x, w) - exp).max() <= THRESHOLD_F32


# ---- src/ml/operations_test.go:831-878 ------------------------------------------------

def test_linear_bf16_golden():
    g = GOLD["linear_bf16"]
    w, x, exp = bf(g["weightVals"]), bf(g["inputVals"]), np.array(g["expected"], np.float32)
    got = f(O.linear_bf16(x, w))
    assert np.abs(got - exp).max() <= THRESHOLD_F32
    # (the literals are 4-decimal PyTorch prints, so 1e-3 is as tight as the reference pins this)
    assert np.all(np.abs(got - exp) < 1e-4)


# ---- src/ml/operations_test.go:880-946 ------------------------------------------------

def test_matmul_bf16_golden():
    g = GOLD["matmul_bf16"]
    a, b, exp = bf(g["inputVals"]), bf(g["otherVals"]), np.array(g["expected"], np.float32)
    got = f(O.matmul_bf16(a, b))
    assert got.shape == (2, 2, 4)
    assert np.abs(got - exp).max() <= THRESHOLD_F32
    assert np.all(np.abs(got - exp) / exp < 1e-4)  # 5 significant digits printed


# ---- src/ml/operations_test.go:589-652 (Pow) ------------------------------------------

def test_pow2_golden():
    x = bf(np.arange(3, 8, dtype=np.float32))
    assert np.array_equal(O.pow2_bf16(x), np.array(GOLD["pow2_arange_3_8"]["expected"], np.float32))


# ---- src/ml/operations_test.go:654-780 (Mean over createTestInputTensor 1,2,3,...) -----

def test_mean_golden():
    t = np.arange(1, 61, dtype=np.float32).reshape(5, 4, 3)
    got = O.mean_f32(t)
    exp = np.array(GOLD["mean_5x4x3_keepdim"]["expected"], np.float32)  # 2, 5, 8, ... exactly representable
    assert got.shape == (5, 4, 1)
    assert np.array_equal(got, exp)
    assert got[0, 0, 0] == 2.0 and got[4, 3, 0] == 59.0


# ---- docs/10-ROPE-ROTARY-POSITIONAL-EMBEDDINGS.md:276-288 (all 64 scaled inverse freqs) --

DOC_FREQS = GOLD["rope_scaled_inv_freqs"]["values"]
assert len(DOC_FREQS) == 64


def test_rope_freqs_match_reference_doc():
    freqs, _ = O.rope_table(128, 8, 500000.0, True)
    got = f(freqs)
    for g, e in zip(got, DOC_FREQS):
        # the doc prints 5 significant digits of the bf16 value
        assert float("%.4e" % g) == pytest.approx(e, rel=0, abs=0), (g, e)


def test_rope_positions_are_bf16_quantised():
    # docs/10-ROPE...md:397,403: t[4094] and t[4095] both give 4.0800e+03 * freq
    _, cis = O.rope_table(128, 4096, 500000.0, True)
    assert np.array_equal(cis[4094], cis[4095])
    assert np.array_equal(cis[257], cis[256])          # bf16(257) == 256
    assert not np.array_equal(cis[255], cis[256])
    # freq[0] == 1 -> angle == bf16(pos): row 4094 col 0 is cos/sin(4080)
    assert cis[4094, 0, 0] == np.float32(math.cos(4080.0)) and cis[4094, 0, 1] == np.float32(math.sin(4080.0))
    assert np.array_equal(cis[0], np.stack([np.ones(64, np.float32), np.zeros(64, np.float32)], -1))


# ---- own known-answer tests for ops the reference never pins (SURVEY 8c last row) -------

def test_argmax_first_max_wins_and_nan():
    x = np.array([1, 5, 5, 2], np.float32)
    assert O.argmax_f32(x) == 1
    x = np.array([np.nan, -1, -1], np.float32)
    assert O.argmax_f32(x) == 1
    assert O.argmax_f32(np.array([np.nan], np.float32)) == -1


def test_softmax_f64_no_max_subtraction():
    x = np.array([[0.5, -1.25, 3.0]], np.float32)
    e = np.exp(x.astype(np.float64))
    exp = (e / e.sum()).astype(np.float32)
    assert np.array_equal(O.softmax_f32(x), exp)


def test_silu_table_known_values():
    tab = O.silu_table_bf16()
    assert tab[0] == 0                                   # silu(0) = 0
    one = int(bf([1.0])[0])
    assert tab[one] == bf([np.float32(1.0 / (1.0 + math.exp(-1.0)))])[0]
    ninf = int(bf([-np.inf])[0])
    assert np.isnan(f(tab[ninf:ninf + 1])[0])            # -inf/(1+inf) = NaN, like the Go table
    x = bf([0.25, -3.0, 7.5])
    got = O.silu_bf16(x)
    for b, g in zip(x, got):
        v = float(f(np.array([b]))[0])
        assert g == bf([np.float32(v / (1.0 + math.exp(-v)))])[0]


def test_rmsnorm_two_truncations():
    rng = np.random.default_rng(1)
    x = bf(rng.standard_normal((3, 64)))
    w = bf(1 + 0.1 * rng.standard_normal(64))
    xs = f(x)
    out = np.empty_like(x)
    for s in range(3):
        acc = np.float32(0)
        for j in range(64):
            acc = np.float32(acc + np.float32(xs[s, j] * xs[s, j]))
        ms = np.float32(acc / np.float32(64)) + np.float32(1e-5)
        r = np.float32(1.0 / math.sqrt(float(ms)))
        n1 = bf(xs[s] * r)
        out[s] = bf(f(n1) * f(w))
    assert np.array_equal(O.rmsnorm(x, w, 1e-5), out)


def test_rope_apply_uses_f64_intermediates():
    rng = np.random.default_rng(2)
    _, cis = O.rope_table(128, 64, 500000.0, True)
    x = bf(rng.standard_normal((2, 3, 128)))
    got = O.rope_apply(x, cis, 5)
    xs = f(x).astype(np.float64)
    a, b = xs[..., 0::2], xs[..., 1::2]
    c = cis[5:7, None, :, 0].astype(np.float64)
    d = cis[5:7, None, :, 1].astype(np.float64)
    re = (a * c - b * d).astype(np.float32)
    im = (a * d + b * c).astype(np.float32)
    exp = np.empty_like(x)
    exp[..., 0::2] = bf(re)
    exp[..., 1::2] = bf(im)
    assert np.array_equal(got, exp)


def test_linear_paths_agree_s1_vs_sN():
    rng = np.random.default_rng(3)
    x = bf(rng.standard_normal((5, 96)))
    w = bf(rng.standard_normal((37, 96)) * 0.1)
    full = O.linear_bf16(x, w)
    for s in range(5):
        assert np.array_equal(O.linear_bf16(x[s:s + 1], w), full[s:s + 1])
    # and against a literal sequential-f32 python loop
    xs, ws = f(x), f(w)
    for s, n in [(0, 0), (4, 36), (2, 17)]:
        acc = np.float32(0)
        for k in range(96):
            acc = np.float32(acc + np.float32(xs[s, k] * ws[n, k]))
        assert full[s, n] == bf([acc])[0]


def test_committed_fixture_is_what_the_reference_sources_say(tmp_path):
    """the fixture is what tests/golden/extract_reference_vectors.py extracted from the Go reference's sources: its
    canonical SHA-256 is the one recorded with that extraction (tests/golden/reference_vectors.sha256).  The sources
    are not part of this repository; when LNB_REFERENCE_DIR names a checkout of them, the extractor runs again and
    must reproduce the fixture and the digest."""
    import hashlib
    import json
    import os
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    recorded = open(os.path.join(here, "golden", "reference_vectors.sha256")).read().strip()
    assert hashlib.sha256(json.dumps(GOLD, sort_keys=True, separators=(",", ":")).encode()).hexdigest() == recorded
    ref = os.environ.get("LNB_REFERENCE_DIR", "")
    if not ref or not os.path.isdir(os.path.join(ref, "src", "ml")):
        return
    src = open(os.path.join(here, "golden", "extract_reference_vectors.py")).read().replace(
        'OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_vectors.json")', "OUT = %r" % str(tmp_path / "v.json"))
    script = tmp_path / "extract.py"
    script.write_text(src)
    subprocess.check_call([sys.executable, str(script)])
    assert json.load(open(tmp_path / "v.json")) == GOLD
    assert open(tmp_path / "reference_vectors.sha256").read().strip() == recorded


# ---- building blocks of the RoPE table and the mask: the reference's own literals (operations_test.go:56-587) ----

@pytest.mark.parametrize("case", GOLD["arange_bf16"], ids=lambda c: "arange" + str(c["args"]))
def test_arange_bf16_golden(case):
    got = f(O.arange_bf16(*case["args"]))
    assert got.shape == (len(case["expected"]),) and np.array_equal(got, np.array(case["expected"], np.float32))
    with pytest.raises(ValueError):
        O.arange_bf16(3, 3, 1)                                       # "start value must be less than end value"


def test_outer_bf16_golden():
    g = GOLD["outer_bf16"]
    got = f(O.outer_bf16(O.arange_bf16(*g["vec1_arange"]), O.arange_bf16(*g["vec2_arange"])))
    assert np.array_equal(got, np.array(g["expected"], np.float32))


def test_polar_golden():
    g = GOLD["polar"]
    angle = np.array([eval(e.replace("math.Pi", "math.pi"), {"math": math}) for e in g["angle_expr"]], np.float32)   # float32(math.Pi/2), ...
    got = O.polar(np.array([g["abs"]], np.float32), angle[None, :])
    exp = np.array([[complex(a, b) for a, b in g["expected_re_im"]]], np.complex64)
    assert got.shape == (1, 5) and got.dtype == np.complex64
    assert np.abs(got - exp).max() <= THRESHOLD_F32


@pytest.mark.parametrize("case", GOLD["triangular_upper"], ids=lambda c: "triu%sx%s_d%s" % (c["size"][0], c["size"][1], c["diagonal"]))
def test_triangular_upper_golden(case):
    got = O.triangular_upper(O.full_f32(case["size"], case["fill"]), case["diagonal"])
    assert np.array_equal(got, np.array(case["expected"], np.float32))


def test_c_rope_table_equals_the_composition_of_the_pinned_blocks():
    """precomputeFreqsCis (llamatransformer.go:694-751) = ARange -> pow -> scaling -> Outer -> Polar.  The C oracle
    computes it in one function; composing the NumPy blocks above (each pinned to the reference's literals) from the
    C oracle's inverse frequencies must give the same table bit for bit, for every position and frequency."""
    for dim, end, theta, scaled in ((128, 4096, 500000.0, True), (128, 300, 500000.0, False), (32, 128, 10000.0, True)):
        freqs, cis = O.rope_table(dim, end, theta, scaled)
        assert np.array_equal(cis, O.rope_table_from_blocks(dim, end, theta, freqs))
    # and the unscaled inverse frequencies themselves: ARange(0, dim, 2) -> float32(1 / theta^(val / dim)) -> bf16
    freqs, _ = O.rope_table(128, 8, 500000.0, False)
    val = f(O.arange_bf16(0, 128, 2))
    exp = bf((1.0 / np.power(500000.0, (val / np.float32(128)).astype(np.float64))).astype(np.float32))
    assert np.array_equal(freqs, exp)


def test_oracle_outputs_did_not_drift():
    """the oracle checks every GPU kernel; its own outputs for fixed seeded inputs are anchored by committed digests
    (tests/golden/oracle_regression.json, written by tests/golden/make_oracle_regression.py)"""
    import importlib.util
    import json
    import os
    here = os.path.dirname(os.path.abspath(__file__))
    spec = importlib.util.spec_from_file_location("make_oracle_regression", os.path.join(here, "golden", "make_oracle_regression.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    with open(os.path.join(here, "golden", "oracle_regression.json")) as fh:
        committed = json.load(fh)
    assert mod.compute() == committed
