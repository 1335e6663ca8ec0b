"""Extracts the reference's weight-free golden vectors for the hot path from its OWN test sources and docs and
writes tests/golden/reference_vectors.json.

The reference is Go (no toolchain in the image), so it cannot be imported or run to generate fixtures; its tests
however hold literal known answers for this path (SURVEY 8c).  This script parses those literals where they lie
under /root/reference (read-only) and records file:line for each, so the committed fixture is provably the
reference's data and not a transcription.  Run here:  python tests/golden/extract_reference_vectors.py
(/root/reference does not exist on the GPU box; tests only read the committed JSON.)"""
import hashlib
import json
import os
import re
import sys

REF = os.environ.get("LNB_REFERENCE_DIR", "/root/reference")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_vectors.json")
# digest of what was extracted, kept beside the fixture: without a reference checkout the tests can still tell that the
# fixture is the extraction and was not edited by hand
DIGEST = os.path.join(os.path.dirname(OUT), "reference_vectors.sha256")
NUM = r"[-+]?(?:\d+\.\d*|\.\d+|\d+)(?:[eE][-+]?\d+)?"


def digest(vectors) -> str:
    """SHA-256 of the extracted vectors in canonical JSON (sorted keys, no whitespace)"""
    return hashlib.sha256(json.dumps(vectors, sort_keys=True, separators=(",", ":")).encode()).hexdigest()


def read(rel):
    with open(os.path.join(REF, rel)) as f:
        return f.read()


def func_body(src, name):
    """(first line number, text) of `func name(` ... up to the next top-level func"""
    m = re.search(r"^func %s\(" % re.escape(name), src, re.M)
    assert m, name
    nxt = re.search(r"^func ", src[m.end():], re.M)
    end = m.end() + nxt.start() if nxt else len(src)
    return src.count("\n", 0, m.start()) + 1, src[m.start():end]


def literal(body, var):
    """nested list of floats of `var := [][]T{ ... }`, BFloat16fromFloat32(x) wrappers removed"""
    m = re.search(r"\b%s\s*:=\s*((?:\[\])+)[\w.]+\{" % re.escape(var), body)
    assert m, var
    depth_decl = m.group(1).count("[]")
    i = m.end() - 1
    depth, j = 0, i
    while True:
        if body[j] == "{":
            depth += 1
        elif body[j] == "}":
            depth -= 1
            if depth == 0:
                break
        j += 1
    text = body[i:j + 1]
    text = re.sub(r"dtype\.BFloat16fromFloat32\((%s)\)" % NUM, r"\1", text)
    text = re.sub(r"float32\((%s)\)" % NUM, r"\1", text)
    text = text.replace("{", "[").replace("}", "]")
    text = re.sub(r",\s*\]", "]", text)
    text = re.sub(r"(?<![\d.])\.(\d)", r"0.\1", text)          # .5 -> 0.5
    text = re.sub(r"(\d)\.(?!\d)", r"\1.0", text)               # 1. -> 1.0
    val = json.loads(text)
    d, v = 0, val
    while isinstance(v, list):
        d += 1
        v = v[0]
    assert d == depth_decl, (var, d, depth_decl)
    return val


def main():
    out = {"_generated_by": "tests/golden/extract_reference_vectors.py", "_reference": "adalkiran/llama-nuts-and-bolts"}

    ops = read("src/ml/operations_test.go")
    for key, fn, vars_ in (("linear_f32", "TestLinearTransformationF32", ("expected", "weightVals", "inputVals")),
                           ("linear_bf16", "TestLinearTransformationBF16", ("expected", "weightVals", "inputVals")),
                           ("matmul_bf16", "TestMatMulBF16", ("expected", "inputVals", "otherVals"))):
        line, body = func_body(ops, fn)
        entry = {"source": "src/ml/operations_test.go:%d (%s)" % (line, fn), "threshold": "common.THRESHOLD_F32 = 1e-3"}
        for v in vars_:
            entry[v] = literal(body, v)
        out[key] = entry
    line, body = func_body(ops, "TestPow")          # ARange(3, 8, 1, DT_BF16) squared
    out["pow2_arange_3_8"] = {"source": "src/ml/operations_test.go:%d (TestPow, case 1)" % line, "expected": literal(body, "expected")}
    line, body = func_body(ops, "TestMean3dKeepDimTrue")   # createTestInputTensor([5,4,3]) = 1, 2, 3, ... ; mean over the last dim
    out["mean_5x4x3_keepdim"] = {"source": "src/ml/operations_test.go:%d (TestMean3dKeepDimTrue)" % line, "expected": literal(body, "expected")}
    # building blocks of the RoPE table and the causal mask (operations_test.go:56-587)
    cases = []
    for fn in ("TestARangeStep1BF16", "TestARangeMultipleCasesBF16"):
        line, body = func_body(ops, fn)
        exps = re.findall(r"expected\s*:?=\s*\[\]float32\{([^}]*)\}", body)
        calls = re.findall(r"ARange\((-?\d+),\s*(-?\d+),\s*(-?\d+),\s*DT_BF16\)", body)
        assert len(exps) == len(calls) and exps, fn
        for e, c in zip(exps, calls):
            cases.append({"args": [int(x) for x in c], "expected": [float(x) for x in re.findall(NUM, e)],
                          "source": "src/ml/operations_test.go:%d (%s)" % (line, fn)})
    out["arange_bf16"] = cases
    line, body = func_body(ops, "TestOuter")
    calls = re.findall(r"ARange\((-?\d+),\s*(-?\d+),\s*(-?\d+),\s*DT_BF16\)", body)
    out["outer_bf16"] = {"source": "src/ml/operations_test.go:%d (TestOuter)" % line, "vec1_arange": [int(x) for x in calls[0]],
                         "vec2_arange": [int(x) for x in calls[1]], "expected": literal(body, "expected")}
    line, body = func_body(ops, "TestPolar")
    exp = [[float(a), float(b)] for a, b in re.findall(r"complex64\(complex\((%s),\s*(%s)\)\)" % (NUM, NUM), body)]
    absv = [float(x) for x in re.findall(r"abs\.SetItem\(\[\]int\{0, \d\}, float32\((%s)\)\)" % NUM, body)]
    ang = re.findall(r"angle\.SetItem\(\[\]int\{0, \d\}, float32\(([^)]*)\)\)", body)
    assert len(exp) == 5 and len(absv) == 5 and len(ang) == 5
    out["polar"] = {"source": "src/ml/operations_test.go:%d (TestPolar)" % line, "abs": absv, "angle_expr": ang, "expected_re_im": exp}
    triu = []
    for fn in ("TestTriangularUpperOnSquare", "TestTriangularUpperOnLandscapeRectangle", "TestTriangularUpperOnPortraitRectangle"):
        line, body = func_body(ops, fn)
        m = re.search(r"Full\(\[\]int\{(\d+), (\d+)\}, DT_F32, float32\((%s)\)\)" % NUM, body)
        size, fill = [int(m.group(1)), int(m.group(2))], float(m.group(3))
        exps = [m2.group(1) for m2 in re.finditer(r"expected\s*:?=\s*\[\]\[\]float32(\{(?:[^{}]|\{[^{}]*\})*\})", body)]
        diags = [int(x) for x in re.findall(r"TriangularUpper\(originalInput,\s*(-?\d+)\)", body)]
        assert len(exps) == len(diags) and exps, fn
        for e, dg in zip(exps, diags):
            rows = [[float(x) for x in re.findall(NUM, r)] for r in re.findall(r"\{([^{}]*)\}", e)]
            assert len(rows) == size[0] and all(len(r) == size[1] for r in rows), (fn, dg)
            triu.append({"size": size, "fill": fill, "diagonal": dg, "expected": rows, "source": "src/ml/operations_test.go:%d (%s)" % (line, fn)})
    out["triangular_upper"] = triu

    # Tensor.Transpose / SetSlice (KV-cache append and the attention layout changes; src/ml/tensor_test.go)
    tt = read("src/ml/tensor_test.go")
    tr = []
    for fn in ("TestTranspose_Simple", "TestTranspose_Simple_Dim1_Dim3", "TestTranspose_Large"):
        line, body = func_body(tt, fn)
        m = re.search(r"\.Transpose\((\d+),\s*(\d+)\)", body)
        tr.append({"source": "src/ml/tensor_test.go:%d (%s)" % (line, fn), "dims": [int(m.group(1)), int(m.group(2))],
                   "input": literal(body, "inputVals"), "expected": literal(body, "expected")})
    out["transpose"] = tr
    line, body = func_body(tt, "TestSetSlice")
    out["set_slice"] = {"source": "src/ml/tensor_test.go:%d (TestSetSlice)" % line, "input_size": [4, 5],
                        "note": "createTestInputTensor([4,5]) = 1..20 in bf16, written with SetSlice([1],[5]) into [10,5] and "
                                "SetSlice([19,1],[19,5]) into [20,10,5], read back with the same Slice",
                        "expected": literal(body, "expected")}

    # weight-dependent goldens (usable only with the real Meta-Llama-3.1-8B-Instruct checkpoint; SURVEY 8c)
    sim = read("src/model/llamatransformer_simulated_test.go")
    line, body = func_body(sim, "testSimulatedInternal")
    body_nc = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    m = re.search(r"promptTokens := \[\]TokenId\{([^}]*)\}", body_nc)
    prompt = [int(x) for x in re.findall(r"\d+", m.group(1))]
    m = re.search(r"expectedOutputTokenIds := \[\]TokenId\{([^}]*)\}", body_nc)
    toks = [int(x) for x in re.findall(r"\d+", m.group(1))]
    m = re.search(r"expectedLogitsOnlyFirstLayer := \[\]\[\]float32\{(.*?)\n\t\t\t\}", body_nc, re.S)
    rows = [[float(x) for x in re.findall(NUM, r)] for r in re.findall(r"\{([^{}]*)\}", m.group(1))]
    assert len(prompt) == 15 and len(toks) == 5 and len(rows) == 6 and all(len(r) == 6 for r in rows)
    m = re.search(r"inferenceArgs\.SequenceLength = (\d+)", body_nc)
    out["simulated_only_first_layer"] = {
        "source": "src/model/llamatransformer_simulated_test.go:%d (testSimulatedInternal, onlyFirstLayer=true)" % line,
        "needs": "models-original/Meta-Llama-3.1-8B-Instruct (not available offline)",
        "prompt_text": "<|begin_of_text|><|start_header_id|>user<|end_header_id|>\n\nWhat is your name?<|eot_id|><|start_header_id|>assistant<|end_header_id|>\n\n",
        "prompt_tokens": prompt, "sequence_length": int(m.group(1)), "expected_output_tokens": toks,
        "logits_rows": [0, 1, 2, 12, 13, 14], "logits_first3_last3": rows,
        "logits_tolerance": "30 * common.THRESHOLD_BF16 = 0.3 (PyTorch round-to-nearest vs Go truncation)"}
    thr = read("src/common/utils.go")
    m = re.search(r"THRESHOLD_F32\s*=\s*(%s)" % NUM, thr)
    out["threshold_f32"] = {"source": "src/common/utils.go:%d" % (thr.count("\n", 0, m.start()) + 1), "value": float(m.group(1))}

    bft = read("src/dtype/bfloat16_test.go")
    cases = []
    for fn in ("TestNotTruncatedDecimalPart", "TestTruncatedDecimalPart"):
        line, body = func_body(bft, fn)
        exp = re.findall(r"expected\s*:?=\s*float32\((%s)\)" % NUM, body)
        inp = re.findall(r"BFloat16fromFloat32\((%s)\)" % NUM, body)
        assert len(exp) == len(inp) and exp, fn
        cases += [{"input": float(i), "expected": float(e), "source": "src/dtype/bfloat16_test.go:%d (%s)" % (line, fn)} for i, e in zip(inp, exp)]
    out["bf16_from_f32"] = cases
    line, body = func_body(bft, "TestReadBFloat16LittleEndian")
    le = []
    for m in re.finditer(r'"input":\s*\[\]byte\{0x([0-9A-Fa-f]+),\s*0x([0-9A-Fa-f]+)\}.*?"expectedUInt16Bits":\s*uint16\(0x([0-9A-Fa-f]+)\).*?'
                         r'"expectedF32":\s*float32\((%s)\)' % NUM, body, re.S):
        le.append({"bytes": [int(m.group(1), 16), int(m.group(2), 16)], "bits": int(m.group(3), 16), "f32": float(m.group(4))})
    assert len(le) == 3
    out["bf16_little_endian"] = {"source": "src/dtype/bfloat16_test.go:%d (TestReadBFloat16LittleEndian)" % line, "cases": le}

    doc = read("docs/10-ROPE-ROTARY-POSITIONAL-EMBEDDINGS.md")
    m = re.search(r"after running Apply_AsFloat32 and then applyScaling, freqs will be:\s*\nfreqs:\s*\{[^\n]*\n(.*?)\n\}", doc, re.S)
    assert m
    freqs = [float(x) for x in re.findall(NUM, m.group(1))]
    assert len(freqs) == 64, len(freqs)
    out["rope_scaled_inv_freqs"] = {"source": "docs/10-ROPE-ROTARY-POSITIONAL-EMBEDDINGS.md:%d" % (doc.count("\n", 0, m.start(1)) + 1),
                                    "note": "all 64 bf16 inverse frequencies after Llama-3.1 scaling, printed with 5 significant digits",
                                    "values": freqs}

    with open(OUT, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    with open(DIGEST, "w") as f:
        f.write(digest(out) + "\n")
    print("wrote", OUT, "and", DIGEST)


if __name__ == "__main__":
    sys.exit(main())
