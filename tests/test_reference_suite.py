"""The reference's own test-suite, and this repository's versions of its examples, checked on the B200 backend without
the reference tree.

test_reference_unittest_programs replays every program that the reference's unit tests
(tests/{features,std,bug_fixes,large_programs}.py of microsoft/EVA) compile and execute.  The programs, compiler
configurations, input descriptions and what the reference's own compiler and plaintext executor produce for them
are stored in tests/golden/reference_suite.json (tests/golden/gen_reference_suite.py regenerates it).  Each case is
graded by the reference's criteria over every slot (tests/common.py: MSE < 1e-10 between the compiled and the source
program in plaintext, MSE < 0.01 between the decrypted result and the source program in plaintext).  The plaintext
result is tied to the reference's own output values at the stored slots (MSE < 1e-10), the decrypted result is
checked against those values as well, and the encryption parameters must equal the reference compiler's.  A
configuration the reference compiler rejects must be rejected with the same message; the serialization case goes
through save / load at every hand-over, as tests/features.py does.

The two example tests run this repository's examples, not the reference's scripts, with the reference examples'
accuracy check (MSE < 0.01 after decryption): examples/image_processing.py runs the same Sobel and Harris programs as
the reference's example, on the reference example's 64x64 baboon.png (stored under tests/golden/);
examples/serialization.py is a client/server save/load flow of its own, with a program different from the
reference's example.  The reference's own save/load flow is the replayed features test_serialization case.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def make_input(spec, n):
    """the input vector a case describes: {"linear": [a, b]} is a + b*j, {"uniform": [lo, hi], "seed": s} a seeded draw"""
    if "linear" in spec:
        a, b = spec["linear"]
        return a + b * np.arange(n, dtype=np.float64)
    lo, hi = spec["uniform"]
    return np.random.default_rng(spec["seed"]).uniform(lo, hi, n)


def _sampled_mse(outputs, reference):
    """MSE over the stored slots of every output"""
    errs = [np.asarray(outputs[name])[r["slots"]] - np.asarray(r["values"]) for name, r in reference.items()]
    return float(np.mean(np.concatenate(errs) ** 2))


def _execute(case, compiled, params, signature, inputs, tmp_path):
    from eva import load, save
    from eva.seal import generate_keys
    if case["flow"] != "serialization":
        public_ctx, secret_ctx = generate_keys(params)
        return secret_ctx.decrypt(public_ctx.execute(compiled, public_ctx.encrypt(inputs, signature)), signature)
    # every artefact crosses a file between the parties, as in the reference's test_serialization
    path = lambda name: str(tmp_path / name)   # noqa: E731
    save(compiled, path("poly.eva")); save(params, path("poly.evaparams")); save(signature, path("poly.evasignature"))
    public_ctx, secret_ctx = generate_keys(load(path("poly.evaparams")))
    save(public_ctx, path("poly.sealpublic")); save(secret_ctx, path("poly.sealsecret"))
    signature = load(path("poly.evasignature"))
    save(load(path("poly.sealpublic")).encrypt(inputs, signature), path("poly_inputs.sealvals"))
    out = load(path("poly.sealpublic")).execute(load(path("poly.eva")), load(path("poly_inputs.sealvals")))
    save(out, path("poly_outputs.sealvals"))
    return load(path("poly.sealsecret")).decrypt(load(path("poly_outputs.sealvals")), signature)


@pytest.mark.gpu
def test_reference_unittest_programs(tmp_path):
    from eva import evaluate
    from eva.ckks import CKKSCompiler
    from eva.metric import valuation_mse
    from test_compiler_golden import build_source
    with open(os.path.join(GOLDEN, "reference_suite.json")) as f:
        cases = json.load(f)["cases"]
    for i, case in enumerate(cases):
        what = "case %d (%s, %s)" % (i, case["test"], case["source"][0])
        src = build_source(case["source"])
        compiler = CKKSCompiler(config=dict(case["config"], warn_vec_size="false"))
        if "error" in case:
            with pytest.raises(RuntimeError) as ei:
                compiler.compile(src)
            assert str(ei.value) == case["error"], what
            continue
        compiled, params, signature = compiler.compile(src)
        assert list(params.prime_bits) == case["prime_bits"], what
        if case["flow"] == "compile":
            continue
        inputs = {name: list(make_input(spec, src.vec_size)) for name, spec in case["inputs"].items()}
        reference = evaluate(src, inputs)
        assert valuation_mse(reference, evaluate(compiled, inputs)) < 1e-10, what
        assert _sampled_mse(reference, case["reference_outputs"]) < 1e-10, what
        case_dir = tmp_path / str(i)
        case_dir.mkdir()
        outputs = _execute(case, compiled, params, signature, inputs, case_dir)
        he_mse = valuation_mse(outputs, reference)                          # every slot, as tests/common.py
        assert he_mse < 0.01, (what, he_mse)
        he_mse_ref = _sampled_mse(outputs, case["reference_outputs"])       # the reference's own values at the stored slots
        assert he_mse_ref < 0.01, (what, he_mse_ref)


def _run_example(args, cwd):
    env = dict(os.environ)
    env["PYTHONPATH"] = ROOT + os.pathsep + env.get("PYTHONPATH", "")   # `import eva` -> the alias package of this repo
    r = subprocess.run([sys.executable] + args, cwd=cwd, env=env, capture_output=True, text=True, timeout=1200)
    log = r.stdout + r.stderr
    assert r.returncode == 0, log[-6000:]
    return log


@pytest.mark.gpu
def test_image_processing_example_on_reference_image(tmp_path):
    """examples/image_processing.py (the reference example's Sobel and Harris programs) on the reference example's
    64x64 baboon.png: MSE of the decrypted result against plaintext evaluation below 0.01 for both"""
    pytest.importorskip("PIL")
    log = _run_example([os.path.join(ROOT, "examples", "image_processing.py"), os.path.join(GOLDEN, "baboon.png")], str(tmp_path))
    mses = [float(line.split()[-1]) for line in log.splitlines() if "MSE" in line]
    assert len(mses) == 2 and all(m < 0.01 for m in mses), log[-2000:]


@pytest.mark.gpu
def test_serialization_example(tmp_path):
    """examples/serialization.py, this repository's client/server flow: compile -> save; keygen -> save; encrypt -> save;
    load everything on the "server", execute, save; load on the "client", decrypt; MSE below 0.01."""
    log = _run_example([os.path.join(ROOT, "examples", "serialization.py"), str(tmp_path)], str(tmp_path))
    mses = [float(line.split()[-1]) for line in log.splitlines() if line.startswith("MSE")]
    assert len(mses) == 1 and mses[0] < 0.01, log[-2000:]
