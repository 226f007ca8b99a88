"""Generates tests/golden/reference_suite.json: every encrypted check of the reference's own unit-test suite
(tests/{features,bug_fixes,large_programs,std}.py of a microsoft/EVA checkout) as data, so that
tests/test_reference_suite.py replays it on this backend without the reference tree.

The reference's test modules run here against this package (`import eva` is the alias package of this repository)
with key generation, encryption, execution and decryption replaced by recorders, so no GPU is needed.  Every
program that one of those tests compiles and executes becomes one case: the source program (in the line format of
tests/golden/programs, see oracle/ref_compiler/driver.cpp), the compiler configuration, a description of the
inputs, and what the reference's own compiler and plaintext executor (oracle/_ref/eva_ref_compile, built by
oracle/ref_compiler/build.sh) produce for it: encryption parameters, or the compile error, and the output values.

Limit: the source programs are built by this repository's `eva` front end (the DSL operators, constant conversion
and the order of operands), because the reference's Python front end needs its native module, which cannot be
built without SEAL.  Only the compilation and the plaintext evaluation of each program come from the reference's
code.  A difference between the two front ends' lowering of the DSL would therefore be stored in the fixture, not
caught by it.

Inputs the reference draws at random are replaced by seeded uniform draws from the same interval; inputs it
computes as a + b*j are kept as that progression.  Outputs are stored at up to SAMPLE slots per output (a fixed,
seeded choice), which keeps the file small.

Usage: python tests/golden/gen_reference_suite.py <reference checkout>
"""
import json
import os
import subprocess
import sys
import unittest

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
PROBE = os.path.join(ROOT, "oracle", "_ref", "eva_ref_compile")
OUT = os.path.join(HERE, "reference_suite.json")
SAMPLE = 64
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
from test_reference_suite import make_input  # noqa: E402  (the replay draws the same inputs)


def source_lines(prog):
    """the source program as the line format the reference driver reads"""
    lines = ["program %s %d" % (prog.name, prog.vec_size)]
    names = {t.index: n for n, t in prog.outputs.items()}
    for t in prog.terms():
        a, op = t.attributes, str(t.op).split(".")[1]
        ids = [o.index for o in t.operands]
        if op == "Input":
            ty = str(a["TypeAttribute"]).split(".")[1].lower()
            lines.append("input %d %s %s" % (t.index, [n for n, x in prog.inputs.items() if x.index == t.index][0], ty))
        elif op == "Constant":
            c = list(a["ConstantValueAttribute"])
            if len(set(c)) == 1:
                lines.append("uconst %d %r" % (t.index, float(c[0])))
            else:
                lines.append("dconst %d %d %s" % (t.index, len(c), " ".join(repr(float(x)) for x in c)))
        elif op in ("RotateLeftConst", "RotateRightConst"):
            lines.append("%s %d %d %d" % ("rotl" if op == "RotateLeftConst" else "rotr", t.index, ids[0], a["RotationAttribute"]))
        elif op == "Output":
            lines.append("output %s %d" % (names[t.index], ids[0]))
        else:
            lines.append("term %d %s %s" % (t.index, op, " ".join(map(str, ids))))
    return lines


def input_spec(values, seed):
    """a + b*j when the values are that progression, else a seeded uniform draw over [-2, 2] (the reference's interval)"""
    v = np.asarray(values, dtype=np.float64)
    j = np.arange(len(v), dtype=np.float64)
    if len(v) > 1:
        a, b = float(v[0]), float(v[1] - v[0])
        if np.allclose(v, a + b * j, rtol=1e-12, atol=1e-12 * max(1.0, float(np.abs(v).max()))):
            return {"linear": [a, b]}
    return {"uniform": [-2.0, 2.0], "seed": seed}


def reference_run(lines, config, inputs):
    txt = list(lines) + ["config %s %s" % kv for kv in sorted(config.items())]
    txt += ["evaluate"] + ["evalinput %s %d %s" % (k, len(v), " ".join(repr(float(x)) for x in v)) for k, v in sorted(inputs.items())]
    res = subprocess.run([PROBE], input=("\n".join(txt) + "\n").encode(), stdout=subprocess.PIPE, check=True).stdout.decode()
    return json.loads(res)


class Recorder:
    def __init__(self):
        self.cases, self.test, self.compiled = [], None, {}

    def add(self, source, config, inputs, flow):
        n = len(self.cases)
        lines = source_lines(source) + ["scales %d" % self.scale_of(source), "ranges %d" % self.range_of(source)]
        specs = {k: input_spec(v, 1000 + 16 * n + i) for i, (k, v) in enumerate(sorted(inputs.items()))}
        vals = {k: make_input(s, source.vec_size) for k, s in specs.items()}
        cfg = {k: str(v) for k, v in config.items() if k != "warn_vec_size"}
        ref = reference_run(lines, cfg, vals)
        case = {"test": self.test, "flow": flow, "source": lines, "config": cfg, "inputs": specs}
        if "error" in ref:
            case["error"] = ref["error"]
        else:
            case["prime_bits"] = ref["prime_bits"]
            outs = {}
            for name, v in ref["reference_outputs"].items():
                idx = np.arange(len(v)) if len(v) <= SAMPLE else np.sort(np.random.default_rng(n).choice(len(v), SAMPLE, replace=False))
                outs[name] = {"slots": [int(i) for i in idx], "values": [v[i] for i in idx]}
            case["reference_outputs"] = outs
        self.cases.append(case)

    # scales and ranges are attributes of the source's inputs / outputs
    @staticmethod
    def scale_of(prog):
        return int(next(iter(prog.inputs.values())).attributes.get("EncodeAtScaleAttribute", 0)) if prog.inputs else Recorder.const_scale(prog)

    @staticmethod
    def const_scale(prog):
        for t in prog.terms():
            if "EncodeAtScaleAttribute" in t.attributes:
                return int(t.attributes["EncodeAtScaleAttribute"])
        return 0

    @staticmethod
    def range_of(prog):
        return int(next(iter(prog.outputs.values())).attributes["RangeAttribute"])


def main(refdir):
    sys.path.insert(0, os.path.join(refdir, "tests"))
    import eva
    import eva.ckks
    import eva.seal
    rec = Recorder()
    real_compiler = eva.ckks.CKKSCompiler

    class Compiler:
        def __init__(self, config=None):
            self._config = dict(config or {})
            self._real = real_compiler(config=self._config)

        def compile(self, prog):
            try:
                res = self._real.compile(prog)
            except Exception:
                rec.add(prog, self._config, {n: [0.0] * prog.vec_size for n in prog.inputs}, "error")
                raise
            rec.compiled[id(res[0])] = [prog, dict(self._config), False]   # source, configuration, executed
            return res

    class Public:
        def encrypt(self, inputs, signature):
            return ("enc", inputs)

        def execute(self, prog, enc):
            entry = rec.compiled[id(prog)]
            entry[2] = True
            rec.add(entry[0], entry[1], enc[1], "serialization" if rec.test.endswith("test_serialization") else "execute")
            return ("out", prog, enc[1])

    class Secret:
        def decrypt(self, out, signature):
            return eva.evaluate(out[1], out[2])

    store = {}
    eva.ckks.CKKSCompiler = Compiler
    eva.seal.generate_keys = lambda params: (Public(), Secret())
    eva.save = lambda obj, path: store.__setitem__(path, obj)
    eva.load = lambda path: store[path]
    suite = unittest.defaultTestLoader.loadTestsFromNames(["features", "bug_fixes", "large_programs", "std"])

    def flat(s):
        for t in s:
            yield from (flat(t) if isinstance(t, unittest.TestSuite) else [t])
    for t in flat(suite):
        rec.test = t.id()
        r = unittest.TestResult()
        t.run(r)
        for src, cfg, executed in rec.compiled.values():   # compiled and checked, never executed: parameters only
            if not executed:
                rec.add(src, cfg, {n: [0.0] * src.vec_size for n in src.inputs}, "compile")
        rec.compiled.clear()
        assert r.wasSuccessful() or r.expectedFailures, (t.id(), r.errors, r.failures)
    with open(OUT, "w") as f:
        f.write('{"generated_from": "tests/{features,bug_fixes,large_programs,std}.py of microsoft/EVA", "sample": %d, "cases": [\n' % SAMPLE)
        f.write(",\n".join(json.dumps(c) for c in rec.cases) + "\n]}\n")
    print("%d cases -> %s (%d bytes)" % (len(rec.cases), OUT, os.path.getsize(OUT)))


if __name__ == "__main__":
    main(sys.argv[1])
