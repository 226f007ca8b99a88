"""End to end through the user-facing API, in the style of the reference's own
acceptance tests (tests/common.py:12-36): DSL -> CKKSCompiler -> generate_keys ->
encrypt -> execute (GPU) -> decrypt, compared with evaluate() by MSE < 0.01
(HE vs plaintext) and < 1e-10 (compiled vs source)."""
import random

import pytest

pytestmark = pytest.mark.gpu


def check(prog, inputs, config=None):
    from eva import evaluate
    from eva.ckks import CKKSCompiler
    from eva.metric import valuation_mse
    from eva.seal import generate_keys
    compiler = CKKSCompiler(config) if config else CKKSCompiler()
    compiled, params, signature = compiler.compile(prog)
    reference = evaluate(prog, inputs)
    reference_compiled = evaluate(compiled, inputs)
    assert valuation_mse(reference, reference_compiled) < 1e-10
    public_ctx, secret_ctx = generate_keys(params)
    enc_inputs = public_ctx.encrypt(inputs, signature)
    enc_outputs = public_ctx.execute(compiled, enc_inputs)
    outputs = secret_ctx.decrypt(enc_outputs, signature)
    assert valuation_mse(outputs, reference) < 0.01
    return params


def test_readme_polynomial():
    from eva import EvaProgram, Input, Output
    poly = EvaProgram('Polynomial', vec_size=1024)
    with poly:
        x = Input('x')
        Output('y', 3 * x ** 2 + 5 * x - 2)
    poly.set_output_ranges(30)
    poly.set_input_scales(30)
    p = check(poly, {'x': [i / 1024.0 for i in range(1024)]})
    assert list(p.prime_bits) == [60, 60, 60] and p.poly_modulus_degree == 8192


@pytest.mark.parametrize("is_enc", [(True, True), (True, False), (False, True)])
@pytest.mark.parametrize("op", ["add", "sub", "mul"])
def test_binary_ops(op, is_enc):
    from eva import EvaProgram, Input, Output
    random.seed(1)
    prog = EvaProgram('bin', vec_size=64)
    with prog:
        a, b = Input('a', is_enc[0]), Input('b', is_enc[1])
        Output('y', a + b if op == "add" else a - b if op == "sub" else a * b)
    prog.set_output_ranges(20)
    prog.set_input_scales(30)
    check(prog, {'a': [random.uniform(-2, 2) for _ in range(64)], 'b': [random.uniform(-2, 2) for _ in range(64)]})


def test_rotations_and_unary():
    from eva import EvaProgram, Input, Output
    random.seed(2)
    prog = EvaProgram('rot', vec_size=8)
    with prog:
        x = Input('x')
        Output('l', x << 1)
        Output('r', x >> 2)
        Output('n', -x)
        Output('c', x ** 3)
    prog.set_output_ranges(20)
    prog.set_input_scales(30)
    check(prog, {'x': [random.uniform(-2, 2) for _ in range(8)]})


def test_horizontal_sum_and_mixed():
    from eva import EvaProgram, Input, Output
    from eva.std.numeric import horizontal_sum
    random.seed(3)
    prog = EvaProgram('hsum', vec_size=2048)
    with prog:
        x = Input('x')
        c = Input('c', False)
        Output('y', horizontal_sum(x) * 0.001 + c)
    prog.set_output_ranges(25)
    prog.set_input_scales(25)
    check(prog, {'x': [random.uniform(-1, 1) for _ in range(2048)], 'c': [random.uniform(-1, 1) for _ in range(2048)]})


@pytest.mark.parametrize("rescaler", ["lazy_waterline", "eager_waterline", "always"])
def test_sobel_image(rescaler):
    """examples/image_processing.py:39-63 on a smooth synthetic image"""
    from eva import EvaProgram, Input, Output
    import math
    h = w = 64
    sobel = EvaProgram('sobel', vec_size=h * w)
    with sobel:
        image = Input('image')
        F = [[-1, 0, 1], [-2, 0, 2], [-1, 0, 1]]
        for i in range(3):
            for j in range(3):
                rot = image << (i * w + j)
                hor, ver = rot * F[i][j], rot * F[j][i]
                if i == 0 and j == 0:
                    Ix, Iy = hor, ver
                else:
                    Ix += hor
                    Iy += ver
        d = Ix ** 2 + Iy ** 2
        d2 = d * d
        d3 = d2 * d
        Output('image', d * 2.2137874823876622 + d2 * -1.0984324107372518 + d3 * 0.17254603006834726)
    sobel.set_input_scales(25)
    sobel.set_output_ranges(10)
    img = [0.5 + 0.25 * math.sin(0.1 * (k % w)) * math.cos(0.07 * (k // w)) for k in range(h * w)]
    p = check(sobel, {'image': img}, {"rescaler": rescaler})
    if rescaler == "lazy_waterline":
        assert list(p.prime_bits) == [60] * 5 and p.poly_modulus_degree == 16384


def test_security_levels_and_error_paths():
    from eva import EvaProgram, Input, Output
    from eva.ckks import CKKSCompiler
    prog = EvaProgram('sec', vec_size=64)
    with prog:
        x = Input('x')
        Output('y', x * x)
    prog.set_output_ranges(20)
    prog.set_input_scales(30)
    for s in ("128", "192", "256"):
        for q in ("false", "true"):
            check(prog, {'x': [0.5] * 64}, {"security_level": s, "quantum_safe": q, "warn_vec_size": "false"})
    with pytest.raises(RuntimeError):
        CKKSCompiler({"security_level": "1024"}).compile(prog)


def test_regressions_like_reference_large_programs():
    """linear (63 inputs), polynomial and multivariate regression: reference tests/large_programs.py:55-146"""
    from eva import EvaProgram, Input, Output
    lin = EvaProgram('linear_regression', vec_size=2048)
    with lin:
        p = 63
        x = [Input('x%d' % i) for i in range(p)]
        y = Input('e') + 6.56
        for i in range(p):
            y += x[i] * (i * 0.732)
        Output('y', y)
    lin.set_input_scales(40); lin.set_output_ranges(30)
    ins = {'e': [(2048 - i) * 0.001 for i in range(2048)]}
    for i in range(63):
        ins['x%d' % i] = [i * j * 0.01 for j in range(2048)]
    check(lin, ins, {'warn_vec_size': 'false'})

    pol = EvaProgram('polynomial_regression', vec_size=4096)
    with pol:
        x, y = Input('x'), Input('e') + 6.56
        for i in range(4):
            xi = x
            for _ in range(i):
                xi = xi * x
            y += xi * (i * 0.732)
        Output('y', y)
    pol.set_input_scales(40); pol.set_output_ranges(30)
    check(pol, {'x': [i * 0.0001 for i in range(4096)], 'e': [(4096 - i) * 0.001 for i in range(4096)]}, {'warn_vec_size': 'false'})


def test_high_inner_term_scale_and_transparent():
    """reference tests/bug_fixes.py:10-26 and tests/features.py:135-152"""
    from eva import EvaProgram, Input, Output
    prog = EvaProgram('HighInnerTermScale', vec_size=4)
    with prog:
        x1, x2 = Input('x1'), Input('x2')
        Output('y', x1 * x1 * x2)
    prog.set_output_ranges(20); prog.set_input_scales(60)
    check(prog, {'x1': [0.5, -1.0, 1.5, 2.0], 'x2': [1.0, 0.25, -0.5, 1.25]}, {'rescaler': 'lazy_waterline', 'warn_vec_size': 'false'})
    tr = EvaProgram('Transparent', vec_size=4096)
    with tr:
        x = Input('x')
        Output('y', x - x + x * 0)
    tr.set_output_ranges(20); tr.set_input_scales(30)
    check(tr, {'x': [0.001 * i for i in range(4096)]}, {'warn_vec_size': 'false'})


def test_harris_and_large_sobel():
    """Harris corner detector (examples/image_processing.py:65-100) and the 90x90 Sobel of
    tests/large_programs.py:10-53 (vec 8192, scale 45, range 20) with balance on/off"""
    import math
    from tests_programs import harris
    img = [0.5 + 0.25 * math.sin(0.1 * (k % 64)) * math.cos(0.07 * (k // 64)) for k in range(4096)]
    check(harris(), {'image': img}, {'warn_vec_size': 'false'})
    from eva import EvaProgram, Input, Output
    from tests_programs import _conv_xy, SOBEL_FILTER
    sob = EvaProgram('sobel', vec_size=8192)
    with sob:
        image = Input('image')
        ix, iy = _conv_xy(image, 90, SOBEL_FILTER)
        x = ix ** 2 + iy ** 2
        Output('image', x * 2.2137874823876622 + x ** 2 * -1.0984324107372518 + x ** 3 * 0.17254603006834726)
    sob.set_input_scales(45); sob.set_output_ranges(20)
    img = [0.5 + 0.25 * math.sin(0.05 * (k % 90)) for k in range(8192)]
    for bal in ('true', 'false'):
        check(sob, {'image': img}, {'balance_reductions': bal, 'warn_vec_size': 'false'})


def _two_input_program():
    from eva import EvaProgram, Input, Output
    from eva.ckks import CKKSCompiler
    prog = EvaProgram('two', vec_size=64)
    with prog:
        a, b = Input('a'), Input('b')
        Output('y', a * b + a)
    prog.set_output_ranges(30)
    prog.set_input_scales(30)
    return CKKSCompiler({'warn_vec_size': 'false'}).compile(prog)


def test_untrusted_valuations_are_validated():
    """plans are cached per program: an omitted input must not silently reuse the previous call's ciphertext, and a
    ciphertext / plaintext whose buffer does not match the plan's shape must never reach the device arena"""
    import numpy as np
    from eva.seal import generate_keys
    from eva_b200 import b200
    compiled, params, signature = _two_input_program()
    public_ctx, secret_ctx = generate_keys(params)
    x = {'a': [0.5] * 64, 'b': [0.25] * 64}
    enc = public_ctx.encrypt(x, signature)
    public_ctx.execute(compiled, enc)                      # builds and caches the plan
    only_a = b200.B200Valuation()
    kind, arr, scale = enc.get('a')
    only_a.set_cipher('a', arr, scale)
    with pytest.raises(RuntimeError, match="Missing input value"):
        public_ctx.execute(compiled, only_a)
    bad = b200.B200Valuation()
    bad.set_cipher('a', arr, scale)
    bad.set_cipher('b', np.ascontiguousarray(arr[:, :, : arr.shape[2] // 2]), scale)      # half the coefficients
    with pytest.raises(RuntimeError, match="does not match the program signature"):
        public_ctx.execute(compiled, bad)
    bad2 = b200.B200Valuation()
    bad2.set_cipher('a', arr, scale)
    bad2.set_cipher('b', np.ascontiguousarray(arr[:, :-1]), scale)                         # one residue short
    with pytest.raises(RuntimeError, match="does not match the program signature"):
        public_ctx.execute(compiled, bad2)
    with pytest.raises(RuntimeError, match=r"\[ell\]\[N\]"):
        bad2.set_plain('b', arr, scale)
    # the context still works after the rejected calls
    out = secret_ctx.decrypt(public_ctx.execute(compiled, enc), signature)
    assert abs(out['y'][0] - (0.5 * 0.25 + 0.5)) < 1e-3


def test_randomness_default_is_os_entropy_and_seed_is_reproducible():
    """generate_keys() draws from a ChaCha20 stream keyed by the OS (two contexts never share key material);
    generate_keys(seed=...) is the deterministic test path"""
    import numpy as np
    from eva_b200 import b200
    compiled, params, signature = _two_input_program()
    pk = lambda ctx: ctx._export()["public_key"]
    a, _ = b200.generate_keys(params)
    b, _ = b200.generate_keys(params)
    assert not np.array_equal(pk(a), pk(b))
    c, _ = b200.generate_keys(params, seed=7)
    d, _ = b200.generate_keys(params, seed=7)
    assert np.array_equal(pk(c), pk(d)) and not np.array_equal(pk(a), pk(c))
    # uniform halves of the public key look uniform: mean of the top byte near 127.5 is too weak a test to be worth it;
    # check instead that no residue repeats between the two independently keyed contexts
    assert len(np.intersect1d(pk(a)[1, 0, :256], pk(b)[1, 0, :256])) == 0


def test_debug_verbosity_prints_every_executed_term():
    """EVA_VERBOSITY=debug: the reference prints `EVA: Execute t<i> = <Op>(t<j>,...)` per term
    (eva/seal/seal_executor.h:280-294); so does the plan replay (with the stream it went to), inside NVTX ranges"""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (
        "from eva import EvaProgram, Input, Output\n"
        "from eva.ckks import CKKSCompiler\n"
        "from eva.seal import generate_keys\n"
        "p = EvaProgram('poly', vec_size=64)\n"
        "with p:\n"
        "    x = Input('x')\n"
        "    Output('y', 3 * x ** 2 + 5 * x - 2)\n"
        "p.set_output_ranges(30); p.set_input_scales(30)\n"
        "c, params, sig = CKKSCompiler({'warn_vec_size': 'false'}).compile(p)\n"
        "pub, sec = generate_keys(params)\n"
        "out = sec.decrypt(pub.execute(c, pub.encrypt({'x': [0.5] * 64}, sig)), sig)\n"
        "print('RESULT', out['y'][0])\n")
    env = dict(os.environ, EVA_VERBOSITY="debug", PYTHONPATH=root)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("EVA: Execute t")]
    ops = {l.split("= ")[1].split("(")[0] for l in lines}
    assert {"Mul", "Relinearize", "Rescale", "Add"} <= ops, ops
    assert all("[stream " in l for l in lines)
    res = [l for l in r.stdout.splitlines() if l.startswith("RESULT")]
    assert abs(float(res[0].split()[1]) - (3 * 0.25 + 2.5 - 2)) < 1e-3


def test_approx_hoist_is_opt_in_and_accurate():
    """set_options(approx_hoist=True): one mod-down per weighted sum of rotations of one ciphertext (SURVEY 8f-4).
    Not bit-exact with the reference by construction -- graded like the reference's own tests, by MSE against
    evaluate() (tests/common.py:30-36), and it has to stay as close to the plaintext result as the exact path."""
    import math
    from eva import evaluate
    from eva.ckks import CKKSCompiler
    from eva.metric import valuation_mse
    from eva.seal import generate_keys
    from tests_programs import harris, sobel
    for prog, n in ((sobel(), 4096), (harris(), 4096)):
        img = [0.5 + 0.25 * math.sin(0.1 * (k % 64)) * math.cos(0.07 * (k // 64)) for k in range(n)]
        compiled, params, signature = CKKSCompiler({'warn_vec_size': 'false'}).compile(prog)
        reference = evaluate(prog, {'image': img})
        public_ctx, secret_ctx = generate_keys(params)
        enc = public_ctx.encrypt({'image': img}, signature)
        exact = secret_ctx.decrypt(public_ctx.execute(compiled, enc), signature)
        public_ctx.set_options(approx_hoist=True)
        approx = secret_ctx.decrypt(public_ctx.execute(compiled, enc), signature)
        public_ctx.set_options(approx_hoist=False)
        again = secret_ctx.decrypt(public_ctx.execute(compiled, enc), signature)
        e_exact, e_approx = valuation_mse(exact, reference), valuation_mse(approx, reference)
        assert e_exact < 0.01 and e_approx < 0.01
        assert e_approx < 4 * e_exact + 1e-12, (e_exact, e_approx)
        assert valuation_mse(approx, exact) < 4 * (e_exact + e_approx) + 1e-12   # two noisy results of the same computation
        assert valuation_mse(again, exact) == 0.0          # switching the option back rebuilds the exact plan


def test_approx_hoist_plan_shapes():
    """approx_hoist on the plan shapes that take its special cases: more than 16 taps of one ciphertext, a rotation that is
    also used outside the weighted sum (it must still be materialised), the same rotation twice in one sum, vector weights,
    weights that depend on an unencrypted input (encoded inside every execute), sums at two levels"""
    import numpy as np
    from eva import EvaProgram, Input, Output, evaluate
    from eva.ckks import CKKSCompiler
    from eva.metric import valuation_mse
    from eva.seal import generate_keys
    n = 1024
    rng = np.random.default_rng(5)
    vecs = [list(rng.uniform(-1, 1, n)) for _ in range(24)]

    def many_taps():
        acc = None
        x = Input('x')
        for k in range(20):
            t = (x << (k + 1)) * (0.05 * (k + 1))
            acc = t if acc is None else acc + t
        Output('y', acc)

    def shared_rotation():
        x = Input('x')
        r1, r2, r3 = x << 1, x << 2, x >> 3
        s = r1 * 0.5 + r2 * vecs[0] + r3 * -0.25
        Output('y', s + r2)              # r2 is needed as a ciphertext as well
        Output('z', r1 * r1)             # and r1 feeds a ciphertext product

    def repeated_rotation():
        x = Input('x')
        r = x << 5
        Output('y', r * 0.5 + (x << 6) * vecs[1] + r * vecs[2] + (x >> 1) * 2.0)

    def input_weights():
        x, w = Input('x'), Input('w', is_encrypted=False)
        Output('y', (x << 1) * w + (x << 2) * 0.75 + (x << 3) * w)

    def two_levels():
        x = Input('x')
        a = (x << 1) * 0.5 + (x << 2) * 0.25 + (x << 4) * vecs[3]
        b = a * a
        Output('y', (b << 1) * 0.5 + (b << 2) * vecs[4] + (b >> 7) * -1.5 + b)

    for body in (many_taps, shared_rotation, repeated_rotation, input_weights, two_levels):
        prog = EvaProgram(body.__name__, vec_size=n)
        with prog:
            body()
        prog.set_input_scales(30)
        prog.set_output_ranges(20)
        compiled, params, signature = CKKSCompiler({'warn_vec_size': 'false'}).compile(prog)
        inputs = {'x': list(rng.uniform(-1, 1, n))}
        if body is input_weights:
            inputs['w'] = list(rng.uniform(-1, 1, n))
        reference = evaluate(prog, inputs)
        # deterministic keys and encryption: these programs get a 20-bit prime, and a zero coefficient of the input's digit
        # modulo it (about 1 % of random encryptions at N = 8192) makes execute() drop the shared mod-up, and with it the
        # lazy sums, for the rest of the context (backend.hpp collect) -- a different plan from the one checked here
        public_ctx, secret_ctx = generate_keys(params, seed=17)
        enc = public_ctx.encrypt(inputs, signature)
        exact = secret_ctx.decrypt(public_ctx.execute(compiled, enc), signature)
        public_ctx.set_options(approx_hoist=True)
        approx = secret_ctx.decrypt(public_ctx.execute(compiled, enc), signature)
        approx2 = secret_ctx.decrypt(public_ctx.execute(compiled, enc), signature)     # the captured graph
        st = public_ctx.plan_stats(compiled)
        want = {'many_taps': (2, 20, 20), 'shared_rotation': (1, 3, 1), 'repeated_rotation': (1, 3, 2), 'input_weights': (1, 3, 3),
                'two_levels': (2, 6, 6)}[body.__name__]   # lazy sums, rotations in them, rotations never materialised
        assert (st['lazy_sums'], st['lazy_rotations'], st['elided_rotations']) == want, (body.__name__, st)
        e_exact, e_approx = valuation_mse(exact, reference), valuation_mse(approx, reference)
        assert e_exact < 1e-6 and e_approx < 4 * e_exact + 1e-12, (body.__name__, e_exact, e_approx)
        assert valuation_mse(approx, approx2) == 0.0, body.__name__


def test_pipelined_execute_batch():
    """execute_batch_async / execute_batch_result: two batches in flight on disjoint plan replicas give the bits of the blocking
    call; a slot takes one batch at a time; a handle that is dropped uncollected waits for its copies"""
    import numpy as np
    from eva.ckks import CKKSCompiler
    from eva.seal import generate_keys
    from tests_programs import sobel
    compiled, params, signature = CKKSCompiler({'warn_vec_size': 'false'}).compile(sobel(32, 32))
    public_ctx, secret_ctx = generate_keys(params)
    rng = np.random.default_rng(2)
    batches = [[public_ctx.encrypt({'image': list(rng.uniform(0, 1, 1024))}, signature) for _ in range(3)] for _ in range(3)]
    want = [public_ctx.execute_batch(compiled, b) for b in batches]

    def same(a, b):
        for x, y in zip(a, b):
            for name in x.names():
                assert np.array_equal(np.asarray(x.get(name)[1]), np.asarray(y.get(name)[1]))
    h0 = public_ctx.execute_batch_async(compiled, batches[0], 0)
    h1 = public_ctx.execute_batch_async(compiled, batches[1], 1)
    with pytest.raises(RuntimeError, match="slot in use"):
        public_ctx.execute_batch_async(compiled, batches[2], 1)
    same(public_ctx.execute_batch_result(h0), want[0])
    h2 = public_ctx.execute_batch_async(compiled, batches[2], 0)
    same(public_ctx.execute_batch_result(h1), want[1])
    same(public_ctx.execute_batch_result(h2), want[2])
    with pytest.raises(RuntimeError, match="collected already"):
        public_ctx.execute_batch_result(h2)
    h3 = public_ctx.execute_batch_async(compiled, batches[0], 2)
    del h3                                   # never collected
    same(public_ctx.execute_batch(compiled, batches[0]), want[0])


def test_approx_hoist_batched_equals_single():
    """approx_hoist is deterministic: instances fused into one launch (fuse=2, execute_batch) give the bits of separate execute() calls"""
    import numpy as np
    from eva.ckks import CKKSCompiler
    from eva.seal import generate_keys
    from tests_programs import sobel
    compiled, params, signature = CKKSCompiler({'warn_vec_size': 'false'}).compile(sobel(32, 32))
    public_ctx, secret_ctx = generate_keys(params)
    rng = np.random.default_rng(9)
    vals = [public_ctx.encrypt({'image': list(rng.uniform(0, 1, 1024))}, signature) for _ in range(4)]
    public_ctx.set_options(approx_hoist=True, fuse=2)
    batched = public_ctx.execute_batch(compiled, vals)
    public_ctx.set_options(approx_hoist=True, fuse=1)
    for v, b in zip(vals, batched):
        single = public_ctx.execute(compiled, v)
        for name in single.names():
            assert np.array_equal(np.asarray(single.get(name)[1]), np.asarray(b.get(name)[1]))
    assert public_ctx.plan_stats(compiled)['lazy_sums'] == 2
