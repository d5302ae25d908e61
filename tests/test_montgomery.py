"""Montgomery-form helpers (SURVEY 8(f)-4): the oracle's restatement and the product's host functions against the
known answers the reference's tests hold (test/test-avx512-util.cpp:359-470, test/test-eltwise-reduce-mod-avx512.cpp:38-64,
test/test-eltwise-mult-mod-avx512.cpp:210-262), the restatement against the compiled reference on random inputs, and --
on the GPU -- the element-wise kernels against the checker."""
import numpy as np
import pytest

from util import sha, uniform_below

MASK64 = (1 << 64) - 1
# (modulus, r, T, T * 2^-r mod modulus): restated from the reference's tests
REDC_KATS = [(5, 3, t, o) for t, o in zip([0, 1, 4, 6, 8, 9, 12, 16], [0, 2, 3, 2, 1, 3, 4, 2])] + \
            [(5, 3, t, o) for t, o in zip([0, 2, 3, 2, 1, 3, 4, 2], [0, 4, 1, 4, 2, 1, 3, 4])] + \
            [(67280421310725, 46, 59999999999996 * 42006526039321, 1546598034044),
             (2251799813684809, 51, (5446 << 52) + 3006504763740625, 1832909426971103)]


def _cases():
    """(q, r): the reference's test parameters plus the range ends"""
    return [(67280421310725, 46), ((1 << 60) + 7, 61), ((1 << 61) - 1, 61), ((1 << 61) + 37, 62), (0x1FFFFC001, 33),
            (769, 10), (5, 3)]


def _kat_arrays(q, r):
    """operands a, b (0, 1 and q-1 first), R^2 mod q, and the known answers a*b/R, a*R and a*b mod q"""
    R = 1 << r
    n = 1031
    a, b = uniform_below(q % 1000, n, q), uniform_below(q % 1000 + 1, n, q)
    a[:3] = [0, 1, q - 1]
    b[:3] = [q - 1, q - 1, q - 1]
    rinv = pow(R, -1, q)
    exp_mul = np.array([int(x) * int(y) * rinv % q for x, y in zip(a, b)], dtype=np.uint64)
    exp_fin = np.array([int(x) * R % q for x in a], dtype=np.uint64)
    plain = np.array([int(x) * int(y) % q for x, y in zip(a, b)], dtype=np.uint64)
    return a, b, R * R % q, exp_mul, exp_fin, plain


def _check_impl(impl):
    assert impl.hensel_lemma_2adic_root(46, 67280421310725) == 62463730494515  # test-avx512-util.cpp:417
    for q, r, T, out in REDC_KATS:
        inv = impl.hensel_lemma_2adic_root(r, q)
        assert (q * inv + 1) % (1 << r) == 0 and inv < (1 << r)
        assert impl.montgomery_reduce(T >> 64, T & MASK64, q, r, inv) == out, (q, r, T)
    for q, r in _cases():
        inv = impl.hensel_lemma_2adic_root(r, q)
        a, b, r2, exp_mul, exp_fin, plain = _kat_arrays(q, r)
        assert (impl.mont_reduce_mod(a, b, q, r, inv) == exp_mul).all(), (q, r)
        fin = impl.montgomery_form_in(a, r2, q, r, inv)
        assert (fin == exp_fin).all(), (q, r)
        assert (impl.montgomery_form_out(fin, q, r, inv) == a).all(), (q, r)               # test-eltwise-reduce-mod-avx512.cpp:59-64
        assert (impl.mont_reduce_mod(fin, b, q, r, inv) == plain).all(), (q, r)            # test-eltwise-mult-mod-avx512.cpp:229-236


def test_restatement_against_the_reference_kats(port):
    _check_impl(port)


def test_compiled_reference_against_its_own_kats_and_the_restatement(reference_outputs, port):
    """What the compiled reference returned (tests/golden/reference_outputs.json: scalars, and SHA-256 of arrays)
    against the known answers, and against the restatement on random inputs."""
    ref = reference_outputs["montgomery"]
    assert ref["hensel_lemma_2adic_root(46, 67280421310725)"] == 62463730494515   # test-avx512-util.cpp:417
    assert ref["montgomery_reduce"] == [out for *_, out in REDC_KATS]
    for q, r in _cases():
        c = ref["cases"][f"{q},{r}"]
        inv = port.hensel_lemma_2adic_root(r, q)
        assert c["inv"] == inv
        a, b, _, exp_mul, exp_fin, plain = _kat_arrays(q, r)
        assert c["kat mont_reduce_mod"] == sha(exp_mul), (q, r)
        assert c["kat montgomery_form_in"] == sha(exp_fin), (q, r)
        assert c["kat montgomery_form_out"] == sha(a), (q, r)
        assert c["kat mont_reduce_mod of form_in"] == sha(plain), (q, r)
        a, b = uniform_below(3, 4099, q), uniform_below(4, 4099, q)
        assert c["mont_reduce_mod"] == sha(port.mont_reduce_mod(a, b, q, r, inv)), (q, r)
        if r in (46, 61) and ref["avx512"]:
            assert c["avx512 helper"]  # the reference's own AVX-512 helper produced these bits


def test_product_host_functions(hb):
    """hexl_b200_hensel_lemma_2adic_root / hexl_b200_montgomery_reduce run on the host (no GPU needed)"""
    assert hb.HenselLemma2adicRoot(46, 67280421310725) == 62463730494515
    for q, r, T, out in REDC_KATS:
        inv = hb.HenselLemma2adicRoot(r, q)
        assert hb.MontgomeryReduce(T >> 64, T & MASK64, q, r, inv) == out
    assert hb.HenselLemma2adicRoot(10, 768) == 0 and hb.HenselLemma2adicRoot(0, 769) == 0   # invalid arguments
    x = np.zeros(8, dtype=np.uint64)
    for bad in (lambda: hb.EltwiseMontReduceMod(x, x, x, 8, 768, 10, 1),        # even modulus
                lambda: hb.EltwiseMontReduceMod(x, x, x, 8, 769, 9, 1),         # R <= q
                lambda: hb.EltwiseMontReduceMod(x, x, x, 8, 769, 63, 1),        # r > 62
                lambda: hb.EltwiseMontReduceMod(x, x, x, 8, 769, 10, 12345),    # not -1/q mod R
                lambda: hb.EltwiseMontgomeryFormIn(x, x, 769, 8, 769, 10, hb.HenselLemma2adicRoot(10, 769)),  # R2 >= q
                lambda: hb.EltwiseMontgomeryFormOut(x, x, 0, 769, 10, hb.HenselLemma2adicRoot(10, 769))):     # n == 0
        with pytest.raises(hb.HexlB200Error):
            bad()


@pytest.mark.gpu
def test_montgomery_kernels_match_the_checker(hb, checker):
    torch = pytest.importorskip("torch")

    def dev(a):
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint64).view(np.int64)).cuda()

    def host(t):
        return t.cpu().numpy().view(np.uint64)

    for q, r in _cases():
        inv = hb.HenselLemma2adicRoot(r, q)
        r2 = (1 << r) * (1 << r) % q
        for n in (1, 7, 4096 + 5, 1 << 18):
            a, b = uniform_below(n + r, n, q), uniform_below(n + r + 1, n, q)
            if n > 3:
                a[:3] = [0, 1, q - 1]
                b[:3] = [q - 1] * 3
            da, db, o = dev(a), dev(b), dev(np.zeros_like(a))
            assert (host(hb.EltwiseMontReduceMod(o, da, db, n, q, r, inv)) == checker.mont_reduce_mod(a, b, q, r, inv)).all()
            fin = host(hb.EltwiseMontgomeryFormIn(o, da, r2, n, q, r, inv)).copy()
            assert (fin == checker.montgomery_form_in(a, r2, q, r, inv)).all()
            assert (host(hb.EltwiseMontgomeryFormOut(o, o, n, q, r, inv)) == a).all()          # in place, round trip
            if q < (1 << 62):
                plain = host(hb.EltwiseMultMod(dev(np.zeros_like(a)), da, db, n, q, 1))
                assert (host(hb.EltwiseMontReduceMod(o, dev(fin), db, n, q, r, inv)) == plain).all()
    # host pointers and an unaligned view
    q, r = (1 << 60) + 7, 61
    inv = hb.HenselLemma2adicRoot(r, q)
    n = (5 << 20) + 3
    a, b = uniform_below(1, n, q), uniform_below(2, n, q)
    h = np.zeros_like(a)
    hb.EltwiseMontReduceMod(h, a, b, n, q, r, inv)
    assert (h == checker.mont_reduce_mod(a, b, q, r, inv)).all()
    buf = torch.zeros(1025, dtype=torch.int64, device="cuda")
    buf[1:] = dev(a[:1024])
    out = torch.zeros(1025, dtype=torch.int64, device="cuda")
    hb.EltwiseMontgomeryFormOut(out[1:], buf[1:], 1024, q, r, inv)
    assert (host(out[1:]) == checker.montgomery_form_out(a[:1024], q, r, inv)).all()


RADIX4_CASES = ((4, 30), (5, 40), (10, 50), (11, 55), (12, 60), (13, 61), (15, 45), (16, 55), (17, 60))


def radix4_inputs(logn, q):
    """("forward" | "inverse", in_mf, out_mf, x) of every transform compared with the reference's radix-4 path"""
    n = 1 << logn
    for in_mf, out_mf in ((1, 1), (4, 1), (2, 4)):
        yield "forward", in_mf, out_mf, uniform_below(logn + in_mf, n, q * in_mf)
    for in_mf, out_mf in ((1, 1), (2, 1), (2, 2)):
        yield "inverse", in_mf, out_mf, uniform_below(logn + 7 + in_mf, n, q * in_mf)


@pytest.mark.gpu
def test_ntt_matches_the_references_radix4_path(hb, reference_outputs):
    """The register passes of the sm_100a kernels consume twiddles by the reference's radix-4 index rule
    (W[m+i], W[2(m+i)], W[2(m+i)+1] = a tree node and its two children, ntt-radix-4.cpp:223-233; odd log2 N starts
    with one radix-2 stage, :49-71): their outputs must equal ForwardTransformToBitReverseRadix4 /
    InverseTransformFromBitReverseRadix4 of the compiled reference bit for bit (lazy outputs mod q).  The reference's
    outputs are recorded in tests/golden/reference_outputs.json (SHA-256; of the residues mod q for lazy outputs)."""
    torch = pytest.importorskip("torch")

    def dev(a):
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint64).view(np.int64)).cuda()

    def host(t):
        return t.cpu().numpy().view(np.uint64)

    for logn, bits in RADIX4_CASES:
        ref = reference_outputs["radix4"][f"{logn},{bits}"]
        n = 1 << logn
        q = hb.GeneratePrimes(1, bits, True, n)[0]
        assert q == ref["q"]
        t = hb.NTT(n, q)
        for direction, in_mf, out_mf, x in radix4_inputs(logn, q):
            fn = t.ComputeForward if direction == "forward" else t.ComputeInverse
            got = host(fn(dev(np.zeros_like(x)), dev(x), in_mf, out_mf))
            exp = ref[direction][f"{in_mf},{out_mf}"]
            if out_mf == 1:
                assert sha(got) == exp, (direction, logn, in_mf)
            else:
                assert sha(got % np.uint64(q)) == exp and (got < np.uint64(out_mf * q)).all(), (direction, logn, in_mf)
