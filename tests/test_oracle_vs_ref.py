"""The oracle restatement against the COMPILED reference on random inputs -- the
reference never tests N > 2^13 itself (SURVEY.md 4), so large-N parity rests on
this.  What the reference returned on these inputs is recorded in
tests/golden/reference_outputs.json (SHA-256 of every output array), so the
comparison runs without the reference.  Lazy outputs are compared bit for bit
with the reference's scalar tier and modulo q with its AVX-512 tiers (which the
reference's own tests do too: test/test-ntt-avx512.cpp:194-204).  CPU only."""
import numpy as np
import pytest

from util import sha, uniform_below

NTT_CASES = [(2, 48), (4, 20), (8, 22), (16, 29), (64, 31), (1024, 30), (2048, 49), (4096, 50),
             (8192, 60), (16384, 58), (32768, 50), (65536, 55), (131072, 60)]
ELTWISE_BITS = [20, 30, 31, 32, 33, 40, 48, 50, 51, 52, 55, 58, 59, 60]
KEY_SWITCH_CASES = [(4, 2, 59), (10, 3, 50), (13, 5, 58)]
# the lazy element-wise output: compared modulo q, and the reference's output must lie below 2q
LAZY_ELTWISE = "reduce_mod q->2"


def ntt_inputs(n, q):
    """("forward" | "inverse", in_mf, out_mf, x) of every transform the comparison makes"""
    batch = 3 if n <= 8192 else 1
    for in_mf, out_mf in [(1, 1), (2, 1), (4, 1), (1, 4), (2, 4), (4, 4)]:
        yield "forward", in_mf, out_mf, uniform_below(n + in_mf, n * batch, q * in_mf)
    for in_mf, out_mf in [(1, 1), (2, 1), (1, 2), (2, 2)]:
        yield "inverse", in_mf, out_mf, uniform_below(7 * n + in_mf, n * batch, q * in_mf)


def eltwise_outputs(impl, q, **tier):
    """(name, output) of every element-wise call the comparison makes; `tier` is passed on to the reference"""
    n = 1024 + 7  # the reference's own odd size (test-eltwise-reduce-mod.cpp:103)
    a, b = uniform_below(1, n, q), uniform_below(2, n, q)
    yield "add_mod", impl.add_mod(a, b, q, **tier)
    yield "add_mod scalar", impl.add_mod(a, int(b[0]), q, **tier)
    yield "sub_mod", impl.sub_mod(a, b, q, **tier)
    yield "sub_mod scalar", impl.sub_mod(a, int(b[0]), q, **tier)
    for mf in (1, 2, 4):
        x, y = uniform_below(3, n, mf * q), uniform_below(4, n, mf * q)
        yield f"mult_mod {mf}", impl.mult_mod(x, y, q, mf, **tier)
    for mf in (1, 2, 4, 8):
        x, c = uniform_below(5, n, mf * q), uniform_below(6, n, mf * q)
        s = int(uniform_below(7, 1, mf * q)[0])
        yield f"fma_mod {mf}", impl.fma_mod(x, s, c, q, mf, **tier)
        yield f"fma_mod {mf} no addend", impl.fma_mod(x, s, None, q, mf, **tier)
    wide = uniform_below(8, n, 1 << 63)
    yield "reduce_mod q->1", impl.reduce_mod(wide, q, q, 1, **tier)
    yield LAZY_ELTWISE, impl.reduce_mod(wide, q, q, 2, **tier)
    x4 = uniform_below(9, n, 4 * q)
    yield "reduce_mod 4->1", impl.reduce_mod(x4, q, 4, 1, **tier)
    yield "reduce_mod 4->2", impl.reduce_mod(x4, q, 4, 2, **tier)
    x2 = uniform_below(10, n, 2 * q)
    yield "reduce_mod 2->1", impl.reduce_mod(x2, q, 2, 1, **tier)
    for cmp in range(8):
        bound, diff = int(a[5]), int(b[6]) or 1
        yield f"cmp_add {cmp}", impl.cmp_add(a, cmp, bound, diff, **tier)
        w = uniform_below(11, n, 1 << 64)
        yield f"cmp_sub_mod {cmp}", impl.cmp_sub_mod(w, q, cmp, int(w[3]), diff, **tier)


def key_switch_inputs(n, decomp, mods):
    """(t_target, keys, result, x, y): the key switch operands and the DyadicMultiply operands"""
    kms, kcc = decomp + 1, 2
    t_target = np.concatenate([uniform_below(30 + j, n, mods[j]) for j in range(decomp)])
    keys = [np.concatenate([uniform_below(100 * j + 7 * k + i, n, mods[i]) for k in range(kcc) for i in range(kms)])
            for j in range(decomp)]
    result = np.concatenate([uniform_below(500 + 10 * k + i, n, mods[i]) for k in range(kcc) for i in range(decomp)])
    x = np.concatenate([uniform_below(1 + i, n, q) for _ in range(2) for i, q in enumerate(mods)])
    y = np.concatenate([uniform_below(9 + i, n, q) for _ in range(2) for i, q in enumerate(mods)])
    return t_target, keys, result, x, y


@pytest.mark.parametrize("n,bits", NTT_CASES)
def test_ntt_port_matches_reference(port, reference_outputs, n, bits):
    ref = reference_outputs["ntt"][f"{n},{bits}"]
    q = ref["q"]
    assert port.generate_primes(1, bits, True, n)[0] == q
    assert port.minimal_primitive_root(2 * n, q) == ref["root"]
    assert [sha(t) for t in port.tables(n, q)[1:]] == ref["tables"]
    qq = np.uint64(q)
    for direction, in_mf, out_mf, x in ntt_inputs(n, q):
        fn = port.ntt_forward if direction == "forward" else port.ntt_inverse
        exp = ref[direction][f"{in_mf},{out_mf}"]
        a = fn(x, n, q, in_mf, out_mf)
        assert sha(a) == exp["native"], (direction, in_mf, out_mf)
        assert sha(a % qq) == exp["dispatch mod q"] and exp["dispatch max"] < out_mf * q, (direction, in_mf, out_mf)
        if out_mf == 1:
            assert sha(a) == exp["dispatch mod q"]
    x = uniform_below(99, n, q)
    assert (port.ntt_inverse(port.ntt_forward(x, n, q), n, q) == x).all()
    if n <= 4096:
        assert sha(port.ntt_forward_textbook(x, n, q)) == ref["forward textbook"]
        assert sha(port.ntt_forward(x, n, q)) == ref["forward radix4"]


@pytest.mark.parametrize("bits", ELTWISE_BITS)
def test_eltwise_port_matches_reference(port, reference_outputs, bits):
    ref = reference_outputs["eltwise"][str(bits)]
    q = ref["q"]
    qq = np.uint64(q)
    for name, out in eltwise_outputs(port, q):
        for tier in ("native", "dispatch"):
            if name == LAZY_ELTWISE:
                assert sha(out % qq) == ref[tier][name] and ref[tier][name + " max"] < 2 * q, tier
            else:
                assert sha(out) == ref[tier][name], (name, tier)


@pytest.mark.parametrize("logn,decomp,bits", KEY_SWITCH_CASES)
def test_key_switch_port_matches_reference(port, reference_outputs, logn, decomp, bits):
    ref = reference_outputs["key_switch"][f"{logn},{decomp},{bits}"]
    n = 1 << logn
    kms = rns = decomp + 1
    kcc = 2
    mods, modswitch = ref["moduli"], ref["modswitch"]
    t_target, keys, result, x, y = key_switch_inputs(n, decomp, mods)
    a = port.key_switch(result.copy(), t_target, n, decomp, kms, rns, kcc, mods, keys, modswitch)
    assert sha(a) == ref["key_switch"]
    assert sha(port.dyadic_multiply(x, y, n, mods)) == ref["dyadic_multiply"]
