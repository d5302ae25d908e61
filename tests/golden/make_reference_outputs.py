#!/usr/bin/env python
"""Record what the compiled reference returns on the random inputs of
tests/test_oracle_vs_ref.py and of the reference comparisons in
tests/test_montgomery.py, so that those tests run where the reference is not.

    python tests/golden/make_reference_outputs.py

Needs oracle/_ref (oracle.build(ref=True) compiles it from the intel/hexl
sources); nothing reads the reference at test time.  Writes
tests/golden/reference_outputs.json: scalars as they are, arrays as the SHA-256
of their uint64 words (tests/util.py sha), lazy outputs as the SHA-256 of their
residues mod q plus their maximum.  The inputs, case lists and call sequences
are imported from the tests themselves, so the two cannot drift apart.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path[:0] = [TESTS, os.path.dirname(TESTS)]

import oracle  # noqa: E402
import test_montgomery as tm  # noqa: E402
import test_oracle_vs_ref as tv  # noqa: E402
from util import sha  # noqa: E402

MASK64 = (1 << 64) - 1


def lazy(out, q):
    return sha(out % np.uint64(q)), int(out.max())


def ntt_case(ref, n, bits):
    q = ref.generate_primes(1, bits, True, n)[0]
    c = {"q": q, "root": ref.root(n, q), "tables": [sha(t) for t in ref.tables(n, q)], "forward": {}, "inverse": {}}
    for direction, in_mf, out_mf, x in tv.ntt_inputs(n, q):
        fn = ref.ntt_forward if direction == "forward" else ref.ntt_inverse
        mod_q, top = lazy(fn(x, n, q, in_mf, out_mf), q)
        c[direction][f"{in_mf},{out_mf}"] = {"native": sha(fn(x, n, q, in_mf, out_mf, native=True)),
                                             "dispatch mod q": mod_q, "dispatch max": top}
    if n <= 4096:
        x = tv.uniform_below(99, n, q)
        c["forward textbook"] = sha(ref.ntt_forward_textbook(x, n, q))
        c["forward radix4"] = sha(ref.ntt_forward_radix4(x, n, q))
    return c


def eltwise_case(ref, bits):
    q = ref.generate_primes(1, bits, True, 1)[0]
    c = {"q": q}
    for tier, native in (("native", True), ("dispatch", False)):
        c[tier] = {}
        for name, out in tv.eltwise_outputs(ref, q, native=native):
            if name == tv.LAZY_ELTWISE:
                c[tier][name], c[tier][name + " max"] = lazy(out, q)
            else:
                c[tier][name] = sha(out)
    return c


def key_switch_case(ref, logn, decomp, bits):
    n = 1 << logn
    kms = rns = decomp + 1
    mods = ref.generate_primes(kms, bits, True, n)
    modswitch = [ref.inverse_mod(mods[-1] % mods[i], mods[i]) for i in range(decomp)]
    t_target, keys, result, x, y = tv.key_switch_inputs(n, decomp, mods)
    out = ref.key_switch(result.copy(), t_target, n, decomp, kms, rns, 2, mods, keys, modswitch)
    return {"moduli": mods, "modswitch": modswitch, "key_switch": sha(out),
            "dyadic_multiply": sha(ref.dyadic_multiply(x, y, n, mods))}


def montgomery(ref):
    m = {"avx512": ref.avx512,
         "hensel_lemma_2adic_root(46, 67280421310725)": ref.hensel_lemma_2adic_root(46, 67280421310725),
         "montgomery_reduce": [ref.montgomery_reduce(T >> 64, T & MASK64, q, r, ref.hensel_lemma_2adic_root(r, q))
                               for q, r, T, _ in tm.REDC_KATS],
         "cases": {}}
    for q, r in tm._cases():
        inv = ref.hensel_lemma_2adic_root(r, q)
        a, b, r2, *_ = tm._kat_arrays(q, r)
        fin = ref.montgomery_form_in(a, r2, q, r, inv)
        c = {"inv": inv, "kat mont_reduce_mod": sha(ref.mont_reduce_mod(a, b, q, r, inv)),
             "kat montgomery_form_in": sha(fin), "kat montgomery_form_out": sha(ref.montgomery_form_out(fin, q, r, inv)),
             "kat mont_reduce_mod of form_in": sha(ref.mont_reduce_mod(fin, b, q, r, inv))}
        a, b = tm.uniform_below(3, 4099, q), tm.uniform_below(4, 4099, q)
        c["mont_reduce_mod"] = sha(ref.mont_reduce_mod(a, b, q, r, inv))
        c["avx512 helper"] = ref.last_mont_was_avx512
        m["cases"][f"{q},{r}"] = c
    return m


def radix4_case(ref, logn, bits):
    n = 1 << logn
    q = ref.generate_primes(1, bits, True, n)[0]
    c = {"q": q, "forward": {}, "inverse": {}}
    for direction, in_mf, out_mf, x in tm.radix4_inputs(logn, q):
        fn = ref.ntt_forward_radix4 if direction == "forward" else ref.ntt_inverse_radix4
        out = fn(x, n, q, in_mf, out_mf)
        c[direction][f"{in_mf},{out_mf}"] = sha(out) if out_mf == 1 else sha(out % np.uint64(q))
    return c


def main():
    ref = oracle.Ref()
    assert ref.has_mont and ref.has_seal, "oracle/_ref lacks the Montgomery or SEAL entry points"
    out = {
        "_comment": "Outputs of the compiled reference (intel/hexl 1.2.5) on the tests' inputs; "
                    "written by tests/golden/make_reference_outputs.py",
        "ntt": {f"{n},{bits}": ntt_case(ref, n, bits) for n, bits in tv.NTT_CASES},
        "eltwise": {str(bits): eltwise_case(ref, bits) for bits in tv.ELTWISE_BITS},
        "key_switch": {f"{logn},{d},{bits}": key_switch_case(ref, logn, d, bits) for logn, d, bits in tv.KEY_SWITCH_CASES},
        "montgomery": montgomery(ref),
        "radix4": {f"{logn},{bits}": radix4_case(ref, logn, bits) for logn, bits in tm.RADIX4_CASES},
    }
    with open(os.path.join(HERE, "reference_outputs.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print(f"reference_outputs.json written ({ref.path}, AVX-512 tiers: {ref.avx512})")


if __name__ == "__main__":
    main()
