"""Pin the CPU oracle (oracle/wilson_oracle.c) against the reference's OWN host sources
(tests/host_reference/{wilson_dslash,clover}_reference.cpp, tests/utils/{host_utils,index_utils,host_blas}.cpp).  The
reference tree stores no golden vectors (SURVEY.md 8c) so this is what anchors parity.  Same compiler flags on both
sides -> bit-identical.

The reference's outputs for the inputs below are stored in tests/golden/oracle_pin.json: the SHA-256 of each output
array's bytes, so the comparison stays bit-exact, and a few sampled values that show how far off a mismatch is.  To
record them again, build oracle/_ref (`make -C oracle ref`, needs the reference tree) and run
`python tests/test_oracle_pin.py`."""
import hashlib
import json
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))  # also when run as a script
import oracle  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_pin.json")
DIMS = [(4, 4, 4, 4), (8, 4, 6, 2), (2, 4, 6, 8), (8, 8, 8, 8)]
KAPPA, MU = 0.12195, 0.1


class Restatement:
    """the oracle's functions behind the call signatures of oracle.Reference, so that one list of cases runs on both"""

    def __init__(self, X):
        self.X = X

    def random_gauge(self, prec, seed, anisotropy=1.0, antiperiodic_t=True):
        return oracle.random_gauge(self.X, prec, seed=seed, anisotropy=anisotropy, antiperiodic_t=antiperiodic_t)

    def random_clover(self, prec, seed):
        return oracle.random_clover(self.X, prec, seed=seed)

    def wil_dslash(self, g, s, parity, dagger):
        return oracle.wil_dslash(g, s, self.X, parity, dagger)

    def wil_matpc(self, g, s, kappa, matpc, dagger):
        return oracle.wil_matpc(g, s, self.X, kappa, matpc, dagger)

    def wil_mat(self, g, s, kappa, dagger):
        return oracle.wil_mat(g, s, self.X, kappa, dagger)

    def apply_clover(self, c, s, parity):
        return oracle.apply_clover(c, s, self.X, parity)

    def clover_dslash(self, g, cinv, s, parity, dagger):
        return oracle.clover_dslash(g, cinv, s, self.X, parity, dagger)

    def clover_matpc(self, g, c, cinv, s, kappa, matpc, dagger):
        return oracle.clover_matpc(g, c, cinv, s, self.X, kappa, matpc, dagger)

    def clover_mat(self, g, c, s, kappa, dagger):
        return oracle.clover_mat(g, c, s, self.X, kappa, dagger)

    def twist_gamma5(self, s, kappa, mu, dagger, inverse):
        return oracle.twist_gamma5(s, kappa, mu, dagger, inverse)

    def tm_dslash(self, g, s, kappa, mu, parity, dagger, matpc):
        return oracle.tm_dslash(g, s, self.X, kappa, mu, parity, dagger, matpc)

    def tm_matpc(self, g, s, kappa, mu, matpc, dagger):
        return oracle.tm_matpc(g, s, self.X, kappa, mu, matpc, dagger)

    def tm_mat(self, g, s, kappa, mu, dagger):
        return oracle.tm_mat(g, s, self.X, kappa, mu, dagger)


# Each case yields (name, output) pairs; the inputs always come from the oracle's generators (pinned by the first case).
def field_generators(impl, X, prec):
    for aniso, apbc in [(1.0, True), (2.38, False)]:
        yield f"gauge aniso={aniso} apbc={apbc}", impl.random_gauge(prec, seed=137, anisotropy=aniso, antiperiodic_t=apbc)
    yield "clover", impl.random_clover(prec, seed=5)


def wilson_operators(impl, X, prec):
    g = oracle.random_gauge(X, prec, seed=137)
    s = oracle.random_spinor(X, prec, seed=137)
    for parity in (0, 1):
        for dagger in (0, 1):
            yield f"wil_dslash parity={parity} dagger={dagger}", impl.wil_dslash(g, s, parity, dagger)
    for matpc in (oracle.MATPC_EVEN_EVEN, oracle.MATPC_ODD_ODD):
        for dagger in (0, 1):
            yield f"wil_matpc matpc={matpc} dagger={dagger}", impl.wil_matpc(g, s, KAPPA, matpc, dagger)
    full = oracle.random_spinor(X, prec, seed=99, nparity=2)
    for dagger in (0, 1):
        yield f"wil_mat dagger={dagger}", impl.wil_mat(g, full, KAPPA, dagger)


def clover_operators(impl, X, prec):
    g = oracle.random_gauge(X, prec, seed=137)
    c = oracle.random_clover(X, prec, seed=11)
    cinv = oracle.clover_invert(c)
    s = oracle.random_spinor(X, prec, seed=137)
    for parity in (0, 1):
        yield f"apply_clover parity={parity}", impl.apply_clover(c, s, parity)
        for dagger in (0, 1):
            yield f"clover_dslash parity={parity} dagger={dagger}", impl.clover_dslash(g, cinv, s, parity, dagger)
    for matpc in range(4):
        for dagger in (0, 1):
            yield f"clover_matpc matpc={matpc} dagger={dagger}", impl.clover_matpc(g, c, cinv, s, KAPPA, matpc, dagger)
    full = oracle.random_spinor(X, prec, seed=99, nparity=2)
    for dagger in (0, 1):
        yield f"clover_mat dagger={dagger}", impl.clover_mat(g, c, full, KAPPA, dagger)


def clover_inverse(impl, X, prec):
    """A^{-1} (A v) through the reference's apply_clover, with the oracle's host inverse"""
    c = oracle.random_clover(X, prec, seed=3)
    cinv = oracle.clover_invert(c)
    s = oracle.random_spinor(X, prec, seed=1)
    for parity in (0, 1):
        yield f"inverse of apply_clover parity={parity}", impl.apply_clover(cinv, impl.apply_clover(c, s, parity), parity)


def twisted_mass_operators(impl, X, prec):
    g = oracle.random_gauge(X, prec, seed=137)
    s = oracle.random_spinor(X, prec, seed=21)
    full = oracle.random_spinor(X, prec, seed=22, nparity=2)
    for dagger in (0, 1):
        for inverse in (False, True):
            yield f"twist_gamma5 dagger={dagger} inverse={inverse}", impl.twist_gamma5(s, KAPPA, MU, dagger, inverse)
        for matpc in range(4):
            for parity in (0, 1):
                yield (f"tm_dslash matpc={matpc} parity={parity} dagger={dagger}",
                       impl.tm_dslash(g, s, KAPPA, MU, parity, dagger, matpc))
            yield f"tm_matpc matpc={matpc} dagger={dagger}", impl.tm_matpc(g, s, KAPPA, MU, matpc, dagger)
        yield f"tm_mat dagger={dagger}", impl.tm_mat(g, full, KAPPA, MU, dagger)


CLOVER_INVERSE_X = (4, 4, 4, 4)
CASES = [(field_generators, DIMS), (wilson_operators, DIMS), (clover_operators, DIMS[:3]),
         (twisted_mass_operators, DIMS[:3]), (clover_inverse, [CLOVER_INVERSE_X])]


def _key(case, X, prec, name):
    return f"{case.__name__} X={'x'.join(map(str, X))} prec={prec}: {name}"


def _record(a):
    a = np.ascontiguousarray(a)
    flat = a.ravel()
    return {"sha256": hashlib.sha256(a.tobytes()).hexdigest(),
            "sample": [float(flat[i]) for i in np.linspace(0, flat.size - 1, 4).astype(int)]}


_golden = None


def _check(case, X, prec):
    """every output of `case` from the oracle is bit-identical to the reference's stored one; returns the outputs"""
    global _golden
    if _golden is None:
        with open(GOLDEN) as f:
            _golden = json.load(f)
    outs = list(case(Restatement(X), X, prec))
    for name, a in outs:
        key = _key(case, X, prec, name)
        got, want = _record(a), _golden[key]
        assert got["sha256"] == want["sha256"], f"{key}: sampled values {got['sample']}, the reference's {want['sample']}"
    return outs


@pytest.mark.parametrize("X", DIMS)
@pytest.mark.parametrize("prec", [8, 4])
def test_field_generators_bit_identical(X, prec):
    _check(field_generators, X, prec)


def test_random_gauge_is_su3():
    X = (4, 4, 4, 4)
    g = oracle.random_gauge(X, 8, antiperiodic_t=False)
    u = g[..., 0] + 1j * g[..., 1]
    uu = np.einsum("dvab,dvcb->dvac", u, u.conj())
    assert np.allclose(uu, np.eye(3), atol=1e-12)
    assert np.allclose(np.linalg.det(u), 1.0, atol=1e-12)


@pytest.mark.parametrize("X", DIMS)
@pytest.mark.parametrize("prec", [8, 4])
def test_wilson_operators_bit_identical(X, prec):
    _check(wilson_operators, X, prec)


@pytest.mark.parametrize("X", DIMS[:3])
@pytest.mark.parametrize("prec", [8, 4])
def test_clover_operators_bit_identical(X, prec):
    _check(clover_operators, X, prec)


@pytest.mark.parametrize("prec", [8, 4])
def test_clover_inverse_is_inverse(prec):
    """The reference inverts the clover term on the device; our host inverse is checked through the
    reference's own apply_clover: A^{-1} (A v) == v."""
    s = oracle.random_spinor(CLOVER_INVERSE_X, prec, seed=1)
    for _, back in _check(clover_inverse, CLOVER_INVERSE_X, prec):
        assert np.allclose(back, s, rtol=0, atol=1e-13 if prec == 8 else 2e-6)


def test_compare_spinor_metric():
    rng = np.random.default_rng(0)
    a = rng.standard_normal(24 * 512)
    lvl, dev, _ = oracle.compare_spinor(a, a)
    assert lvl == 16
    b = a.copy()
    b[7] += 3e-6 * np.abs(a).max()
    lvl, dev, fails = oracle.compare_spinor(a, b)
    assert lvl == 5 and fails[5] == 1 and fails[4] == 0


@pytest.mark.parametrize("X", DIMS[:3])
@pytest.mark.parametrize("prec", [8, 4])
def test_twisted_mass_operators_bit_identical(X, prec):
    """twist_gamma5 / tm_dslash / tm_mat / tm_matpc (wilson_dslash_reference.cpp:139-315), singlet flavour, all four
    matpc types, both parities, dagger"""
    _check(twisted_mass_operators, X, prec)


if __name__ == "__main__":
    # record the reference's outputs (oracle/_ref) for every case above
    rec = {}
    for case, dims in CASES:
        for X in dims:
            for prec in (8, 4):
                for name, a in case(oracle.Reference(X), X, prec):
                    rec[_key(case, X, prec, name)] = _record(a)
    with open(GOLDEN, "w") as f:
        f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(v)}" for k, v in rec.items()) + "\n}\n")
    print(f"{len(rec)} outputs -> {GOLDEN}")
