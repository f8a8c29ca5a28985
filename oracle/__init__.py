"""TEST INFRASTRUCTURE ONLY -- ctypes front end for the CPU oracle.

Two shared objects live here (both built by ``oracle/Makefile``; ``__graft_entry__.build()`` calls it):

* ``_build/liboracle.so``      -- ``wilson_oracle.c``: our restatement of the reference's host operators
  (``tests/host_reference/wilson_dslash_reference.cpp``, ``clover_reference.cpp``, field generators of
  ``tests/utils/host_utils.cpp``), used as the checker in ``tests/`` and as the CPU baseline.
* ``_ref/libquda_hostref.so``  -- the reference's *own* host sources compiled in place
  (``ref_glue.cpp`` only supplies link-time stand-ins); records the outputs that pin the restatement
  (``tests/golden/oracle_pin.json``, see ``tests/test_oracle_pin.py``) and is ``cpu_baseline.kind == "reference"`` in
  ``bench.py``.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py`` (cpu_baseline / ``--impl reference``) may
import this package.  ``quda_b200`` never does; it fails loudly without its CUDA library instead.

Host field orders (as in the reference's tests):
  gauge   float array [4][2*Vh][3][3][2]   "QDP" order, parity-major (even sites first)
  spinor  float array [Vh][4][3][2]        single parity, DeGrand-Rossi basis
  clover  float array [2*Vh][2][36]        6 real diagonals + 15 complex lower-triangular, per chiral block
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(_HERE, "_build", "liboracle.so")
REF_SO = os.path.join(_HERE, "_ref", "libquda_hostref.so")

MATPC_EVEN_EVEN, MATPC_ODD_ODD, MATPC_EVEN_EVEN_ASYM, MATPC_ODD_ODD_ASYM = 0, 1, 2, 3


def build(ref=True):
    """Compile the restatement, and (if /root/reference is mounted) the reference host sources."""
    subprocess.check_call(["make", "-s", "-C", _HERE, "oracle"])
    if ref and os.path.isdir("/root/reference/tests/host_reference"):
        subprocess.check_call(["make", "-s", "-C", _HERE, "ref"])


def have_ref():
    return os.path.exists(REF_SO)


_lib = None
_ref = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(ORACLE_SO):
            build(ref=False)
        _lib = C.CDLL(ORACLE_SO)
    return _lib


def ref():
    global _ref
    if _ref is None:
        _ref = C.CDLL(REF_SO)
    return _ref


def _dt(prec):
    return {8: np.float64, 4: np.float32}[prec]


def _sfx(a):
    return "_f64" if a.dtype == np.float64 else "_f32"


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _X(X):
    return (C.c_int * 4)(*[int(v) for v in X])


def _gptr(gauge):
    """void*[4] of per-direction base pointers of a contiguous [4][...] gauge array."""
    assert gauge.flags["C_CONTIGUOUS"] and gauge.shape[0] == 4
    return (C.c_void_p * 4)(*[gauge[mu].ctypes.data for mu in range(4)])


def volume(X):
    return int(X[0]) * int(X[1]) * int(X[2]) * int(X[3])


# ------------------------------------------------------------------ field generators (restatement)
def random_gauge(X, prec=8, seed=137, anisotropy=1.0, antiperiodic_t=True):
    """Random SU(3) links + scaling, libc rand() after srand(seed) (tests/utils/host_utils.cpp:444-455,1022-1098)."""
    V = volume(X)
    g = np.zeros((4, V, 3, 3, 2), dtype=_dt(prec))
    L = lib()
    L.orc_srand(C.c_uint(seed))
    getattr(L, "orc_random_gauge" + _sfx(g))(_gptr(g), _X(X), C.c_double(anisotropy), C.c_int(int(antiperiodic_t)))
    return g


def random_clover(X, prec=8, norm=0.01, diag=1.0, seed=None):
    V = volume(X)
    c = np.zeros((V, 2, 36), dtype=_dt(prec))
    L = lib()
    if seed is not None:
        L.orc_srand(C.c_uint(seed))
    getattr(L, "orc_random_clover" + _sfx(c))(_p(c), C.c_long(V), C.c_double(norm), C.c_double(diag))
    return c


def random_spinor(X, prec=8, seed=137, nparity=1):
    """Uniform [0,1) components from the reference's rand48 clone (lib/comm_common.cpp:26-41)."""
    n = volume(X) // 2 * nparity
    s = np.zeros((n, 4, 3, 2), dtype=_dt(prec))
    st = C.c_ulong(seed)
    getattr(lib(), "orc_random_spinor" + _sfx(s))(_p(s), C.c_long(s.size), C.byref(st))
    return s


def clover_invert(clover):
    inv = np.zeros_like(clover)
    getattr(lib(), "orc_clover_invert" + _sfx(clover))(_p(inv), _p(clover), C.c_long(clover.shape[0]))
    return inv


# ------------------------------------------------------------------ operators (restatement)
def wil_dslash(gauge, inp, X, parity, dagger=0):
    out = np.zeros_like(inp)
    getattr(lib(), "orc_wil_dslash" + _sfx(inp))(_p(out), _gptr(gauge), _p(inp), _X(X), C.c_int(parity), C.c_int(dagger))
    return out


def wil_mat(gauge, inp, X, kappa, dagger=0):
    out = np.zeros_like(inp)
    getattr(lib(), "orc_wil_mat" + _sfx(inp))(_p(out), _gptr(gauge), _p(inp), _X(X), C.c_double(kappa), C.c_int(dagger))
    return out


def wil_matpc(gauge, inp, X, kappa, matpc=MATPC_EVEN_EVEN, dagger=0):
    out = np.zeros_like(inp)
    getattr(lib(), "orc_wil_matpc" + _sfx(inp))(
        _p(out), _gptr(gauge), _p(inp), _X(X), C.c_double(kappa), C.c_int(matpc), C.c_int(dagger))
    return out


TWIST_SINGLET = 1  # QudaTwistFlavorType value the reference multiplies mu with


def twist_gamma5(inp, kappa, mu, dagger=0, inverse=False, flavor=TWIST_SINGLET):
    """b (1 + i a gamma5) inp in the DeGrand-Rossi basis (wilson_dslash_reference.cpp:139-169)"""
    out = np.zeros_like(inp)
    getattr(lib(), "orc_twist_gamma5" + _sfx(inp))(
        _p(out), _p(inp), C.c_int(dagger), C.c_double(kappa), C.c_double(mu), C.c_int(flavor), C.c_long(inp.size // 24),
        C.c_int(1 if inverse else 0))
    return out


def tm_dslash(gauge, inp, X, kappa, mu, parity, dagger=0, matpc=MATPC_EVEN_EVEN, flavor=TWIST_SINGLET):
    out = np.zeros_like(inp)
    getattr(lib(), "orc_tm_dslash" + _sfx(inp))(
        _p(out), _gptr(gauge), _p(inp), _X(X), C.c_double(kappa), C.c_double(mu), C.c_int(flavor), C.c_int(matpc),
        C.c_int(parity), C.c_int(dagger))
    return out


def tm_mat(gauge, inp, X, kappa, mu, dagger=0, flavor=TWIST_SINGLET):
    out = np.zeros_like(inp)
    getattr(lib(), "orc_tm_mat" + _sfx(inp))(
        _p(out), _gptr(gauge), _p(inp), _X(X), C.c_double(kappa), C.c_double(mu), C.c_int(flavor), C.c_int(dagger))
    return out


def tm_matpc(gauge, inp, X, kappa, mu, matpc=MATPC_EVEN_EVEN, dagger=0, flavor=TWIST_SINGLET):
    out = np.zeros_like(inp)
    getattr(lib(), "orc_tm_matpc" + _sfx(inp))(
        _p(out), _gptr(gauge), _p(inp), _X(X), C.c_double(kappa), C.c_double(mu), C.c_int(flavor), C.c_int(matpc),
        C.c_int(dagger))
    return out


def apply_clover(clover, inp, X, parity):
    out = np.zeros_like(inp)
    getattr(lib(), "orc_apply_clover" + _sfx(inp))(_p(out), _p(clover), _p(inp), _X(X), C.c_int(parity))
    return out


def clover_dslash(gauge, clover, inp, X, parity, dagger=0):
    out = np.zeros_like(inp)
    getattr(lib(), "orc_clover_dslash" + _sfx(inp))(
        _p(out), _gptr(gauge), _p(clover), _p(inp), _X(X), C.c_int(parity), C.c_int(dagger))
    return out


def clover_matpc(gauge, clover, clover_inv, inp, X, kappa, matpc=MATPC_EVEN_EVEN, dagger=0):
    out = np.zeros_like(inp)
    getattr(lib(), "orc_clover_matpc" + _sfx(inp))(
        _p(out), _gptr(gauge), _p(clover), _p(clover_inv), _p(inp), _X(X), C.c_double(kappa), C.c_int(matpc),
        C.c_int(dagger))
    return out


def clover_mat(gauge, clover, inp, X, kappa, dagger=0):
    out = np.zeros_like(inp)
    getattr(lib(), "orc_clover_mat" + _sfx(inp))(
        _p(out), _gptr(gauge), _p(clover), _p(inp), _X(X), C.c_double(kappa), C.c_int(dagger))
    return out


def compare_spinor(ref_field, test_field):
    """Reference metric: returns (accuracy_level, deviation=10**-level, fails[16])."""
    a = np.ascontiguousarray(ref_field, dtype=np.float64).ravel()
    b = np.ascontiguousarray(test_field, dtype=np.float64).ravel()
    assert a.size == b.size
    fails = (C.c_long * 16)()
    lvl = lib().orc_compare_spinor(_p(a), _p(b), C.c_long(a.size), fails)
    return lvl, 10.0 ** (-lvl), list(fails)


def tolerance(prec_name, recon=18):
    """tests/utils/host_utils.h:292-310 and tests/dslash_test.cpp:74-76."""
    tol = {"double": 1e-11, "single": 1e-4, "half": 1e-3, "quarter": 1e-1}[prec_name]
    if recon == 8 and prec_name in ("half", "quarter"):
        tol *= 10
    return tol


# ------------------------------------------------------------------ the reference's own code (oracle/_ref)
class Reference:
    """Thin wrappers around the reference host sources compiled in place (see ref_glue.cpp)."""

    def __init__(self, X):
        self.X = [int(v) for v in X]
        self.L = ref()
        self.L.ref_set_dims(_X(self.X))

    def _pb(self, a):
        return C.c_int(a.dtype.itemsize)

    def random_gauge(self, prec=8, seed=137, anisotropy=1.0, antiperiodic_t=True):
        g = np.zeros((4, volume(self.X), 3, 3, 2), dtype=_dt(prec))
        self.L.ref_srand(C.c_uint(seed))
        self.L.ref_random_gauge(_gptr(g), C.c_int(prec), _X(self.X), C.c_double(anisotropy), C.c_int(int(antiperiodic_t)))
        return g

    def random_clover(self, prec=8, norm=0.01, diag=1.0, seed=None):
        c = np.zeros((volume(self.X), 2, 36), dtype=_dt(prec))
        if seed is not None:
            self.L.ref_srand(C.c_uint(seed))
        self.L.ref_random_clover(_p(c), C.c_double(norm), C.c_double(diag), C.c_int(prec))
        return c

    def wil_dslash(self, gauge, inp, parity, dagger=0):
        out = np.zeros_like(inp)
        self.L.ref_wil_dslash(_p(out), _gptr(gauge), _p(inp), C.c_int(parity), C.c_int(dagger), self._pb(inp), _X(self.X))
        return out

    def wil_mat(self, gauge, inp, kappa, dagger=0):
        out = np.zeros_like(inp)
        self.L.ref_wil_mat(_p(out), _gptr(gauge), _p(inp), C.c_double(kappa), C.c_int(dagger), self._pb(inp), _X(self.X))
        return out

    def wil_matpc(self, gauge, inp, kappa, matpc=MATPC_EVEN_EVEN, dagger=0):
        out = np.zeros_like(inp)
        self.L.ref_wil_matpc(_p(out), _gptr(gauge), _p(inp), C.c_double(kappa), C.c_int(self.L.ref_matpc_enum(matpc)),
                             C.c_int(dagger), self._pb(inp), _X(self.X))
        return out

    def twist_gamma5(self, inp, kappa, mu, dagger=0, inverse=False):
        out = np.zeros_like(inp)
        self.L.ref_twist_gamma5(_p(out), _p(np.ascontiguousarray(inp.copy())), C.c_int(dagger), C.c_double(kappa), C.c_double(mu),
                                C.c_int(inp.size // 24), C.c_int(1 if inverse else 0), self._pb(inp))
        return out

    def tm_dslash(self, gauge, inp, kappa, mu, parity, dagger=0, matpc=MATPC_EVEN_EVEN):
        out = np.zeros_like(inp)
        work = np.ascontiguousarray(inp.copy())  # the reference twists its input in place
        self.L.ref_tm_dslash(_p(out), _gptr(gauge), _p(work), C.c_double(kappa), C.c_double(mu),
                             C.c_int(self.L.ref_matpc_enum(matpc)), C.c_int(parity), C.c_int(dagger), self._pb(inp), _X(self.X))
        return out

    def tm_mat(self, gauge, inp, kappa, mu, dagger=0):
        out = np.zeros_like(inp)
        self.L.ref_tm_mat(_p(out), _gptr(gauge), _p(inp), C.c_double(kappa), C.c_double(mu), C.c_int(dagger), self._pb(inp),
                          _X(self.X))
        return out

    def tm_matpc(self, gauge, inp, kappa, mu, matpc=MATPC_EVEN_EVEN, dagger=0):
        out = np.zeros_like(inp)
        work = np.ascontiguousarray(inp.copy())
        self.L.ref_tm_matpc(_p(out), _gptr(gauge), _p(work), C.c_double(kappa), C.c_double(mu),
                            C.c_int(self.L.ref_matpc_enum(matpc)), C.c_int(dagger), self._pb(inp), _X(self.X))
        return out

    def apply_clover(self, clover, inp, parity):
        out = np.zeros_like(inp)
        self.L.ref_apply_clover(_p(out), _p(clover), _p(inp), C.c_int(parity), self._pb(inp))
        return out

    def clover_dslash(self, gauge, clover, inp, parity, dagger=0):
        out = np.zeros_like(inp)
        self.L.ref_clover_dslash(_p(out), _gptr(gauge), _p(clover), _p(inp), C.c_int(parity), C.c_int(dagger),
                                 self._pb(inp), _X(self.X))
        return out

    def clover_matpc(self, gauge, clover, clover_inv, inp, kappa, matpc=MATPC_EVEN_EVEN, dagger=0):
        out = np.zeros_like(inp)
        self.L.ref_clover_matpc(_p(out), _gptr(gauge), _p(clover), _p(clover_inv), _p(inp), C.c_double(kappa),
                                C.c_int(self.L.ref_matpc_enum(matpc)), C.c_int(dagger), self._pb(inp), _X(self.X))
        return out

    def clover_mat(self, gauge, clover, inp, kappa, dagger=0):
        out = np.zeros_like(inp)
        self.L.ref_clover_mat(_p(out), _gptr(gauge), _p(clover), _p(inp), C.c_double(kappa), C.c_int(dagger),
                              self._pb(inp), _X(self.X))
        return out
