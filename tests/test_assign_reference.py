"""CPU checks of the gated linear assignment: the scipy oracle (tests/assign_reference.py) against brute-force enumeration, and
the C ABI's argument handling (pcreid_lsap / pcreid_lsap_workspace_bytes) through ctypes, which answers before any CUDA call."""
import numpy as np
import pytest

import assign_reference as R


def _problem(rng, T, D, kind):
    if kind == "ties":
        S = rng.integers(-2, 3, size=(T, D)).astype(np.float32)
    else:
        S = rng.normal(size=(T, D)).astype(np.float32)
    if kind == "nonfinite" and T * D:
        for v in (np.nan, np.inf, -np.inf):
            S.flat[rng.integers(0, T * D)] = v
    mask = rng.random((T, D)) < 0.7 if kind != "dense" else None
    return S, mask


@pytest.mark.parametrize("kind", ["dense", "masked", "ties", "nonfinite"])
def test_oracle_equals_brute_force(kind):
    rng = np.random.default_rng({"dense": 0, "masked": 1, "ties": 2, "nonfinite": 3}[kind])
    for _ in range(120):
        T, D = (int(x) for x in rng.integers(0, 6, 2))
        S, mask = _problem(rng, T, D, kind)
        tau = float(rng.choice([-1.5, -0.5, 0.0, 0.5]))
        d4t, t4d = R.assign(S, tau, mask)
        assert d4t.shape == (T,) and t4d.shape == (D,)
        assert R.consistent(d4t, t4d)
        assert R.objective(S, tau, d4t, mask) == pytest.approx(R.brute_force_value(S, tau, mask), abs=1e-12)


def test_oracle_degenerate_shapes():
    for T, D in ((0, 0), (0, 4), (3, 0)):
        d4t, t4d = R.assign(np.zeros((T, D), np.float32), 0.0)
        assert (d4t == -1).all() and (t4d == -1).all() and d4t.shape == (T,) and t4d.shape == (D,)
    # nothing above the threshold: nothing is matched, whatever it would add
    d4t, _ = R.assign(np.full((3, 3), -1.0, np.float32), -1.0)
    assert (d4t == -1).all()
    # a positive-weight pair is never dropped for an unmatched row
    d4t, _ = R.assign(np.array([[0.25]], np.float32), 0.0)
    assert d4t.tolist() == [0]


@pytest.fixture(scope="module")
def L():
    from pcreid_b200 import _lib
    return _lib.lib()


def test_workspace_bytes(L):
    assert L.pcreid_lsap_workspace_bytes(0, 5) == 0
    for T, D in ((1, 1), (7, 3), (64, 64), (4096, 4096), (4096, 0)):
        n = L.pcreid_lsap_workspace_bytes(T, D)
        assert n >= 12 * (T + min(T, D) + 1) and n % 16 == 0
    for T, D in ((-1, 4), (4, -1), (4097, 4), (4, 4097)):
        assert L.pcreid_lsap_workspace_bytes(T, D) == -1


def test_lsap_argument_errors_before_any_cuda_call(L):
    lsap = L.pcreid_lsap
    # negative sizes, a non-finite threshold: PCREID_ERR_ARG
    assert lsap(-1, 4, 4, None, None, 0.0, None, None, None, None) == 1
    assert lsap(1, -4, 4, None, None, 0.0, None, None, None, None) == 1
    assert lsap(1, 4, -4, None, None, 0.0, None, None, None, None) == 1
    assert lsap(1, 4, 4, None, None, float("nan"), None, None, None, None) == 1
    assert lsap(1, 4, 4, None, None, float("inf"), None, None, None, None) == 1
    # shapes beyond the kernel: PCREID_ERR_UNSUPPORTED
    assert lsap(1, 4097, 4, None, None, 0.0, None, None, None, None) == 3
    assert lsap(1, 4, 4097, None, None, 0.0, None, None, None, None) == 3
    assert lsap(65536, 4, 4, None, None, 0.0, None, None, None, None) == 3
    # missing buffers: PCREID_ERR_ARG
    assert lsap(1, 4, 4, None, None, 0.0, None, None, None, None) == 1
    # nothing to do: PCREID_OK without touching a pointer
    assert lsap(0, 4, 4, None, None, 0.0, None, None, None, None) == 0
    assert lsap(3, 0, 0, None, None, 0.0, None, None, None, None) == 0
