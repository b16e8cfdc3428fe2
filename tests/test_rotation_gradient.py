"""Pauli-rotation gradients, host side: the sweep counts of qsb_pauli_rotation_gradient_dry_run and its argument checks.
No device needed."""
import ctypes as C

import numpy as np
import pytest

import gpu_quantum_simulator_b200 as q
from gpu_quantum_simulator_b200 import _lib

N = 30
RING = [f"Z{k} Z{(k + 1) % N}" for k in range(N)]
QAOA_LAYER = RING + [f"X{k}" for k in range(N)]


def dry(paulis, observable, prec=q.F32, world=1, low_bits=0, n=N):
    return q.rotation_gradient_dry_run(n, paulis, observable, prec, world_size=world, low_bits=low_bits)


@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_diagonal_observable_takes_one_lambda_sweep(prec):
    rng = np.random.default_rng(1)
    diag = ["", "Z0", f"Z{N - 1}"]
    while len(diag) < 1000:
        qs = rng.choice(N, int(rng.integers(1, 5)), replace=False)
        diag.append(" ".join(f"Z{k}" for k in qs))
    assert dry(["X3"], diag, prec)["apply_sweeps"] == 1
    assert dry(QAOA_LAYER, RING, prec)["apply_sweeps"] == 1


@pytest.mark.parametrize("prec,one_layer,four_layers", [(q.F32, 4, 13), (q.F64, 4, 14)])
def test_qaoa_adjoint_sweeps(prec, one_layer, four_layers):
    """The adjoint tile has one bit fewer than the forward one (11 f32 / 10 f64) and keeps the low 4 / 3 bits: a
    sweep takes the ring's ZZ rotations and the X rotations of 8 (f32) / 7 (f64) qubits above the low bits, so one
    layer of X on 30 qubits takes 4 sweeps; consecutive layers share sweeps across their boundaries."""
    assert dry(QAOA_LAYER, RING, prec) == {"apply_sweeps": 1, "adjoint_sweeps": one_layer, "exchanges": 0}
    assert dry(QAOA_LAYER * 4, RING, prec) == {"apply_sweeps": 1, "adjoint_sweeps": four_layers, "exchanges": 0}
    # the forward pass of the same list, with the full tile, takes fewer
    assert q.pauli_rotation_dry_run(N, QAOA_LAYER * 4, prec)["sweeps"] < four_layers


def test_zero_angles_do_not_change_the_counts():
    """The dry run has no angles: it counts as if every angle were non-zero, and the device call keeps zero angles in
    the adjoint pass, so the same list always plans the same sweeps."""
    rots = QAOA_LAYER * 2
    assert dry(rots, RING)["adjoint_sweeps"] == 7


def test_runs_longer_than_one_launch_split():
    assert dry(["Z0 Z1"] * 1024, ["Z0"])["adjoint_sweeps"] == 1
    assert dry(["Z0 Z1"] * 1025, ["Z0"])["adjoint_sweeps"] == 2
    assert dry(["X5"] * 3000, ["Z0"])["adjoint_sweeps"] == 3


@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_exchanges_on_ranks(prec):
    """Qubit 29 (and 28, 27 at world 4, 8) lie on rank bits.  H: X29 flips rank bits, Y28 / X27 X0 do from world 4 / 8 on;
    each distinct rank pattern of H fetches the partner's psi once.  Rotations: one adjoint sweep per rank pattern run,
    each fetching the partner's phi and lambda (counted as one copy)."""
    rots = ["X29", "Z0", "X28 X3", "Y29 Z1"]
    obs = ["X29", "Y28", "Z29 Z28", "X27 X0"]
    assert dry(rots, obs, prec, world=1) == {"apply_sweeps": 1, "adjoint_sweeps": 1, "exchanges": 0}
    assert dry(rots, obs, prec, world=2) == {"apply_sweeps": 2, "adjoint_sweeps": 1, "exchanges": 2}
    assert dry(rots, obs, prec, world=4) == {"apply_sweeps": 3, "adjoint_sweeps": 3, "exchanges": 5}
    assert dry(rots, obs, prec, world=8) == {"apply_sweeps": 4, "adjoint_sweeps": 3, "exchanges": 6}
    # diagonal rotations and terms never fetch a partner shard
    assert dry(["Z29", "Z28 Z0"], ["Z29 Z27"], prec, world=8)["exchanges"] == 0


def _raw(n, rx, rz, nrot, hx, hz, nterms, opt=True):
    o = q.simulator._options(q.F32, q.MODE_TILED, 0, 0, 1, -1)
    a, b, c = C.c_uint32(), C.c_uint32(), C.c_uint32()
    return _lib.lib.qsb_pauli_rotation_gradient_dry_run(n, C.byref(o) if opt else None, rx, rz, nrot, hx, hz, nterms,
                                                        C.byref(a), C.byref(b), C.byref(c))


def test_dry_run_argument_errors():
    m = np.array([1], dtype=np.uint64)
    big = np.array([1 << 12], dtype=np.uint64)
    d = m.ctypes.data
    assert _raw(12, d, d, 1, d, d, 1) == 0
    assert _raw(12, d, d, 1, d, d, 1, opt=False) == 0               # default options
    assert _raw(12, None, None, 0, d, d, 1) == 0                     # no rotations: valid
    assert _raw(12, d, d, 1, d, d, 0) == -1                          # an observable needs a term
    assert _raw(12, None, d, 1, d, d, 1) == -1
    assert _raw(12, d, None, 1, d, d, 1) == -1
    assert _raw(12, d, d, 1, None, d, 1) == -1
    assert _raw(12, d, d, 1, d, None, 1) == -1
    assert _raw(12, big.ctypes.data, d, 1, d, d, 1) == -1            # qubit >= n
    assert _raw(12, d, d, 1, d, big.ctypes.data, 1) == -1
    assert _raw(0, d, d, 1, d, d, 1) == -1
    assert "at least one term" in (_raw(12, d, d, 1, d, d, 0), _lib.lib.qsb_last_error().decode())[1]
    with pytest.raises(q.QsbError):
        q.rotation_gradient_dry_run(N, ["X0"], ["Z0"], world_size=3)
    with pytest.raises(q.QsbError):
        q.rotation_gradient_dry_run(N, ["X0"], ["Q0"])
