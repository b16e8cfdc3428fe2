"""Pauli rotations, host side: the in-order sweep grouping of qsb_pauli_rotation_dry_run and argument checks.  No device
needed."""
import ctypes as C

import numpy as np
import pytest

import gpu_quantum_simulator_b200 as q
from gpu_quantum_simulator_b200 import _lib

N = 30
TILE = {q.F32: 12, q.F64: 11}
LOW_BITS = {q.F32: [3, 4, 5, 6], q.F64: [2, 3, 4, 5]}      # the values qsb_create accepts (0 = the default 4 / 3)


def dry(paulis, prec=q.F32, world=1, low_bits=0, n=N):
    return q.pauli_rotation_dry_run(n, paulis, prec, world_size=world, low_bits=low_bits)


@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_diagonal_rotations_take_one_sweep(prec):
    rng = np.random.default_rng(1)
    diag = ["", "Z0", f"Z{N - 1}"]
    while len(diag) < 1000:
        qs = rng.choice(N, int(rng.integers(1, 5)), replace=False)
        diag.append(" ".join(f"Z{k}" for k in qs))
    assert dry(diag, prec) == {"sweeps": 1, "exchanges": 0}
    assert dry([f"Z{k} Z{k + 1}" for k in range(N - 1)] * 30, prec) == {"sweeps": 1, "exchanges": 0}   # 870 rotations


def test_runs_longer_than_one_launch_split():
    """A launch carries at most 1024 rotations: a longer run of diagonal rotations is split into sweeps."""
    assert dry(["Z0 Z1"] * 1024)["sweeps"] == 1
    assert dry(["Z0 Z1"] * 1025)["sweeps"] == 2
    assert dry(["X0"] * 3000)["sweeps"] == 3


@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_single_qubit_x_rotations_on_distinct_qubits(prec):
    """X0, X1, ..., X_{n-1}: the low L qubits lie in every tile, the next one becomes the flip pattern outside the tile,
    the next T - L fill the tile, so the first sweep holds T + 1 rotations and every later one T - L + 1:
    ceil((n - L) / (T - L + 1)) sweeps, one fewer than ceil((n - L) / (T - L)) now and then (the flip pattern outside
    the tile carries one more qubit per sweep at no extra traffic)."""
    T = TILE[prec]
    for low in LOW_BITS[prec]:
        for n in range(1, N + 1):
            want = max(1, -(-(n - low) // (T - low + 1)))
            got = dry([f"X{k}" for k in range(n)], prec, low_bits=low)
            assert got == {"sweeps": want, "exchanges": 0}, (low, n, got)
            assert want <= max(1, -(-(n - low) // (T - low)))
            assert dry([f"Y{k}" for k in range(n)], prec, low_bits=low)["sweeps"] == want


@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_x_on_every_qubit_takes_one_sweep(prec):
    for text in (" ".join(f"X{k}" for k in range(N)), " ".join(f"{'XY'[k % 2]}{k}" for k in range(N))):
        assert dry([text], prec) == {"sweeps": 1, "exchanges": 0}
        assert dry([text, "Z0 Z7", text, f"Z{N - 1}"], prec) == {"sweeps": 1, "exchanges": 0}


@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_hand_counted_sequences(prec):
    # X0 lies in every tile, X29 becomes the flip pattern, diagonal rotations fit anywhere: one sweep
    assert dry(["X0", f"X{N - 1}", "Z3 Z4"] * 40, prec) == {"sweeps": 1, "exchanges": 0}
    # X29 -> flip pattern; X28 -> tile bit 28; X28 X29 = tile flip + pattern; X20..X26 -> 7 more tile bits (8 = T - L);
    # X27 needs a ninth: a second sweep
    seq = [f"X{N - 1}", f"X{N - 2}", f"X{N - 2} X{N - 1}"] + [f"X{k}" for k in range(20, 28)]
    assert dry(seq, prec) == {"sweeps": 2, "exchanges": 0}
    # the order is kept: X29, X28, X27, ... in reverse also take a second sweep only after T - L + 1 of them
    T, L = TILE[prec], (4 if prec == q.F32 else 3)
    assert dry([f"X{k}" for k in range(N - 1, N - 2 - (T - L), -1)], prec)["sweeps"] == 1
    assert dry([f"X{k}" for k in range(N - 1, N - 3 - (T - L), -1)], prec)["sweeps"] == 2


@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_one_exchange_per_rank_flipping_sweep(world):
    g = world.bit_length() - 1
    top = N - 1                                   # from the identity layout the top log2(world) qubits are the rank bits
    for prec in (q.F32, q.F64):
        assert dry([" ".join(f"X{k}" for k in range(N))], prec, world) == {"sweeps": 1, "exchanges": 1}
        assert dry([f"Z{top}", f"Z0 Z{top}", "Z3"], prec, world) == {"sweeps": 1, "exchanges": 0}
        # X0 / X_top / Z pairs: one run with one rank pattern, one exchange
        assert dry(["X0", f"X{top}", "Z3 Z4"] * 40, prec, world) == {"sweeps": 1, "exchanges": 1}
        # every repetition of the same rank flip is a new sweep only when something breaks the run
        assert dry([f"X{top}"] * 5, prec, world) == {"sweeps": 1, "exchanges": 1}
        if g >= 2:   # two different rank patterns alternate: every rotation starts a sweep with its own exchange
            seq = [f"X{top}", "Z0 Z1", f"X{top - 1}", "Z0 Z1"] * 3
            assert dry(seq, prec, world) == {"sweeps": 6, "exchanges": 6}
        # one Trotter step of the Ising chain: the ZZ stretch and the local X share sweeps; X on each rank qubit flips
        # a different rank pattern, the first joins the last local run, each other one takes a sweep of its own
        step = [f"Z{k} Z{k + 1}" for k in range(N - 1)] + [f"X{k}" for k in range(N)]
        got = dry(step, prec, world)
        assert got["exchanges"] == g, got
        assert got["sweeps"] == dry(step[:N - 1 + N - g], prec, world)["sweeps"] + g - 1, got


def test_refusals():
    x = np.array([1 << 8], dtype=np.uint64)
    z = np.zeros(1, dtype=np.uint64)
    sw, ex = C.c_uint32(), C.c_uint32()
    with pytest.raises(q.QsbError) as e:
        q.simulator.check(_lib.lib.qsb_pauli_rotation_dry_run(8, None, x.ctypes.data, z.ctypes.data, 1, C.byref(sw), C.byref(ex)))
    assert e.value.code == -1 and "qubit >= 8" in str(e.value)
    assert _lib.lib.qsb_pauli_rotation_dry_run(8, None, None, None, 3, None, None) == -1
    assert _lib.lib.qsb_pauli_rotation_dry_run(0, None, None, None, 0, None, None) == -1
    assert _lib.lib.qsb_pauli_rotation_dry_run(8, None, None, None, 0, C.byref(sw), C.byref(ex)) == 0
    assert (sw.value, ex.value) == (0, 0)
    with pytest.raises(q.QsbError):
        dry(["X0"], world=3)
    with pytest.raises(q.QsbError):
        dry(["X0"], world=8, n=14)                # too few qubits to shard
    t = np.array([0.5])
    assert _lib.lib.qsb_apply_pauli_rotations(None, x.ctypes.data, z.ctypes.data, t.ctypes.data, 1) == -1
    assert "null handle" in _lib.lib.qsb_last_error().decode()
    assert _lib.lib.qsb_apply_pauli_rotations(None, None, None, None, 0) == -1
