"""Pauli-string expectation values, host side: the string parser, the sweep grouping of qsb_expectation_dry_run
and argument checks.  No device needed."""
import ctypes as C

import numpy as np
import pytest

import gpu_quantum_simulator_b200 as q
from gpu_quantum_simulator_b200 import _lib

N = 30


def masks(text, n=8):
    x, z = q.pauli_masks(text, n)
    return int(x[0]), int(z[0])


def test_parser_round_trip():
    rng = np.random.default_rng(3)
    for _ in range(200):
        n = int(rng.integers(1, 41))
        x = z = 0
        toks = []
        for qb in rng.permutation(n)[: rng.integers(0, min(n, 6) + 1)]:
            p = "IXYZ"[rng.integers(4)]
            toks.append(f"{p}{qb}")
            x |= (p in "XY") << int(qb)
            z |= (p in "YZ") << int(qb)
        assert masks(" ".join(toks), n) == (x, z)
        assert masks("\t ".join(reversed(toks)) + " ", n) == (x, z)


def test_parser_y_sets_both_bits_and_identity():
    assert masks("Y3") == (8, 8)
    assert masks("X0 Z3 Y5") == (0b100001, 0b101000)
    assert masks("") == (0, 0)
    assert masks("I") == (0, 0)
    assert masks("I I") == (0, 0)
    assert masks("I4") == (0, 0)
    x, z = q.pauli_masks(["Z0 Z1", "X2"], 3)
    assert x.tolist() == [0, 4] and z.tolist() == [3, 0]


@pytest.mark.parametrize("text,code", [("X0 X0", -4), ("Z1 Y1", -4), ("A1", -4), ("x1", -4), ("X", -4), ("X1a", -4),
                                       ("X8", -1), ("Z0 Y100", -1)])
def test_parser_refusals(text, code):
    with pytest.raises(q.QsbError) as e:
        q.pauli_masks(text, 8)
    assert e.value.code == code


def ising(n):
    return [f"X{k}" for k in range(n)] + [f"Z{k} Z{k + 1}" for k in range(n - 1)]


def random_strings(n, count, seed):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(count):
        qs = rng.choice(n, int(rng.integers(1, 5)), replace=False)
        out.append(" ".join(f"{'XYZ'[rng.integers(3)]}{k}" for k in qs))
    return out


@pytest.mark.parametrize("prec,low", [(q.F32, 4), (q.F64, 3)])
def test_dry_run_targets(prec, low):
    tile = 12 if prec == q.F32 else 11
    diag = [f"Z{k}" for k in range(N)] + [f"Z{k} Z{k + 1}" for k in range(N - 1)] + ["", f"Z0 Z{N - 1}"]
    assert q.expectation_dry_run(N, diag, prec) == {"sweeps": 1, "exchanges": 0}
    want = -(-(N - low) // (tile - low))
    assert q.expectation_dry_run(N, ising(N), prec)["sweeps"] <= want
    assert q.expectation_dry_run(N, " ".join(f"X{k}" for k in range(N)), prec)["sweeps"] == 1
    assert q.expectation_dry_run(N, " ".join(f"Y{k}" for k in range(N)), prec)["sweeps"] == 1
    terms = random_strings(N, 1000, seed=7)
    x, _ = q.pauli_masks(terms, N)
    distinct = len(set(x.tolist()))
    got = q.expectation_dry_run(N, terms, prec)["sweeps"]
    print(f"precision {prec}: 1000 random strings of weight <= 4 -> {got} sweeps, {distinct} distinct x masks")
    assert got <= distinct


def test_dry_run_splits_large_batches():
    """A batch larger than one launch holds is split; every chunk rereads the state."""
    terms = [f"Z{a} Z{b}" for a in range(N) for b in range(a + 1, N)]       # 435 diagonal terms
    one = q.expectation_dry_run(N, terms)["sweeps"]
    three = q.expectation_dry_run(N, terms * 3)["sweeps"]
    assert one == 1 and three == 3


@pytest.mark.parametrize("world", [2, 4, 8])
def test_dry_run_sharded_exchanges(world):
    g = world.bit_length() - 1
    for prec in (q.F32, q.F64):
        top = N - 1                       # from the identity layout the top log2(world) qubits are the rank bits
        assert q.expectation_dry_run(N, [f"X{top}"], prec, world_size=world)["exchanges"] >= 1
        assert q.expectation_dry_run(N, [f"Y{N - g} Z0"], prec, world_size=world)["exchanges"] >= 1
        assert q.expectation_dry_run(N, [f"Z{top}", f"Z0 Z{top}", "Z3"], prec, world_size=world) == {"sweeps": 1, "exchanges": 0}
        assert q.expectation_dry_run(N, ising(N), prec, world_size=world)["exchanges"] == g


def test_dry_run_refusals():
    with pytest.raises(q.QsbError) as e:
        x = np.array([1 << 8], dtype=np.uint64)
        z = np.zeros(1, dtype=np.uint64)
        sw, ex = C.c_uint32(), C.c_uint32()
        q.simulator.check(_lib.lib.qsb_expectation_dry_run(8, None, x.ctypes.data, z.ctypes.data, 1, C.byref(sw), C.byref(ex)))
    assert e.value.code == -1 and "qubit >= 8" in str(e.value)
    rc = _lib.lib.qsb_expectation_dry_run(8, None, None, None, 3, None, None)
    assert rc == -1


def test_expectation_on_null_handle_fails_cleanly():
    x = np.array([1], dtype=np.uint64)
    out = np.zeros(1)
    assert _lib.lib.qsb_expectation_pauli(None, x.ctypes.data, x.ctypes.data, 1, out.ctypes.data) == -1
    assert "null handle" in _lib.lib.qsb_last_error().decode()
    assert _lib.lib.qsb_expectation_pauli(None, None, None, 0, None) == -1
