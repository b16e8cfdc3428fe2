"""Dense matrices, host side: the in-order sweep grouping of qsb_matrix_dry_run, the SWAP rewrite of ops with several rank
targets, and the argument checks.  No device needed."""
import ctypes as C

import numpy as np
import pytest

import gpu_quantum_simulator_b200 as q
from gpu_quantum_simulator_b200 import _lib

N = 30
TILE = {q.F32: 12, q.F64: 11}
LOW = {q.F32: 4, q.F64: 3}                                  # the default low bits
LOW_BITS = {q.F32: [3, 4, 5, 6], q.F64: [2, 3, 4, 5]}      # the values qsb_create accepts


def dry(shapes, prec=q.F32, world=1, low_bits=0, n=N):
    return q.matrix_dry_run(n, shapes, prec, world_size=world, low_bits=low_bits)


@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_ops_inside_the_low_bits_share_one_sweep(prec):
    L = LOW[prec]
    low = list(range(L))
    shapes = [[0], low, low[::-1], [1, 0], ([0], [1]), (low[:2], [N - 1])] * 50
    assert dry(shapes, prec) == {"sweeps": 1, "exchanges": 0}
    # any single op fits a tile, and one op outside the low bits still shares the sweep with them
    assert dry(shapes + [list(range(N - 6, N))] + shapes, prec) == {"sweeps": 1, "exchanges": 0}


@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_brickwork_layer_at_30_qubits(prec):
    """15 disjoint pairs (0, 1), (2, 3), ..., (28, 29); a sweep adds at most T - L = 8 tile bits to the low bits.
    f32 (L = 4): (0,1) (2,3) are free, (4,5)..(10,11) add 8 -> 6 pairs; then 4 + 4 + 1 pairs: 4 sweeps.
    f64 (L = 3): (0,1) free, (2,3) adds bit 3, (4,5)..(8,9) 6 more -> 5 pairs; then 4 + 4 + 2 pairs: 4 sweeps."""
    layer = [[k, k + 1] for k in range(0, N, 2)]
    assert dry(layer, prec) == {"sweeps": 4, "exchanges": 0}
    # the sweep boundaries, from the counts above
    first = 6 if prec == q.F32 else 5
    assert dry(layer[:first], prec)["sweeps"] == 1
    assert dry(layer[:first + 1], prec)["sweeps"] == 2
    assert dry(layer[:first + 4], prec)["sweeps"] == 2
    assert dry(layer[:first + 5], prec)["sweeps"] == 3
    # two layers: the last sweep of the first goes on into the second (f32: (28,29) + (0,1)..(8,9); f64: (26,27) (28,29)
    # + (0,1)..(4,5)), then 4 + 4 + 2 pairs (f32) / 4 + 4 + 4 pairs (f64): 7 sweeps, not 8
    assert dry(layer + layer, prec)["sweeps"] == 7


@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_wide_ops_on_disjoint_high_qubits_take_a_sweep_each(prec):
    ops = [list(range(a, a + 6)) for a in (6, 12, 18, 24)]
    for low in LOW_BITS[prec]:
        assert dry(ops, prec, low_bits=low) == {"sweeps": 4, "exchanges": 0}, low
        assert dry(ops[:1] * 5, prec, low_bits=low) == {"sweeps": 1, "exchanges": 0}   # the same targets: one run


@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_order_is_kept(prec):
    """6 + 2 high bits fill the 8 free tile bits (T - L = 8 for both defaults): a ninth bit breaks the run, even when a
    later op would fit the first tile again."""
    assert TILE[prec] - LOW[prec] == 8
    assert dry([list(range(10, 16)), [20, 21]], prec)["sweeps"] == 1
    assert dry([list(range(10, 16)), [20, 21], [22]], prec)["sweeps"] == 2
    assert dry([list(range(10, 16)), [22], [20, 21]], prec)["sweeps"] == 2
    # [22] starts the second sweep, which still has room for (10, 11)
    assert dry([list(range(10, 16)), [20, 21], [22], [10, 11]], prec)["sweeps"] == 2
    assert dry([list(range(10, 16)), [20, 21], [22], [0, 1], [12, 13, 14, 15, 16, 17], [23], [24]], prec)["sweeps"] == 3
    # controls never need tile bits
    assert dry([(list(range(10, 16)), list(range(16, 30))), ([20, 21], [22, 23, 24])], prec)["sweeps"] == 1


@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_counts(world):
    g = world.bit_length() - 1
    top = N - 1                                   # from the identity layout the top log2(world) qubits are the rank bits
    for prec in (q.F32, q.F64):
        assert dry([[top]], prec, world) == {"sweeps": 1, "exchanges": 1}
        assert dry([[0, top]], prec, world) == {"sweeps": 1, "exchanges": 1}
        assert dry([[5], [top, 3]] + [[top]] * 5 + [[0, 1]], prec, world) == {"sweeps": 1, "exchanges": 1}
        # controls on rank qubits cost nothing
        assert dry([([0, 1], [top]), ([2], [top, 6])], prec, world) == {"sweeps": 1, "exchanges": 0}
        if g >= 2:
            # alternating rank targets: one sweep and one exchange each
            assert dry([[top], [top - 1]] * 3, prec, world) == {"sweeps": 6, "exchanges": 6}
            assert dry([[top, top - 1]], prec, world) == {"sweeps": 3, "exchanges": 3}          # m = 2: 2m - 1
            assert dry([[0, top - 1, 7, top]], prec, world) == {"sweeps": 3, "exchanges": 3}
        if g >= 3:
            assert dry([[top, top - 1, top - 2]], prec, world) == {"sweeps": 5, "exchanges": 5}  # m = 3: 2m - 1
            assert dry([([top - 2, top, top - 1, 0], [1])], prec, world) == {"sweeps": 5, "exchanges": 5}


def test_sharded_swap_rewrite_needs_a_free_local_qubit():
    n, world = 26, 4                              # 24 local qubits
    ok = ([n - 1, n - 2], list(range(23)))        # qubit 23 is free
    assert dry([ok], world=world, n=n) == {"sweeps": 3, "exchanges": 3}
    with pytest.raises(q.QsbError) as e:
        dry([([n - 1, n - 2], list(range(24)))], world=world, n=n)
    assert e.value.code == -1 and "no free local qubit" in str(e.value)


def raw_dry(ops, count, n=8):
    sw, ex = C.c_uint32(), C.c_uint32()
    return _lib.lib.qsb_matrix_dry_run(n, None, ops, count, C.byref(sw), C.byref(ex)), sw.value, ex.value


def test_refusals():
    def one(k=1, targets=(0,), controls=0, flags=0):
        arr = (q.MatrixOp * 1)()
        arr[0].k, arr[0].controls, arr[0].flags = k, controls, flags
        for j, t in enumerate(targets):
            arr[0].targets[j] = t
        return arr

    assert raw_dry(one(), 1)[0] == 0
    assert raw_dry(None, 0) == (0, 0, 0)
    assert raw_dry(None, 2)[0] == -1
    for arr, text in ((one(k=0), "0 targets"), (one(k=7, targets=range(6)), "7 targets"),
                      (one(k=2, targets=(3, 3)), "target 3 twice"), (one(k=2, targets=(1, 8)), "target 8 outside"),
                      (one(k=1, targets=(-1,)), "target -1 outside"), (one(controls=1), "both a control and a target"),
                      (one(controls=1 << 8), "control >= 8"), (one(flags=1), "flags 1")):
        assert raw_dry(arr, 1)[0] == -1
        assert text in _lib.lib.qsb_last_error().decode(), text
    assert raw_dry(one(k=4, targets=(0, 1, 2, 3)), 1, n=3)[0] == -1         # k > n
    with pytest.raises(q.QsbError):
        dry([[0]], world=3)
    with pytest.raises(q.QsbError):
        dry([[0]], world=8, n=14)                 # too few qubits to shard
    with pytest.raises(ValueError):
        dry([list(range(7))])
    assert _lib.lib.qsb_apply_matrices(None, one(), 1) == -1
    assert "null handle" in _lib.lib.qsb_last_error().decode()
    assert _lib.lib.qsb_apply_matrices(None, None, 0) == -1


def test_struct_layout():
    assert C.sizeof(q.MatrixOp) == 8 + 4 + 6 * 4 + 4 + 8
    assert q.MatrixOp.m.offset == 40


@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_low_bits_outside_the_accepted_range_are_refused(prec):
    """A tile keeps T - L >= 6 free bits only for the low_bits the tile scheduler accepts; any other value is refused
    with QSB_ERR_ARG (it would leave an op that fits no tile), also for ops inside the low bits."""
    for low in (1, 2, 7, 8, 11, 12, 40) if prec == q.F32 else (1, 6, 7, 11, 40):
        for shapes in ([list(range(20, 26))], [[20]], [[0]]):
            with pytest.raises(q.QsbError) as e:
                dry(shapes, prec, low_bits=low)
            assert e.value.code == -1 and f"low_bits {low} unsupported" in str(e.value), (low, shapes)
    for low in LOW_BITS[prec] + [0, -1]:                   # 0 and negative values mean the default
        assert dry([list(range(20, 26)), list(range(0, 6))], prec, low_bits=low)["sweeps"] >= 1


def test_apply_matrices_takes_any_iterable():
    """Simulator.apply_matrices builds its list once: a generator of ops reaches the library (and, without a device,
    its refusal of the null handle) instead of a TypeError."""
    s = q.Simulator.__new__(q.Simulator)
    s._h = C.c_void_p()
    with pytest.raises(q.QsbError) as e:
        s.apply_matrices((np.eye(2), [k]) for k in range(3))
    assert e.value.code == -1 and "null handle" in str(e.value)
