"""Overlaps, host side: the steps and partner-shard copies of qsb_inner_product_dry_run for hand-built layouts, and its
argument checks.  No device needed."""
import ctypes as C

import numpy as np
import pytest

import gpu_quantum_simulator_b200 as q
from gpu_quantum_simulator_b200 import _lib

N = 20


def swapped(n, pairs):
    """identity layout with the physical bits of each (a, b) pair of qubits exchanged"""
    p = list(range(n))
    for a, b in pairs:
        p[a], p[b] = p[b], p[a]
    return p


@pytest.mark.parametrize("pa,pb", [(q.F32, q.F32), (q.F32, q.F64), (q.F64, q.F32), (q.F64, q.F64)])
@pytest.mark.parametrize("n", [1, 3, 12, 20])
def test_one_gpu_is_one_step_for_any_layouts(n, pa, pb):
    rng = np.random.default_rng(n)
    for _ in range(5):
        a, b = rng.permutation(n), rng.permutation(n)
        assert q.overlap_dry_run(n, a, b, pa, pb) == {"steps": 1, "exchanges": 0}
    # small registers: the qubits may sit anywhere among the (padded) local bits
    nloc = {q.F32: 12, q.F64: 11}
    if n < 11:
        a = rng.permutation(nloc[pa])[:n]
        b = rng.permutation(nloc[pb])[:n]
        assert q.overlap_dry_run(n, a, b, pa, pb) == {"steps": 1, "exchanges": 0}


@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_same_rank_qubit_on_two_ranks(prec):
    a = swapped(N, [(3, 7)])
    b = swapped(N, [(0, 11), (2, 5)])          # local bits differ, q19 stays the rank qubit of both
    for r in range(2):
        assert q.overlap_dry_run(N, a, b, prec, prec, world_size=2, rank=r) == {"steps": 1, "exchanges": 0}


def test_swapped_rank_positions_on_four_ranks():
    """rank bits (q5, q6) for a and (q6, q5) for b: d = 0, ranks 0 and 3 combine their own shard, 1 and 2 trade."""
    nloc = N - 2
    a = swapped(N, [(5, nloc), (6, nloc + 1)])
    b = swapped(N, [(6, nloc), (5, nloc + 1)])
    want = {0: (1, 0), 1: (1, 1), 2: (1, 1), 3: (1, 0)}
    for r, (st, ex) in want.items():
        assert q.overlap_dry_run(N, a, b, world_size=4, rank=r) == {"steps": st, "exchanges": ex}
        assert q.overlap_dry_run(N, a, b, q.F64, q.F32, world_size=4, rank=r) == {"steps": st, "exchanges": ex}


@pytest.mark.parametrize("world", [4, 8])
def test_disjoint_rank_sets(world):
    g = world.bit_length() - 1
    n = 24
    nloc = n - g
    a = list(range(n))
    b = swapped(n, [(i, nloc + i) for i in range(g)])       # b's rank qubits are q0..q(g-1), local in a
    for r in range(world):
        assert q.overlap_dry_run(n, a, b, world_size=world, rank=r) == {"steps": world, "exchanges": world - 1}


def test_one_shared_and_one_differing_rank_qubit():
    """world 4: C = {q19}, D_a = {q18}, D_b = {q2}: 2 steps, and each rank copies a partner shard in one of them."""
    a = list(range(N))
    b = swapped(N, [(2, N - 2)])
    for r in range(4):
        assert q.overlap_dry_run(N, a, b, world_size=4, rank=r) == {"steps": 2, "exchanges": 1}


def _raw(n, perm_a, perm_b, oa, ob):
    pa = np.full(64, -1, dtype=np.int8)
    pb = np.full(64, -1, dtype=np.int8)
    pa[:n], pb[:n] = perm_a, perm_b
    st, ex = C.c_uint32(), C.c_uint32()
    rc = q.lib.qsb_inner_product_dry_run(n, C.byref(oa), pa.ctypes.data, C.byref(ob), pb.ctypes.data, C.byref(st), C.byref(ex))
    return rc, q.lib.qsb_last_error().decode()


def _opt(world=1, rank=0, prec=q.F32, low_bits=0):
    o = _lib.Options()
    q.lib.qsb_options_default(C.byref(o))
    o.precision, o.world_size, o.rank, o.low_bits = prec, world, rank, low_bits
    return o


def test_refused_arguments():
    ident = list(range(N))
    assert _raw(N, ident, ident, _opt(), _opt())[0] == 0
    bad = list(range(N)); bad[3] = 4
    for perm_a, perm_b in ((bad, ident), (ident, bad)):
        rc, msg = _raw(N, perm_a, perm_b, _opt(), _opt())
        assert rc == -1 and "not a permutation" in msg
    rc, msg = _raw(N, ident[:-1] + [N], ident, _opt(), _opt())     # a physical bit beyond the shard
    assert rc == -1 and "not a permutation" in msg
    rc, msg = _raw(N, ident, ident, _opt(world=2), _opt(world=4))
    assert rc == -1 and "differ in world" in msg
    rc, msg = _raw(N, ident, ident, _opt(world=2, rank=0), _opt(world=2, rank=1))
    assert rc == -1 and "differ in world" in msg
    rc, msg = _raw(N, ident, ident, _opt(world=2, rank=2), _opt(world=2, rank=2))
    assert rc == -1 and "outside world" in msg
    for prec, lows in ((q.F32, (1, 2, 7, 8)), (q.F64, (1, 6, 7))):
        for lb in lows:
            for oa, ob in ((_opt(prec=prec, low_bits=lb), _opt()), (_opt(), _opt(prec=prec, low_bits=lb))):
                rc, msg = _raw(N, ident, ident, oa, ob)
                assert rc == -1 and f"low_bits {lb} unsupported" in msg, (prec, lb)
    for prec, lows in ((q.F32, (3, 4, 5, 6)), (q.F64, (2, 3, 4, 5))):
        for lb in lows:
            assert _raw(N, ident, ident, _opt(prec=prec, low_bits=lb), _opt(prec=prec, low_bits=lb))[0] == 0
    with pytest.raises(q.QsbError):
        q.overlap_dry_run(N, bad, ident)
    with pytest.raises(q.QsbError):
        q.overlap_dry_run(N, ident, ident, low_bits_a=9)
