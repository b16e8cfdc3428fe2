"""Noise channels, host side: the counts of qsb_channel_dry_run (groups of state-dependent channels, fixed-weight channels
resolved without a read, partner shards of sharded layouts), the argument checks, and the Kraus-set builders.
No device needed."""
import ctypes as C

import numpy as np
import pytest

import gpu_quantum_simulator_b200 as q
from gpu_quantum_simulator_b200 import _lib

N = 30
LOW_BITS = {q.F32: [3, 4, 5, 6], q.F64: [2, 3, 4, 5]}      # the values qsb_create accepts


def dry(channels, prec=q.F32, world=1, low_bits=0, n=N):
    return q.channel_dry_run(n, channels, prec, world_size=world, low_bits=low_bits)


def damping_layer(n=N):
    return [(q.amplitude_damping(0.01), [k]) for k in range(n)]


@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_amplitude_damping_layer(prec):
    """30 single-qubit state-dependent channels form 8 groups of at most 4 qubits: one read of the state per group (its
    reduced density matrix), and the 4 operators chosen in a group go in one matrix sweep before the next read."""
    assert dry(damping_layer(), prec) == {"sweeps": 8, "gram_sweeps": 8, "exchanges": 0}
    # without operators every channel is taken as state-dependent: the same counts
    assert dry([[k] for k in range(N)], prec) == {"sweeps": 8, "gram_sweeps": 8, "exchanges": 0}
    # the per-channel composition (a read and a sweep per channel) would take 30 of each
    assert dry(damping_layer()[:1], prec) == {"sweeps": 1, "gram_sweeps": 1, "exchanges": 0}


def test_amplitude_damping_layer_at_every_low_bits():
    """Every accepted low_bits leaves a tile room for 4 single-qubit operators: the counts do not change."""
    for prec in (q.F32, q.F64):
        for low in LOW_BITS[prec]:
            assert dry(damping_layer(), prec, low_bits=low) == {"sweeps": 8, "gram_sweeps": 8, "exchanges": 0}, (prec, low)
    # wider channels at the largest low_bits: 4-qubit operators on disjoint high qubits take a sweep each
    wide = [(None, list(range(a, a + 4))) for a in (10, 14, 18, 22, 26)]
    assert dry(wide, q.F32, low_bits=6) == {"sweeps": 5, "gram_sweeps": 5, "exchanges": 0}


@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_depolarizing_needs_no_read(prec):
    one = [(q.depolarizing(0.01), [k]) for k in range(N)]
    # 30 operators on 30 qubits: the matrix path's grouping of 30 single-qubit ops (4 sweeps), no read
    assert dry(one, prec) == {"sweeps": 4, "gram_sweeps": 0, "exchanges": 0}
    assert q.matrix_dry_run(N, [[k] for k in range(N)], prec)["sweeps"] == 4
    two = [(q.depolarizing(0.02, 2), [k, (k + 1) % N]) for k in range(N)]
    assert dry(two, prec)["gram_sweeps"] == 0
    flips = [(q.pauli_channel(0.01, 0, 0), [k]) for k in range(5)] + [(q.pauli_channel(0, 0, 0.02), [k]) for k in range(5)]
    assert dry(flips, prec) == {"sweeps": 1, "gram_sweeps": 0, "exchanges": 0}


@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_fixed_weight_channel_inside_a_group(prec):
    """A fixed-weight channel whose targets fit the group's union joins it (resolved on the host from rho_U); one that
    does not fit ends the group and is resolved from r alone."""
    ad, dep = q.amplitude_damping(0.1), q.depolarizing(0.05)
    inside = [(ad, [20]), (dep, [21]), (ad, [22]), (dep, [20]), (ad, [23])]
    assert dry(inside, prec) == {"sweeps": 1, "gram_sweeps": 1, "exchanges": 0}
    # the fixed-weight [24] breaks the union of 4 and is pending with the group's operators; [25] starts a second group
    split = inside + [(dep, [24]), (ad, [25])]
    assert dry(split, prec) == {"sweeps": 2, "gram_sweeps": 2, "exchanges": 0}
    # fixed-weight channels before any group are applied before the group is read
    assert dry([(dep, [k]) for k in range(4)] + [(ad, [10])], prec) == {"sweeps": 2, "gram_sweeps": 1, "exchanges": 0}
    # two-qubit state-dependent channels on overlapping pairs: (0,1) (1,2) (2,3) share U = {0..3}, (3,4) starts anew
    pairs = [(None, [k, k + 1]) for k in range(4)]
    assert dry(pairs, prec) == {"sweeps": 2, "gram_sweeps": 2, "exchanges": 0}


@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_fallbacks(world):
    g = world.bit_length() - 1
    top = N - 1                                   # from the identity layout the top log2(world) qubits are the rank bits
    for prec in (q.F32, q.F64):
        # local groups: no partner shard
        assert dry([[k] for k in range(8)], prec, world) == {"sweeps": 2, "gram_sweeps": 2, "exchanges": 0}
        # a group on a rank qubit: its Gram matrix from the reduced density matrix (2 reads, 1 partner shard), then the
        # pending operator on the rank qubit through the matrix path (1 sweep, 1 partner shard)
        assert dry([[top]], prec, world) == {"sweeps": 1, "gram_sweeps": 2, "exchanges": 2}
        # fixed-weight channels on rank qubits need no read, only the matrix path for their operators
        assert dry([(q.depolarizing(0.1), [top])], prec, world) == {"sweeps": 1, "gram_sweeps": 0, "exchanges": 1}
        # a pending run with a rank target, then a local group: the run's sweep, the read, the group's operator
        assert dry([(q.depolarizing(0.1), [top]), [0]], prec, world) == {"sweeps": 2, "gram_sweeps": 1, "exchanges": 1}
        if g >= 2:
            # two rank qubits in one group: 4 reads and 3 partner shards for rho, two rank targets for the run
            assert dry([[top, top - 1]], prec, world) == {"sweeps": 3, "gram_sweeps": 4, "exchanges": 6}


def raw(channels, n=8, opt=None):
    sw, gs, ex = C.c_uint32(), C.c_uint32(), C.c_uint32()
    return _lib.lib.qsb_channel_dry_run(n, opt, channels, len(channels) if channels is not None else 0, C.byref(sw),
                                        C.byref(gs), C.byref(ex))


def one(k=1, targets=(0,), nkraus=None, flags=0, kraus=None):
    """A one-element Channel array; kraus: an (m, d, d) complex array or None."""
    arr = (q.Channel * 1)()
    c = arr[0]
    c.k, c.flags = k, flags
    for j, t in enumerate(targets):
        c.targets[j] = t
    keep = None
    if kraus is not None:
        keep = np.ascontiguousarray(np.asarray(kraus, dtype=np.complex128))
        c.kraus = keep.view(np.float64).ctypes.data_as(C.POINTER(C.c_double))
        c.nkraus = keep.shape[0] if nkraus is None else nkraus
    else:
        c.nkraus = 1 if nkraus is None else nkraus
    arr._keep = keep
    return arr


def error():
    return _lib.lib.qsb_last_error().decode()


def test_refusals():
    ad = q.amplitude_damping(0.2)
    assert raw(one(kraus=ad)) == 0
    assert _lib.lib.qsb_channel_dry_run(8, None, None, 0, None, None, None) == 0
    assert _lib.lib.qsb_channel_dry_run(8, None, None, 2, None, None, None) == -1 and "null channel array" in error()
    nan = np.array(ad); nan[1, 0, 1] = np.nan           # operator 1, entry (0, 1): double 8 + 2
    inf = np.array(ad); inf[0, 1, 1] = np.inf
    lossy = [np.array(ad[0])]                           # drops K_1: not trace-preserving
    big = np.tile(np.eye(2, dtype=np.complex128) / np.sqrt(5), (5, 1, 1))
    for arr, text in ((one(k=0), "0 targets"), (one(k=5, targets=range(4)), "5 targets"),
                      (one(k=2, targets=(3, 3)), "target 3 twice"), (one(k=2, targets=(1, 8)), "target 8 outside"),
                      (one(targets=(-1,)), "target -1 outside"), (one(flags=2), "flags 2"),
                      (one(nkraus=0), "0 Kraus operators"), (one(kraus=big), "5 Kraus operators, expected 1..4"),
                      (one(kraus=nan), "non-finite entry at 10"), (one(kraus=inf), "non-finite"),
                      (one(kraus=lossy), "not trace-preserving")):
        assert raw(arr) == -1, text
        assert text in error(), (text, error())
    assert raw(one(k=4, targets=(0, 1, 2, 3)), n=3) == -1 and "4 targets, expected 1..3" in error()
    # a set within 1e-10 of trace-preserving is accepted, one beyond is not
    near = [np.array(ad[0]) * (1 + 1e-12), np.array(ad[1])]
    assert raw(one(kraus=near)) == 0
    far = [np.array(ad[0]) * (1 + 1e-9), np.array(ad[1])]
    assert raw(one(kraus=far)) == -1 and "not trace-preserving" in error()
    with pytest.raises(q.QsbError):
        dry([[0]], world=3)
    with pytest.raises(q.QsbError):
        dry([[0]], world=8, n=14)                 # too few qubits to shard
    with pytest.raises(ValueError):
        dry([list(range(5))])


def test_apply_refusals_without_a_device():
    """The null handle and null arrays are refused before anything else; n = 0 needs no arrays."""
    ad = one(kraus=q.amplitude_damping(0.2))
    r = (C.c_double * 1)(0.5)
    b = (C.c_uint32 * 1)()
    assert _lib.lib.qsb_apply_channels(None, ad, 1, r, b, None) == -1 and "null handle" in error()
    assert _lib.lib.qsb_apply_channels(None, None, 0, None, None, None) == -1 and "null handle" in error()
    s = q.Simulator.__new__(q.Simulator)
    s._h = C.c_void_p()
    with pytest.raises(q.QsbError) as e:
        s.apply_channels([(q.amplitude_damping(0.1), [0])])
    assert e.value.code == -1 and "null handle" in str(e.value)
    with pytest.raises(ValueError):
        s.apply_channels([(q.amplitude_damping(0.1), [0])], r=[0.1, 0.2])


@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_low_bits_outside_the_accepted_range_are_refused(prec):
    for low in (1, 7, 40) if prec == q.F32 else (1, 6, 40):
        with pytest.raises(q.QsbError) as e:
            dry(damping_layer(), prec, low_bits=low)
        assert e.value.code == -1 and f"low_bits {low} unsupported" in str(e.value)


def test_struct_layout():
    assert C.sizeof(q.Channel) == 4 + 16 + 4 + 4 + 4 + 8      # 4 bytes of padding before the pointer
    assert q.Channel.kraus.offset == 32


def complete(ops):
    d = ops[0].shape[0]
    return np.max(np.abs(sum(np.conj(K).T @ K for K in ops) - np.eye(d)))


def fixed_weight(ops):
    d = ops[0].shape[0]
    return all(np.max(np.abs(np.conj(K).T @ K - np.trace(np.conj(K).T @ K).real / d * np.eye(d))) <= 1e-12 for K in ops)


@pytest.mark.parametrize("name,ops,fixed", [
    ("depolarizing-1", q.depolarizing(0.3), True),
    ("depolarizing-2", q.depolarizing(0.2, 2), True),
    ("pauli", q.pauli_channel(0.1, 0.05, 0.2), True),
    ("bit-flip", q.pauli_channel(0.1, 0, 0), True),
    ("phase-flip", q.pauli_channel(0, 0, 0.1), True),
    ("amplitude-damping", q.amplitude_damping(0.3), False),
    ("phase-damping", q.phase_damping(0.3), False),
])
def test_builders(name, ops, fixed):
    """Each set is complete and classified as intended: the library reads the state exactly for the state-dependent
    ones."""
    ops = [np.asarray(K) for K in ops]
    assert complete(ops) <= 1e-14, name
    assert fixed_weight(ops) == fixed, name
    k = ops[0].shape[0].bit_length() - 1
    c = dry([(ops, list(range(k)))])
    assert c == {"sweeps": 1, "gram_sweeps": 0 if fixed else 1, "exchanges": 0}, (name, c)


def test_depolarizing_structure():
    """The identity comes first with weight 1 - p (4^k - 1) / 4^k, then every other Pauli product with p / 4^k; a
    depolarizing channel with p = 1 maps every state to I / 2^k."""
    for k in (1, 2):
        ops = q.depolarizing(0.4, k)
        d = 1 << k
        assert len(ops) == d * d
        assert np.allclose(ops[0], np.sqrt(1 - 0.4 * (d * d - 1) / (d * d)) * np.eye(d))
        rho = np.zeros((d, d), dtype=np.complex128)
        rho[0, 0] = 1
        out = sum(K @ rho @ np.conj(K).T for K in q.depolarizing(1.0, k))
        assert np.allclose(out, np.eye(d) / d)
    with pytest.raises(ValueError):
        q.depolarizing(0.1, 3)


def test_cli_refuses_malformed_channel_files_before_the_device(tmp_path):
    """qsim reads and checks every --channel file before it creates a handle: one line, exit 1, no device needed."""
    import os
    import subprocess
    exe = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpu_quantum_simulator_b200", "bin", "qsim")
    circ = tmp_path / "c.qasm"
    circ.write_text('OPENQASM 3.0;\ninclude "stdgates.inc";\nqubit[3] q;\nh q[0];\n')
    many = tmp_path / "many.txt"
    many.write_text("0.4 0 0 0 0 0 0.4 0\n" * 5)                 # 5 operators on one qubit: at most 4
    text = tmp_path / "text.txt"
    text.write_text("1 0 0 0 0 0 1 0 x\n")
    short = tmp_path / "short.txt"
    short.write_text("1 0 0 0 0 0\n")
    lossy = tmp_path / "lossy.txt"
    lossy.write_text("1 0 0 0 0 0 0.5 0\n")
    for f, q_, want in ((many, "0", "found more than 4 operators"),
                        (text, "0", "found text that is not a number after 8 numbers"),
                        (short, "0", "expected 1..4 operators of 8 numbers each"),
                        (short, "0 1", "expected 1..16 operators of 32 numbers each"),
                        (lossy, "0", "not trace-preserving"), (lossy, "3", "target 3 outside")):
        r = subprocess.run([exe, str(circ), "--channel", q_, str(f)], capture_output=True, text=True, timeout=60)
        assert r.returncode == 1 and want in r.stdout and len(r.stdout.splitlines()) == 1, (want, r.stdout)


def test_identity_operator_of_a_state_dependent_set_is_read():
    """{sqrt(.5) I, sqrt(.5) |0><0|, sqrt(.5) |1><1|} has an identity operator but is state-dependent: it is read."""
    ops = [np.sqrt(0.5) * np.eye(2), np.sqrt(0.5) * np.diag([1.0, 0.0]), np.sqrt(0.5) * np.diag([0.0, 1.0])]
    assert not fixed_weight(ops) and complete(ops) <= 1e-15
    assert dry([(ops, [2])]) == {"sweeps": 1, "gram_sweeps": 1, "exchanges": 0}
