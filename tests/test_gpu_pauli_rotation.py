"""Pauli rotations on the device (qsb_apply_pauli_rotations) against numpy applying the header's formula in list order:
a <- cos(t/2) a - i sin(t/2) (P a), (P a)_j = i^{popc(x&z)} (-1)^{popc((j^x)&z)} a_{j^x}, on the state as downloaded
before the call."""
import itertools
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers
import gpu_quantum_simulator_b200 as q
from gpu_quantum_simulator_b200 import circuits
from test_gpu_expectation import pauli_apply, random_terms

pytestmark = pytest.mark.gpu

F32, F64 = q.F32, q.F64
PRECS = pytest.mark.parametrize("prec", [F32, F64], ids=["f32", "f64"])
TOL = {F32: 1e-5, F64: 1e-12}
LOW_BITS = {F32: [0, 3, 5, 6], F64: [0, 2, 4, 5]}        # 0 = the default (4 / 3)


def rotate_np(a, terms, thetas, n):
    x, z = q.pauli_masks(terms, n)
    a = np.array(a, dtype=np.complex128)
    for xx, zz, t in zip(x.tolist(), z.tolist(), np.atleast_1d(thetas)):
        a = np.cos(t / 2) * a - 1j * np.sin(t / 2) * pauli_apply(a, xx, zz)
    return a


def angles(count, rng):
    """Random angles with pi (-iP) and 2 pi (-I) among them."""
    t = rng.uniform(-np.pi, np.pi, size=count)
    t[::7] = np.pi
    t[3::11] = 2 * np.pi
    return t


def check(s, terms, thetas, tol):
    """Apply on the device, compare with numpy from the state as it was; the qubit layout must not move."""
    n = s.num_qubits
    a0, perm0 = s.state(), s.layout()[0]
    s.apply_pauli_rotations(terms, thetas)
    want = rotate_np(a0, terms, thetas, n)
    err = float(np.max(np.abs(s.state() - want)))
    assert err <= tol, (n, err)
    assert np.array_equal(s.layout()[0], perm0)
    return err


def permuted(n, prec, low_bits=0, mode=q.MODE_TILED):
    s = q.Simulator(n, precision=prec, low_bits=low_bits, mode=mode, device=0)
    for seed in range(1, 30):
        s.apply(q.gates_from_circuit(circuits.random_layered(n, depth=2, seed=seed)))
        if mode == q.MODE_SWEEP or n < 3 or not np.array_equal(s.layout()[0][:n], np.arange(n)):
            return s
    s.close()
    raise AssertionError("no circuit left a permuted layout")


def low_weight_strings(n):
    out = [""]
    for a in range(n):
        out += [f"{p}{a}" for p in "XYZ"]
    for a, b in itertools.combinations(range(n), 2):
        out += [f"{p}{a} {r}{b}" for p in "XYZ" for r in "XYZ"]
    return out


EXHAUSTIVE = [(p, n, lb) for p in (F32, F64) for n in ((12 if p == F32 else 11), 13, 14, 16) for lb in LOW_BITS[p]]


@pytest.mark.parametrize("prec,n,low_bits", EXHAUSTIVE, ids=[f"f{p}-n{n}-low{lb}" for p, n, lb in EXHAUSTIVE])
def test_every_low_weight_string(prec, n, low_bits):
    """Every string of weight <= 2, plus X / Y / mixed on every qubit, on a permuted layout, in batches of 64 so each
    batch is checked against numpy from the state it started from."""
    terms = low_weight_strings(n) + [" ".join(f"X{k}" for k in range(n)), " ".join(f"Y{k}" for k in range(n)),
                                     " ".join(f"{'XYZ'[k % 3]}{k}" for k in range(n))]
    rng = np.random.default_rng(n * 100 + low_bits)
    th = angles(len(terms), rng)
    with permuted(n, prec, low_bits) as s:
        for k in range(0, len(terms), 64):
            check(s, terms[k:k + 64], th[k:k + 64], TOL[prec])


SIZES = [1, 2, 5, 11, 12, 13, 17, 21, 26]


@pytest.mark.parametrize("mode", [q.MODE_TILED, q.MODE_SWEEP], ids=["tiled", "sweep"])
@pytest.mark.parametrize("n", SIZES)
@PRECS
def test_sizes_modes_and_layouts(n, mode, prec):
    count = 200 if n <= 21 else 30
    rng = np.random.default_rng(n)
    terms = random_terms(n, count, seed=n)
    with permuted(n, prec, mode=mode) as s:
        check(s, terms, angles(count, rng), TOL[prec])
        a = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)     # unnormalised upload
        s.set_state(3.0 * a / np.linalg.norm(a))
        check(s, terms, angles(count, rng), 3 * TOL[prec])


@PRECS
def test_long_sequence_order_and_fusion(prec):
    n = 20
    rng = np.random.default_rng(5)
    terms = random_terms(n, 1000, seed=11)
    sweeps = q.pauli_rotation_dry_run(n, terms, prec)["sweeps"]
    assert sweeps > 10                              # spans several sweeps and launches
    with permuted(n, prec) as s:
        check(s, terms, angles(1000, rng), 3 * TOL[prec])
    # a non-commuting pair: each order matches numpy, and the two orders differ
    pair, th = ["X3 Z17", "Z3 Y9"], [0.7, -1.1]
    got = []
    for order in (pair, pair[::-1]):
        with permuted(n, prec) as s:
            check(s, order, th, TOL[prec])
            got.append(s.state())
    assert np.max(np.abs(got[0] - got[1])) > 0.01


@PRECS
def test_pins_against_the_gate_path(prec):
    n = 14
    circ = circuits.random_layered(n, depth=3, seed=4)
    th = 0.8123
    for k in (0, 5, n - 1):
        for rot, gates, phase in ((f"X{k}", [("rx", [k], [th])], 1.0), (f"Y{k}", [("ry", [k], [th])], 1.0),
                                  (f"Z{k}", [("p", [k], [th])], np.exp(-0.5j * th)),
                                  (f"Z{k} Z{(k + 3) % n}", [("cx", [k, (k + 3) % n], []), ("p", [(k + 3) % n], [th]),
                                                             ("cx", [k, (k + 3) % n], [])], np.exp(-0.5j * th))):
            with q.Simulator(n, precision=prec, device=0) as s1, q.Simulator(n, precision=prec, device=0) as s2:
                s1.apply(q.gates_from_circuit(circ))
                s2.apply(q.gates_from_circuit(circ))
                s1.apply_pauli_rotations(rot, th)
                s2.apply(q.gates_from_circuit(gates))
                assert np.max(np.abs(s1.state() - phase * s2.state())) <= 2 * TOL[prec], rot


@PRECS
def test_invariants(prec):
    n = 16
    rng = np.random.default_rng(2)
    terms = random_terms(n, 300, seed=3)
    th = angles(300, rng)
    with permuted(n, prec) as s:
        raw0, perm0 = s.state_native().copy(), s.layout()[0]
        s.apply_pauli_rotations(terms, np.zeros(300))           # theta = 0 and an empty list: the same bytes
        s.apply_pauli_rotations([], [])
        assert np.array_equal(s.state_native(), raw0)
        norm0 = s.norm_argmax()[0]
        a0 = s.state()
        s.apply_pauli_rotations(terms, th)
        assert abs(s.norm_argmax()[0] - norm0) <= 10 * TOL[prec]
        s.apply_pauli_rotations(terms[::-1], -th[::-1])          # the inverse returns the state
        assert np.max(np.abs(s.state() - a0)) <= 3 * TOL[prec]
        assert np.array_equal(s.layout()[0], perm0)
    for t in (0.3, 1.9, np.pi):                                  # <Z> after R_X(t) |0> = cos t
        with q.Simulator(n, precision=prec, device=0) as s:
            s.apply_pauli_rotations("X4", t)
            assert abs(s.expectation("Z4") - np.cos(t)) <= TOL[prec]


@PRECS
def test_plans_and_graphs_made_before_the_call(prec):
    n = 18
    circ = q.gates_from_circuit(circuits.random_layered(n, depth=4, seed=8))
    terms = random_terms(n, 100, seed=9)
    th = angles(100, np.random.default_rng(9))
    for use_graph in (False, True):
        with q.Simulator(n, precision=prec, device=0, use_graph=use_graph) as s, q.Simulator(n, precision=prec, device=0) as r:
            p = s.plan(circ)
            if use_graph:
                s.execute(p)                                     # captures the graph
                s.reset()
            check(s, terms, th, 3 * TOL[prec])
            r.set_state(s.state())
            s.execute(p)
            r.apply(circ)
            assert np.max(np.abs(s.state() - r.state())) <= 3 * TOL[prec], use_graph
            p.close()


def ising(n):
    return [f"Z{k} Z{k + 1}" for k in range(n - 1)] + [f"X{k}" for k in range(n)], np.array([1.0] * (n - 1) + [0.7] * n)


def test_evolve():
    n = 10
    paulis, coeffs = ising(n)
    H = np.zeros((1 << n, 1 << n), dtype=np.complex128)
    eye = np.eye(1 << n)
    for p, c in zip(paulis, coeffs):
        x, z = q.pauli_masks(p, n)
        H += c * np.stack([pauli_apply(eye[:, j], int(x[0]), int(z[0])) for j in range(1 << n)], axis=1)
    import scipy.linalg
    a0 = np.zeros(1 << n, dtype=np.complex128); a0[0] = 1
    exact = scipy.linalg.expm(-1j * 0.8 * H) @ a0
    for order in (1, 2):
        errs = []
        for steps in (4, 8, 16):
            with q.Simulator(n, precision=F64, device=0) as s:
                s.evolve(paulis, coeffs, 0.8, steps, order=order)
                got = s.state()
            dt = 0.8 / steps
            if order == 1:
                want = rotate_np(a0, paulis * steps, np.tile(2 * coeffs * dt, steps), n)
            else:
                want = rotate_np(a0, (paulis + paulis[::-1]) * steps, np.tile(np.concatenate([coeffs * dt, (coeffs * dt)[::-1]]), steps), n)
            assert np.max(np.abs(got - want)) <= 1e-12
            errs.append(np.linalg.norm(got - exact))
        ratios = [errs[i] / errs[i + 1] for i in range(2)]
        lo, hi = (1.6, 2.5) if order == 1 else (3.2, 4.8)
        assert all(lo <= r <= hi for r in ratios), (order, errs, ratios)


@PRECS
def test_refused_arguments_leave_the_state(prec):
    n = 12
    with permuted(n, prec) as s:
        raw0 = s.state_native().copy()
        for bad in (["X12"], ["Z0 X40"]):
            with pytest.raises(q.QsbError) as e:
                x = np.array([1 << 12 if bad[0] == "X12" else (1 << 40) | 1], dtype=np.uint64)
                z = np.zeros(1, dtype=np.uint64)
                t = np.array([0.5])
                q.simulator.check(q.lib.qsb_apply_pauli_rotations(s._h, x.ctypes.data, z.ctypes.data, t.ctypes.data, 1))
            assert e.value.code == -1
        for t in (np.nan, np.inf, -np.inf):
            with pytest.raises(q.QsbError) as e:
                s.apply_pauli_rotations(["X0", "Z1"], [0.5, t])
            assert e.value.code == -1 and "non-finite" in str(e.value)
        x = np.array([1], dtype=np.uint64)
        t = np.array([0.5])
        assert q.lib.qsb_apply_pauli_rotations(s._h, None, x.ctypes.data, t.ctypes.data, 1) == -1
        assert q.lib.qsb_apply_pauli_rotations(s._h, x.ctypes.data, None, t.ctypes.data, 1) == -1
        assert q.lib.qsb_apply_pauli_rotations(s._h, x.ctypes.data, x.ctypes.data, None, 1) == -1
        assert q.lib.qsb_apply_pauli_rotations(s._h, None, None, None, 0) == 0
        assert np.array_equal(s.state_native(), raw0)
        with pytest.raises(ValueError):
            s.apply_pauli_rotations(["X0", "Z1"], [0.5])


def test_cli_pauli_rot_then_expect(tmp_path):
    exe = os.path.join(helpers.ROOT, "gpu_quantum_simulator_b200", "bin", "qsim")
    n = 14
    circ = circuits.random_layered(n, depth=4, seed=9)
    path = tmp_path / "c.qasm"
    path.write_text(circuits.to_qasm(circ, n))
    rots = [("X0 Z3", 0.25), ("Y13", -1.5), ("Z2 Z5", 2.0)]
    texts = ["Z0", "X0 Z3", "Y13 Z2", ""]
    args = [exe, str(path)]
    for p, t in rots:
        args += ["--pauli-rot", p, repr(t)]
    for t in texts:
        args += ["--expect", t]
    r = subprocess.run(args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    exp = r.stdout.splitlines()[1:1 + len(texts)]
    assert [ln.rsplit(":", 1)[0] for ln in exp] == [f"EXPECTATION {t}" for t in texts]
    with q.Simulator(n, precision=F32, device=0) as s:
        s.apply(q.gates_from_circuit(circ))
        s.apply_pauli_rotations([p for p, _ in rots], [t for _, t in rots])
        want = s.expectation(texts)
    got = np.array([float(ln.rsplit(":", 1)[1]) for ln in exp])
    assert np.max(np.abs(got - want)) <= 1e-12
    bad = subprocess.run([exe, str(path), "--pauli-rot", "X0", "abc"], capture_output=True, text=True, timeout=300)
    assert bad.returncode == 1 and "expected an angle" in bad.stdout


def test_sharded_pauli_rotation():
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 8 if ngpu >= 8 else 4 if ngpu >= 4 else 2
    script = os.path.join(os.path.dirname(__file__), "dist_pauli_rotation_worker.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", "29571", script],
                       capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "sharded_pauli_rotation_ok" in r.stdout


@pytest.mark.slow
def test_30q_ising_evolution_f32_against_f64():
    n = 30
    paulis, coeffs = ising(n)
    circ = q.gates_from_circuit(circuits.random_layered(n, depth=20))
    vals = []
    for prec in (F32, F64):
        with q.Simulator(n, precision=prec, device=0) as s:
            s.apply(circ)
            s.evolve(paulis, coeffs, 0.5, 4, order=2)
            vals.append(s.expectation(paulis))
            assert abs(s.norm_argmax()[0] - 1.0) <= (1e-4 if prec == F32 else 1e-10)
    assert np.max(np.abs(vals[0] - vals[1])) <= 1e-4
