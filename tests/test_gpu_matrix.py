"""Dense k-qubit matrices on the device (qsb_apply_matrices) against numpy applying each matrix to the downloaded state by
tensordot over the target axes, in list order."""
import os
import subprocess
import sys

import numpy as np
import pytest
from scipy.stats import unitary_group

import helpers
import gpu_quantum_simulator_b200 as q
from gpu_quantum_simulator_b200 import circuits
from test_gpu_pauli_rotation import permuted, rotate_np

pytestmark = pytest.mark.gpu

F32, F64 = q.F32, q.F64
PRECS = pytest.mark.parametrize("prec", [F32, F64], ids=["f32", "f64"])
TOL = {F32: 1e-5, F64: 1e-12}
LOW_BITS = {F32: [0, 3, 5, 6], F64: [0, 2, 4, 5]}        # 0 = the default (4 / 3)


def apply_np(a, ops, n):
    """ops: (U, targets[, controls]); bit i of a row / column index of U is the value of targets[i]."""
    a = np.array(a, dtype=np.complex128)
    idx = np.arange(1 << n, dtype=np.int64)
    for op in ops:
        U, ts = np.asarray(op[0], dtype=np.complex128), list(op[1])
        cs = list(op[2]) if len(op) > 2 else []
        k = len(ts)
        psi = a.reshape([2] * n)                       # axis n - 1 - qb is qubit qb
        axes = [n - 1 - t for t in ts[::-1]]           # row / column axis j of U.reshape is bit k - 1 - j
        out = np.tensordot(U.reshape([2] * (2 * k)), psi, axes=(list(range(k, 2 * k)), axes))
        out = np.moveaxis(out, list(range(k)), axes).reshape(-1)
        if cs:
            on = np.all([(idx >> c) & 1 for c in cs], axis=0)
            out = np.where(on, out, a)
        a = out
    return a


def unitary(k, seed):
    return unitary_group.rvs(1 << k, random_state=seed)


def contraction(k, seed):
    """A random non-unitary matrix of spectral norm 1."""
    rng = np.random.default_rng(seed)
    m = rng.normal(size=(1 << k, 1 << k)) + 1j * rng.normal(size=(1 << k, 1 << k))
    return m / np.linalg.norm(m, 2)


def random_ops(n, count, seed, kmax=6, controls=True):
    rng = np.random.default_rng(seed)
    ops = []
    for i in range(count):
        k = int(rng.integers(1, min(kmax, n) + 1))
        qs = [int(x) for x in rng.permutation(n)]
        ts, rest = qs[:k], qs[k:]
        cs = rest[:int(rng.integers(0, min(2, len(rest)) + 1))] if controls and rng.random() < 0.3 else []
        U = unitary(k, seed * 1000 + i) if i % 2 == 0 else contraction(k, seed * 1000 + i)
        ops.append((U, ts, cs))
    return ops


def check(s, ops, tol):
    """Apply on the device, compare with numpy from the state as it was; the qubit layout must not move."""
    n = s.num_qubits
    a0, perm0 = s.state(), s.layout()[0]
    s.apply_matrices(ops)
    want = apply_np(a0, ops, n)
    err = float(np.max(np.abs(s.state() - want)))
    assert err <= tol, (n, err)
    assert np.array_equal(s.layout()[0], perm0)
    return err


WIDTHS = [(p, lb) for p in (F32, F64) for lb in LOW_BITS[p]]


@pytest.mark.parametrize("prec,low_bits", WIDTHS, ids=[f"f{p}-low{lb}" for p, lb in WIDTHS])
def test_every_width_on_every_low_bits(prec, low_bits):
    """k = 1..6 on qubits in and out of the low bits and across the tile size, unitary and non-unitary, on a permuted
    layout: one op per call, then all of them as one call."""
    for n in (6, 11, 12, 13, 16):
        with permuted(n, prec, low_bits) as s:
            ops = []
            for k in range(1, 7):
                for j, ts in enumerate((list(range(k)), list(range(n - k, n))[::-1], [int(x) for x in np.random.default_rng(k + n).permutation(n)[:k]])):
                    U = unitary(k, 10 * k + j) if j != 1 else contraction(k, 10 * k + j)
                    ops.append((U, ts))
                    check(s, [ops[-1]], TOL[prec])
            check(s, ops, 3 * TOL[prec])


SIZES = [1, 2, 5, 11, 12, 13, 17, 21, 26]


@pytest.mark.parametrize("mode", [q.MODE_TILED, q.MODE_SWEEP], ids=["tiled", "sweep"])
@pytest.mark.parametrize("n", SIZES)
@PRECS
def test_sizes_modes_and_layouts(n, mode, prec):
    count = 40 if n <= 21 else 8
    rng = np.random.default_rng(n)
    with permuted(n, prec, mode=mode) as s:
        check(s, random_ops(n, count, seed=n), 3 * TOL[prec])
        a = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)     # unnormalised upload
        s.set_state(3.0 * a / np.linalg.norm(a))
        check(s, random_ops(n, count, seed=n + 100), 10 * TOL[prec])


@PRECS
def test_f32_bound_at_k6(prec):
    """The error of one k = 6 op, reported so the f32 tolerance rests on a measured value."""
    n = 20
    with permuted(n, prec) as s:
        errs = [check(s, [(unitary(6, 70 + j), ts)], TOL[prec]) for j, ts in
                enumerate(([0, 1, 2, 3, 4, 5], [19, 3, 11, 7, 15, 0], [14, 15, 16, 17, 18, 19]))]
    print(f"k=6 prec={prec} max errors {errs}")


@PRECS
def test_controls(prec):
    n = 20
    U2, U1 = unitary(2, 1), contraction(1, 2)
    with permuted(n, prec) as s:
        perm, _ = s.layout()
        hi = sorted(range(n), key=lambda qb: -perm[qb])            # the highest-placed qubits lie outside most tiles
        lo = sorted(range(n), key=lambda qb: perm[qb])
        cases = [(U2, [lo[0], lo[1]], [lo[2]]),                  # control on a low (tile) bit
                 (U2, [lo[0], hi[0]], [hi[1]]),                  # control outside the tile
                 (U1, [hi[2]], [lo[3], hi[0], hi[5]]),            # several, mixed
                 (unitary(3, 3), [hi[3], lo[1], hi[7]], [lo[0], hi[1], hi[2], hi[4]]),
                 (unitary(6, 4), hi[:6], [lo[0]])]
        for op in cases:
            check(s, [op], 2 * TOL[prec])
        check(s, cases * 3, 10 * TOL[prec])


def gate_m(g):
    return np.array([[g.m[0] + 1j * g.m[1], g.m[2] + 1j * g.m[3]], [g.m[4] + 1j * g.m[5], g.m[6] + 1j * g.m[7]]])


@PRECS
def test_pins_against_other_paths(prec):
    n = 14
    circ = q.gates_from_circuit(circuits.random_layered(n, depth=3, seed=4))

    def pair():
        s1, s2 = q.Simulator(n, precision=prec, device=0), q.Simulator(n, precision=prec, device=0)
        s1.apply(circ)
        s2.apply(circ)
        return s1, s2

    # k = 1 against qsb_apply_gates with the same m, with and without controls; CCX as X with two controls
    for name, qs, params in (("u", [5], [0.3, 1.1, -0.7]), ("cu", [2, 9], [0.4, -0.2, 0.9, 0.0]), ("ccx", [1, 12, 6], []),
                             ("ry", [13], [0.77])):
        g = q.gates_from_circuit([(name, qs, params)])
        assert len(g) == 1
        ctrl = [c for c in range(n) if (g[0].controls >> c) & 1]
        s1, s2 = pair()
        s1.apply_matrix(gate_m(g[0]), [g[0].target], ctrl)
        s2.apply(g)
        assert np.max(np.abs(s1.state() - s2.state())) <= 2 * TOL[prec], name
        s1.close(); s2.close()
    # the matrix of a small random circuit on k qubits against apply() of that circuit
    for k, qs in ((2, [3, 10]), (4, [13, 0, 7, 2]), (6, [1, 12, 4, 9, 6, 11])):
        sub = circuits.random_layered(k, depth=4, seed=k)
        with q.Simulator(k, precision=F64, device=0) as m:
            cols = []
            for c in range(1 << k):
                e = np.zeros(1 << k, dtype=np.complex128); e[c] = 1
                m.set_state(e)
                m.apply(q.gates_from_circuit(sub))
                cols.append(m.state())
        U = np.stack(cols, axis=1)
        mapped = [(nm, [qs[x] for x in qq], p) for nm, qq, p in sub]
        s1, s2 = pair()
        s1.apply_matrix(U, qs)
        s2.apply(q.gates_from_circuit(mapped))
        assert np.max(np.abs(s1.state() - s2.state())) <= 3 * TOL[prec], k
        s1.close(); s2.close()
    # the matrix of exp(-i t P / 2) on P's support against apply_pauli_rotations
    for text, qs in (("X3 Z8", [3, 8]), ("Y0 Y13 Z6", [0, 13, 6])):
        k, t = len(qs), 0.9
        local = " ".join(f"{tok[0]}{j}" for j, tok in enumerate(text.split()))
        U = np.stack([rotate_np(np.eye(1 << k)[:, c], [local], [t], k) for c in range(1 << k)], axis=1)
        s1, s2 = pair()
        s1.apply_matrix(U, qs)
        s2.apply_pauli_rotations(text, t)
        assert np.max(np.abs(s1.state() - s2.state())) <= 2 * TOL[prec], text
        s1.close(); s2.close()


@PRECS
def test_invariants(prec):
    n = 16
    ops = random_ops(n, 30, seed=5, controls=True)
    inv = [(np.conj(U).T, ts, cs) for U, ts, cs in ops[::-1] if np.allclose(U @ np.conj(U).T, np.eye(len(U)))]
    uni = [op for op in ops if np.allclose(op[0] @ np.conj(op[0]).T, np.eye(len(op[0])))]
    with permuted(n, prec) as s, permuted(n, prec) as r:
        raw0, perm0 = s.state_native().copy(), s.layout()[0]
        s.apply_matrices([])
        assert np.array_equal(s.state_native(), raw0)
        a0 = s.state()
        s.apply_matrices(uni)
        s.apply_matrices(inv)                                     # U then U^dagger returns the state
        assert np.max(np.abs(s.state() - a0)) <= 10 * TOL[prec]
        assert np.array_equal(s.layout()[0], perm0)
        s.set_state(a0)
        r.set_state(a0)
        s.apply_matrices(ops)
        r.apply_matrices(ops)                                     # repeated calls: identical bytes
        assert np.array_equal(s.state_native(), r.state_native())


@PRECS
def test_plans_and_graphs_made_before_the_call(prec):
    n = 18
    circ = q.gates_from_circuit(circuits.random_layered(n, depth=4, seed=8))
    ops = random_ops(n, 20, seed=9)
    for use_graph in (False, True):
        with q.Simulator(n, precision=prec, device=0, use_graph=use_graph) as s, q.Simulator(n, precision=prec, device=0) as r:
            p = s.plan(circ)
            if use_graph:
                s.execute(p)                                     # captures the graph
                s.reset()
            check(s, ops, 3 * TOL[prec])
            r.set_state(s.state())
            s.execute(p)
            r.apply(circ)
            assert np.max(np.abs(s.state() - r.state())) <= 3 * TOL[prec], use_graph
            p.close()


@PRECS
def test_refused_arguments_leave_the_state(prec):
    n = 12
    U = unitary(2, 0)
    with permuted(n, prec) as s:
        raw0 = s.state_native().copy()
        bad_u = U.copy(); bad_u[1, 1] = np.nan
        for ops, text in (([(U, [0, 12])], "outside"), ([(U, [3, 3])], "twice"), ([(U, [0, 1], [1])], "both a control"),
                          ([(U, [0, 1], [12])], "control >= 12"), ([(U, [0, 1]), (bad_u, [2, 3])], "non-finite"),
                          ([(np.eye(128), list(range(7)))], "at most 6")):
            with pytest.raises((q.QsbError, ValueError)) as e:
                s.apply_matrices(ops)
            assert text in str(e.value), text
        arr = (q.MatrixOp * 1)()
        arr[0].k, arr[0].targets[0] = 1, 0
        assert q.lib.qsb_apply_matrices(s._h, arr, 1) == -1                        # null m
        assert "null matrix" in q.lib.qsb_last_error().decode()
        arr[0].m = np.eye(2, dtype=np.complex128).view(np.float64).ctypes.data_as(q._lib.C.POINTER(q._lib.C.c_double))
        arr[0].flags = 1
        assert q.lib.qsb_apply_matrices(s._h, arr, 1) == -1
        arr[0].flags, arr[0].k = 0, 0
        assert q.lib.qsb_apply_matrices(s._h, arr, 1) == -1
        assert q.lib.qsb_apply_matrices(s._h, None, 1) == -1
        assert q.lib.qsb_apply_matrices(s._h, None, 0) == 0
        assert np.array_equal(s.state_native(), raw0)
        with pytest.raises(ValueError):
            s.apply_matrix(np.eye(4), [0])


@PRECS
def test_handle_with_unsupported_low_bits_is_refused(prec):
    """qsb_create takes any low_bits; the matrix call refuses the values that would leave an op no tile, before it
    touches the state."""
    n = 16
    with q.Simulator(n, precision=prec, low_bits=8, device=0) as s:
        s.set_state(np.arange(1 << n) * (1 + 1j) / (1 << n))
        raw0 = s.state_native().copy()
        for ops in ([(unitary(6, 1), list(range(10, 16)))], [(unitary(1, 2), [0])]):
            with pytest.raises(q.QsbError) as e:
                s.apply_matrices(ops)
            assert e.value.code == -1 and "low_bits 8 unsupported" in str(e.value)
        assert np.array_equal(s.state_native(), raw0)


def test_cli_matrix_then_expect(tmp_path):
    exe = os.path.join(helpers.ROOT, "gpu_quantum_simulator_b200", "bin", "qsim")
    n = 14
    circ = circuits.random_layered(n, depth=4, seed=9)
    path = tmp_path / "c.qasm"
    path.write_text(circuits.to_qasm(circ, n))
    ops = [(unitary(2, 1), [0, 3]), (contraction(1, 2), [13]), (unitary(3, 3), [7, 2, 11])]
    args = [exe, str(path)]
    for j, (U, qs) in enumerate(ops):
        f = tmp_path / f"m{j}.txt"
        f.write_text("\n".join(" ".join(f"{float(v.real)!r} {float(v.imag)!r}" for v in row) for row in U) + "\n")
        args += ["--matrix", " ".join(map(str, qs)), str(f)]
    texts = ["Z0", "X0 Z3", "Y13 Z2", ""]
    for t in texts:
        args += ["--expect", t]
    r = subprocess.run(args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    exp = r.stdout.splitlines()[1:1 + len(texts)]
    assert [ln.rsplit(":", 1)[0] for ln in exp] == [f"EXPECTATION {t}" for t in texts]
    with q.Simulator(n, precision=F32, device=0) as s:
        s.apply(q.gates_from_circuit(circ))
        s.apply_matrices(ops)
        want = s.expectation(texts)
    got = np.array([float(ln.rsplit(":", 1)[1]) for ln in exp])
    assert np.max(np.abs(got - want)) <= 1e-12
    short = tmp_path / "short.txt"
    short.write_text("1 0 0 0 0 0\n")
    for extra, text in ((["--matrix", "0", str(short)], "expected 8 numbers"),
                        (["--matrix", "0", str(tmp_path / "missing.txt")], "cannot open"),
                        (["--matrix", "0 x", str(short)], "expected a whitespace-separated list"),
                        (["--matrix", "14", str(tmp_path / "m1.txt")], "target 14 outside")):
        bad = subprocess.run([exe, str(path)] + extra, capture_output=True, text=True, timeout=300)
        assert bad.returncode == 1 and text in bad.stdout, bad.stdout


def test_sharded_matrices():
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 8 if ngpu >= 8 else 4 if ngpu >= 4 else 2
    script = os.path.join(os.path.dirname(__file__), "dist_matrix_worker.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", "29573", script],
                       capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "sharded_matrix_ok" in r.stdout


def quantum_volume_layers(n, layers, seed):
    rng = np.random.default_rng(seed)
    ops = []
    for layer in range(layers):
        perm = rng.permutation(n)
        for j in range(n // 2):
            ops.append((unitary(2, seed * 100000 + layer * 100 + j), [int(perm[2 * j]), int(perm[2 * j + 1])]))
    return ops


@pytest.mark.slow
def test_30q_quantum_volume_f32_against_f64():
    n = 30
    ops = quantum_volume_layers(n, 10, seed=1)
    paulis = ["Z0", "Z0 Z1", "X5 X17", "Y29 Z3"]
    vals = []
    for prec in (F32, F64):
        with q.Simulator(n, precision=prec, device=0) as s:
            for k in range(0, len(ops), 15):
                s.apply_matrices(ops[k:k + 15])
            vals.append((s.norm_argmax()[0], s.marginal_probabilities(list(range(10, 20))), s.expectation(paulis)))
    assert abs(vals[0][0] - vals[1][0]) <= 1e-4 and abs(vals[1][0] - 1.0) <= 1e-10
    assert np.max(np.abs(vals[0][1] - vals[1][1])) <= 1e-4
    assert np.max(np.abs(vals[0][2] - vals[1][2])) <= 1e-4
