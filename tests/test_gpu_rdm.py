"""Reduced density matrices on the device (qsb_reduced_density_matrix) against numpy on s.state() of the same handle.

rho[a, b] = sum of a_j conj(a_j') over index pairs that agree on every other qubit, bit i of a / b = value of qubits[i].
The reference reshapes the amplitudes to (2^k, 2^(n - k)) in that bit order and forms M M^H, in clongdouble where the
size allows and in complex128 otherwise.  Every comparison with numpy is absolute, <= 1e-12, in both precisions: the
products of two stored f32 components are exact in fp64."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers
import gpu_quantum_simulator_b200 as q
from gpu_quantum_simulator_b200 import circuits
from gpu_quantum_simulator_b200._lib import lib

TOL = {q.F32: 1e-6, q.F64: 1e-12}     # against analytic values (the stored state is rounded to the precision)
RTOL = 1e-12                          # against numpy on the stored state


def rho_np(a, qubits):
    """M M^H with M = the amplitudes as (2^k, 2^(n-k)), row index bit i = qubits[i]."""
    n = a.size.bit_length() - 1
    k = len(qubits)
    t = a.reshape((2,) * n) if n else a
    keep = [n - 1 - qb for qb in reversed(qubits)]          # axis 0 = the top bit of the row index
    rest = [ax for ax in range(n) if ax not in keep]
    M = np.transpose(t, keep + rest).reshape(1 << k, -1)
    if (1 << k) * M.size <= 1 << 24:
        M = M.astype(np.clongdouble)
        return np.asarray(M @ M.conj().T, dtype=np.complex128)
    return M @ M.conj().T


def run(n, circ, prec, mode=q.MODE_TILED, **kw):
    s = q.Simulator(n, precision=prec, mode=mode, device=0, **kw)
    s.apply(q.gates_from_circuit(circ))
    return s


def circuit_for(n, seed):
    if n in (2, 5, 11, 12):
        return circuits.random_superset(n, 12 * n, seed=seed)
    return circuits.random_layered(n, depth=6 if n > 5 else 3, seed=seed)


def qubit_sets(n, perm, rng):
    """qubit 0, qubit n - 1, the qubits on physical bits 0..3, contiguous, reversed and scattered sets, the largest k
    (min(n, 12) up to 20 qubits, 8 at 24), and every qubit for n <= 12"""
    sets = [[0], [n - 1]]
    for b in range(4):
        sets += [[qb] for qb in range(n) if perm[qb] == b]
    sets.append([qb for b in range(4) for qb in range(n) if perm[qb] == b])
    sets += [list(range(min(n, 4))), list(range(min(n, 4)))[::-1]]
    if n >= 3:
        sets += [sorted(rng.choice(n, min(n, 5), replace=False).tolist()), rng.permutation(n)[:min(n, 7)].tolist()]
    sets.append(rng.permutation(n)[:min(n, 12) if n <= 20 else 8].tolist())
    if n <= 12:
        sets.append(rng.permutation(n).tolist())
    return [qs for qs in sets if qs]


def bits(x):
    return np.ascontiguousarray(x).view(np.uint64)


def check_structure(rho, k):
    """exactly Hermitian, +0.0 diagonal imaginary parts"""
    assert rho.shape == (1 << k, 1 << k)
    off = ~np.eye(1 << k, dtype=bool)
    assert np.array_equal(bits(rho.real)[off], bits(rho.real.T)[off])
    assert np.array_equal(bits(rho.imag)[off], bits(-rho.imag.T)[off])
    assert np.all(bits(np.diagonal(rho).imag) == 0)


def check_rdms(s, n, rng):
    perm0, _ = s.layout()
    raw0 = s.state_native().copy()
    a = s.state()
    for qs in qubit_sets(n, perm0, rng):
        got = s.reduced_density_matrix(qs)
        check_structure(got, len(qs))
        again = s.reduced_density_matrix(qs)
        assert np.array_equal(bits(got), bits(again)), qs
        err = float(np.max(np.abs(got - rho_np(a, qs))))
        assert err <= RTOL, (n, qs, err)
        if len(qs) == n:
            order = np.zeros(1 << n, dtype=np.int64)       # psi psi^H in the qubits[] order
            for j in range(1 << n):
                order[sum(((j >> i) & 1) << qs[i] for i in range(n))] = j
            v = np.empty_like(a)
            v[order] = a
            assert np.max(np.abs(got - np.outer(v, v.conj()))) <= RTOL
    assert np.array_equal(s.state_native(), raw0) and np.array_equal(s.layout()[0], perm0)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [q.MODE_TILED, q.MODE_SWEEP])
@pytest.mark.parametrize("prec", [q.F32, q.F64])
@pytest.mark.parametrize("n", [1, 2, 5, 11, 12, 16, 20, 24])
def test_rdm_values(n, prec, mode):
    with run(n, circuit_for(n, 500 + n), prec, mode) as s:
        check_rdms(s, n, np.random.default_rng(n))


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_rdm_on_permuted_layouts(prec):
    permuted = 0
    for n in (13, 18):
        with run(n, circuits.random_layered(n, depth=8, seed=n), prec) as s:
            perm, _ = s.layout()
            permuted += any(perm[qb] != qb for qb in range(n))
            check_rdms(s, n, np.random.default_rng(3 * n))
    assert permuted, "no circuit left a permuted qubit layout"


def pauli(c):
    return {"I": np.eye(2), "X": np.array([[0, 1], [1, 0]]), "Y": np.array([[0, -1j], [1j, 0]]),
            "Z": np.diag([1.0, -1.0])}[c].astype(np.complex128)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_rdm_structure(prec):
    n = 14
    with run(n, circuits.random_layered(n, depth=6, seed=41), prec) as s:
        norm = s.norm_argmax()[0]
        for qs in ([5], [0, 13], [3, 0], [9, 2, 7], [1, 4, 6, 8, 10]):
            k = len(qs)
            rho = s.reduced_density_matrix(qs)
            check_structure(rho, k)
            assert abs(np.trace(rho).real - norm) <= RTOL
            assert np.max(np.abs(np.diagonal(rho).real - s.marginal_probabilities(qs))) <= RTOL
            if k <= 3:   # Tr(rho P) = <P> for every Pauli string on the chosen qubits
                texts, mats = [], []
                for code in range(4 ** k):
                    letters = ["IXYZ"[(code >> (2 * i)) & 3] for i in range(k)]
                    texts.append(" ".join(f"{c}{qs[i]}" for i, c in enumerate(letters) if c != "I"))
                    m = np.ones((1, 1), dtype=np.complex128)
                    for c in reversed(letters):             # bit i of the index = qubits[i]: qubits[k-1] is the top
                        m = np.kron(m, pauli(c))
                    mats.append(m)
                ev = s.expectation(texts)
                for t, m, e in zip(texts, mats, ev):
                    assert abs(np.trace(rho @ m) - e) <= TOL[prec], (qs, t)
        r03, r30 = s.reduced_density_matrix([0, 3]), s.reduced_density_matrix([3, 0])
        swap = [0, 2, 1, 3]
        assert np.array_equal(r30, r03[np.ix_(swap, swap)])


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_rdm_known_states(prec):
    n = 12
    tol = TOL[prec]
    with run(n, [("x", [1], []), ("x", [6], []), ("x", [11], [])], prec) as s:   # basis state
        for qs in ([1], [0, 6], [11, 3, 1], list(range(12))):
            rho = s.reduced_density_matrix(qs)
            want = np.zeros_like(rho)
            o = sum(1 << i for i, qb in enumerate(qs) if qb in (1, 6, 11))
            want[o, o] = 1.0
            assert np.array_equal(rho, want), qs
    rng = np.random.default_rng(5)
    product = [("ry", [qb], [float(rng.uniform(0, 3))]) for qb in range(n)] + [("rz", [qb], [float(rng.uniform(0, 3))]) for qb in range(n)]
    with run(n, product, prec) as s:
        for qs in ([0], [2, 7], [11, 5, 3, 9]):
            rho = s.reduced_density_matrix(qs)
            assert abs(np.trace(rho @ rho).real - 1.0) <= 10 * tol
            assert abs(s.entanglement_entropy(qs)) <= (1e-4 if prec == q.F32 else 1e-9)
    ghz = [("h", [0], [])] + [("cx", [0, k], []) for k in range(1, n)]
    with run(n, ghz, prec) as s:
        for qs in ([0], [4, 9], [3, 1, 10, 7]):
            rho = s.reduced_density_matrix(qs)
            want = np.zeros_like(rho)
            want[0, 0] = want[-1, -1] = 0.5
            assert np.max(np.abs(rho - want)) <= tol
            assert abs(s.entanglement_entropy(qs) - 1.0) <= 1e-5
    bell = []
    for p in range(0, n, 2):
        bell += [("h", [p], []), ("cx", [p, p + 1], [])]
    with run(n, bell, prec) as s:
        for p in (0, 4, 10):
            assert np.max(np.abs(s.reduced_density_matrix([p + 1]) - np.eye(2) / 2)) <= tol
            assert abs(s.entanglement_entropy([p]) - 1.0) <= 1e-5
            assert abs(s.entanglement_entropy([p, p + 1])) <= 1e-5
            assert abs(s.entanglement_entropy([p, p + 1, (p + 3) % n]) - 1.0) <= 1e-5
            assert abs(s.entanglement_entropy([p], base=np.e) - np.log(2)) <= 1e-5
    for m in (5, 16):   # uploaded unnormalised states: the trace is the squared norm
        a = rng.normal(size=1 << m) + 1j * rng.normal(size=1 << m)
        with q.Simulator(m, precision=prec, device=0) as s:
            s.set_state(3.0 * a)
            stored = s.state()
            for qs in ([0], [m - 1, 2], [4, 1, 3]):
                rho = s.reduced_density_matrix(qs)
                norm2 = float(np.sum(np.abs(stored.astype(np.clongdouble)) ** 2))
                assert abs(np.trace(rho).real - norm2) <= RTOL * norm2
                assert np.max(np.abs(rho - rho_np(stored, qs))) <= RTOL * norm2


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_rdm_after_collapse_and_reset(prec):
    n = 15
    rng = np.random.default_rng(8)
    with run(n, circuits.random_layered(n, depth=6, seed=81), prec) as s:
        for qs in ([3], [0, 9, 14], [1, 2, 5, 7]):
            table = s.marginal_probabilities(qs)
            o = int(rng.choice(np.flatnonzero(table > 1e-6)))
            s.collapse(qs, o)
            rho = s.reduced_density_matrix(qs)
            want = np.zeros_like(rho)
            want[o, o] = 1.0
            assert np.all(rho[want == 0] == 0.0)
            assert np.max(np.abs(rho - rho_np(s.state(), qs))) <= RTOL
            assert abs(rho[o, o].real - 1.0) <= TOL[prec]
        for qs in ([4], [13, 6, 0]):
            s.reset_qubits(qs, 0.4)
            rho = s.reduced_density_matrix(qs)
            assert np.all(rho.ravel()[1:] == 0.0)
            assert abs(rho[0, 0].real - 1.0) <= TOL[prec]


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_rdm_graph_replay(prec):
    n = 14
    with q.Simulator(n, precision=prec, device=0, use_graph=True) as s:
        plan = s.plan(q.gates_from_circuit(circuits.random_layered(n, depth=5, seed=9)))
        s.execute(plan)
        first = [s.reduced_density_matrix(qs) for qs in ([2, 11], [0, 1, 2, 3, 4, 5, 6])]
        s.reset()
        s.execute(plan)
        second = [s.reduced_density_matrix(qs) for qs in ([2, 11], [0, 1, 2, 3, 4, 5, 6])]
        for x, y in zip(first, second):
            assert np.array_equal(bits(x), bits(y))
        plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_rdm_errors_leave_the_state_unchanged(prec):
    n = 14
    with run(n, circuits.random_layered(n, depth=2, seed=3), prec) as s:
        raw = s.state_native().copy()
        out = np.zeros(2 << 24)
        good = (C.c_int * 2)(0, 1)

        def refused(rc):
            assert rc == -1, lib.qsb_last_error()
            assert np.array_equal(s.state_native(), raw)
        for bad in ([1, 1], [n], [-1], [], list(range(13)), [0, 5, 0]):
            qs = (C.c_int * max(len(bad), 1))(*bad)
            refused(lib.qsb_reduced_density_matrix(s._h, qs, len(bad), out.ctypes.data))
        refused(lib.qsb_reduced_density_matrix(None, good, 2, out.ctypes.data))
        refused(lib.qsb_reduced_density_matrix(s._h, None, 2, out.ctypes.data))
        refused(lib.qsb_reduced_density_matrix(s._h, good, 2, None))
        with pytest.raises(q.QsbError) as e:
            s.reduced_density_matrix([3, 3])
        assert e.value.code == -1
    with q.Simulator(3, precision=prec, device=0) as s:   # k above n
        with pytest.raises(q.QsbError) as e:
            s.reduced_density_matrix([0, 1, 2, 0])
        assert e.value.code == -1
        assert s.reduced_density_matrix([0, 1, 2]).shape == (8, 8)


@pytest.mark.gpu
def test_cli_rdm_matches_python(tmp_path):
    exe = os.path.join(helpers.ROOT, "gpu_quantum_simulator_b200", "bin", "qsim")
    n = 14
    circ = circuits.random_layered(n, depth=4, seed=19)
    path = tmp_path / "c.qasm"
    path.write_text(circuits.to_qasm(circ, n))
    sets = [[0, 3], [13], [7, 2, 11]]
    args = [exe, str(path), "--marginal", "0 3"]
    for qs in sets:
        args += ["--rdm", " ".join(map(str, qs))]
    r = subprocess.run(args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.splitlines()
    assert lines[1].startswith("MARGINAL 0 3:")          # the RDM lines follow the MARGINAL lines
    rdm = lines[2:]
    assert [ln.split(":")[0] for ln in rdm] == ["RDM " + " ".join(map(str, qs)) for qs in sets]
    with run(n, circ, q.F32) as s:
        for ln, qs in zip(rdm, sets):
            v = np.array([float(x) for x in ln.split(":")[1].split()])
            assert v.size == 2 << (2 * len(qs))
            got = v.view(np.complex128).reshape(1 << len(qs), 1 << len(qs))
            assert np.max(np.abs(got - s.reduced_density_matrix(qs))) <= 1e-12
    plain = subprocess.run([exe, str(path)], capture_output=True, text=True, timeout=300)
    assert plain.returncode == 0 and len(plain.stdout.splitlines()) == 1 and "RDM" not in plain.stdout
    marg = subprocess.run([exe, str(path), "--marginal", "0 3"], capture_output=True, text=True, timeout=300)
    assert marg.stdout.splitlines()[1:] == lines[1:2]
    bad = subprocess.run([exe, str(path), "--rdm", "0 x"], capture_output=True, text=True, timeout=300)
    assert bad.returncode == 1 and "--rdm" in bad.stdout


@pytest.mark.gpu
def test_sharded_rdm():
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs >= 2 GPUs")
    script = os.path.join(os.path.dirname(__file__), "dist_rdm_worker.py")
    for world in [w for w in (2, 4, 8) if w <= ngpu]:
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                            "--master-addr", "127.0.0.1", "--master-port", "29571", script],
                           capture_output=True, text=True, timeout=1800)
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
        assert "sharded_rdm_ok" in r.stdout


@pytest.mark.gpu
@pytest.mark.slow
def test_30q_f32_against_f64_and_24q_entropy():
    n = 30
    circ = circuits.random_layered(n, depth=20)
    rng = np.random.default_rng(30)
    sets = [rng.permutation(n)[:4].tolist(), rng.permutation(n)[:12].tolist()]
    vals = []
    for prec in (q.F32, q.F64):
        with run(n, circ, prec) as s:
            vals.append([s.reduced_density_matrix(qs) for qs in sets])
    for a, b in zip(*vals):
        assert np.max(np.abs(a - b)) <= 1e-5
    n = 24
    with run(n, circuits.random_layered(n, depth=12, seed=24), q.F64) as s:
        half = list(range(0, n, 2))
        a = s.state()
        w = np.linalg.eigvalsh(rho_np(a, half))
        w = w[w > 0]
        want = float(-np.sum(w * np.log2(w)))
        assert abs(s.entanglement_entropy(half) - want) <= 1e-9
