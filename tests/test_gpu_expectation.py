"""Pauli-string expectation values on the device (qsb_expectation_pauli) against numpy on the same amplitudes.

The reference is the formula of include/qsim_b200.h, (P a)_j = i^{popc(x&z)} (-1)^{popc((j^x)&z)} a_{j^x}, applied
to s.state(); the formula itself is pinned against dense Kronecker products for n <= 4."""
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers
import gpu_quantum_simulator_b200 as q
from gpu_quantum_simulator_b200 import circuits

TOL = {q.F32: 1e-6, q.F64: 1e-12}


def pauli_apply(a, x, z):
    """(P a) by the header's index formula."""
    j = np.arange(a.size, dtype=np.uint64)
    jx = j ^ np.uint64(x)
    par = np.bitwise_count(jx & np.uint64(z)) & 1
    y = bin(x & z).count("1") % 4
    return (1j ** y) * (1.0 - 2.0 * par.astype(np.float64)) * a[jx]


def expect_np(a, terms, n):
    x, z = q.pauli_masks(terms, n)
    return np.array([np.vdot(a, pauli_apply(a, int(xx), int(zz))).real for xx, zz in zip(x, z)])


def test_formula_matches_dense_kron():
    mats = {"I": np.eye(2), "X": np.array([[0, 1], [1, 0]]), "Y": np.array([[0, -1j], [1j, 0]]), "Z": np.diag([1, -1])}
    rng = np.random.default_rng(0)
    for n in range(1, 5):
        for _ in range(40):
            letters = [("IXYZ"[rng.integers(4)]) for _ in range(n)]
            M = np.array([[1.0]])
            for k in range(n):                     # qubit k <-> bit k: qubit n-1 is the leftmost factor
                M = np.kron(mats[letters[k]], M)
            x = sum(1 << k for k in range(n) if letters[k] in "XY")
            z = sum(1 << k for k in range(n) if letters[k] in "YZ")
            a = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)
            assert np.allclose(pauli_apply(a, x, z), M @ a, atol=1e-14)


def run(n, circ, prec, mode=q.MODE_TILED):
    s = q.Simulator(n, precision=prec, mode=mode, device=0)
    s.apply(q.gates_from_circuit(circ))
    return s


def random_terms(n, count, seed):
    """Strings with X/Y on bit 0, on the top qubit, on qubits far apart, weight-n strings, then random weight <= 4."""
    rng = np.random.default_rng(seed)
    out = ["", "X0", "Y0", "Z0", f"X{n - 1}", f"Y{n - 1}",
           " ".join(f"X{k}" for k in range(n)), " ".join(f"{'XYZ'[k % 3]}{k}" for k in range(n)),
           " ".join(f"{'YZ'[k % 2]}{k}" for k in range(n))]
    if n > 1:
        out += [f"X0 Y{n - 1}", f"Z0 Z{n - 1}"]
    while len(out) < count:
        w = int(rng.integers(1, min(n, 4) + 1)) if rng.random() > 0.05 else n
        qs = rng.choice(n, w, replace=False)
        out.append(" ".join(f"{'XYZ'[rng.integers(3)]}{k}" for k in qs))
    return out[:count]


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_analytic_states(prec):
    tol = 10 * TOL[prec]
    n = 13
    with run(n, [("h", [k], []) for k in range(n)], prec) as s:
        v = s.expectation([f"X{k}" for k in range(n)] + [" ".join(f"X{k}" for k in range(n)), "Z0", "", "Y3"])
        assert np.all(np.abs(v[:n + 1] - 1) < tol) and abs(v[n + 1]) < tol and abs(v[n + 2] - 1) < tol and abs(v[n + 3]) < tol
    with run(n, [("h", [0], []), ("s", [0], [])], prec) as s:
        assert abs(s.expectation("Y0") - 1.0) < tol
        assert abs(s.expectation("X0")) < tol and abs(s.expectation("Z5") - 1.0) < tol
    for n in (3, 12, 14):
        ghz = [("h", [0], [])] + [("cx", [0, k], []) for k in range(1, n)]
        with run(n, ghz, prec) as s:
            v = s.expectation(["Z0 Z1", f"Z0 Z{n - 1}", f"Z{n // 2} Z{n - 1}", " ".join(f"X{k}" for k in range(n)),
                               "Y0 Y1 " + " ".join(f"X{k}" for k in range(2, n)), "", "Z0", "X0"])
            assert np.all(np.abs(v[:4] - 1) < tol), v
            assert abs(v[4] + 1) < tol and abs(v[5] - 1) < tol and abs(v[6]) < tol and abs(v[7]) < tol, v
            norm = s.norm_argmax()[0]
            assert abs(v[5] - norm) < tol


SIZES = [1, 2, 5, 11, 12, 13, 17, 21, 26]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [q.MODE_TILED, q.MODE_SWEEP])
@pytest.mark.parametrize("n", SIZES)
def test_random_layered_matches_numpy(n, mode):
    """Both precisions after the same circuit: each against numpy on its own amplitudes, f32 against f64; repeated
    calls identical to the bit; state and qubit layout untouched by the call."""
    count = 300 if n <= 21 else 40
    terms = random_terms(n, count, seed=n)
    circ = circuits.random_layered(n, depth=6 if n > 5 else 3, seed=100 + n)
    vals = {}
    for prec in (q.F64, q.F32):
        with run(n, circ, prec, mode) as s:
            perm0, _ = s.layout()
            raw0 = s.state_native().copy()
            got = s.expectation(terms)
            again = s.expectation(terms)
            assert np.array_equal(got.view(np.uint64), again.view(np.uint64))
            assert np.array_equal(s.state_native(), raw0) and np.array_equal(s.layout()[0], perm0)
            want = expect_np(s.state(), terms, n)
            err = np.max(np.abs(got - want))
            assert err <= TOL[prec], (prec, err, terms[int(np.argmax(np.abs(got - want)))])
            vals[prec] = got
    assert np.max(np.abs(vals[q.F32] - vals[q.F64])) <= 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_set_state_and_load_state(prec, tmp_path):
    for n in (5, 16):
        rng = np.random.default_rng(n)
        a = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)
        a /= np.linalg.norm(a)
        terms = random_terms(n, 300, seed=7 * n)
        with q.Simulator(n, precision=prec, device=0) as s:
            s.apply(q.gates_from_circuit(circuits.random_layered(n, depth=2, seed=1)))   # a permuted layout
            s.set_state(a)
            got = s.expectation(terms)
            assert np.max(np.abs(got - expect_np(s.state(), terms, n))) <= TOL[prec]
            path = str(tmp_path / f"shard_{n}_{prec}.bin")
            s.save_state(path)
        with q.Simulator(n, precision=prec, device=0) as s:
            s.load_state(path)
            assert np.array_equal(s.expectation(terms), got)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_alone_and_in_a_large_batch(prec):
    n = 18
    batch = random_terms(n, 1000, seed=5)
    with run(n, circuits.random_layered(n, depth=5, seed=2), prec) as s:
        together = s.expectation(batch)
        for k in (0, 1, 8, 9, 500, 999):
            assert abs(s.expectation(batch[k]) - together[k]) <= TOL[prec]
        assert s.expectation([]).size == 0


@pytest.mark.gpu
def test_cli_expect_matches_python(tmp_path):
    exe = os.path.join(helpers.ROOT, "gpu_quantum_simulator_b200", "bin", "qsim")
    n = 14
    circ = circuits.random_layered(n, depth=4, seed=9)
    path = tmp_path / "c.qasm"
    path.write_text(circuits.to_qasm(circ, n))
    texts = ["Z0 Z1", "X3 Y13", "", "Y0"]
    args = [exe, str(path)]
    for t in texts:
        args += ["--expect", t]
    r = subprocess.run(args + ["--profile"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.splitlines()
    assert lines[1].startswith("{")                       # the --profile line comes first
    exp = lines[2:2 + len(texts)]
    assert [ln.rsplit(":", 1)[0] for ln in exp] == [f"EXPECTATION {t}" for t in texts]
    with run(n, circ, q.F32) as s:
        want = s.expectation(texts)
    got = np.array([float(ln.rsplit(":", 1)[1]) for ln in exp])
    assert np.max(np.abs(got - want)) <= 1e-12
    plain = subprocess.run([exe, str(path)], capture_output=True, text=True, timeout=300)
    assert plain.returncode == 0 and len(plain.stdout.splitlines()) == 1 and "EXPECTATION" not in plain.stdout


@pytest.mark.gpu
def test_sharded_expectation():
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 8 if ngpu >= 8 else 4 if ngpu >= 4 else 2
    script = os.path.join(os.path.dirname(__file__), "dist_expectation_worker.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", "29561", script],
                       capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "sharded_expectation_ok" in r.stdout


@pytest.mark.gpu
@pytest.mark.slow
def test_30q_headline_circuit_f32_against_f64():
    n = 30
    circ = circuits.random_layered(n, depth=20)
    terms = [f"X{k}" for k in range(n)] + [f"Z{k} Z{k + 1}" for k in range(n - 1)] + [f"Y{k} Y{k + 1}" for k in range(0, n - 1, 7)]
    vals = []
    for prec in (q.F32, q.F64):
        with run(n, circ, prec) as s:
            vals.append(s.expectation(terms))
    assert np.max(np.abs(vals[0] - vals[1])) <= 1e-4
