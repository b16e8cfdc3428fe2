"""Energy gradients with respect to Pauli-rotation angles on the device (qsb_pauli_rotation_gradient) against the exact
parameter-shift rule in numpy, g_k = [E(theta + pi/2 e_k) - E(theta - pi/2 e_k)] / 2, against parameter shift through
the existing device calls, and against the bit-exact contracts of the header: the state left in the handle is that of
qsb_apply_pauli_rotations, the energy is the term-ordered sum of qsb_expectation_pauli values."""
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers
import gpu_quantum_simulator_b200 as q
from gpu_quantum_simulator_b200 import circuits
from test_gpu_expectation import pauli_apply, random_terms
from test_gpu_pauli_rotation import LOW_BITS, permuted, rotate_np

pytestmark = pytest.mark.gpu

F32, F64 = q.F32, q.F64
PRECS = pytest.mark.parametrize("prec", [F32, F64], ids=["f32", "f64"])
REL = {F32: 2e-4, F64: 1e-10}          # times sum |c|


def energy_np(a, obs, coef, n):
    hx, hz = q.pauli_masks(obs, n)
    return sum(c * np.vdot(a, pauli_apply(a, int(x), int(z))).real for x, z, c in zip(hx.tolist(), hz.tolist(), coef))


def shift_grad_np(a0, rots, th, obs, coef, n):
    """The exact parameter-shift rule, one pair of numpy runs per angle."""
    th = np.asarray(th, dtype=np.float64)
    g = np.empty(th.size)
    for k in range(th.size):
        e = []
        for sh in (0.5 * np.pi, -0.5 * np.pi):
            t = th.copy()
            t[k] += sh
            e.append(energy_np(rotate_np(a0, rots, t, n), obs, coef, n))
        g[k] = 0.5 * (e[0] - e[1])
    return g


def adjoint_grad_np(a0, rots, th, obs, coef, n):
    """The adjoint method in numpy (complex128), for lists too long for parameter shift; checked against it below."""
    x, z = q.pauli_masks(rots, n)
    hx, hz = q.pauli_masks(obs, n)
    psi = rotate_np(a0, rots, th, n)
    lam = sum(c * pauli_apply(psi, int(xx), int(zz)) for xx, zz, c in zip(hx.tolist(), hz.tolist(), coef))
    phi = psi.copy()
    g = np.empty(len(th))
    for k in range(len(th) - 1, -1, -1):
        xx, zz, t = int(x[k]), int(z[k]), th[k]
        pphi = pauli_apply(phi, xx, zz)
        g[k] = np.vdot(lam, pphi).imag
        phi = np.cos(t / 2) * phi + 1j * np.sin(t / 2) * pphi
        lam = np.cos(t / 2) * lam + 1j * np.sin(t / 2) * pauli_apply(lam, xx, zz)
    return energy_np(psi, obs, coef, n), g, psi


def angles(count, rng):
    """Random angles with 0, pi and 2 pi among them."""
    t = rng.uniform(-np.pi, np.pi, size=count)
    t[::5] = 0.0
    t[1::7] = np.pi
    t[3::11] = 2 * np.pi
    return t


def observable(n, count, seed):
    obs = random_terms(n, count, seed=seed)
    coef = np.random.default_rng(seed).normal(size=count)
    return obs, coef


def check_numpy(s, rots, th, obs, coef, prec, ref=shift_grad_np):
    """Gradient call against numpy from the state as it was; the layout must not move and psi is left."""
    n = s.num_qubits
    a0, perm0 = s.state(), s.layout()[0]
    e, g = s.rotation_gradient(rots, th, obs, coef)
    want = ref(a0, rots, th, obs, coef, n)
    want = want[1] if isinstance(want, tuple) else want
    tol = REL[prec] * np.sum(np.abs(coef))
    err = float(np.max(np.abs(g - want))) if len(rots) else 0.0
    assert err <= tol, (n, err, tol)
    psi = rotate_np(a0, rots, th, n)
    assert abs(e - energy_np(psi, obs, coef, n)) <= tol
    assert np.array_equal(s.layout()[0], perm0)
    return g


SIZES = [1, 2, 5, 11, 12, 13]


@pytest.mark.parametrize("mode", [q.MODE_TILED, q.MODE_SWEEP], ids=["tiled", "sweep"])
@pytest.mark.parametrize("n", SIZES)
@PRECS
def test_against_parameter_shift(n, mode, prec):
    rng = np.random.default_rng(n + 7)
    rots = random_terms(n, 30, seed=n)
    obs, coef = observable(n, 12, seed=n + 1)
    with permuted(n, prec, mode=mode) as s:
        check_numpy(s, rots, angles(len(rots), rng), obs, coef, prec)
        a = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)     # unnormalised upload
        s.set_state(2.5 * a / np.linalg.norm(a))
        check_numpy(s, rots, angles(len(rots), rng), obs, 3.0 * coef, prec)


@pytest.mark.parametrize("prec,low_bits", [(p, lb) for p in (F32, F64) for lb in LOW_BITS[p]])
def test_low_bits(prec, low_bits):
    n = 13
    rng = np.random.default_rng(low_bits)
    rots = random_terms(n, 40, seed=low_bits + 3) + [f"X{k}" for k in range(n)]
    obs, coef = observable(n, 10, seed=low_bits)
    with permuted(n, prec, low_bits) as s:
        check_numpy(s, rots, angles(len(rots), rng), obs, coef, prec)


def test_numpy_adjoint_matches_parameter_shift():
    n = 6
    rng = np.random.default_rng(1)
    rots = random_terms(n, 25, seed=2)
    th = angles(25, rng)
    obs, coef = observable(n, 8, seed=3)
    a0 = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)
    assert np.max(np.abs(adjoint_grad_np(a0, rots, th, obs, coef, n)[1] - shift_grad_np(a0, rots, th, obs, coef, n))) <= 1e-12


@pytest.mark.parametrize("n", [17, 21])
@PRECS
def test_against_device_parameter_shift(n, prec):
    """Parameter shift through apply_pauli_rotations + expectation: an independent device path."""
    rng = np.random.default_rng(n)
    rots = random_terms(n, 16, seed=n + 5)
    th = angles(16, rng)
    obs, coef = observable(n, 20, seed=n + 6)
    circ = q.gates_from_circuit(circuits.random_layered(n, depth=3, seed=n))
    with q.Simulator(n, precision=prec, device=0) as s, q.Simulator(n, precision=prec, device=0) as r:
        s.apply(circ)
        a0 = s.state_native().copy()
        _, g = s.rotation_gradient(rots, th, obs, coef)
        want = np.empty(len(rots))
        for k in range(len(rots)):
            e = []
            for sh in (0.5 * np.pi, -0.5 * np.pi):
                r.set_state(s_native_to_complex(a0))
                t = th.copy()
                t[k] += sh
                r.apply_pauli_rotations(rots, t)
                e.append(float(np.dot(coef, r.expectation(obs))))
            want[k] = 0.5 * (e[0] - e[1])
    assert np.max(np.abs(g - want)) <= REL[prec] * np.sum(np.abs(coef))


def s_native_to_complex(raw):
    return raw.astype(np.float64).view(np.complex128)


@PRECS
def test_bit_exact_contracts(prec):
    n = 16
    rng = np.random.default_rng(4)
    rots = random_terms(n, 120, seed=5)
    th = angles(120, rng)
    obs, coef = observable(n, 30, seed=6)
    circ = q.gates_from_circuit(circuits.random_layered(n, depth=4, seed=2))
    with q.Simulator(n, precision=prec, device=0) as s, q.Simulator(n, precision=prec, device=0) as twin:
        s.apply(circ)
        twin.apply(circ)
        perm0 = s.layout()[0]
        raw0 = s.state_native().copy()
        e, g = s.rotation_gradient(rots, th, obs, coef)
        twin.apply_pauli_rotations(rots, th)
        assert np.array_equal(s.state_native(), twin.state_native())     # the state of apply_pauli_rotations
        assert np.array_equal(s.layout()[0], perm0)
        v = twin.expectation(obs)
        acc = 0.0
        for c, x in zip(coef.tolist(), v.tolist()):
            acc = acc + c * x
        assert e == acc                                                   # the term-ordered sum, bit for bit
        for _ in range(2):                                                # repeated calls: identical bits
            s.set_state(s_native_to_complex(raw0))
            e2, g2 = s.rotation_gradient(rots, th, obs, coef)
            assert e2 == e and np.array_equal(g2.view(np.uint64), g.view(np.uint64))


@PRECS
def test_plans_and_graphs_made_before_the_call(prec):
    n = 18
    circ_list = circuits.random_layered(n, depth=4, seed=8)
    circ = q.gates_from_circuit(circ_list)
    rots = random_terms(n, 60, seed=9)
    th = angles(60, np.random.default_rng(9))
    obs, coef = observable(n, 10, seed=10)
    for use_graph in (False, True):
        with q.Simulator(n, precision=prec, device=0, use_graph=use_graph) as s:
            p = s.plan(circ)
            if use_graph:
                s.execute(p)                                     # captures the graph
                s.reset()
            s.rotation_gradient(rots, th, obs, coef)
            psi = s.state()
            s.execute(p)
            want = helpers.oracle_run_circuit(circ_list, n, state=psi)
            assert np.max(np.abs(s.state() - want)) <= 3 * (1e-5 if prec == F32 else 1e-12), use_graph
            p.close()


@PRECS
def test_grouping_coverage(prec):
    """More than 1024 rotations (several adjoint launches), rotations on tile-outer qubits, X on every qubit, diagonal
    stretches between pairing rotations, and many theta = 0 entries, against the numpy adjoint."""
    n = 16
    rng = np.random.default_rng(12)
    rots = []
    while len(rots) < 1100:
        r = rng.random()
        if r < 0.3:                                              # a diagonal stretch
            for _ in range(int(rng.integers(1, 6))):
                qs = rng.choice(n, int(rng.integers(1, 4)), replace=False)
                rots.append(" ".join(f"Z{k}" for k in qs))
        elif r < 0.5:                                            # tile-outer qubits
            hi = n - 1 - int(rng.integers(3))
            rots.append(f"{'XY'[rng.integers(2)]}{hi} Z{int(rng.integers(hi))}")
        elif r < 0.52:
            rots.append(" ".join(f"X{k}" for k in range(n)))
        else:
            qs = rng.choice(n, int(rng.integers(1, 5)), replace=False)
            rots.append(" ".join(f"{'XYZ'[rng.integers(3)]}{k}" for k in qs))
    th = angles(len(rots), rng)
    th[::3] = 0.0
    obs, coef = observable(n, 25, seed=13)
    assert q.rotation_gradient_dry_run(n, rots, obs, prec)["adjoint_sweeps"] > 2
    with permuted(n, prec) as s:
        g = check_numpy(s, rots, th, obs, coef, prec, ref=adjoint_grad_np)
    assert np.count_nonzero(np.abs(g[th == 0.0]) > 1e-3) > 10      # zero angles get their (non-zero) gradients
    # rotations inside one tile: a full 1024-rotation adjoint launch and a second one
    rots = [f"X0 Z{int(rng.integers(1, n))}" if k % 3 == 0 else f"Z{int(rng.integers(n))} Z{int(rng.integers(n))}" for k in range(1100)]
    rots = [r if r.split()[0] != r.split()[1] else "Z3" for r in rots]
    assert q.rotation_gradient_dry_run(n, rots, obs, prec)["adjoint_sweeps"] == 2
    with permuted(n, prec) as s:
        check_numpy(s, rots, angles(len(rots), rng), obs, coef, prec, ref=adjoint_grad_np)


def test_qaoa_from_zero_angles():
    """QAOA MaxCut layers on a ring from theta = 0: every angle gets its gradient."""
    n = 12
    ring = [f"Z{k} Z{(k + 1) % n}" for k in range(n)]
    layer = ring + [f"X{k}" for k in range(n)]
    rots = layer * 2
    th = np.zeros(len(rots))
    th[:n] = 0.3                                                # the first cost layer on, the rest at 0
    with q.Simulator(n, precision=F64, device=0) as s:
        s.apply(q.gates_from_circuit([("h", [k], []) for k in range(n)]))
        check_numpy(s, rots, th, ring, np.ones(n), F64)


@PRECS
def test_refused_arguments_leave_the_state(prec):
    n = 12
    with permuted(n, prec) as s:
        raw0 = s.state_native().copy()
        x = np.array([1], dtype=np.uint64)
        z = np.array([2], dtype=np.uint64)
        big = np.array([1 << 12], dtype=np.uint64)
        t = np.array([0.5])
        c = np.array([1.0])
        e = q.simulator.C.c_double()
        g = np.empty(1)
        f = q.lib.qsb_pauli_rotation_gradient
        ok = (s._h, x.ctypes.data, z.ctypes.data, t.ctypes.data, 1, x.ctypes.data, z.ctypes.data, c.ctypes.data, 1,
              q.simulator.C.byref(e), g.ctypes.data)
        bad = [(0, None), (1, None), (2, None), (3, None), (5, None), (6, None), (7, None), (8, 0), (9, None), (10, None),
               (1, big.ctypes.data), (6, big.ctypes.data)]
        for pos, val in bad:
            args = list(ok)
            args[pos] = val
            assert f(*args) == -1, pos
        for arr in (t, c):
            for v in (np.nan, np.inf, -np.inf):
                old = arr[0]
                arr[0] = v
                assert f(*ok) == -1
                assert "non-finite" in q.lib.qsb_last_error().decode()
                arr[0] = old
        assert np.array_equal(s.state_native(), raw0)
        args = list(ok)
        args[4], args[10] = 0, None                           # nrot = 0: the energy only, the state unchanged
        assert f(*args) == 0
        assert np.array_equal(s.state_native(), raw0)
        assert abs(e.value - s.expectation("X0 Z1")) == 0.0
        with pytest.raises(ValueError):
            s.rotation_gradient(["X0", "Z1"], [0.5], ["Z0"], [1.0])
        with pytest.raises(ValueError):
            s.rotation_gradient(["X0"], [0.5], ["Z0", "Z1"], [1.0])


def test_cli_gradient_matches_python(tmp_path):
    exe = os.path.join(helpers.ROOT, "gpu_quantum_simulator_b200", "bin", "qsim")
    n = 14
    circ = circuits.random_layered(n, depth=4, seed=9)
    path = tmp_path / "c.qasm"
    path.write_text(circuits.to_qasm(circ, n))
    rots = [("X0 Z3", 0.25), ("Y13", -1.5), ("Z2 Z5", 0.0), ("X7 X8", 2.0)]
    terms = [("Z0 Z1", 0.5), ("X13", -1.25), ("Y2 Z5", 0.75)]
    args = [exe, str(path)]
    for p, t in rots:
        args += ["--pauli-rot", p, repr(t)]
    for p, c in terms:
        args += ["--gradient", p, repr(c)]
    r = subprocess.run(args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.splitlines()
    assert lines[1].startswith("ENERGY ") and lines[2].startswith("GRADIENT ")
    with q.Simulator(n, precision=F32, device=0) as s:
        s.apply(q.gates_from_circuit(circ))
        e, g = s.rotation_gradient([p for p, _ in rots], [t for _, t in rots], [p for p, _ in terms], [c for _, c in terms])
    assert float(lines[1].split()[1]) == e
    assert np.array_equal(np.array([float(v) for v in lines[2].split()[1:]]), g)
    bad = subprocess.run([exe, str(path), "--gradient", "X0", "abc"], capture_output=True, text=True, timeout=300)
    assert bad.returncode == 1 and "expected a coefficient" in bad.stdout


def test_sharded_rotation_gradient():
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs >= 2 GPUs")
    for world in (2, 4, 8):
        if world > ngpu:
            break
        script = os.path.join(os.path.dirname(__file__), "dist_rotation_gradient_worker.py")
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                            "--master-addr", "127.0.0.1", "--master-port", "29583", script],
                           capture_output=True, text=True, timeout=1200)
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
        assert "sharded_rotation_gradient_ok" in r.stdout
