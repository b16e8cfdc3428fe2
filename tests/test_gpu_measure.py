"""Marginal probabilities and projective measurement on the device (qsb_marginal_probabilities, qsb_collapse,
qsb_measure_qubits, qsb_reset_qubits) against numpy on s.state() of the same handle, with np.longdouble sums of |a|^2.

Bit i of a bin index or an outcome is the value of qubits[i]."""
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers
import gpu_quantum_simulator_b200 as q
from gpu_quantum_simulator_b200 import circuits

TOL = {q.F32: 1e-6, q.F64: 1e-12}     # state-level tolerances (norm, projected amplitudes)
MTOL = 1e-12                          # marginals: the same fp64 numbers summed in another order


def probs_ld(a):
    """|a|^2 in long double, shaped (2,) * n: axis j holds qubit n - 1 - j."""
    n = a.size.bit_length() - 1
    re, im = a.real.astype(np.longdouble), a.imag.astype(np.longdouble)
    return (re * re + im * im).reshape((2,) * n) if n else re * re + im * im


def marginal_np(p, qubits):
    """Marginal table of `qubits` from probs_ld(): bin b has bit i = value of qubits[i]."""
    n = p.ndim
    keep = [n - 1 - qb for qb in qubits]
    m = p.sum(axis=tuple(ax for ax in range(n) if ax not in keep))
    rest = sorted(keep)
    order = [rest.index(keep[i]) for i in reversed(range(len(qubits)))]   # axis 0 = the top bit of b
    return np.asarray(m.transpose(order).reshape(-1), dtype=np.float64)


def bins_of(n, qubits):
    """bin index of every amplitude index"""
    idx = np.arange(1 << n, dtype=np.uint64)
    b = np.zeros(1 << n, dtype=np.uint64)
    for i, qb in enumerate(qubits):
        b |= ((idx >> np.uint64(qb)) & np.uint64(1)) << np.uint64(i)
    return b


def project_np(a, qubits, outcome):
    keep = bins_of(a.size.bit_length() - 1, qubits) == np.uint64(outcome)
    out = np.where(keep, a, 0)
    p = float(np.sum(np.abs(a[keep].astype(np.clongdouble)) ** 2))
    return out / np.sqrt(p), keep


def rule(table, r):
    """measure()'s search on a table (quantum_simulator.c:279): first b with C_b != 0 and C_b >= r * T, with C the
    inclusive serial fp64 prefix sum and T its last value."""
    c, cs = 0.0, []
    for v in table:
        c += float(v)
        cs.append(c)
    t = r * cs[-1]
    for b, cb in enumerate(cs):
        if cb != 0.0 and cb >= t:
            return b
    raise AssertionError("no bin reached")


def run(n, circ, prec, mode=q.MODE_TILED, **kw):
    s = q.Simulator(n, precision=prec, mode=mode, device=0, **kw)
    s.apply(q.gates_from_circuit(circ))
    return s


def circuit_for(n, seed):
    if n in (2, 5, 11, 12):
        return circuits.random_superset(n, 12 * n, seed=seed)
    return circuits.random_layered(n, depth=6 if n > 5 else 3, seed=seed)


def qubit_sets(n, perm, rng):
    """qubit 0, qubit n - 1, the qubits on physical bits 0..3, contiguous, reversed and scattered sets, k = min(n, 20)"""
    sets = [[0], [n - 1]]
    for b in range(4):
        sets += [[qb] for qb in range(n) if perm[qb] == b]
    sets += [list(range(min(n, 4))), list(range(min(n, 4)))[::-1]]
    if n >= 3:
        sets += [sorted(rng.choice(n, min(n, 5), replace=False).tolist()), rng.permutation(n)[:min(n, 7)].tolist()]
    sets.append(rng.permutation(n)[:min(n, 20)].tolist())
    return sets


def check_marginals(s, n, rng):
    """Every qubit set against numpy; repeated calls bit-identical; state and layout untouched."""
    perm0, _ = s.layout()
    raw0 = s.state_native().copy()
    p = probs_ld(s.state())
    for qs in qubit_sets(n, perm0, rng):
        got = s.marginal_probabilities(qs)
        assert got.shape == (1 << len(qs),)
        again = s.marginal_probabilities(qs)
        assert np.array_equal(got.view(np.uint64), again.view(np.uint64)), qs
        err = float(np.max(np.abs(got - marginal_np(p, qs))))
        assert err <= MTOL, (n, qs, err)
    assert np.array_equal(s.state_native(), raw0) and np.array_equal(s.layout()[0], perm0)


SIZES = [1, 2, 5, 11, 12, 16, 20, 24, 26]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [q.MODE_TILED, q.MODE_SWEEP])
@pytest.mark.parametrize("prec", [q.F32, q.F64])
@pytest.mark.parametrize("n", SIZES)
def test_marginal_values(n, prec, mode):
    with run(n, circuit_for(n, 300 + n), prec, mode) as s:
        check_marginals(s, n, np.random.default_rng(n))


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_marginal_on_permuted_layouts_and_uploaded_states(prec):
    permuted = 0
    for n in (13, 16, 20):
        with run(n, circuits.random_layered(n, depth=8, seed=n), prec) as s:
            perm, _ = s.layout()
            permuted += any(perm[qb] != qb for qb in range(n))
            check_marginals(s, n, np.random.default_rng(7 * n))
    assert permuted, "no circuit left a permuted qubit layout"
    for n in (5, 16):
        rng = np.random.default_rng(n)
        a = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)
        a /= np.linalg.norm(a)
        with run(n, circuits.random_layered(n, depth=2, seed=1), prec) as s:
            s.set_state(a)
            check_marginals(s, n, rng)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_consistency_with_probabilities_norm_and_expectation(prec):
    for n in (5, 12, 16, 20):
        with run(n, circuits.random_layered(n, depth=5, seed=40 + n), prec) as s:
            rng = np.random.default_rng(n)
            order = rng.permutation(n).tolist()
            full = s.marginal_probabilities(order)                  # k = n: one amplitude per bin
            probs = s.probabilities()
            assert np.max(np.abs(full - probs[bins_of(n, order).argsort()])) <= 1e-15
            assert np.max(np.abs(s.marginal_probabilities(list(range(n))) - probs)) <= 1e-15
            norm = s.norm_argmax()[0]
            for qs in ([0], [n - 1, 2], order[:4]):
                m = s.marginal_probabilities(qs)
                assert abs(float(np.sum(m)) - norm) <= 1e-12
                k = len(qs)
                # inverse Walsh transform of the 2^k Z strings: p_b = 2^-k sum_s (-1)^popc(b & s) <Z_s>
                texts = [" ".join(f"Z{qs[i]}" for i in range(k) if (sm >> i) & 1) for sm in range(1 << k)]
                z = s.expectation(texts)
                signs = np.array([[(-1.0) ** bin(b & sm).count("1") for sm in range(1 << k)] for b in range(1 << k)])
                assert np.max(np.abs(signs @ z / (1 << k) - m)) <= TOL[prec], (n, qs)


def assert_collapsed(s, before, qs, outcome, p, table, prec, perm0):
    want, keep = project_np(before, qs, outcome)
    got = s.state()
    assert p == table[outcome]                              # bit for bit the table entry
    assert np.all(got[~keep] == 0.0)
    assert np.max(np.abs(got - want)) <= TOL[prec]
    assert abs(s.norm_argmax()[0] - 1.0) <= TOL[prec]
    assert np.array_equal(s.layout()[0], perm0)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [q.F32, q.F64])
@pytest.mark.parametrize("n", [3, 12, 16, 22])
def test_collapse(n, prec):
    rng = np.random.default_rng(n)
    with run(n, circuits.random_layered(n, depth=6, seed=60 + n), prec) as s:
        perm0, _ = s.layout()
        on_low = [qb for qb in range(n) if perm0[qb] in (0, 1, 4, 9)]   # the f32 pack bit, thread and unit bits
        cases = [[0], [n - 1], rng.permutation(n)[:min(n, 4)].tolist()] + ([on_low[:3]] if on_low else [])
        for qs in cases:
            before = s.state()
            table = s.marginal_probabilities(qs)
            outcome = int(rng.choice(np.flatnonzero(table > 1e-6)))
            p = s.collapse(qs, outcome)
            assert_collapsed(s, before, qs, outcome, p, table, prec, perm0)
            # another outcome of the same qubits now has p = 0: refused, state unchanged
            other = (outcome + 1) % (1 << len(qs))
            frozen = s.state_native().copy()
            with pytest.raises(q.QsbError) as e:
                s.collapse(qs, other)
            assert e.value.code == -1 and np.array_equal(s.state_native(), frozen)
            s.set_state(before)                            # back to the state before the collapse


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_measure_rule(prec):
    n = 12
    with run(n, circuits.random_layered(n, depth=5, seed=77), prec) as s:
        a0 = s.state()
        for qs in ([3, 0, 7], [n - 1], [5, 1]):
            table = s.marginal_probabilities(qs)
            c = np.cumsum(table)
            rs = [0.0, np.nextafter(1.0, 0.0), 0.5, 1e-300]
            for b in range(len(c)):
                e = float(c[b] / c[-1])
                rs += [x for x in (e, np.nextafter(e, 0.0), np.nextafter(e, 1.0)) if 0.0 <= x < 1.0]
            for r in rs:
                s.set_state(a0)
                b, p = s.measure_qubits(qs, r)
                assert b == rule(table, r), (qs, r)
                assert p == table[b] and p > 0.0
                assert abs(s.norm_argmax()[0] - 1.0) <= TOL[prec]
            s.set_state(a0)
    for n in (3, 14):
        ghz = [("h", [0], [])] + [("cx", [0, k], []) for k in range(1, n)]
        for r in (0.0, 0.25, 0.4999, 0.5, 0.75, np.nextafter(1.0, 0.0)):
            with run(n, ghz, prec) as s:
                table = s.marginal_probabilities(list(range(n)))
                b, p = s.measure_qubits(list(range(n)), r)
                assert b in (0, (1 << n) - 1) and b == rule(table, r)
                assert p == table[b] and abs(p - 0.5) <= TOL[prec]


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_measure_skips_leading_zero_bins(prec):
    """Tables whose first bins are 0: with r = 0 the rule's C_b != 0 clause must pass over them (bin 0 would have p = 0)."""
    n = 12
    circ = [("x", [3], []), ("h", [5], []), ("x", [9], []), ("x", [10], [])]
    for qs, r, want in (([3], 0.0, 1), ([3, 5], 0.0, 1), ([9, 10, 5], 0.0, 3), ([3, 5], 0.6, 3), ([3, 5], 0.5, None)):
        with run(n, circ, prec) as s:
            table = s.marginal_probabilities(qs)
            assert table[0] == 0.0
            b, p = s.measure_qubits(qs, r)
            assert b == rule(table, r) and (want is None or b == want), (qs, r, b)
            assert p == table[b] and p > 0.0
            assert abs(s.norm_argmax()[0] - 1.0) <= TOL[prec]
    with run(n, circ, prec) as s:
        assert s.reset_qubits([3, 9], 0.0) == 3                 # both read 1 (bin 0 has p = 0), both end in |0>
        b, p = s.measure_qubits([9, 3], 0.0)
        assert b == 0 and abs(p - 1.0) <= TOL[prec]


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_mid_circuit_measurement(prec):
    n = 14
    tol = 10 * TOL[prec]
    circ_a = circuits.random_layered(n, depth=5, seed=11)
    circ_b = circuits.random_layered(n, depth=4, seed=12)
    qs = [2, 9, 0]
    for use_graph in (False, True):
        with q.Simulator(n, precision=prec, device=0, use_graph=use_graph) as s:
            plan_a = s.plan(q.gates_from_circuit(circ_a))
            s.execute(plan_a)
            before = s.state()
            native_a = s.state_native().copy()
            b, p = s.measure_qubits(qs, q.sample_uniform(5, 0))
            projected, _ = project_np(before, qs, b)
            s.apply(q.gates_from_circuit(circ_b))
            with q.Simulator(n, precision=prec, device=0) as ref:
                ref.set_state(projected)
                ref.apply(q.gates_from_circuit(circ_b))
                assert np.max(np.abs(s.state() - ref.state())) <= tol
            s.reset()
            s.execute(plan_a)                               # the plan (and its graph) runs again on the same buffer
            assert np.array_equal(s.state_native(), native_a)
            plan_a.close()
    # chain rule: group a, then group b gives p(a) p(b | a) = the joint marginal of a + b
    with run(n, circ_a, prec) as s:
        ga, gb = [1, 6], [3, 12, 8]
        joint = s.marginal_probabilities(ga + gb)
        oa, pa = s.measure_qubits(ga, 0.3)
        ob, pb = s.measure_qubits(gb, 0.6)
        assert abs(pa * pb - joint[oa | (ob << len(ga))]) <= TOL[prec]


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_reset_qubits(prec):
    n = 13
    with run(n, circuits.random_layered(n, depth=5, seed=21), prec) as s:
        for qs, r in (([4], 0.7), ([0, 12, 6], 0.2), ([n - 1, 1], 0.9)):
            before = s.state()
            b = s.reset_qubits(qs, r)
            m = s.marginal_probabilities(qs)
            assert abs(m[0] - 1.0) <= TOL[prec] and np.all(np.abs(m[1:]) <= TOL[prec])
            projected, _ = project_np(before, qs, b)
            flip = sum(1 << qs[i] for i in range(len(qs)) if (b >> i) & 1)
            want = projected[np.arange(1 << n) ^ flip]
            assert np.max(np.abs(s.state() - want)) <= 10 * TOL[prec]


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [q.F32, q.F64])
def test_errors_leave_the_state_unchanged(prec):
    n = 22
    with run(n, circuits.random_layered(n, depth=2, seed=3), prec) as s:
        raw = s.state_native().copy()

        def refused(fn, *args):
            with pytest.raises(q.QsbError) as e:
                fn(*args)
            assert e.value.code == -1, e.value
            assert np.array_equal(s.state_native(), raw)
        for bad in ([1, 1], [n], [-1], [], list(range(21))):
            refused(s.marginal_probabilities, bad)
            refused(s.collapse, bad, 0)
            refused(s.measure_qubits, bad, 0.5)
            refused(s.reset_qubits, bad, 0.5)
        for r in (1.0, -1e-300, -0.5, float("nan"), 2.0):
            refused(s.measure_qubits, [0, 1], r)
            refused(s.reset_qubits, [0], r)
        refused(s.collapse, [0, 5], 4)
        refused(s.collapse, [3], 2)
    with q.Simulator(9, precision=prec, device=0) as s:
        s.set_state(np.zeros(1 << 9, dtype=np.complex128))
        raw = s.state_native().copy()
        assert np.array_equal(s.marginal_probabilities([0, 4]), np.zeros(4))
        refused(s.measure_qubits, [0, 4], 0.5)
        refused(s.reset_qubits, [2], 0.0)
        refused(s.collapse, [0, 4], 0)


@pytest.mark.gpu
def test_cli_marginal_matches_python(tmp_path):
    exe = os.path.join(helpers.ROOT, "gpu_quantum_simulator_b200", "bin", "qsim")
    n = 14
    circ = circuits.random_layered(n, depth=4, seed=9)
    path = tmp_path / "c.qasm"
    path.write_text(circuits.to_qasm(circ, n))
    sets = [[0, 3, 5], [13], [7, 2, 11, 1]]
    args = [exe, str(path), "--expect", "Z0"]
    for qs in sets:
        args += ["--marginal", " ".join(map(str, qs))]
    r = subprocess.run(args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.splitlines()
    assert lines[1].startswith("EXPECTATION Z0:")       # the MARGINAL lines follow the EXPECTATION lines
    marg = lines[2:]
    assert [ln.split(":")[0] for ln in marg] == ["MARGINAL " + " ".join(map(str, qs)) for qs in sets]
    with run(n, circ, q.F32) as s:
        for ln, qs in zip(marg, sets):
            got = np.array([float(v) for v in ln.split(":")[1].split()])
            assert got.size == 1 << len(qs)
            assert np.max(np.abs(got - s.marginal_probabilities(qs))) <= 1e-12
    plain = subprocess.run([exe, str(path)], capture_output=True, text=True, timeout=300)
    assert plain.returncode == 0 and len(plain.stdout.splitlines()) == 1 and "MARGINAL" not in plain.stdout


@pytest.mark.gpu
def test_sharded_measure():
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 8 if ngpu >= 8 else 4 if ngpu >= 4 else 2
    script = os.path.join(os.path.dirname(__file__), "dist_measure_worker.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", "29567", script],
                       capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "sharded_measure_ok" in r.stdout


@pytest.mark.gpu
@pytest.mark.slow
def test_30q_f32_against_f64_and_collapse():
    n = 30
    circ = circuits.random_layered(n, depth=20)
    rng = np.random.default_rng(30)
    sets = [[17], rng.permutation(n)[:10].tolist(), rng.permutation(n)[:20].tolist()]
    vals = []
    for prec in (q.F32, q.F64):
        with run(n, circ, prec) as s:
            vals.append([s.marginal_probabilities(qs) for qs in sets])
            if prec == q.F32:
                table = vals[-1][1]
                p = s.collapse(sets[1], int(np.argmax(table)))
                assert p == table[int(np.argmax(table))]
                assert abs(s.norm_argmax()[0] - 1.0) <= 1e-5
    for a, b in zip(*vals):
        assert np.max(np.abs(a - b)) <= 1e-5
