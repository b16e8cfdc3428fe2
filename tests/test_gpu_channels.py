"""Noise channels on the device (qsb_apply_channels) against a numpy replay on the downloaded state: every Kraus operator
applied by tensordot, w_i = ||K_i psi||^2, the branch by the rule of qsb_measure_qubits, psi <- sqrt(T / w_i) K_i psi.

A draw r whose host margin min_i |C_i - r T| is below 1e-9 T is skipped (redrawn): there the numpy weights and the
library's (from a Gram matrix in another summation order, or from q_i for a fixed-weight channel) may round to
different sides of r T, and either branch is correct."""
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers
import gpu_quantum_simulator_b200 as q
from gpu_quantum_simulator_b200 import circuits
from test_gpu_matrix import apply_np
from test_gpu_pauli_rotation import permuted

pytestmark = pytest.mark.gpu

F32, F64 = q.F32, q.F64
PRECS = pytest.mark.parametrize("prec", [F32, F64], ids=["f32", "f64"])
TOL = {F32: 1e-5, F64: 1e-12}
PTOL = {F32: 1e-6, F64: 1e-12}                            # relative, on prob
LOW_BITS = {F32: [0, 3, 5, 6], F64: [0, 2, 4, 5]}        # 0 = the default (4 / 3)


def stinespring(k, m, seed):
    """m Kraus operators of a random channel on k qubits: the blocks of a random (m 2^k) x 2^k isometry."""
    rng = np.random.default_rng(seed)
    d = 1 << k
    a = rng.normal(size=(m * d, d)) + 1j * rng.normal(size=(m * d, d))
    v, _ = np.linalg.qr(a)
    return [v[i * d:(i + 1) * d, :] for i in range(m)]


def replay(a, kraus, ts, r, n):
    """-> (branch, prob, new state, margin / T) of one channel on the complex128 state a."""
    outs = [apply_np(a, [(np.asarray(K), ts)], n) for K in kraus]
    w = [float(np.vdot(o, o).real) for o in outs]
    T = 0.0
    for x in w:
        T += x
    c, branch = 0.0, None
    margin = np.inf
    for i, x in enumerate(w):
        c += x
        margin = min(margin, abs(c - r * T))
        if branch is None and c != 0.0 and c >= r * T:
            branch = i
    return branch, w[branch] / T, outs[branch] * np.sqrt(T / w[branch]), margin / T


def replay_list(a, channels, rs, n):
    """-> (branches, probs, state, smallest margin) of a list, channel by channel."""
    bs, ps, mg = [], [], np.inf
    for (kraus, ts), r in zip(channels, rs):
        b, p, a, m = replay(a, kraus, ts, r, n)
        bs.append(b)
        ps.append(p)
        mg = min(mg, m)
    return np.array(bs), np.array(ps), a, mg


def draws(seed, count):
    return [q.sample_uniform(seed, c) for c in range(count)]


def random_channel(n, rng, seed, kmax=4):
    k = int(rng.integers(1, min(kmax, n) + 1))
    ts = [int(x) for x in rng.permutation(n)[:k]]
    kind = rng.integers(0, 4)
    if kind == 0 and k == 1:
        return q.amplitude_damping(float(rng.uniform(0.05, 0.9))), ts
    if kind == 1 and k <= 2:
        return q.depolarizing(float(rng.uniform(0.05, 0.9)), k), ts
    m = int(rng.choice([1, 2, 1 << (2 * k)])) if rng.random() < 0.5 else int(rng.integers(1, (1 << (2 * k)) + 1))
    return stinespring(k, m, seed), ts


def run_and_compare(s, channels, prec, seed0):
    """Apply the list with the first r draw whose margins are safe; compare with the replay."""
    n = s.num_qubits
    a0, perm0 = s.state(), s.layout()[0]
    for seed in range(seed0, seed0 + 50):
        rs = draws(seed, len(channels))
        bw, pw, want, mg = replay_list(a0, channels, rs, n)
        if mg >= 1e-9:
            break
    else:
        raise AssertionError("no safe draw")
    b, p = s.apply_channels(channels, r=rs)
    assert np.array_equal(b, bw.astype(np.uint32)), (b, bw)
    assert np.allclose(p, pw, rtol=PTOL[prec], atol=0), (p, pw)
    err = float(np.max(np.abs(s.state() - want)))
    assert err <= 3 * TOL[prec], err
    assert np.array_equal(s.layout()[0], perm0)
    return err


@pytest.mark.parametrize("prec,low_bits", [(p, lb) for p in (F32, F64) for lb in LOW_BITS[p]],
                         ids=[f"f{p}-low{lb}" for p in (F32, F64) for lb in LOW_BITS[p]])
def test_replay_per_channel(prec, low_bits):
    """One channel per call, every width and Kraus count, targets in any order, low and high bits, several sizes."""
    rng = np.random.default_rng(100 + low_bits + prec)
    for n in (1, 2, 3, 5, 9, 14, 17, 22):
        with permuted(n, prec, low_bits=low_bits) as s:
            for i in range(6 if n < 20 else 3):
                kraus, ts = random_channel(n, rng, seed=n * 100 + i)
                run_and_compare(s, [(kraus, ts)], prec, seed0=1000 * n + i)
            if n >= 4:   # the extremes of the Kraus count on 4 targets, lowest and highest qubits
                for m, ts in ((1, [0, 1, 2, 3]), (256, [n - 1, 0, n - 2, 1]), (7, [1, n - 1, 0, n - 2])):
                    run_and_compare(s, [(stinespring(4, m, n + m), ts)], prec, seed0=77 * n + m)


@PRECS
def test_multi_channel_layers(prec):
    """Layers of 1..30 channels of mixed kinds in one call, against the replay channel by channel."""
    n = 16
    rng = np.random.default_rng(5)
    with permuted(n, prec) as s:
        for count in (1, 2, 5, 13, 30):
            chans = [random_channel(n, rng, seed=count * 1000 + i) for i in range(count)]
            run_and_compare(s, chans, prec, seed0=count * 31)
        layer = [(q.amplitude_damping(0.2), [k]) for k in range(n)] + [(q.depolarizing(0.3), [k]) for k in range(n)]
        run_and_compare(s, layer, prec, seed0=9)
        pairs = [(stinespring(2, 3, i), [i, (i + 1) % n]) for i in range(10)]
        run_and_compare(s, pairs, prec, seed0=19)


@PRECS
def test_identity_branch_changes_no_byte(prec):
    n = 14
    with permuted(n, prec) as s:
        raw0 = s.state_native().copy()
        dep = q.depolarizing(0.01)
        b, p = s.apply_channels([(dep, [k]) for k in range(n)] + [(q.depolarizing(0.02, 2), [3, 9])], r=[0.0] * (n + 1))
        assert np.all(b == 0)
        assert np.allclose(p[:n], 1 - 0.75 * 0.01) and np.isclose(p[n], 1 - 15 / 16 * 0.02)
        assert np.array_equal(s.state_native(), raw0)
        # a fixed-weight channel written as a general set: its identity operator is skipped without a read
        b, p = s.apply_channels([([np.sqrt(0.9) * np.eye(2), np.sqrt(0.1) * np.array([[0, 1], [1, 0]])], [5])], r=[0.1])
        assert b[0] == 0 and np.isclose(p[0], 0.9) and np.array_equal(s.state_native(), raw0)
        # a state-dependent set with an identity operator: the group reads rho, picks branch 0 (weight 1/2 whatever the
        # state) and the identity skip inside the group leaves every byte as it was; so do two such channels in one group
        proj = [np.sqrt(0.5) * np.eye(2), np.sqrt(0.5) * np.diag([1.0, 0.0]), np.sqrt(0.5) * np.diag([0.0, 1.0])]
        assert q.channel_dry_run(n, [(proj, [5])], prec)["gram_sweeps"] == 1
        b, p = s.apply_channels([(proj, [5]), (proj, [11]), (proj, [5])], r=[0.1, 0.3, 0.49])
        assert np.all(b == 0) and np.allclose(p, 0.5, rtol=1e-6)
        assert np.array_equal(s.state_native(), raw0)


@PRECS
def test_invariants(prec):
    """Layout unchanged, plans and captured graphs made before the call execute after it, repeated calls give the same
    bits."""
    n = 18
    circ = q.gates_from_circuit(circuits.random_layered(n, depth=4, seed=8))
    chans = [(q.amplitude_damping(0.3), [k]) for k in range(0, n, 2)] + [(stinespring(2, 4, 1), [1, 17])]
    rng = np.random.default_rng(4)
    a0 = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)
    a0 /= np.linalg.norm(a0)
    for use_graph in (False, True):
        with q.Simulator(n, precision=prec, device=0, use_graph=use_graph) as s, q.Simulator(n, precision=prec, device=0) as r:
            p = s.plan(circ)
            if use_graph:
                s.execute(p)                                     # captures the graph
                s.reset()
            s.set_state(a0)
            r.set_state(a0)
            perm0 = s.layout()[0]
            b1, p1 = s.apply_channels(chans, seed=3)
            b2, p2 = r.apply_channels(chans, seed=3)
            assert np.array_equal(b1, b2) and np.array_equal(p1.view(np.uint64), p2.view(np.uint64))
            assert np.array_equal(s.state_native(), r.state_native())
            assert np.array_equal(s.layout()[0], perm0)
            s.execute(p)
            r.apply(circ)
            assert np.max(np.abs(s.state() - r.state())) <= 3 * TOL[prec], use_graph
            p.close()


def test_trajectory_statistics():
    """The average of |psi><psi| over 4000 trajectories matches the exact Kraus evolution of rho."""
    n, count = 4, 4000
    circ = [("h", [0], []), ("cx", [0, 1], []), ("ry", [2], [0.7]), ("cx", [2, 3], []), ("rx", [1], [0.4])]
    gates = q.gates_from_circuit(circ)
    chans = ([(q.amplitude_damping(0.3), [k]) for k in range(n)] + [(q.depolarizing(0.2), [k]) for k in range(n)]
             + [(stinespring(2, 3, 42), [1, 3])])
    with q.Simulator(n, precision=F64, device=0) as s:
        s.apply(gates)
        psi0 = s.state()
        acc = np.zeros((1 << n, 1 << n), dtype=np.complex128)
        for t in range(count):
            s.set_state(psi0)
            s.apply_channels(chans, seed=t)
            a = s.state()
            a = a / np.linalg.norm(a)
            acc += np.outer(a, np.conj(a))
    acc /= count
    rho = np.outer(psi0, np.conj(psi0))
    for kraus, ts in chans:   # rho <- sum_i K_i rho K_i^dag, with K_i on the full register via apply_np on each column
        ops = []
        for K in kraus:
            M = np.stack([apply_np(np.eye(1 << n)[:, j], [(K, ts)], n) for j in range(1 << n)], axis=1)
            ops.append(M)
        rho = sum(M @ rho @ np.conj(M).T for M in ops)
    assert abs(np.trace(rho).real - 1) < 1e-12
    assert np.max(np.abs(acc - rho)) <= 5 / np.sqrt(count), np.max(np.abs(acc - rho))


def compose(s, channels, rs):
    """The composition a caller could write: per channel the reduced density matrix of its targets, the host rule,
    then apply_matrix of the chosen operator scaled to keep the norm."""
    bs, ps = [], []
    for (kraus, ts), r in zip(channels, rs):
        rho = s.reduced_density_matrix(ts)
        w = [max(float(np.trace(K @ rho @ np.conj(K).T).real), 0.0) for K in map(np.asarray, kraus)]
        T = 0.0
        for x in w:
            T += x
        c, b = 0.0, None
        for i, x in enumerate(w):
            c += x
            if c != 0.0 and c >= r * T:
                b = i
                break
        s.apply_matrix(np.asarray(kraus[b]) * np.sqrt(T / w[b]), ts)
        bs.append(b)
        ps.append(w[b] / T)
    return np.array(bs, dtype=np.uint32), np.array(ps)


def composition_case(n, prec):
    circ = q.gates_from_circuit(circuits.random_layered(n, depth=6, seed=n))
    rng = np.random.default_rng(n)
    chans = [(q.amplitude_damping(0.05), [k]) for k in range(n)] + [(q.depolarizing(0.05), [k]) for k in range(n)]
    chans += [(stinespring(2, 4, 900 + i), [int(x) for x in rng.permutation(n)[:2]]) for i in range(10)]
    rs = draws(11, len(chans))
    with q.Simulator(n, precision=prec, device=0) as s, q.Simulator(n, precision=prec, device=0) as c:
        s.apply(circ)
        c.copy_from(s)
        b, p = s.apply_channels(chans, r=rs)
        bc, pc = compose(c, chans, rs)
        assert np.array_equal(b, bc), (b, bc)
        assert np.allclose(p, pc, rtol=1e-5 if prec == F32 else 1e-10)
        f = s.fidelity(c)
        assert f >= 1 - (1e-5 if prec == F32 else 1e-12), f


@PRECS
def test_composition_24q(prec):
    composition_case(24, prec)


@pytest.mark.slow
@PRECS
def test_composition_30q(prec):
    composition_case(30, prec)


@PRECS
def test_refusals_leave_the_state(prec):
    n = 12
    ad = q.amplitude_damping(0.3)
    with permuted(n, prec) as s:
        raw0 = s.state_native().copy()
        nan = np.array(ad); nan[0, 1, 1] = np.nan
        for chans, r, text in (([(ad, [12])], [0.5], "outside"), ([(stinespring(2, 2, 0), [3, 3])], [0.5], "twice"),
                               ([(ad, [0]), (nan, [1])], [0.5, 0.5], "non-finite"),
                               ([(ad[:1], [0])], [0.5], "not trace-preserving"),
                               ([(ad, [0]), (ad, [1])], [0.5, 1.0], "outside [0, 1)"),
                               ([(ad, [0])], [np.nan], "outside [0, 1)"), ([(ad, [0])], [-0.1], "outside [0, 1)"),
                               ([(stinespring(1, 5, 0), [0])], [0.5], "5 Kraus operators")):
            with pytest.raises(q.QsbError) as e:
                s.apply_channels(chans, r=r)
            assert e.value.code == -1 and text in str(e.value), (text, str(e.value))
            assert np.array_equal(s.state_native(), raw0), text
        with pytest.raises(ValueError):
            s.apply_channels([(stinespring(3, 2, 0), [0, 1])])
        with pytest.raises(ValueError):
            s.apply_channels([(np.eye(32)[None], list(range(5)))])
        assert np.array_equal(s.state_native(), raw0)
    with q.Simulator(n, precision=prec, device=0) as z:
        z.set_state(np.zeros(1 << n))
        with pytest.raises(q.QsbError) as e:
            z.apply_channels([(q.depolarizing(0.1), [0]), (ad, [2])], r=[0.99, 0.5])
        assert e.value.code == -1 and "norm 0" in str(e.value)
        assert not np.any(z.state_native())
    with q.Simulator(n, precision=prec, low_bits=8, device=0) as s:
        s.set_state(np.arange(1 << n) * (1 + 1j) / (1 << n))
        raw0 = s.state_native().copy()
        with pytest.raises(q.QsbError) as e:
            s.apply_channels([(ad, [0])], r=[0.5])
        assert e.value.code == -1 and "low_bits 8 unsupported" in str(e.value)
        assert np.array_equal(s.state_native(), raw0)


def write_kraus(path, kraus):
    path.write_text("\n".join(" ".join(f"{float(v.real)!r} {float(v.imag)!r}" for v in np.asarray(K).reshape(-1))
                              for K in kraus) + "\n")


def test_cli_channels(tmp_path):
    exe = os.path.join(helpers.ROOT, "gpu_quantum_simulator_b200", "bin", "qsim")
    n = 12
    circ = circuits.random_layered(n, depth=4, seed=9)
    path = tmp_path / "c.qasm"
    path.write_text(circuits.to_qasm(circ, n))
    chans = [(q.amplitude_damping(0.4), [3]), (q.depolarizing(0.3, 2), [0, 7]), (stinespring(2, 3, 5), [11, 2]),
             (q.phase_damping(0.5), [5])]
    base = [exe, str(path), "--expect", "Z3", "--expect", "X0 Z7"]
    args = list(base)
    for j, (kraus, qs) in enumerate(chans):
        f = tmp_path / f"k{j}.txt"
        write_kraus(f, kraus)
        args += ["--channel", " ".join(map(str, qs)), str(f)]
    r = subprocess.run(args + ["--channel-seed", "5", "--profile"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.splitlines()
    assert lines[1].startswith("{")                                   # the --profile line, then the CHANNEL lines
    got = lines[2:2 + len(chans)]
    assert [ln.split(":")[0] for ln in got] == ["CHANNEL " + " ".join(map(str, qs)) for _, qs in chans]
    assert lines[2 + len(chans)].startswith("EXPECTATION Z3:")
    with q.Simulator(n, precision=F32, device=0) as s:
        s.apply(q.gates_from_circuit(circ))
        b, p = s.apply_channels(chans, seed=5)
        ev = s.expectation(["Z3", "X0 Z7"])
    assert [int(ln.split(":")[1].split()[0]) for ln in got] == list(b)
    assert [float(ln.split(":")[1].split()[1]) for ln in got] == list(p)
    assert [float(ln.rsplit(":", 1)[1]) for ln in lines[2 + len(chans):4 + len(chans)]] == list(ev)
    # without --channel: the time line and the EXPECTATION lines only, the values of the circuit alone
    r0 = subprocess.run(base, capture_output=True, text=True, timeout=300)
    assert r0.returncode == 0 and not any(ln.startswith("CHANNEL") for ln in r0.stdout.splitlines())
    with q.Simulator(n, precision=F32, device=0) as s:
        s.apply(q.gates_from_circuit(circ))
        assert r0.stdout.splitlines()[1:] == [f"EXPECTATION Z3: {s.expectation('Z3'):.17g}",
                                              f"EXPECTATION X0 Z7: {s.expectation('X0 Z7'):.17g}"]
    short = tmp_path / "short.txt"
    short.write_text("1 0 0 0 0 0\n")
    lossy = tmp_path / "lossy.txt"
    write_kraus(lossy, q.amplitude_damping(0.4)[:1])
    for extra, text in ((["--channel", "0", str(short)], "expected 1..4 operators of 8 numbers"),
                        (["--channel", "0", str(tmp_path / "missing.txt")], "cannot open"),
                        (["--channel", "0 x", str(short)], "expected a whitespace-separated list"),
                        (["--channel", "12", str(tmp_path / "k0.txt")], "target 12 outside"),
                        (["--channel", "1", str(lossy)], "not trace-preserving")):
        bad = subprocess.run([exe, str(path)] + extra, capture_output=True, text=True, timeout=300)
        assert bad.returncode == 1 and text in bad.stdout and len(bad.stdout.splitlines()) == 1, bad.stdout


def test_sharded_channels():
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 8 if ngpu >= 8 else 4 if ngpu >= 4 else 2
    script = os.path.join(os.path.dirname(__file__), "dist_channel_worker.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", "29589", script],
                       capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "sharded_channel_ok" in r.stdout
