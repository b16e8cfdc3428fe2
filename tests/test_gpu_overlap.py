"""Overlaps <a|b> and the state copy on the device, against np.vdot on the downloaded states: every precision pair, sizes
around the tile and padding boundaries, layouts from circuits and crafted through load_state, exactness on a state and
its copy, determinism, invariants, refusals and the CLI."""
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers
import gpu_quantum_simulator_b200 as q
from gpu_quantum_simulator_b200 import circuits

pytestmark = pytest.mark.gpu

F32, F64 = q.F32, q.F64
PAIRS = pytest.mark.parametrize("pa,pb", [(F32, F32), (F32, F64), (F64, F32), (F64, F64)])
NLOC_MIN = {F32: 12, F64: 11}


def tol(pa, pb):
    return 1e-12 if pa == pb == F64 else 1e-5


def random_state(n, seed):
    rng = np.random.default_rng(seed)
    v = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)
    return v / np.linalg.norm(v)


def write_shard(path, n, prec, perm, psi, world=1, rank=0):
    """A shard file (qsb_save_state format) holding the logical state psi under the layout perm (perm[q] = physical bit
    of qubit q, bits >= nloc are rank bits); padding bits read 0."""
    g = world.bit_length() - 1
    nloc = max(n - g, NLOC_MIN[prec])
    j = np.arange(1 << n, dtype=np.int64)
    p = np.zeros_like(j)
    for qb in range(n):
        p |= ((j >> qb) & 1) << int(perm[qb])
    mine = (p >> nloc) == rank
    phys = np.zeros(1 << nloc, dtype=np.complex128)
    phys[p[mine] & ((1 << nloc) - 1)] = psi[mine]
    if prec == F32:
        re, im = phys.real.astype(np.float32), phys.imag.astype(np.float32)
        body = np.stack([re[0::2], re[1::2], im[0::2], im[1::2]], axis=1)
    else:
        body = np.stack([phys.real, phys.imag], axis=1)
    hdr = bytearray(128)
    hdr[0:8] = b"QSBSHARD"
    hdr[8:32] = np.array([1, n, prec, world, rank, nloc], dtype=np.uint32).tobytes()
    pm = np.full(64, -1, dtype=np.int8)
    pm[:n] = perm
    hdr[32:96] = pm.tobytes()
    with open(path, "wb") as f:
        f.write(bytes(hdr))
        f.write(np.ascontiguousarray(body).tobytes())


def crafted(tmp_path, name, n, prec, perm, psi, **kw):
    path = tmp_path / f"{name}.qsb"
    write_shard(path, n, prec, perm, psi)
    s = q.Simulator(n, precision=prec, device=0, **kw)
    s.load_state(str(path))
    assert np.array_equal(s.layout()[0][:n], np.asarray(perm))
    return s


def check_against_numpy(a, b, t):
    x, y = a.state(), b.state()
    got, na, nb = a._inner(b)
    want = np.vdot(x, y)
    scale = np.sqrt(np.vdot(x, x).real * np.vdot(y, y).real) or 1.0
    assert abs(got - want) <= t * scale, (got, want)
    assert abs(na - np.vdot(x, x).real) <= t * max(na, 1e-300) and abs(nb - np.vdot(y, y).real) <= t * max(nb, 1e-300)
    assert a.overlap(b) == got
    return got


@PAIRS
@pytest.mark.parametrize("n", [1, 3, 11, 12, 13, 20, 24])
def test_random_layouts_against_vdot(tmp_path, n, pa, pb):
    rng = np.random.default_rng(100 + n)
    x = random_state(n, 2 * n)
    y = 0.6 * x + 0.8 * random_state(n, 2 * n + 1)       # a sizeable overlap
    for k in range(2):
        perm_a = rng.permutation(max(n, NLOC_MIN[pa]))[:n]  # small registers: qubits anywhere among the padded bits
        perm_b = rng.permutation(max(n, NLOC_MIN[pb]))[:n]
        with crafted(tmp_path, "a", n, pa, perm_a, x) as a, crafted(tmp_path, "b", n, pb, perm_b, y) as b:
            got = check_against_numpy(a, b, tol(pa, pb))
            assert abs(got) > 0.3
            check_against_numpy(b, a, tol(pa, pb))


@PAIRS
def test_low_bits_of_one_on_the_top_bits_of_the_other(tmp_path, pa, pb):
    n = 20
    x, y = random_state(n, 1), random_state(n, 2)
    perm_a = np.arange(n)
    perm_b = n - 1 - np.arange(n)                          # b's low bits hold a's top local qubits
    with crafted(tmp_path, "a", n, pa, perm_a, x) as a, crafted(tmp_path, "b", n, pb, perm_b, y + 0.5 * x) as b:
        check_against_numpy(a, b, tol(pa, pb))
        check_against_numpy(b, a, tol(pa, pb))


def test_f32_f64_pair_with_different_padding(tmp_path):
    n = 3
    x, y = random_state(n, 3), random_state(n, 4)
    with crafted(tmp_path, "a", n, F32, [11, 5, 0], x) as a, crafted(tmp_path, "b", n, F64, [3, 10, 7], y) as b:
        check_against_numpy(a, b, 1e-5)
        check_against_numpy(b, a, 1e-5)


@PAIRS
@pytest.mark.parametrize("n", [13, 20])
def test_layouts_from_circuits(n, pa, pb):
    with q.Simulator(n, precision=pa, device=0) as a, q.Simulator(n, precision=pb, device=0) as b:
        a.apply(q.gates_from_circuit(circuits.random_layered(n, depth=6, seed=1)))
        for seed in range(2, 30):                       # the first circuit that leaves b in another layout
            b.reset()
            b.apply(q.gates_from_circuit(circuits.random_layered(n, depth=5, seed=seed)))
            if not np.array_equal(a.layout()[0][:n], b.layout()[0][:n]):
                break
        assert not np.array_equal(a.layout()[0][:n], b.layout()[0][:n])
        check_against_numpy(a, b, tol(pa, pb))


@PAIRS
def test_same_circuit_in_both_precisions(pa, pb):
    n = 18
    circ = q.gates_from_circuit(circuits.random_layered(n, depth=8, seed=3))
    with q.Simulator(n, precision=pa, device=0) as a, q.Simulator(n, precision=pb, device=0) as b:
        a.apply(circ)
        b.apply(circ)
        check_against_numpy(a, b, tol(pa, pb))
        assert abs(a.fidelity(b) - 1.0) <= 1e-5


@pytest.mark.parametrize("prec", [F32, F64])
@pytest.mark.parametrize("n", [3, 13, 20])
def test_self_overlap_and_copy_are_exact(prec, n):
    with q.Simulator(n, precision=prec, device=0) as a, q.Simulator(n, precision=prec, device=0) as b:
        a.apply(q.gates_from_circuit(circuits.random_layered(n, depth=4, seed=n)))
        ov, na, nb = a._inner(a)
        assert ov.imag == 0.0 and ov.real == na == nb
        b.copy_from(a)
        assert np.array_equal(b.layout()[0], a.layout()[0])
        assert np.array_equal(b.state_native(), a.state_native())
        for x, y in ((a, b), (b, a)):
            ov2, na2, nb2 = x._inner(y)
            assert ov2.imag == 0.0 and ov2.real == na2 == nb2 == na
        assert a.fidelity(b) == 1.0
        b.copy_from(b)                                      # a no-op
        assert np.array_equal(b.state_native(), a.state_native())


@PAIRS
def test_repeat_calls_and_invariants(pa, pb):
    """Repeat calls return the same bits; bytes and layouts stay; a plan (and a captured graph) made on each handle before
    the call still executes after it."""
    n = 16
    ca = q.gates_from_circuit(circuits.random_layered(n, depth=4, seed=5))
    cb = q.gates_from_circuit(circuits.random_layered(n, depth=3, seed=6))
    for use_graph in (False, True):
        with q.Simulator(n, precision=pa, device=0, use_graph=use_graph) as a, \
                q.Simulator(n, precision=pb, device=0, use_graph=use_graph) as b, \
                q.Simulator(n, precision=pa, device=0) as ra, q.Simulator(n, precision=pb, device=0) as rb:
            if use_graph:                                   # capture at the identity layout, then back to it
                plan_a, plan_b = a.plan(ca), b.plan(cb)
                a.execute(plan_a); a.reset()
                b.execute(plan_b); b.reset()
                a.set_state(random_state(n, 1)); b.set_state(random_state(n, 2))
                ra.set_state(random_state(n, 1)); rb.set_state(random_state(n, 2))
            else:                                           # plans for the permuted layouts the circuits leave
                a.apply(cb); b.apply(ca)
                ra.apply(cb); rb.apply(ca)
                plan_a, plan_b = a.plan(ca), b.plan(cb)
            raw_a, raw_b = a.state_native().copy(), b.state_native().copy()
            lay_a, lay_b = a.layout(), b.layout()
            first = a._inner(b)
            for _ in range(3):
                assert a._inner(b) == first
            b._inner(a)
            assert np.array_equal(a.state_native(), raw_a) and np.array_equal(b.state_native(), raw_b)
            assert np.array_equal(a.layout()[0], lay_a[0]) and np.array_equal(b.layout()[0], lay_b[0])
            a.execute(plan_a); b.execute(plan_b)
            ra.apply(ca); rb.apply(cb)
            assert np.max(np.abs(a.state() - ra.state())) <= 3 * tol(pa, pa), use_graph
            assert np.max(np.abs(b.state() - rb.state())) <= 3 * tol(pb, pb), use_graph
            plan_a.close(); plan_b.close()


def test_refused_arguments(tmp_path):
    n = 12
    with q.Simulator(n, precision=F32, device=0) as a, q.Simulator(n + 1, precision=F32, device=0) as b, \
            q.Simulator(n, precision=F64, device=0) as c, q.Simulator(n, precision=F32, low_bits=7, device=0) as d, \
            q.Simulator(n, precision=F64, low_bits=1, device=0) as e:
        a.apply(q.gates_from_circuit(circuits.random_layered(n, depth=3, seed=1)))
        raw = [s.state_native().copy() for s in (a, b, c, d, e)]
        for x, y, text in ((a, b, "differ"), (b, a, "differ"), (a, d, "low_bits 7 unsupported"), (d, a, "low_bits 7 unsupported"),
                           (e, c, "low_bits 1 unsupported")):
            with pytest.raises(q.QsbError) as err:
                x.overlap(y)
            assert err.value.code == -1 and text in str(err.value)
        for x, y, text in ((a, b, "differ"), (a, c, "precision"), (c, a, "precision")):
            with pytest.raises(q.QsbError) as err:
                x.copy_from(y)
            assert err.value.code == -1 and text in str(err.value)
        import ctypes as C
        out = np.empty(2)
        assert q.lib.qsb_inner_product(None, a._h, out.ctypes.data, None) == -1
        assert q.lib.qsb_inner_product(a._h, None, out.ctypes.data, None) == -1
        assert q.lib.qsb_inner_product(a._h, c._h, None, None) == -1
        assert q.lib.qsb_inner_product(a._h, c._h, out.ctypes.data, None) == 0   # norms may be NULL
        assert q.lib.qsb_copy_state(None, a._h) == -1 and q.lib.qsb_copy_state(a._h, C.c_void_p()) == -1
        for s, r in zip((a, b, c, d, e), raw):
            assert np.array_equal(s.state_native(), r)
        c.set_state(np.zeros(1 << n))
        with pytest.raises(ValueError):
            a.fidelity(c)
        assert a.overlap(c) == 0


def test_cli_overlap(tmp_path):
    exe = os.path.join(helpers.ROOT, "gpu_quantum_simulator_b200", "bin", "qsim")
    n = 14
    main = circuits.random_layered(n, depth=4, seed=9)
    others = [circuits.random_layered(n, depth=3, seed=10), main[: len(main) // 2]]
    path = tmp_path / "main.qasm"
    path.write_text(circuits.to_qasm(main, n))
    args = [exe, str(path), "--pauli-rot", "X0 Z3", "0.25"]
    files = []
    for k, c in enumerate(others):
        f = tmp_path / f"o{k}.qasm"
        f.write_text(circuits.to_qasm(c, n))
        files.append(str(f))
        args += ["--overlap", str(f)]
    for prec in (32, 64):
        r = subprocess.run(args + ["--precision", str(prec), "--rdm", "0"], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stdout + r.stderr
        lines = r.stdout.splitlines()
        assert lines[1].startswith("RDM 0:")
        ov = lines[2:2 + len(files)]
        assert [ln.rsplit(":", 1)[0] for ln in ov] == [f"OVERLAP {f}" for f in files]
        with q.Simulator(n, precision=prec, device=0) as s:
            s.apply(q.gates_from_circuit(main))
            s.apply_pauli_rotations("X0 Z3", 0.25)
            for ln, c in zip(ov, others):
                with q.Simulator(n, precision=prec, device=0) as o:
                    o.apply(q.gates_from_circuit(c))
                    re, im, fid = map(float, ln.rsplit(":", 1)[1].split())
                    assert complex(re, im) == s.overlap(o)
                    assert fid == pytest.approx(s.fidelity(o), rel=1e-14, abs=0)
    bad = tmp_path / "bad.qasm"
    bad.write_text(circuits.to_qasm(circuits.random_layered(n + 1, 2, 1), n + 1))
    r = subprocess.run([exe, str(path), "--overlap", str(bad)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 1 and "15 qubits" in r.stdout and len(r.stdout.splitlines()) == 1, r.stdout


def test_sharded_overlaps():
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 8 if ngpu >= 8 else 4 if ngpu >= 4 else 2
    script = os.path.join(os.path.dirname(__file__), "dist_overlap_worker.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", "29577", script],
                       capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "sharded_overlap_ok" in r.stdout
