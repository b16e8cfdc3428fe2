"""Device-side readout (SURVEY 8f-1, 8f-4) against the oracle's compute_state_cumulative_distribution /
measurement restatement (oc_cdf, oc_measure <- quantum_simulator.c:256-283): CDF, streaming sampler,
shard dump / reload.  Through the C ABI."""
import math
import os
import subprocess

import numpy as np
import pytest

import helpers
import gpu_quantum_simulator_b200 as q
from gpu_quantum_simulator_b200 import circuits

pytestmark = pytest.mark.gpu

F32, F64 = q.F32, q.F64
TOL = {F32: 1e-5, F64: 1e-12}


def oracle_cdf(state, n):
    L = helpers.oracle_lib()
    v = np.ascontiguousarray(state, dtype=np.complex128)
    out = np.zeros(1 << n)
    L.oc_cdf(v.ctypes.data, n, out.ctypes.data)
    return out


def oracle_measure(cdf, n, r):
    L = helpers.oracle_lib()
    return int(L.oc_measure(cdf.ctypes.data, n, r))


def check_shots(shots, cdf, n, seed, rs=None):
    """Every shot is what the reference's search rule gives for the same r on the device CDF; a shot may only
    differ when r sits within rounding of a CDF step.  rs: the r of each shot, when the caller has them already
    (q.sample_uniform replays the generator from shot 0, so a long run would cost time quadratic in its length)."""
    for k, got in enumerate(shots):
        r = q.sample_uniform(seed, k) if rs is None else float(rs[k])
        want = oracle_measure(cdf, n, r)
        if int(got) != want:
            assert abs(cdf[want] - r) < 1e-12 or abs(cdf[int(got)] - r) < 1e-12, (k, r, int(got), want)
        p = cdf[int(got)] - (cdf[int(got) - 1] if got else 0.0)
        assert p > 0.0


def cdf_ranges(n, firsts=None):
    """(first, count) pairs of qsb_cdf ranges that start off 0 (at 1, 255, 256 and just past the middle by default) and
    end on a 4096-value block boundary, just past one, a few blocks on, or at the end."""
    N = 1 << n
    out = []
    for first in firsts or (1, 255, 256, N // 2 + 3):
        if first >= N:
            continue
        block_end = min(-(-(first + 1) // 4096) * 4096, N)
        for end in sorted({first + 1, block_end, block_end + 1, first + 3 * 4096 + 17, N}):
            if end <= N:
                out.append((first, end - first))
    return out


@pytest.mark.parametrize("precision", [F32, F64], ids=["f32", "f64"])
@pytest.mark.parametrize("n", [1, 5, 12, 13, 17, 21])
def test_cdf_and_shots_after_a_fused_circuit(n, precision):
    """The circuit leaves the qubits permuted inside the tile, so the logical-order gather is exercised."""
    circ = circuits.random_layered(n, depth=4, seed=100 + n) if n > 1 else [("h", (0,), ()), ("t", (0,), ())]
    with q.Simulator(n, precision=precision) as s:
        s.apply(q.gates_from_circuit(circ))
        state = s.state()
        cdf = s.compute_state_cumulative_distribution()
        want = oracle_cdf(state, n)
        assert np.max(np.abs(cdf - want)) < 1e-12
        assert np.all(np.diff(cdf) >= 0.0)                      # monotone like the serial sum
        assert abs(cdf[-1] - s.norm_argmax()[0]) < 1e-12
        part = s.compute_state_cumulative_distribution(first=0, count=(1 << n) // 2 + 1)
        assert np.array_equal(part, cdf[: (1 << n) // 2 + 1])
        for first, count in cdf_ranges(n):                       # a range is the slice of the global CDF, bit for bit
            part = s.compute_state_cumulative_distribution(first=first, count=count)
            assert np.array_equal(part, cdf[first:first + count]), (first, count, part[0], cdf[first], cdf[first] - cdf[first - 1])
        shots = s.measurement(48, seed=11 + n)
        check_shots(shots, cdf, n, 11 + n)
        assert np.array_equal(shots, s.measurement(48, seed=11 + n))   # seeded: reproducible


def test_cdf_of_a_given_state_matches_the_reference_rule():
    n = 14
    rng = np.random.default_rng(5)
    v = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)
    v[rng.random(1 << n) < 0.6] = 0.0                            # flat stretches: the "cdf != 0" clause matters
    v[:37] = 0.0
    v[-100:] = 0.0
    v /= np.linalg.norm(v)
    with q.Simulator(n, precision=F64) as s:
        s.set_state(v)
        cdf = s.compute_state_cumulative_distribution()
        want = oracle_cdf(v, n)
        assert np.max(np.abs(cdf - want)) < 1e-12
        shots = s.measurement(500, seed=3)
        check_shots(shots, cdf, n, 3)
        assert shots.min() >= 37 and shots.max() < (1 << n) - 100


def test_sampler_on_basis_and_bell_states():
    with q.Simulator(6, precision=F32) as s:
        assert np.all(s.measurement(32, seed=1) == 0)           # |0...0>: cdf is 1 everywhere, first index wins
        s.apply(q.gates_from_circuit([("x", (5,), ()), ("x", (1,), ())]))
        assert np.all(s.measurement(32, seed=1) == 34)
    nq, gates = 2, q.gates_from_circuit([("h", (0,), ()), ("cx", (0, 1), ())])     # entanglement.qasm
    with q.Simulator(nq, precision=F64) as s:
        s.apply(gates)
        shots = s.measurement(400, seed=9)
        assert set(shots.tolist()) == {0, 3}
        assert 140 < int(np.sum(shots == 0)) < 260


def test_shot_frequencies_follow_the_distribution():
    n, shots_n = 8, 40000
    circ = circuits.random_layered(n, depth=6, seed=77)
    with q.Simulator(n, precision=F64) as s:
        s.apply(q.gates_from_circuit(circ))
        p = s.probabilities()
        shots = s.measurement(shots_n, seed=2024)
    freq = np.bincount(shots.astype(np.int64), minlength=1 << n) / shots_n
    sigma = np.sqrt(p * (1 - p) / shots_n)
    assert np.all(np.abs(freq - p) < 6 * sigma + 1e-4)


@pytest.mark.parametrize("precision", [F32, F64], ids=["f32", "f64"])
def test_streaming_sampler_on_a_large_register(precision):
    """26 qubits: 2^14 segments, several per scan thread.  H on every qubit gives the uniform distribution,
    whose CDF is the index itself, so the shot for r must be close to r * 2^n -- no 2^n array on the host."""
    n = 26
    with q.Simulator(n, precision=precision) as s:
        s.apply(q.gates_from_circuit([("h", (k,), ()) for k in range(n)]))
        seed, count = 5, 64
        shots = s.measurement(count, seed=seed)
        for k in range(count):
            r = q.sample_uniform(seed, k)
            assert abs(float(shots[k]) + 1 - r * 2 ** n) <= 2 ** n * 1e-5 + 1
        # a structured state: only indices with bit 25 set and bit 0 clear survive
        s.reset()
        s.apply(q.gates_from_circuit([("x", (25,), ())] + [("h", (k,), ()) for k in range(1, 25)]))
        shots = s.measurement(count, seed=seed)
        assert np.all((shots >> np.uint64(25)) == 1) and np.all((shots & np.uint64(1)) == 0)
        for k in range(count):
            r = q.sample_uniform(seed, k)
            assert abs(float(shots[k] & np.uint64((1 << 25) - 1)) + 2 - r * 2 ** 25) <= 2 ** 25 * 1e-5 + 2


@pytest.mark.parametrize("precision", [F32, F64], ids=["f32", "f64"])
def test_shard_dump_and_reload_continue_the_run(precision, tmp_path):
    n = 16
    first = circuits.random_layered(n, depth=3, seed=1)
    second = circuits.random_layered(n, depth=3, seed=2)
    path = str(tmp_path / "shard.bin")
    with q.Simulator(n, precision=precision) as s:
        s.apply(q.gates_from_circuit(first))
        mid = s.state()
        s.save_state(path)
        s.apply(q.gates_from_circuit(second))
        end = s.state()
    assert os.path.getsize(path) == 128 + (1 << n) * (8 if precision == F32 else 16)
    with q.Simulator(n, precision=precision) as s:
        s.load_state(path)
        assert np.array_equal(s.state(), mid)                    # bit-exact, qubit map included
        s.apply(q.gates_from_circuit(second))
        assert np.array_equal(s.state(), end)
        assert np.max(np.abs(end - helpers.oracle_run_circuit(first + second, n))) <= TOL[precision]
    # shape mismatches and garbage are refused
    with q.Simulator(n + 1, precision=precision) as s:
        with pytest.raises(q.QsbError):
            s.load_state(path)
    with q.Simulator(n, precision=F64 if precision == F32 else F32) as s:
        with pytest.raises(q.QsbError):
            s.load_state(path)
    junk = str(tmp_path / "junk.bin")
    open(junk, "wb").write(b"\0" * 4096)
    with q.Simulator(n, precision=precision) as s:
        with pytest.raises(q.QsbError):
            s.load_state(junk)
        with pytest.raises(q.QsbError):
            s.load_state(str(tmp_path / "missing.bin"))
        open(junk, "wb").write(open(path, "rb").read()[:-16])
        with pytest.raises(q.QsbError):
            s.load_state(junk)


def test_cli_checkpoint_flags(tmp_path):
    n = 14
    first = circuits.random_layered(n, depth=2, seed=3)
    second = circuits.random_layered(n, depth=2, seed=4)
    fa, fb, fab = (str(tmp_path / f) for f in ("a.qasm", "b.qasm", "ab.qasm"))
    open(fa, "w").write(circuits.to_qasm(first, n))
    open(fb, "w").write(circuits.to_qasm(second, n))
    open(fab, "w").write(circuits.to_qasm(first + second, n))
    exe = os.path.join(helpers.ROOT, "gpu_quantum_simulator_b200", "bin", "qsim")
    ck, out1, out2 = (str(tmp_path / f) for f in ("ck.bin", "o1.bin", "o2.bin"))
    for args in ([fa, "--precision", "64", "--save-state", ck],
                 [fb, "--precision", "64", "--load-state", ck, "--dump-bin", out1],
                 [fab, "--precision", "64", "--dump-bin", out2]):
        r = subprocess.run([exe] + args, capture_output=True, text=True, timeout=120)
        assert r.returncode == 0, r.stdout
        float(r.stdout.splitlines()[0])
    a, b = np.fromfile(out1), np.fromfile(out2)
    assert a.size == 2 << n and np.max(np.abs(a - b)) <= 1e-12
    r = subprocess.run([exe, fb, "--load-state", str(tmp_path / "nope.bin")], capture_output=True, text=True, timeout=120)
    assert r.returncode == 1 and "cannot open state file" in r.stdout
