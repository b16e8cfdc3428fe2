"""Pin the CPU checker: restatement (oracle/qsim_oracle.c) vs the outputs of the unmodified reference
program stored in tests/golden/ (oracle/make_golden.py) and vs circuits it runs itself.  CPU only."""
import math
import os

import numpy as np
import pytest

import helpers
from gpu_quantum_simulator_b200 import circuits


def golden(name):
    return helpers.load_case(os.path.join(helpers.GOLDEN, name + ".npz"))


def golden_with_note(note):
    return [os.path.basename(p)[:-4] for p in helpers.golden_cases() if helpers.load_case(p)[3] == note]


def oracle_run_text(text, tmp_path, phi=0.0):
    """The restatement on a QASM file with this text, times the global phase e^{i phi}."""
    path = tmp_path / "c.qasm"
    path.write_bytes(text.encode())
    n, v = helpers.oracle_run_file(path)
    return n, v * complex(math.cos(phi), math.sin(phi))


def test_known_answers_bell():
    v = helpers.oracle_run_circuit([("h", (0,), ()), ("cx", (0, 1), ())], 2)
    r = 0.70710678118654746          # SURVEY.md §8c, printed by the reference in the build container
    assert v[0] == r and v[3] == r and v[1] == 0 and v[2] == 0


@pytest.mark.parametrize("name", ["entanglement.qasm", "grover_3_18.qasm"])
def test_restatement_equals_reference_on_shipped_files(name, tmp_path):
    """The reference's two circuit files, rewritten from the stored fixture with CRLF line ends as shipped, through
    the restatement's file reader: bit-identical to the reference's own run of them."""
    circ, n, amps, _ = golden(name[:-5])
    n1, a = oracle_run_text(circuits.to_qasm(circ, n).replace("\n", "\r\n"), tmp_path)
    assert n1 == n
    assert np.array_equal(a, amps), "restatement must be bit-identical to quantum_simulator.c"


def test_grover_known_values():
    _, _, v, _ = golden("grover_3_18")
    p = np.abs(v) ** 2
    assert abs(p[3] - 0.49959115777166263) < 1e-15 and abs(p[18] - 0.49959115777166119) < 1e-15
    assert set(np.argsort(p)[-2:]) == {3, 18}


@pytest.mark.parametrize("name", golden_with_note("reference gate set"))
def test_restatement_equals_reference_on_random_reference_gate_circuits(name, tmp_path):
    circ, n, amps, _ = golden(name)
    _, a = oracle_run_text(circuits.to_qasm(circ, n), tmp_path)
    assert np.array_equal(a, amps)
    assert np.array_equal(a, helpers.oracle_run_circuit(circ, n))


@pytest.mark.parametrize("n,ng,seed", [(3, 60, 5), (8, 250, 6), (12, 300, 7)])
def test_superset_gates_match_reference_through_identities(n, ng, seed, tmp_path):
    """rx/ry/y/cz/cp/swap/ccx are not in the reference's gate set: the restatement's native
    versions must equal the reference run on the exact respelling (times the dropped phase).  The
    restatement stands in for the reference on the respelling, a file in the reference's gate set:
    the test above pins it bit-identical to the reference's stored outputs on such files."""
    circ = circuits.random_superset(n, ng, seed)
    a = helpers.oracle_run_circuit(circ, n)
    text, phi = circuits.to_reference_qasm(circ, n)
    _, b = oracle_run_text(text, tmp_path, phi)
    assert np.max(np.abs(a - b)) < 1e-13


def test_oracle_file_parser_accepts_both_declarations_and_dollar_operands(tmp_path):
    t1 = 'OPENQASM 3.0;\r\ninclude "stdgates.inc";\r\nqubit[3] q;\r\nh q[0];\r\ncx q[0], q[2];\r\nrz(0.5) q[2];\r\n'
    t2 = 'OPENQASM 3.0;\ninclude "stdgates.inc";\nqubit q[3];\nh $0;\ncx $0, $2;\nrz(0.5) $2;\n'
    p1, p2 = tmp_path / "a.qasm", tmp_path / "b.qasm"
    p1.write_bytes(t1.encode()); p2.write_bytes(t2.encode())
    _, a = helpers.oracle_run_file(p1)
    _, b = helpers.oracle_run_file(p2)
    assert np.array_equal(a, b)
    want = helpers.oracle_run_circuit([("h", (0,), ()), ("cx", (0, 2), ()), ("rz", (2,), (0.5,))], 3)
    assert np.array_equal(a, want)


@pytest.mark.parametrize("path", helpers.golden_cases(), ids=lambda p: os.path.basename(p)[:-4])
def test_restatement_matches_golden_vectors(path):
    circ, n, amps, note = helpers.load_case(path)
    got = helpers.oracle_run_circuit(circ, n)
    if "reference gate set" in note or "reference file" in note:
        assert np.array_equal(got, amps)
    else:
        assert np.max(np.abs(got - amps)) < 1e-13


def test_golden_dir_is_populated():
    assert len(helpers.golden_cases()) >= 10


def test_cdf_and_measure_rule():
    L = helpers.oracle_lib()
    v = helpers.oracle_run_circuit([("h", (0,), ()), ("cx", (0, 1), ())], 2)
    cdf = np.zeros(4)
    L.oc_cdf(v.ctypes.data, 2, cdf.ctypes.data)
    assert cdf[0] == pytest.approx(0.5, abs=1e-15) and cdf[1] == cdf[0] and cdf[3] == pytest.approx(1.0, abs=1e-15)
    assert L.oc_measure(cdf.ctypes.data, 2, 0.25) == 0
    assert L.oc_measure(cdf.ctypes.data, 2, 0.75) == 3      # skips the flat part, like the reference
    assert L.oc_measure(cdf.ctypes.data, 2, 2.0) == 3       # clamps at the last index
