"""QASM front end (csrc/qasm.c) against the reference grammar (quantum_simulator.c:133-242). CPU only."""
import math
import os

import numpy as np
import pytest

import helpers
import gpu_quantum_simulator_b200 as q
from gpu_quantum_simulator_b200 import circuits


def mat(g):
    m = np.array(list(g.m)).reshape(4, 2)
    return (m[:, 0] + 1j * m[:, 1]).reshape(2, 2)


def test_bell_both_declaration_styles_and_crlf():
    for text in ('OPENQASM 3.0;\r\ninclude "stdgates.inc";\r\nqubit q[2];\r\nh q[0];\r\ncx q[0], q[1];\r\n',
                 'OPENQASM 3.0;\ninclude "stdgates.inc";\nqubit[2] q;\nh $0;\ncx $0, $1;\n'):
        n, g = q.parse_qasm_string(text)
        assert n == 2 and len(g) == 2
        assert g[0].target == 0 and g[0].controls == 0
        assert np.allclose(mat(g[0]), np.array([[1, 1], [1, -1]]) / math.sqrt(2))
        assert g[1].controls == 1 and g[1].target == 1          # first operand is the control (:229-235)
        assert np.array_equal(mat(g[1]), np.array([[0, 1], [1, 0]]))


def test_rz_is_the_phase_gate():
    n, g = q.parse_qasm_string('OPENQASM 3.0;\ninclude "stdgates.inc";\nqubit[1] q;\nrz(1.5707963267948966) q[0];\n')
    m = mat(g[0])
    assert m[0, 0] == 1 and m[0, 1] == 0 and m[1, 0] == 0
    assert m[1, 1] == complex(math.cos(1.5707963267948966), math.sin(1.5707963267948966))


def test_reference_gate_table_matches_oracle_table():
    L = helpers.oracle_lib()
    import ctypes as C
    for name in ["x", "sx", "z", "s", "sdg", "t", "tdg", "h", "y"]:
        n, g = q.parse_qasm_string(f'OPENQASM 3.0;\ninclude "stdgates.inc";\nqubit[1] q;\n{name} q[0];\n')
        m = (C.c_double * 8)()
        assert L.oc_gate_matrix(name.encode(), 0.0, m) == 0
        assert list(g[0].m) == list(m), name
    for name in ["rz", "rx", "ry", "p"]:
        n, g = q.parse_qasm_string(f'OPENQASM 3.0;\ninclude "stdgates.inc";\nqubit[1] q;\n{name}(-0.7321) q[0];\n')
        m = (C.c_double * 8)()
        assert L.oc_gate_matrix(name.encode(), -0.7321, m) == 0
        assert list(g[0].m) == list(m), name


def test_unknown_token_is_an_error_with_reference_wording():
    with pytest.raises(q.QsbError) as e:
        q.parse_qasm_string('OPENQASM 3.0;\ninclude "stdgates.inc";\nqubit[2] q;\nfoo q[0];\n')
    assert "Unknown token: foo" in str(e.value)


def test_missing_file():
    with pytest.raises(q.QsbError) as e:
        q.parse_qasm_file("/nonexistent/file.qasm")
    assert "cannot open circuit file" in str(e.value)


def test_operand_out_of_range_and_repeated_operand():
    with pytest.raises(q.QsbError):
        q.parse_qasm_string('OPENQASM 3.0;\ninclude "stdgates.inc";\nqubit[2] q;\nh q[2];\n')
    with pytest.raises(q.QsbError):
        q.parse_qasm_string('OPENQASM 3.0;\ninclude "stdgates.inc";\nqubit[2] q;\ncx q[1], q[1];\n')


def test_pi_expressions_comments_and_ignored_statements():
    text = ('OPENQASM 3.0;\ninclude "stdgates.inc";\n// comment\nqubit[3] q;\nbit[3] c;\n'
            'rx(pi/2) q[0];\nu(pi/2, 0, -pi / 4) q[1];\nbarrier q[0], q[1];\ncp(2*pi/8) q[0], q[2];\nc = measure q;\n')
    n, g = q.parse_qasm_string(text)
    assert n == 3 and len(g) == 3
    assert np.allclose(mat(g[0]), np.array([[1, -1j], [-1j, 1]]) / math.sqrt(2))
    assert g[2].controls == 1 and g[2].target == 2
    assert np.allclose(mat(g[2])[1, 1], np.exp(1j * math.pi / 4))


def test_cuda_variant_header():
    circ = [("h", (0,), ()), ("cx", (0, 1), ()), ("rz", (1,), (0.25,))]
    n, g = q.parse_qasm_string(circuits.to_cuda_variant_text(circ, 2))
    assert n == 2 and len(g) == 3


def test_swap_and_ccx():
    n, g = q.parse_qasm_string('OPENQASM 3.0;\ninclude "stdgates.inc";\nqubit[3] q;\nswap q[0], q[2];\nccx q[0], q[1], q[2];\n')
    assert len(g) == 4
    assert [(x.controls, x.target) for x in g] == [(1, 2), (4, 0), (1, 2), (3, 2)]


def test_shipped_files_parse(tmp_path):
    """The reference's two circuit files, rewritten from their fixtures in tests/golden/ with CRLF line ends as shipped."""
    for name, nq, ng in (("grover_3_18", 6, 2445), ("entanglement", 2, 2)):
        circ, n, _, _ = helpers.load_case(os.path.join(helpers.GOLDEN, name + ".npz"))
        path = tmp_path / (name + ".qasm")
        path.write_bytes(circuits.to_qasm(circ, n).replace("\n", "\r\n").encode())
        n, g = q.parse_qasm_file(path)
        assert n == nq and len(g) == ng


def test_writer_roundtrip_matches_generator():
    circ = circuits.random_superset(7, 120, seed=3)
    n, g = q.parse_qasm_string(circuits.to_qasm(circ, 7))
    g2 = q.gates_from_circuit(circ)
    assert n == 7 and len(g) == len(g2)
    for a, b in zip(g, g2):
        assert a.controls == b.controls and a.target == b.target and list(a.m) == list(b.m)


HDR = 'OPENQASM 3.0;\ninclude "stdgates.inc";\n'


def same_gates(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x.controls == y.controls and x.target == y.target
        assert np.allclose(list(x.m), list(y.m), atol=1e-15)


def test_gate_definitions_expand_with_parameters_and_nesting():
    text = HDR + '''qubit[3] q;
gate bell a, b { h a; cx a, b; }
gate twist(theta, phi) a, b { bell a, b; rz(theta / 2) a; rx(phi + pi) b; bell b, a; }
twist(0.5, -0.25) q[2], q[0];
'''
    flat = HDR + '''qubit[3] q;
h q[2]; cx q[2], q[0]; rz(0.25) q[2]; rx(-0.25 + pi) q[0]; h q[0]; cx q[0], q[2];
'''
    n, g = q.parse_qasm_string(text)
    n2, g2 = q.parse_qasm_string(flat)
    assert n == n2 == 3
    same_gates(g, g2)


def test_modifiers_ctrl_negctrl_inv_pow():
    n, g = q.parse_qasm_string(HDR + 'qubit[4] q;\nctrl @ x q[0], q[1];\nctrl(2) @ rz(0.3) q[0], q[1], q[2];\n'
                                     'inv @ s q[3];\npow(3) @ t q[3];\nnegctrl @ x q[2], q[0];\n')
    n2, g2 = q.parse_qasm_string(HDR + 'qubit[4] q;\ncx q[0], q[1];\nccrz(0.3) q[0], q[1], q[2];\nsdg q[3];\n'
                                       't q[3]; t q[3]; t q[3];\nx q[2]; cx q[2], q[0]; x q[2];\n')
    same_gates(g, g2)
    # inverse of a defined gate: reversed order, adjoint matrices; ctrl @ of a defined gate: every gate controlled
    text = HDR + 'qubit[3] q;\ngate g2(t) a, b { rx(t) a; cx a, b; s b; }\ninv @ g2(0.7) q[0], q[1];\nctrl @ g2(0.7) q[2], q[0], q[1];\n'
    flat = HDR + 'qubit[3] q;\nsdg q[1]; cx q[0], q[1]; rx(-0.7) q[0];\ncrx(0.7) q[2], q[0]; ccx q[2], q[0], q[1]; cs q[2], q[1];\n'
    same_gates(q.parse_qasm_string(text)[1], q.parse_qasm_string(flat)[1])


def test_gphase_registers_and_broadcast():
    n, g = q.parse_qasm_string(HDR + 'qubit[2] a;\nqubit[3] b;\nh a;\ncx a[1], b[2];\ngphase(0.5);\nctrl @ gphase(0.25) b[0];\ncx a, b[0];\n')
    assert n == 5
    assert [(x.controls, x.target) for x in g[:3]] == [(0, 0), (0, 1), (2, 4)]
    assert np.allclose(list(g[3].m), [math.cos(0.5), math.sin(0.5), 0, 0, 0, 0, math.cos(0.5), math.sin(0.5)])
    assert g[4].target == 2 and g[4].controls == 0 and np.allclose(list(g[4].m)[6:], [math.cos(0.25), math.sin(0.25)])
    assert [(x.controls, x.target) for x in g[5:]] == [(1, 2), (2, 2)]          # cx a, b[0] broadcasts over register a
    # a global phase changes the amplitudes, not the probabilities: check through the host interpreter of the plan
    circ_text = HDR + 'qubit[2] q;\nh q[0];\ngphase(0.5);\n'
    n, g = q.parse_qasm_string(circ_text)
    got, _ = helpers.hostcheck_run(g, n, 64)
    want = np.exp(0.5j) * np.array([1, 1, 0, 0]) / math.sqrt(2)
    assert np.max(np.abs(got - want)) < 1e-15


def test_front_end_errors_of_the_superset():
    for bad in ('qubit[2] q;\ngate g a { h a; }\ng q[0], q[1];\n',             # operand count
                'qubit[2] q;\ngate g(t) a { rz(t) a; }\ng q[0];\n',               # parameter count
                'qubit[2] q;\ngate r a { r a; }\nr q[0];\n',                      # recursion
                'qubit[2] q;\nctrl @ x q[0], q[0];\n',                            # control == target
                'qubit[2] q;\npow(0.5) @ x q[0];\n',                              # fractional power
                'qubit[2] q;\ngate g a { h b; }\ng q[0];\n'):                     # unknown qubit argument
        with pytest.raises(q.QsbError):
            q.parse_qasm_string(HDR + bad)


def test_cuda_variant_header_rejects_absurd_qubit_counts():
    for head in ("0 4", "63 4", "39999999999 4", "-3 4"):
        with pytest.raises((q.QsbError, Exception)):
            q.parse_qasm_string(head + "\nh q[0];\n")


def test_mutated_programs_never_yield_invalid_gates():
    """Robustness: random edits of valid programs either fail with a message or parse into gates whose target
    and controls lie inside the declared register (the reference exits on the first unknown token, :213)."""
    import ctypes as C
    import random
    rnd = random.Random(7)
    base = [
        'OPENQASM 3.0;\ninclude "stdgates.inc";\nqubit[4] q;\nh q[0];\ncx q[0], q[1];\nrz(0.5) q[2];\nsx q[3];\ntdg q[1];\n',
        'OPENQASM 3.0;\ninclude "stdgates.inc";\nqubit q[3];\nh $0;\ncx $0, $1;\nrz(1.25) $2;\n',
        'OPENQASM 3.0;\ninclude "stdgates.inc";\nqubit[3] a;\nqubit[2] b;\ngate foo(t) x, y { rx(t/2) x; cx x, y; p(pi*t) y; }\n'
        'foo(0.3) a[0], b[1];\nctrl @ inv @ foo(1) a[1], a[2], b[0];\npow(3) @ s a;\ngphase(0.1);\nnegctrl(2) @ x a[0], a[1], b[0];\n',
        '3 4\nh q[0];\ncx q[0], q[1];\nrz(0.5) q[2];\nx q[1];\n',
    ]
    tokens = ["q[", "]", "(", ")", ",", ";", "{", "}", "@", "pi", "ctrl", "gate", "qubit", "$", "9999999999", "-", "1e309", "/0",
              "inv", "pow(", "rz(", "\n", "\r\n", "//", "/*", "\"", "[" * 50, "(" * 50, "a" * 300, "q[-1]", "q[4]", "q[99999999999]"]
    parsed = failed = 0
    for _ in range(3000):
        s = rnd.choice(base)
        for _ in range(rnd.randint(1, 6)):
            k, pos = rnd.random(), rnd.randrange(len(s) + 1)
            if k < 0.3 and len(s) > 2:
                s = s[:pos] + s[min(len(s), pos + rnd.randint(1, 8)):]
            elif k < 0.7:
                s = s[:pos] + rnd.choice(tokens) + s[pos:]
            else:
                s = s[:pos] + chr(rnd.randint(1, 255)) + s[pos + 1:]
        nq, gp, n = C.c_int(), C.POINTER(q.Gate)(), C.c_size_t()
        rc = q.lib.qsb_parse_qasm_string(s.encode("latin-1", "replace"), C.byref(nq), C.byref(gp), C.byref(n))
        if rc == 0:
            parsed += 1
            assert 0 < nq.value <= 62
            for i in range(n.value):
                g = gp[i]
                assert 0 <= g.target < nq.value and not (g.controls >> nq.value) and not (g.controls >> g.target) & 1
            q.lib.qsb_free(gp)
        else:
            failed += 1
            assert q.lib.qsb_last_error()
    assert parsed > 100 and failed > 100


def test_cli_plan_only_needs_no_gpu(tmp_path):
    import json
    import subprocess
    path = tmp_path / "c.qasm"
    path.write_text(circuits.to_qasm(circuits.random_layered(30, 20, 12345), 30))
    exe = os.path.join(helpers.ROOT, "gpu_quantum_simulator_b200", "bin", "qsim")
    r = subprocess.run([exe, str(path), "--plan-only", "--gpus", "4"], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stdout
    d = json.loads(r.stdout)
    assert d["qubits"] == 30 and d["gates"] == 900 and d["ranks"] == 4 and d["exchanges"] >= 1 and 0 < d["passes"] < 60
    r = subprocess.run([exe, str(tmp_path / "missing.qasm"), "--plan-only"], capture_output=True, text=True, timeout=60)
    assert r.returncode == 1 and "cannot open circuit file" in r.stdout


HDR = 'OPENQASM 3.0;\ninclude "stdgates.inc";\n'


def test_statement_boundaries_follow_the_reference_tokenizer():
    """ADVICE r1: (a) a trailing comment with '=' must not turn a gate into a classical assignment, (b) an operand list
    may continue on the next line after a comma (the reference's streaming parser just reads on, :225-235)."""
    n, g = q.parse_qasm_string(HDR + "qubit[3] q;\nh q[0] // c = 1\ncx q[0],\n   q[1];\nx q[2]; /* y = 2 */ h q[2];\n")
    assert n == 3 and len(g) == 4
    assert [x.target for x in g] == [0, 1, 2, 2] and g[1].controls == 1
    n, g = q.parse_qasm_string(HDR + "qubit[2] q;\nbit[2] c;\nc[0] = measure q[0];\nh q[1];\n")
    assert len(g) == 1 and g[0].target == 1                       # a real assignment is still ignored


def test_controlled_gate_with_gphase_in_its_body():
    """ADVICE r1 (c): gphase inside a gate body has no operand; under ctrl @ it becomes a phase on the control, also
    when the control is qubit 0 (round 1 used a dummy target 0 and reported a control / operand clash)."""
    text = HDR + "qubit[2] q;\ngate foo a { gphase(0.5); h a; }\nctrl @ foo q[0], q[1];\n"
    n, g = q.parse_qasm_string(text)
    assert n == 2 and len(g) == 2
    ph, hh = g
    assert ph.target == 0 and ph.controls == 0
    assert np.allclose(mat(ph), np.diag([1, np.exp(0.5j)]))
    assert hh.target == 1 and hh.controls == 1
    want = np.zeros(4, complex); want[0] = 1                      # |00>: control off, nothing happens
    # oracle-free check of the two gates on |01> (control q0 = 1): e^{0.5i} (|0> + |1>)/sqrt(2) on q1
    v = np.zeros(4, complex); v[1] = 1
    v[1] *= np.exp(0.5j)
    out = v.copy(); out[1] = v[1] / math.sqrt(2); out[3] = v[1] / math.sqrt(2)
    assert abs(abs(out[1]) - 1 / math.sqrt(2)) < 1e-15


def test_pow_and_operand_range_overflows_are_rejected():
    """ADVICE r1: stacked pow modifiers used to wrap a 32-bit int (the gate was silently dropped); operand indices were
    truncated to int (q[4294967296] acted as q[0])."""
    with pytest.raises(q.QsbError, match="pow"):
        q.parse_qasm_string(HDR + "qubit[2] q;\npow(1000000) @ pow(1000000) @ x q[0];\n")
    n, g = q.parse_qasm_string(HDR + "qubit[2] q;\npow(3) @ pow(2) @ x q[0];\n")
    assert len(g) == 6
    for bad in ("x q[4294967296];", "x $4294967297;", "cx q[0], q[99999999999];"):
        with pytest.raises(q.QsbError):
            q.parse_qasm_string(HDR + "qubit[2] q;\n" + bad + "\n")


def test_non_seekable_input(tmp_path):
    """ADVICE r1 (medium): qsb_parse_qasm_file on a FIFO / pipe (ftell = -1) overflowed the heap; it now reads in a
    growing loop.  Parsed through a named pipe here."""
    import threading
    fifo = tmp_path / "c.fifo"
    os.mkfifo(fifo)
    text = HDR + "qubit[4] q;\n" + "".join(f"h q[{k % 4}];\n" for k in range(5000))     # > one 64 KiB read buffer
    t = threading.Thread(target=lambda: open(fifo, "w").write(text))
    t.start()
    n, g = q.parse_qasm_file(str(fifo))
    t.join()
    assert n == 4 and len(g) == 5000
