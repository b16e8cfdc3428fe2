"""Dense-matrix throughput on one GPU: one JSON line.

After random_layered(30, 20) in f32 and f64 it times Simulator.apply_matrices: the median of >= 10 blocking calls after a
warm-up call, host clock.
  1. One matrix of width k = 1..6 on qubits outside the low bits (20 .. 20 + k - 1).  Bytes = 2 x shard (one read and
     one write).  For k <= 5 the same operator also runs through QSB_MODE_DENSE (k_dense, one sweep per fused block): a
     random k-qubit circuit on those qubits is fused into one block with dense_k = k, its matrix is taken column by
     column on a small handle, and the two results are compared from the same product state (h and a phase on every
     qubit).  k_dense_ms is the host-clock time of that apply (fusion included), k_dense_device_ms its CUDA-event time.
  2. One quantum-volume layer: 15 random SU(4) on a random pairing, as one apply_matrices call and as 15 single-op
     calls, with the sweep counts of qsb_matrix_dry_run.
The peak is a measured device-to-device torch copy of 8 GiB (read + write bytes over time).

    python profiles/matrix_bench.py [--qubits 30] [--reps 10]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch
from scipy.stats import unitary_group

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gpu_quantum_simulator_b200 as q  # noqa: E402
from gpu_quantum_simulator_b200 import circuits  # noqa: E402
from pauli_rotation_bench import card, copy_rate, max_diff, timed  # noqa: E402


def circuit_matrix(sub, k):
    """The 2^k x 2^k matrix of a k-qubit circuit, column by column on an f64 handle."""
    cols = []
    with q.Simulator(k, precision=q.F64, device=0) as m:
        gates = q.gates_from_circuit(sub)
        for c in range(1 << k):
            e = np.zeros(1 << k, dtype=np.complex128)
            e[c] = 1
            m.set_state(e)
            m.apply(gates)
            cols.append(m.state())
    return np.stack(cols, axis=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--qubits", type=int, default=30)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("matrix_bench.py needs a CUDA device")
    n, reps = args.qubits, args.reps
    name, power = card()
    peak = copy_rate()
    res = {"bench": "matrix", "qubits": n, "gpu": name, "power_limit": power, "copy_rate_gbps": round(peak / 1e9, 1),
           "lib": q.lib.qsb_version().decode(), "circuit": f"random_layered({n}, 20)"}
    circ = q.gates_from_circuit(circuits.random_layered(n, depth=20))
    rng = np.random.default_rng(3)
    for prec in (q.F32, q.F64):
        shard = (1 << n) * (8 if prec == q.F32 else 16)
        entry = {"width": {}}
        s = q.Simulator(n, precision=prec, device=0)
        s.apply(circ)
        for k in range(1, 7):
            qs = list(range(20, 20 + k))
            sub = circuits.random_layered(k, depth=6, seed=k)
            U = circuit_matrix(sub, k)
            ms, _ = timed(lambda: s.apply_matrix(U, qs), reps)
            nbytes = 2 * shard
            row = {"ms": round(ms, 3), "bytes": nbytes, "gbps": round(nbytes / (ms * 1e-3) / 1e9, 1),
                   "frac_copy_rate": round(nbytes / (ms * 1e-3) / peak, 3),
                   "sweeps": q.matrix_dry_run(n, [qs], prec)["sweeps"]}
            if k <= 5:
                gates = q.gates_from_circuit([(g, [qs[x] for x in qq], p) for g, qq, p in sub])
                try:
                    d = q.Simulator(n, precision=prec, device=0, mode=q.MODE_DENSE, dense_k=k)
                except q.QsbError as e:
                    row["k_dense"] = f"refused: {e}"
                else:
                    # the same product state on both handles (h and a phase on every qubit), then the operator once
                    prep = q.gates_from_circuit([("h", [j], []) for j in range(n)] + [("rz", [j], [0.1 * j]) for j in range(n)])
                    ref_state = q.Simulator(n, precision=prec, device=0)
                    ref_state.apply(prep)
                    d.apply(prep)
                    st = d.apply(gates)
                    ref_state.apply_matrix(U, qs)
                    diff = max_diff(ref_state, d, 1.0, n)
                    ref_state.close()
                    ms_d, _ = timed(lambda: d.apply(gates), reps)
                    row.update({"k_dense_ms": round(ms_d, 3), "k_dense_passes": st["passes"],
                                "k_dense_device_ms": round(d.last_stats()["device_ms"], 3),
                                "speedup_vs_k_dense": round(ms_d / ms, 2), "max_abs_diff_vs_k_dense": diff})
                    d.close()
            entry["width"][k] = row
            print(prec, k, row, file=sys.stderr, flush=True)
        # one quantum-volume layer: 15 random SU(4) on a random pairing
        perm = rng.permutation(n)
        layer = []
        for j in range(n // 2):
            u = unitary_group.rvs(4, random_state=100 + j)
            layer.append((u / np.linalg.det(u) ** 0.25, [int(perm[2 * j]), int(perm[2 * j + 1])]))
        ms_one, _ = timed(lambda: s.apply_matrices(layer), reps)
        ms_each, _ = timed(lambda: [s.apply_matrices([op]) for op in layer], reps)
        sw_one = q.matrix_dry_run(n, [qq for _, qq in layer], prec)["sweeps"]
        entry["qv_layer"] = {"ops": len(layer), "one_call_ms": round(ms_one, 3), "one_call_sweeps": sw_one,
                             "single_calls_ms": round(ms_each, 3), "single_calls_sweeps": len(layer),
                             "one_call_gbps": round(sw_one * 2 * shard / (ms_one * 1e-3) / 1e9, 1),
                             "speedup": round(ms_each / ms_one, 2)}
        print(prec, entry["qv_layer"], file=sys.stderr, flush=True)
        s.close()
        res["f32" if prec == q.F32 else "f64"] = entry
    print(json.dumps(res))


if __name__ == "__main__":
    main()
