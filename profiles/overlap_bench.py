"""Overlap and copy throughput on one GPU: one JSON line, appended to --out.

At 30 qubits it times the median of --reps blocking calls after a warm-up call, host clock:
  1. Simulator.overlap of f32/f32 and f64/f64 pairs with equal layouts (b filled by copy_from(a)) and with different
     layouts (random_layered(30, 20) with two seeds; the layouts are recorded as differing or not).
  2. f32 against f64 after the same circuit, with the fidelity between them (the cost of running in f32).
  3. Simulator.copy_from in both precisions.
Bytes = both shards read once (overlap) or one shard read and written (copy).  The peak is a measured device-to-device
torch copy of 8 GiB (read + write bytes over time).

    python profiles/overlap_bench.py [--qubits 30] [--reps 10] [--out profiles/overlap_bench.jsonl]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gpu_quantum_simulator_b200 as q  # noqa: E402
from gpu_quantum_simulator_b200 import circuits  # noqa: E402
from pauli_rotation_bench import card, copy_rate, timed  # noqa: E402

NAME = {q.F32: "f32", q.F64: "f64"}


def shard_bytes(n, prec):
    return (1 << n) * (8 if prec == q.F32 else 16)


def row(ms, nbytes, peak, **extra):
    r = {"ms": round(ms, 3), "bytes": nbytes, "gbps": round(nbytes / (ms * 1e-3) / 1e9, 1),
         "frac_copy_rate": round(nbytes / (ms * 1e-3) / peak, 3)}
    r.update(extra)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--qubits", type=int, default=30)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "overlap_bench.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("overlap_bench.py needs a CUDA device")
    n, reps = args.qubits, args.reps
    name, power = card()
    peak = copy_rate()
    res = {"bench": "overlap", "qubits": n, "gpu": name, "power_limit": power, "copy_rate_gbps": round(peak / 1e9, 1),
           "lib": q.lib.qsb_version().decode(), "circuits": f"random_layered({n}, 20, seed=1 / 2)", "reps": reps}
    c1 = q.gates_from_circuit(circuits.random_layered(n, depth=20, seed=1))
    c2 = q.gates_from_circuit(circuits.random_layered(n, depth=20, seed=2))
    for prec in (q.F32, q.F64):
        sb = shard_bytes(n, prec)
        with q.Simulator(n, precision=prec, device=0) as a, q.Simulator(n, precision=prec, device=0) as b:
            a.apply(c1)
            ms, _ = timed(lambda: b.copy_from(a), reps)
            res[f"copy_{NAME[prec]}"] = row(ms, 2 * sb, peak)
            ms, ov = timed(lambda: a.overlap(b), reps)
            res[f"equal_layout_{NAME[prec]}"] = row(ms, 2 * sb, peak, overlap=[ov.real, ov.imag])
            b.reset()
            b.apply(c2)
            differ = not np.array_equal(a.layout()[0][:n], b.layout()[0][:n])
            ms, ov = timed(lambda: a.overlap(b), reps)
            res[f"different_layout_{NAME[prec]}"] = row(ms, 2 * sb, peak, layouts_differ=differ, overlap=[ov.real, ov.imag])
        print(res, file=sys.stderr, flush=True)
    with q.Simulator(n, precision=q.F32, device=0) as a, q.Simulator(n, precision=q.F64, device=0) as b:
        a.apply(c1)
        b.apply(c1)
        ms, ov = timed(lambda: a.overlap(b), reps)
        res["f32_vs_f64"] = row(ms, shard_bytes(n, q.F32) + shard_bytes(n, q.F64), peak, overlap=[ov.real, ov.imag],
                                fidelity=a.fidelity(b), one_minus_fidelity=1.0 - a.fidelity(b),
                                layouts_differ=not np.array_equal(a.layout()[0][:n], b.layout()[0][:n]))
    line = json.dumps(res)
    print(line)
    with open(args.out, "a") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
