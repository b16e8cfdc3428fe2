"""Pauli-rotation throughput on one GPU: one JSON line.

After random_layered(30, 20) in f32 and f64 it times Simulator.apply_pauli_rotations on four workloads (one Trotter
step of the transverse-field Ising chain: 29 ZZ + 30 X; 1000 diagonal ZZ rotations; 1000 random rotations of weight
<= 4; one rotation of X on every qubit): the median of >= 10 blocking calls after a warm-up call, host clock.  Bytes =
sweeps x 2 x shard bytes (a sweep reads and writes the state once; the sweep count is that of
qsb_pauli_rotation_dry_run from the identity layout, the layout after the circuit is permuted and may group a little
differently).  The peak is a measured device-to-device torch copy of 8 GiB (read + write bytes over time).

The in-library baseline is the same rotations lowered to gates and run through Simulator.apply: per rotation the basis
change (h for X, sdg h for Y), a CX ladder onto the last qubit of the string, the phase gate p(theta) there, the ladder
and the basis change undone.  That product equals the rotation up to exp(-i theta / 2), which the comparison
multiplies in; the line reports its time, its passes and the largest amplitude difference between the two states.

    python profiles/pauli_rotation_bench.py [--qubits 30] [--reps 10]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gpu_quantum_simulator_b200 as q  # noqa: E402
from gpu_quantum_simulator_b200 import circuits  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power = (r.stdout.strip().split(",") + ["?"])[:2]
    return name.strip(), power.strip()


def copy_rate(nbytes=8 << 30, reps=10):
    src = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda").uniform_()
    dst = torch.empty_like(src)
    dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(reps):
        e0.record(); dst.copy_(src); e1.record(); torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    del src, dst
    torch.cuda.empty_cache()
    return 2 * nbytes / (statistics.median(times) * 1e-3)


def workloads(n, seed=7):
    rng = np.random.default_rng(seed)
    rand = []
    for _ in range(1000):
        qs = rng.choice(n, int(rng.integers(1, 5)), replace=False)
        rand.append(" ".join(f"{'XYZ'[rng.integers(3)]}{k}" for k in qs))
    zz = []
    for _ in range(1000):
        a, b = rng.choice(n, 2, replace=False)
        zz.append(f"Z{a} Z{b}")
    out = {"ising_step": [f"Z{k} Z{k + 1}" for k in range(n - 1)] + [f"X{k}" for k in range(n)],
           "zz1000": zz, "random1000": rand, "x_all": [" ".join(f"X{k}" for k in range(n))]}
    return {k: (v, rng.uniform(-np.pi, np.pi, size=len(v))) for k, v in out.items()}


def lowered(paulis, thetas, n):
    """(gate list, global phase) whose product equals the rotations."""
    circ, phase = [], 1.0 + 0j
    x, z = q.pauli_masks(paulis, n)
    for xx, zz, t in zip(x.tolist(), z.tolist(), thetas):
        qs = [k for k in range(n) if ((xx | zz) >> k) & 1]
        phase *= np.exp(-0.5j * t)
        if not qs:
            continue
        basis = []
        for k in qs:
            if (xx >> k) & 1 and (zz >> k) & 1:
                basis += [("sdg", (k,), ()), ("h", (k,), ())]
            elif (xx >> k) & 1:
                basis += [("h", (k,), ())]
        undo = [("s" if g == "sdg" else g, k, p) for g, k, p in reversed(basis)]
        ladder = [("cx", (qs[i], qs[i + 1]), ()) for i in range(len(qs) - 1)]
        circ += basis + ladder + [("p", (qs[-1],), (float(t),))] + ladder[::-1] + undo
    return q.gates_from_circuit(circ), phase


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); out = fn(); ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts), out


def max_diff(s1, s2, phase, n, chunk=1 << 24):
    d = 0.0
    for f in range(0, 1 << n, chunk):
        d = max(d, float(np.max(np.abs(s1.state(f, chunk) - phase * s2.state(f, chunk)))))
    return d


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--qubits", type=int, default=30)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("pauli_rotation_bench.py needs a CUDA device")
    n = args.qubits
    name, power = card()
    peak = copy_rate()
    res = {"bench": "pauli_rotation", "qubits": n, "gpu": name, "power_limit": power, "copy_rate_gbps": round(peak / 1e9, 1),
           "lib": q.lib.qsb_version().decode(), "circuit": f"random_layered({n}, 20)"}
    wl = workloads(n)
    circ = q.gates_from_circuit(circuits.random_layered(n, depth=20))
    for prec in (q.F32, q.F64):
        shard = (1 << n) * (8 if prec == q.F32 else 16)
        entry = {}
        for key, (paulis, th) in wl.items():
            sweeps = q.pauli_rotation_dry_run(n, paulis, prec)["sweeps"]
            gates, phase = lowered(paulis, th, n)
            s1 = q.Simulator(n, precision=prec, device=0)
            s2 = q.Simulator(n, precision=prec, device=0)
            s1.apply(circ)
            s2.apply(circ)
            s1.apply_pauli_rotations(paulis, th)   # one call each from the same state, for the comparison
            st = s2.apply(gates)
            diff = max_diff(s1, s2, phase, n)
            s2.close()
            ms, _ = timed(lambda: s1.apply_pauli_rotations(paulis, th), args.reps)
            ms_g, _ = timed(lambda: s1.apply(gates), args.reps)
            s1.close()
            nbytes = sweeps * 2 * shard
            entry[key] = {"rotations": len(paulis), "sweeps": sweeps, "ms": round(ms, 3), "bytes": nbytes,
                          "gbps": round(nbytes / (ms * 1e-3) / 1e9, 1), "frac_copy_rate": round(nbytes / (ms * 1e-3) / peak, 3),
                          "lowered_gates": len(gates), "lowered_ms": round(ms_g, 3), "lowered_passes": st["passes"],
                          "speedup_vs_lowered": round(ms_g / ms, 2), "max_abs_diff_vs_lowered": diff}
            print(key, prec, entry[key], file=sys.stderr, flush=True)
        res["f32" if prec == q.F32 else "f64"] = entry
    print(json.dumps(res))


if __name__ == "__main__":
    main()
