"""Rotation-angle gradients on one GPU: one JSON line.

After random_layered(30, 20) in f32 and f64 it times Simulator.rotation_gradient on two workloads:
  qaoa_ring_p4: QAOA MaxCut on a 30-qubit ring, p = 4 (per layer 30 ZZ cost rotations, then 30 X mixer rotations:
                240 rotations), H = sum of the 30 ZZ edges;
  random500:    500 random rotations of weight <= 4, H = 100 random terms of weight <= 4.
Each time is the median of >= 10 blocking calls after a warm-up call, host clock.  The line also gives the time of one
forward pass + energy through the existing calls (apply_pauli_rotations, then expectation), their ratio, and
2 * rotations x (forward + energy) as the computed (not measured) cost of the parameter-shift rule.

Byte model, in shard transfers (dry-run counts from the identity layout): forward 2 per rotation sweep, energy 1 per
expectation sweep, the copy psi -> phi 2, the H psi build 2 for its first sweep and 3 for each later one, every adjoint
sweep 4.  The peak is a measured device-to-device torch copy of 8 GiB (read + write bytes over time); the card name and
power limit come from nvidia-smi in the same run.

    python profiles/rotation_gradient_bench.py [--qubits 30] [--reps 10]
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


def random_strings(n, count, rng):
    out = []
    for _ in range(count):
        qs = rng.choice(n, int(rng.integers(1, 5)), replace=False)
        out.append(" ".join(f"{'XYZ'[rng.integers(3)]}{k}" for k in qs))
    return out


def workloads(n, seed=7):
    rng = np.random.default_rng(seed)
    ring = [f"Z{k} Z{(k + 1) % n}" for k in range(n)]
    qaoa = (ring + [f"X{k}" for k in range(n)]) * 4
    rand = random_strings(n, 500, rng)
    obs = random_strings(n, 100, rng)
    return {"qaoa_ring_p4": (qaoa, rng.uniform(-np.pi, np.pi, size=len(qaoa)), ring, np.ones(n)),
            "random500": (rand, rng.uniform(-np.pi, np.pi, size=500), obs, rng.normal(size=100))}


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--qubits", type=int, default=30)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("rotation_gradient_bench.py needs a CUDA device")
    n = args.qubits
    name, power = card()
    peak = copy_rate()
    res = {"bench": "rotation_gradient", "qubits": n, "gpu": name, "power_limit": power, "copy_rate_gbps": round(peak / 1e9, 1),
           "lib": q.lib.qsb_version().decode(), "circuit": f"random_layered({n}, 20)"}
    wl = workloads(n)
    circ = q.gates_from_circuit(circuits.random_layered(n, depth=20))
    for prec in (q.F32, q.F64):
        shard = (1 << n) * (8 if prec == q.F32 else 16)
        entry = {}
        for key, (rots, th, obs, coef) in wl.items():
            fwd = q.pauli_rotation_dry_run(n, rots, prec)["sweeps"]
            esw = q.expectation_dry_run(n, obs, prec)["sweeps"]
            g = q.rotation_gradient_dry_run(n, rots, obs, prec)
            transfers = 2 * fwd + esw + 2 + (2 + 3 * (g["apply_sweeps"] - 1)) + 4 * g["adjoint_sweeps"]
            with q.Simulator(n, precision=prec, device=0) as s:
                s.apply(circ)
                ms = timed(lambda: s.rotation_gradient(rots, th, obs, coef), args.reps)
                ms_fe = timed(lambda: (s.apply_pauli_rotations(rots, th), s.expectation(obs)), args.reps)
            nbytes = transfers * shard
            entry[key] = {"rotations": len(rots), "terms": len(obs), "forward_sweeps": fwd, "energy_sweeps": esw, **g,
                          "gradient_ms": round(ms, 3), "forward_energy_ms": round(ms_fe, 3),
                          "ratio_to_forward_energy": round(ms / ms_fe, 2), "model_bytes": nbytes,
                          "frac_copy_rate": round(nbytes / (ms * 1e-3) / peak, 3),
                          "parameter_shift_ms_computed": round(2 * len(rots) * ms_fe, 1)}
            print(key, prec, entry[key], file=sys.stderr, flush=True)
        res["f32" if prec == q.F32 else "f64"] = entry
    print(json.dumps(res))


if __name__ == "__main__":
    main()
