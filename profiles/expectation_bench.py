"""Expectation-value throughput on one GPU: one JSON line.

After random_layered(30, 20) in f32 and f64 it times Simulator.expectation on four workloads (one Z term, the
transverse-field Ising Hamiltonian of 59 terms, 1000 random strings of weight <= 4, X on every qubit): the median
of >= 10 blocking calls after a warm-up call, host clock.  Bytes read = sweeps x shard bytes (a sweep reads the state
once; the sweep count is that of qsb_expectation_dry_run from the identity layout, the layout after the circuit is
permuted and may group a little differently).  The peak is a measured device-to-device torch copy of 8 GiB (read +
write bytes over time).  A torch baseline downloads the state once into a complex tensor and evaluates each Ising
term with an index gather, a sign and vdot; the line reports its agreement with the library and the speedup.

    python profiles/expectation_bench.py [--qubits 30] [--reps 10]
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
    return {"z1": ["Z0"],
            "ising59": [f"X{k}" for k in range(n)] + [f"Z{k} Z{k + 1}" for k in range(n - 1)],
            "random1000": rand,
            "x_all": [" ".join(f"X{k}" for k in range(n))]}


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); out = fn(); ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts), out


def torch_baseline(sim, n, terms, prec):
    """Index gather + sign + vdot per term on a complex copy of the state (downloaded once)."""
    a = torch.from_numpy(sim.state()).to("cuda", torch.complex64 if prec == q.F32 else torch.complex128)
    j = torch.arange(1 << n, device="cuda", dtype=torch.int64)
    x, z = q.pauli_masks(terms, n)

    def run():
        out = []
        for xx, zz in zip(x.tolist(), z.tolist()):
            jx = torch.bitwise_xor(j, xx) if xx else j
            b = a[jx] if xx else a
            par = None
            for k in range(n):
                if (zz >> k) & 1:
                    bit = torch.bitwise_and(torch.bitwise_right_shift(jx, k), 1)
                    par = bit if par is None else torch.bitwise_xor(par, bit)
            if par is not None:
                b = b * (1 - 2 * par).to(b.real.dtype)
            y = bin(xx & zz).count("1") % 4
            out.append(float(((1j ** y) * torch.vdot(a, b)).real))
        torch.cuda.synchronize()
        return np.array(out)
    try:
        return timed(run, 3)
    finally:
        del a, j
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--qubits", type=int, default=30)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("expectation_bench.py needs a CUDA device")
    n = args.qubits
    name, power = card()
    peak = copy_rate()
    res = {"bench": "expectation", "qubits": n, "gpu": name, "power_limit": power, "copy_rate_gbps": round(peak / 1e9, 1),
           "lib": q.lib.qsb_version().decode(), "circuit": f"random_layered({n}, 20)"}
    wl = workloads(n)
    for prec in (q.F32, q.F64):
        sim = q.Simulator(n, precision=prec, device=0)
        sim.apply(q.gates_from_circuit(circuits.random_layered(n, depth=20)))
        shard = (1 << n) * (8 if prec == q.F32 else 16)
        entry = {}
        for key, terms in wl.items():
            sweeps = q.expectation_dry_run(n, terms, prec)["sweeps"]
            ms, vals = timed(lambda: sim.expectation(terms), args.reps)
            again = sim.expectation(terms)
            entry[key] = {"terms": len(terms), "sweeps": sweeps, "ms": round(ms, 3), "bytes_read": sweeps * shard,
                          "gbps": round(sweeps * shard / (ms * 1e-3) / 1e9, 1),
                          "frac_copy_rate": round(sweeps * shard / (ms * 1e-3) / peak, 3),
                          "terms_per_s": round(len(terms) / (ms * 1e-3), 1),
                          "repeat_bit_identical": bool(np.array_equal(vals.view(np.uint64), again.view(np.uint64)))}
        ms_t, base = torch_baseline(sim, n, wl["ising59"], prec)
        lib_vals = sim.expectation(wl["ising59"])
        entry["torch_baseline_ising59"] = {"ms": round(ms_t, 1), "speedup": round(ms_t / entry["ising59"]["ms"], 1),
                                           "max_abs_diff": float(np.max(np.abs(base - lib_vals)))}
        res["f32" if prec == q.F32 else "f64"] = entry
        sim.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
