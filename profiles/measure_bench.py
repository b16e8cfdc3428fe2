"""Marginal and projective-measurement throughput on one GPU: one JSON line.

After random_layered(30, 20) in f32 and f64 it times Simulator.marginal_probabilities for k = 1, 4, 10 and 20 (the k = 4
set holds the qubit on the first lane position, physical bit 1 in f32 / 0 in f64), collapse for k = 1 and 4,
measure_qubits for k = 4 and reset_qubits for k = 1: the median of >= 10 blocking calls after a warm-up call, host clock.
Repeated collapses and measurements land on the same outcome and do the same work as the first; before each timed reset
an untimed X puts the qubit back into |1>, so every reset measures 1 and applies its X.

Modelled bytes per call, shard = N_loc * B (B = 8 f32 / 16 f64 bytes per amplitude), K = 2^-k:
  marginal        shard                       (one read)
  collapse        (1 + 2K) * shard            (read of the kept amplitudes for p, then read kept + write all)
  measure_qubits  (2 + K) * shard             (marginal, then the collapse pass)
  reset_qubits    (2 + K) * shard + the X plan's bytes_moved
The peak is a measured device-to-device torch copy of 8 GiB (read + write bytes over time, expectation_bench.copy_rate).
A torch baseline copies the state into a complex tensor once and computes abs()**2, reshaped and summed over the
unmeasured dimensions, for the k = 4 set; the line reports its agreement with the library and the speedup.

    python profiles/measure_bench.py [--qubits 30] [--reps 10]
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import gpu_quantum_simulator_b200 as q  # noqa: E402
from gpu_quantum_simulator_b200 import circuits  # noqa: E402
from expectation_bench import card, copy_rate, timed  # noqa: E402


def qubit_sets(n, perm, prec):
    lane = int(np.flatnonzero(perm[:n] == (1 if prec == q.F32 else 0))[0])
    rng = np.random.default_rng(1)
    others = [qb for qb in rng.permutation(n).tolist() if qb != lane]
    return {"k1": [n - 1], "k4": [lane] + others[:3], "k10": others[:10], "k20": others[:20]}


def torch_baseline(sim, n, qubits, prec):
    a = torch.from_numpy(sim.state()).to("cuda", torch.complex64 if prec == q.F32 else torch.complex128)
    keep = [n - 1 - qb for qb in qubits]
    rest = sorted(keep)
    order = [rest.index(keep[i]) for i in reversed(range(len(qubits)))]

    def run():
        m = (a.abs() ** 2).reshape((2,) * n).sum(dim=tuple(ax for ax in range(n) if ax not in keep))
        out = m.permute(order).reshape(-1).double().cpu().numpy()
        return out
    try:
        return timed(run, 3)
    finally:
        del a
        torch.cuda.empty_cache()


def entry(ms, nbytes, peak):
    return {"ms": round(ms, 3), "bytes": int(nbytes), "gbps": round(nbytes / (ms * 1e-3) / 1e9, 1),
            "frac_copy_rate": round(nbytes / (ms * 1e-3) / peak, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--qubits", type=int, default=30)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("measure_bench.py needs a CUDA device")
    n = args.qubits
    name, power = card()
    peak = copy_rate()
    res = {"bench": "measure", "qubits": n, "gpu": name, "power_limit": power, "copy_rate_gbps": round(peak / 1e9, 1),
           "lib": q.lib.qsb_version().decode(), "circuit": f"random_layered({n}, 20)"}
    for prec in (q.F32, q.F64):
        sim = q.Simulator(n, precision=prec, device=0)
        sim.apply(q.gates_from_circuit(circuits.random_layered(n, depth=20)))
        perm, _ = sim.layout()
        shard = (1 << n) * (8 if prec == q.F32 else 16)
        sets = qubit_sets(n, perm, prec)
        out = {"sets": sets}
        for key, qs in sets.items():
            ms, vals = timed(lambda: sim.marginal_probabilities(qs), args.reps)
            again = sim.marginal_probabilities(qs)
            out["marginal_" + key] = dict(entry(ms, shard, peak), repeat_bit_identical=bool(np.array_equal(vals.view(np.uint64), again.view(np.uint64))))
        ms_t, base = torch_baseline(sim, n, sets["k4"], prec)
        lib_k4 = sim.marginal_probabilities(sets["k4"])
        out["torch_baseline_k4"] = {"ms": round(ms_t, 2), "speedup": round(ms_t / out["marginal_k4"]["ms"], 1),
                                    "max_abs_diff": float(np.max(np.abs(base - lib_k4)))}
        for key in ("k1", "k4"):
            qs = sets[key]
            outcome = int(np.argmax(sim.marginal_probabilities(qs)))
            ms, _ = timed(lambda: sim.collapse(qs, outcome), args.reps)
            out["collapse_" + key] = entry(ms, (1 + 2.0 ** (1 - len(qs))) * shard, peak)
        qs = sets["k4"]
        ms, _ = timed(lambda: sim.measure_qubits(qs, 0.5), args.reps)
        out["measure_k4"] = entry(ms, (2 + 2.0 ** -len(qs)) * shard, peak)
        qs = sets["k1"]
        x = q.gates_from_circuit([("x", (qs[0],), ())])
        ts, xbytes = [], 0
        sim.reset_qubits(qs, 0.5)                     # the qubit is |0> from here on
        for i in range(args.reps + 1):
            sim.apply(x)
            t0 = time.perf_counter()
            b = sim.reset_qubits(qs, 0.5)
            dt = (time.perf_counter() - t0) * 1e3
            assert b == 1
            xbytes = sim.last_stats()["bytes_moved"]
            if i:
                ts.append(dt)
        out["reset_k1"] = dict(entry(statistics.median(ts), 2.5 * shard + xbytes, peak), x_bytes_moved=int(xbytes))
        res["f32" if prec == q.F32 else "f64"] = out
        sim.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
