"""Reduced-density-matrix throughput on one GPU: one JSON line.

After random_layered(30, 20) in f32 and f64 it times Simulator.reduced_density_matrix for k = 1, 2, 4, 6, 8, 10 and 12
qubits (the k = 4 set holds the qubit on the first lane position, physical bit 1 in f32 / 0 in f64): the median of
>= 10 blocking calls after a warm-up call, host clock, the host-side assembly of rho included.

Model per call, shard = 2^n * B (B = 8 f32 / 16 f64 bytes per amplitude), nb = max(1, 2^k / 64) row blocks of the kernel:
  bytes  nb * shard                 (the upper block triangle: every block row is read once per block pair it is in)
  flops  4 * 2^n * (2^k + 1)        (the Hermitian rank update, upper triangle)
The bytes bound is a measured device-to-device torch copy of 8 GiB (expectation_bench.copy_rate); the flops bound is a
measured complex128 torch matmul of two 8192 x 8192 matrices (a cuBLAS rate on this card, not the hardware peak).  Each
entry says which bound is the larger and the share of it the call reached.  For k <= 2 the line also times
marginal_probabilities of the same set (one read of the shard) and reports the ratio.

A torch baseline copies the state into a complex128 tensor, permutes it to (2^k, 2^(n-k)) and computes M @ M.mH; the
line reports its time (the permute included), its agreement with the library and the speedup.

    python profiles/rdm_bench.py [--qubits 30] [--reps 10]
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

KS = (1, 2, 4, 6, 8, 10, 12)


def zgemm_rate(m=8192, reps=5):
    a = torch.randn(m, m, dtype=torch.complex128, device="cuda")
    b = torch.randn(m, m, dtype=torch.complex128, device="cuda")
    torch.matmul(a, b)
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        torch.matmul(a, b)
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    del a, b
    torch.cuda.empty_cache()
    return 8.0 * m ** 3 / statistics.median(ts)


def qubit_sets(n, perm, prec):
    lane = int(np.flatnonzero(perm[:n] == (1 if prec == q.F32 else 0))[0])
    rng = np.random.default_rng(1)
    others = [qb for qb in rng.permutation(n).tolist() if qb != lane]
    return {f"k{k}": ([lane] + others[:3] if k == 4 else others[:k]) for k in KS}


def torch_baseline(a, n, qubits):
    keep = [n - 1 - qb for qb in reversed(qubits)]
    rest = [ax for ax in range(n) if ax not in keep]

    def run():
        m = a.reshape((2,) * n).permute(keep + rest).reshape(1 << len(qubits), -1)
        return (m @ m.mH).cpu().numpy()
    return timed(run, 3)


def model(n, k, prec):
    shard = (1 << n) * (8 if prec == q.F32 else 16)
    return max(1, (1 << k) // 64) * shard, 4.0 * (1 << n) * ((1 << k) + 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--qubits", type=int, default=30)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("rdm_bench.py needs a CUDA device")
    n = args.qubits
    name, power = card()
    peak = copy_rate()
    zrate = zgemm_rate()
    res = {"bench": "rdm", "qubits": n, "gpu": name, "power_limit": power, "copy_rate_gbps": round(peak / 1e9, 1),
           "zgemm_rate_gflops_cublas": round(zrate / 1e9, 1), "lib": q.lib.qsb_version().decode(),
           "circuit": f"random_layered({n}, 20)"}
    for prec in (q.F32, q.F64):
        sim = q.Simulator(n, precision=prec, device=0)
        sim.apply(q.gates_from_circuit(circuits.random_layered(n, depth=20)))
        perm, _ = sim.layout()
        sets = qubit_sets(n, perm, prec)
        out = {"sets": sets}
        a = torch.from_numpy(sim.state()).to("cuda")
        for key, qs in sets.items():
            k = len(qs)
            ms, rho = timed(lambda: sim.reduced_density_matrix(qs), args.reps)
            again = sim.reduced_density_matrix(qs)
            nbytes, flops = model(n, k, prec)
            t_bytes, t_flops = nbytes / peak, flops / zrate
            e = {"ms": round(ms, 3), "bytes": int(nbytes), "flops": flops, "gbps": round(nbytes / (ms * 1e-3) / 1e9, 1),
                 "gflops": round(flops / (ms * 1e-3) / 1e9, 1), "bound": "bytes" if t_bytes >= t_flops else "flops",
                 "share_of_bound": round(max(t_bytes, t_flops) / (ms * 1e-3), 3),
                 "repeat_bit_identical": bool(np.array_equal(rho.view(np.uint64), again.view(np.uint64)))}
            if k <= 2:
                ms_m, _ = timed(lambda: sim.marginal_probabilities(qs), args.reps)
                e["marginal_ms"] = round(ms_m, 3)
                e["over_marginal"] = round(ms / ms_m, 2)
            ms_t, base = torch_baseline(a, n, qs)
            e["torch_ms"] = round(ms_t, 2)
            e["speedup_vs_torch"] = round(ms_t / ms, 2)
            e["max_abs_diff_vs_torch"] = float(np.max(np.abs(base - rho)))
            del base
            out[key] = e
        del a
        torch.cuda.empty_cache()
        res["f32" if prec == q.F32 else "f64"] = out
        sim.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
