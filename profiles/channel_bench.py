"""Noise-channel throughput on one GPU: one JSON line, appended to --out.

After random_layered(30, 20), for f32 and f64, it times the median of --reps blocking Simulator.apply_channels calls
(host clock), each from the same state (restored by copy_from outside the timed window, after one warm-up call):
  (a) amplitude damping gamma = 0.01 on every qubit;
  (b) depolarizing p = 0.01 on every qubit;
  (c) ten two-qubit state-dependent channels (random Stinespring sets of 4 operators) on the overlapping pairs (k, k + 1).
r of channel c is sample_uniform(1, c).  For each case it records the dry-run counts and the launches the call makes by
construction (k_matrix sweeps write the shard, k_rdm launches only read it): one read per group, and the dry run's
sweeps, or for the all-fixed-weight case the matrix sweeps of the non-identity operators chosen.  Beside them it records
the largest count a torch.profiler trace of the call showed, which on the B200 is a lower bound (the trace can lack the
first kernels of a profiled region); the bench fails if that count ever exceeds the constructed one.  It records the
algorithmic bytes (a sweep reads
and writes the shard, a read reads it) and their rate against a measured device-to-device copy of 8 GiB; the
composition a caller could write from the existing calls (per channel reduced_density_matrix, the host rule, then
apply_matrix of the chosen operator; same r, same process), timed the same way (a warm-up call, then the median of
--reps calls from the restored state), the largest amplitude difference and whether the branches agree; and whether a
repeated call from the same state gives the same bytes.

    python profiles/channel_bench.py [--qubits 30] [--reps 10] [--out profiles/channel_bench.jsonl]
"""
import argparse
import json
import os
import statistics
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gpu_quantum_simulator_b200 as q  # noqa: E402
from gpu_quantum_simulator_b200 import circuits  # noqa: E402
from pauli_rotation_bench import card, copy_rate  # noqa: E402

NAME = {q.F32: "f32", q.F64: "f64"}


def stinespring(k, m, seed):
    rng = np.random.default_rng(seed)
    d = 1 << k
    a = rng.normal(size=(m * d, d)) + 1j * rng.normal(size=(m * d, d))
    v, _ = np.linalg.qr(a)
    return [v[i * d:(i + 1) * d, :] for i in range(m)]


def cases(n):
    return {"amplitude_damping": [(q.amplitude_damping(0.01), [k]) for k in range(n)],
            "depolarizing": [(q.depolarizing(0.01), [k]) for k in range(n)],
            "stinespring_pairs": [(stinespring(2, 4, 100 + k), [k, k + 1]) for k in range(10)]}


def compose(s, channels, rs):
    """Per channel: reduced_density_matrix of its targets, the rule of qsb_measure_qubits on the weights, apply_matrix."""
    bs = []
    for (kraus, ts), r in zip(channels, rs):
        rho = s.reduced_density_matrix(ts)
        w = [max(float(np.trace(K @ rho @ np.conj(K).T).real), 0.0) for K in map(np.asarray, kraus)]
        T = 0.0
        for x in w:
            T += x
        c, b = 0.0, len(w) - 1
        for i, x in enumerate(w):
            c += x
            if c != 0.0 and c >= r * T:
                b = i
                break
        s.apply_matrix(np.asarray(kraus[b]) * np.sqrt(T / w[b]), ts)
        bs.append(b)
    return np.array(bs, dtype=np.uint32)


def max_diff(a, b, n, chunk=1 << 26):
    d = 0.0
    for f in range(0, 1 << n, chunk):
        d = max(d, float(np.max(np.abs(a.state(f, chunk) - b.state(f, chunk)))))
    return d


def same_bytes(a, b, n, chunk=1 << 26):
    return all(np.array_equal(a.state_native(f, chunk), b.state_native(f, chunk)) for f in range(0, 1 << n, chunk))


def is_identity(K):
    K = np.asarray(K)
    return K[0, 0].real > 0 and np.array_equal(K, K[0, 0].real * np.eye(len(K)))


def expected_launches(n, chans, b, prec):
    """(sweeps, reads) the call must make: one read per group; the matrix sweeps of the chosen operators.  Every case
    here is either all state-dependent without identity operators (the dry run is exact) or all fixed-weight (one pending
    run of the non-identity operators, no read)."""
    dry = q.channel_dry_run(n, chans, prec)
    chosen = [chans[c][0][int(b[c])] for c in range(len(chans))]
    if dry["gram_sweeps"] == 0:
        ops = [chans[c][1] for c in range(len(chans)) if not is_identity(chosen[c])]
        return (q.matrix_dry_run(n, ops, prec)["sweeps"] if ops else 0), 0
    assert not any(is_identity(K) for K in chosen)
    return dry["sweeps"], dry["gram_sweeps"]


def profiled_launches(fn, want, attempts=3):
    """k_matrix and k_rdm kernels of one call seen by torch.profiler (kernel records of its trace, exported to a
    temporary file), the largest of `attempts` profiled calls.  On the B200 this count is a lower bound only: the trace
    has been seen to lack the first kernels of a profiled region: the first k_rdm of a call while it held the later ones,
    and torch's own marker kernels launched (and synchronised) before the call while it held the call's kernels.  So it is checked not to exceed `want`, the
    launches the call makes by construction, and it is recorded beside it.  -> (sweeps, reads)"""
    best = (0, 0)
    for _ in range(attempts):
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            torch.cuda.synchronize()
            fn()
            torch.cuda.synchronize()
        with tempfile.TemporaryDirectory() as d:
            path = os.path.join(d, "trace.json")
            prof.export_chrome_trace(path)
            with open(path) as f:
                names = [e["name"] for e in json.load(f)["traceEvents"] if e.get("cat") == "kernel"]
        got = (sum(x.startswith("void k_matrix<") for x in names), sum(x.startswith("void k_rdm<") for x in names))
        if got[0] > want[0] or got[1] > want[1]:
            raise SystemExit(f"the profiler saw {got} launches, more than the {tuple(want)} the call makes")
        best = max(best, got, key=sum)
        if best == tuple(want):
            break
    return best


def timed_from(base, s, fn, reps):
    """fn() once to warm up, then the median of reps calls, each after s.copy_from(base) outside the timed window."""
    s.copy_from(base)
    fn()
    ts = []
    out = None
    for _ in range(reps):
        s.copy_from(base)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return ts, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--qubits", type=int, default=30)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "channel_bench.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("channel_bench.py needs a CUDA device")
    n, reps = args.qubits, args.reps
    name, power = card()
    peak = copy_rate()
    res = {"bench": "channels", "qubits": n, "gpu": name, "power_limit": power, "copy_rate_gbps": round(peak / 1e9, 1),
           "lib": q.lib.qsb_version().decode(), "circuit": f"random_layered({n}, 20, seed=1)", "reps": reps,
           "r": "sample_uniform(1, c)"}
    circ = q.gates_from_circuit(circuits.random_layered(n, depth=20, seed=1))
    for prec in (q.F32, q.F64):
        sb = (1 << n) * (8 if prec == q.F32 else 16)
        with q.Simulator(n, precision=prec, device=0) as base, q.Simulator(n, precision=prec, device=0) as s, \
                q.Simulator(n, precision=prec, device=0) as c:
            base.apply(circ)
            for case, chans in cases(n).items():
                rs = [q.sample_uniform(1, i) for i in range(len(chans))]
                ts, (b, p) = timed_from(base, s, lambda: s.apply_channels(chans, r=rs), reps)
                ms = statistics.median(ts)
                c.copy_from(base)
                nw, nr = want = expected_launches(n, chans, b, prec)
                seen = profiled_launches(lambda: c.apply_channels(chans, r=rs), want)
                c.copy_from(base)
                c.apply_channels(chans, r=rs)
                same = bool(same_bytes(s, c, n))                 # s and c: the same call from the same state
                ts_c, bc = timed_from(base, c, lambda: compose(c, chans, rs), reps)
                ms_c = statistics.median(ts_c)
                dry = q.channel_dry_run(n, chans, prec)
                nbytes = (2 * nw + nr) * sb
                res[f"{case}_{NAME[prec]}"] = {
                    "ms": round(ms, 3), "ms_min": round(min(ts), 3), "ms_max": round(max(ts), 3),
                    "launches_writing": nw, "launches_read_only": nr, "launches_profiled_lower_bound": list(seen),
                    "dry_run": dry,
                    "non_identity_branches": int(sum(not is_identity(chans[i][0][int(b[i])]) for i in range(len(chans)))),
                    "bytes": nbytes, "gbps": round(nbytes / (ms * 1e-3) / 1e9, 1),
                    "frac_copy_rate": round(nbytes / (ms * 1e-3) / peak, 3),
                    "composition_ms": round(ms_c, 3), "composition_ms_min": round(min(ts_c), 3),
                    "composition_ms_max": round(max(ts_c), 3), "speedup_vs_composition": round(ms_c / ms, 2),
                    "branches_equal_composition": bool(np.array_equal(b, bc)),
                    "max_abs_diff_composition": max_diff(s, c, n), "repeat_bit_identical": same}
                print(json.dumps({case: res[f"{case}_{NAME[prec]}"]}), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    with open(args.out, "a") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
