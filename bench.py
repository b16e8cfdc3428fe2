#!/usr/bin/env python
"""bench.py -- gates/sec and effective HBM GB/s of the state-vector apply path (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--qubits n] [--precision 32|64] [--dump-outputs DIR]

A "step" is one execution of the whole fused circuit (all passes) on the device-resident state.
Workload at every N: random_layered(34 q, depth 20, seed 12345), f32 -- BASELINE.json's "34q (1/2/4/8 B200)"
configuration, so that the driver's 1 -> 8 GPU scaling compares like with like (strong scaling; 128 GiB
in place on one B200, sharded on the top log2(N) qubits under torchrun).  At N = 1 the line also carries
"at_30q": the same measurement on the 30 q circuit, the size BASELINE.json's single-GPU target is quoted on.
Rank 0 prints ONE JSON line (see the task contract): value = source gates / second, whole job;
roofline = achieved algorithmic bytes/s of the tile-pass kernel vs the measured HBM peak;
e2e = the same metric through the public API with host buffers (QASM text in; norm, arg max and the
first 2^20 amplitudes out);
cpu_baseline = the reference's own C program (oracle/_ref/ref_cexe) on a bounded sample.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 12345
DEPTH = 20
# --dump-outputs: 256 runs of 2^13 consecutive amplitudes = 2^21 amplitudes, 16 MiB (f32) or 32 MiB (f64), plus 16 MiB of indices
DUMP_RUNS, DUMP_RUN_BITS = 256, 13


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------ CPU reference arm
def load_circuits():
    """The circuit generators WITHOUT importing the package: the reference arm must not map libqsim_b200.so
    (VERDICT r1: the package __init__ loads the library as an import side effect)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("qsb_circuits", os.path.join(ROOT, "gpu_quantum_simulator_b200", "circuits.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def reference_full_depth(n_workload, n_s=22):
    """The UNMODIFIED reference program on the WHOLE depth-20 circuit at n_s qubits (about 20 s of one core at 22 q):
    a real run, not a one-layer sample; gates/s at the workload size is that figure scaled by 2^(n_s - n) and
    labelled extrapolated (one sweep per gate: cost is linear in the state size; BASELINE.md section 3)."""
    circuits = load_circuits()
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_cexe")
    if not os.path.exists(exe):
        raise RuntimeError("oracle/_ref/ref_cexe missing (build it in the container: make -C oracle)")
    circ = circuits.random_layered(n_s, DEPTH, SEED)
    ref, _ = circuits.to_reference_gates(circ)
    with tempfile.TemporaryDirectory() as d:
        p1 = os.path.join(d, "full.qasm")
        open(p1, "w").write(circuits.to_qasm(ref, n_s))
        t = float(subprocess.run([exe, p1, "0"], capture_output=True, text=True, check=True).stdout.split()[0])
    measured = len(circ) / t
    return {"value": measured * 2.0 ** (n_s - n_workload), "unit": "gates/s", "cores": 1, "kind": "reference",
            "sample": (f"full depth-{DEPTH} random_layered({n_s}q, seed {SEED}): {len(circ)} source gates = {len(ref)} reference-set gates "
                       f"through oracle/_ref/ref_cexe (unmodified quantum_simulator.c, gcc -O2, 1 thread), its own stdout line; "
                       f"value = measured gates/s scaled by 2^({n_s}-{n_workload}) to the {n_workload}q workload (extrapolated)"),
            "measured": {"qubits": n_s, "seconds": t, "gates_per_sec": measured},
            "host_cores_available": os.cpu_count(), "sample_seconds": t, "sample_qubits": n_s}, t


def reference_sample(n_workload, step_budget_s, reps=1):
    """Time the UNMODIFIED reference program on the first layer of random_layered at the largest
    n_s <= n_workload that fits the budget; scale gates/s by 2^(n_s - n_workload) (cost is linear in
    the state size: one sweep per gate)."""
    circuits = load_circuits()
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_cexe")
    kind = "reference"
    if not os.path.exists(exe):
        raise RuntimeError("oracle/_ref/ref_cexe missing (build it in the container: make -C oracle)")
    try:
        avail = int([l for l in open("/proc/meminfo") if l.startswith("MemAvailable")][0].split()[1]) * 1024
    except Exception:
        avail = 8 << 30
    per_amp_gate = 5.0e-9                      # measured in the build container (BASELINE.md)
    n_s = n_workload
    while n_s > 16:
        layer_gates = n_s * 2                  # ~ one transpiled layer incl. CX
        if (16 << n_s) * 1.25 < avail and layer_gates * per_amp_gate * (1 << n_s) <= step_budget_s:
            break
        n_s -= 1
    full = circuits.random_layered(n_s, DEPTH, SEED)
    layer = full[: n_s + n_s // 2]             # first layer: n_s one-qubit gates + n_s/2 CX
    ref_layer, _ = circuits.to_reference_gates(layer)
    text = circuits.to_qasm(ref_layer, n_s)
    one = circuits.to_qasm(ref_layer[:1], n_s)   # the reference cannot parse a gate-less file; time 1 gate instead
    R = len(ref_layer)
    times = []
    with tempfile.TemporaryDirectory() as d:
        p1, p0 = os.path.join(d, "layer.qasm"), os.path.join(d, "one.qasm")
        open(p1, "w").write(text); open(p0, "w").write(one)
        for _ in range(reps):
            t_full = float(subprocess.run([exe, p1, "0"], capture_output=True, text=True, check=True).stdout.split()[0])
            t_one = float(subprocess.run([exe, p0, "0"], capture_output=True, text=True, check=True).stdout.split()[0])
            # its timer includes malloc + |0> init (:143,:168-177): remove it with the 1-gate run
            times.append(max((t_full - t_one) * R / (R - 1), 1e-9))
    t = sorted(times)[len(times) // 2]
    src_gates = len(layer)
    value = src_gates / t * 2.0 ** (n_s - n_workload)
    sample = (f"first layer ({src_gates} source gates = {R} reference-set gates) of "
              f"random_layered({n_s}q, seed {SEED}) through oracle/_ref/ref_cexe (gcc -O2, 1 thread), init time subtracted; "
              f"gates/s scaled by 2^({n_s}-{n_workload}) to the {n_workload}q workload")
    return {"value": value, "unit": "gates/s", "cores": 1, "kind": kind, "sample": sample,
            "host_cores_available": os.cpu_count(), "sample_seconds": t, "sample_qubits": n_s}, t


def run_reference_gpu(circuits, sizes=(28, 30)):
    """oracle/_ref/ref_4x4 = /root/reference/quantum_simulator_4x4.cu, UNMODIFIED, nvcc -arch=sm_100a (oracle/Makefile): the reference's
    fastest CUDA variant on the same B200, fed the reference-gate spelling of the same circuits in its own "<num_q> <num_g>" format
    (quantum_simulator_4x4.cu:293-529).  Its one stdout line is end to end (parse, malloc, cudaMalloc, kernels, D2H of both planes);
    launches are counted by an LD_PRELOAD shim (oracle/launch_count.c).  It drops fused gates within 1e-3 of identity and is not a
    numerical oracle (SURVEY F10): only its time is reported."""
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_4x4")
    shim = os.path.join(ROOT, "oracle", "_ref", "liblaunchcount.so")
    if not os.path.exists(exe):
        return {"unavailable": "oracle/_ref/ref_4x4 missing (built by make -C oracle where /root/reference and nvcc exist)"}
    out = {"program": "oracle/_ref/ref_4x4 (unmodified quantum_simulator_4x4.cu, nvcc -arch=sm_100a -O2)", "runs": {}}
    for n in sizes:
        circ = circuits.random_layered(n, DEPTH, SEED)
        ref, _ = circuits.to_reference_gates(circ)
        with tempfile.TemporaryDirectory() as d:
            p = os.path.join(d, "c.txt")
            open(p, "w").write(circuits.to_cuda_variant_text(ref, n))
            env = dict(os.environ)
            if os.path.exists(shim):
                env["LD_PRELOAD"] = shim
            try:
                r = subprocess.run([exe, p], capture_output=True, text=True, env=env, timeout=300)
                secs = float(r.stdout.split()[0])
                launches = None
                for ln in r.stderr.splitlines():
                    if ln.startswith("launches="):
                        launches = int(ln.split("=")[1])
                out["runs"][f"{n}q"] = {"seconds_end_to_end": secs, "gates_per_sec": len(circ) / secs, "source_gates": len(circ),
                                        "reference_set_gates": len(ref), "kernel_launches": launches}
            except Exception as e:
                out["runs"][f"{n}q"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    return out


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.qubits or 34
    budget = max(1.0, min(20.0, 150.0 / max(1, args.steps + args.warmup)))
    vals, secs, base = [], [], None
    for i in range(args.warmup + args.steps):
        base, t = reference_full_depth(n) if budget >= 19.0 else reference_sample(n, budget)
        if i >= args.warmup:
            vals.append(base["value"]); secs.append(t)
    value = sum(vals) / len(vals)
    base["value"] = value
    line = {"impl": "reference", "metric": "gates_per_sec", "value": value, "unit": "gates/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(secs) / len(secs),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"random_layered_{n}q_d{DEPTH}", "qubits": n, "depth": DEPTH, "seed": SEED},
            "cpu_baseline": base,
            "e2e": {"value": value, "unit": "gates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------- our arm
def dump_outputs(out_dir, sim):
    """The state the last timed step left, as a fixed sample: DUMP_RUNS runs of 2^DUMP_RUN_BITS consecutive logical
    amplitudes at seeded positions (the whole state when it is no larger).  state.npy holds one (re, im) row per
    amplitude in the device precision, state_index.npy the logical index of each row."""
    import numpy as np
    n = sim.num_qubits
    bits = min(DUMP_RUN_BITS, n)
    runs = 1 << (n - bits)
    picked = np.arange(runs) if runs <= DUMP_RUNS else np.sort(np.random.default_rng(SEED).choice(runs, DUMP_RUNS, replace=False))
    firsts = [int(r) << bits for r in picked]
    amps = np.concatenate([sim.state_native(f, 1 << bits) for f in firsts]).reshape(-1, 2)
    index = np.concatenate([np.arange(f, f + (1 << bits), dtype=np.float64) for f in firsts])
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "state.npy"), amps)
    np.save(os.path.join(out_dir, "state_index.npy"), index)


def run_ours(args):
    import numpy as np
    import torch
    import gpu_quantum_simulator_b200 as q
    from gpu_quantum_simulator_b200 import circuits

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch multi-GPU runs with torch.distributed.run (one rank per GPU)")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs reads the state of a single-GPU run")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    prec = q.F64 if args.precision == 64 else q.F32
    amp_bytes = 16 if prec == q.F64 else 8
    peak, peak_src = load_peaks()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def make_sim(n, prec=prec):
        sim = q.Simulator(n, precision=prec, rank=rank, world_size=world, device=local_rank, low_bits=args.low_bits,
                          reserved=[0, args.no_lazy_diag, args.trim, args.cost_cap, args.res4, args.fused, args.no_sink])
        if world > 1:
            from gpu_quantum_simulator_b200 import dist as qdist
            qdist.init_comm(sim, dist)
        return sim

    def measure(n, steps, warmup, with_clocks, prec=prec, workload=args.workload):
        """-> dict with the device-timed numbers of random_layered(n) and the live objects (sim, plan, circ)."""
        amp_bytes = 16 if prec == q.F64 else 8
        circ = circuits.random_layered(n, DEPTH, SEED) if workload == "layered" else circuits.qft(n)
        gates = q.gates_from_circuit(circ)
        sim = make_sim(n, prec)
        plan = sim.plan(gates)
        pst = plan.stats()
        for _ in range(max(warmup, 3)):
            sim.reset()                      # a plan addresses the layout it was made for (|0..0>, identity map)
            sim.execute(plan)
        sampler = ClockSampler(local_rank)
        barrier()
        if rank == 0 and with_clocks:
            sampler.start()
        dev_ms = xch_ms = 0.0
        t0 = time.perf_counter()
        for _ in range(steps):
            sim.reset()                      # untimed on the device clock: device_ms brackets the passes only
            st = sim.execute(plan)           # device_ms: CUDA events on the launching stream, first pass -> last pass
            dev_ms += st["device_ms"]; xch_ms += st["exchange_ms"]
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        clocks = sampler.stop() if (rank == 0 and with_clocks) else None
        t = torch.tensor([dev_ms, wall_ms, xch_ms], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, wall_ms, xch_ms = (float(x) for x in t.cpu())
        ms_per_step = dev_ms / steps
        # roofline of the dominant kernel (k_tile_pass): algorithmic bytes per launch / average launch time
        n_loc_amps = (1 << n) // world
        bytes_per_launch = 2 * n_loc_amps * amp_bytes
        pass_ms = (dev_ms - xch_ms) / steps / max(pst["passes"], 1)
        achieved = bytes_per_launch / (pass_ms * 1e-3) / 1e9
        traffic = None
        tfile = os.path.join(ROOT, "profiles", "traffic_per_launch.json")
        if os.path.exists(tfile):
            try:
                tj = json.load(open(tfile))
                traffic = tj.get(f"{n}q_f{32 if prec == q.F32 else 64}_{world}gpu_{workload}") or tj.get(f"{n}q_f{32 if prec == q.F32 else 64}_{world}gpu")
                if traffic is None and "dram_over_algorithmic" in tj:
                    traffic = tj["dram_over_algorithmic"] * bytes_per_launch
            except Exception:
                traffic = None
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic, "kernel": "k_tile_pass", "bytes_per_launch": bytes_per_launch,
                    "avg_launch_ms": pass_ms, "peak_source": peak_src,
                    "launches_per_circuit": pst["passes"], "rounds_per_launch": pst["rounds"] / max(pst["passes"], 1),
                    "note": "one launch fuses ~45 gates in ~6 register/shared-memory rounds, so it runs longer than a stream of its 2*N*B bytes; "
                            "the planner minimises circuit time (fewer, deeper launches lower this fraction while gates/s rise); "
                            "at_30q.shallow_fusion is the same kernel with the fusion depth capped (HBM-bound regime)"}
        # second limit of the same kernel (DESIGN.md 3.1): every round but the first of a pass moves the whole tile
        # through shared memory once in each direction; peak = SMs x 128 B/clk x SM clock
        try:
            props = torch.cuda.get_device_properties(local_rank)
            smem_peak = props.multi_processor_count * 128 * (props.clock_rate * 1e3) / 1e9          # GB/s at the max SM clock
            exchanges = max(pst["rounds"] - pst["passes"], 0)
            smem_bytes = exchanges * bytes_per_launch
            smem_achieved = smem_bytes / ((dev_ms - xch_ms) / steps * 1e-3) / 1e9
            roofline["shared_memory"] = {"achieved": smem_achieved, "peak": smem_peak, "unit": "GB/s", "frac": smem_achieved / smem_peak,
                                         "exchanges_per_circuit": exchanges, "bytes_per_exchange": bytes_per_launch}
        except Exception:
            pass
        return {"n": n, "circ": circ, "sim": sim, "plan": plan, "pst": pst, "ms_per_step": ms_per_step,
                "value": len(circ) / (ms_per_step * 1e-3), "wall_ms": wall_ms, "xch_ms": xch_ms, "clocks": clocks,
                "roofline": roofline, "n_loc_amps": n_loc_amps}

    # ---- world > 1: correctness of the sharded path at this revision, BEFORE anything is timed (VERDICT r1, task 1a)
    parity = None
    if world > 1:
        from gpu_quantum_simulator_b200 import dist as qdist
        pn, pdepth, pseed, tol = 24, 8, 777, 1e-5
        pcirc = circuits.random_layered(pn, pdepth, pseed)
        pg = q.gates_from_circuit(pcirc)
        ssim = make_sim(pn)                                  # default exchange flavour of this world size
        pst = ssim.apply(pg)
        got = qdist.gather_state(ssim, dist)                 # logical order, every rank
        ssim.close()
        err = 0.0
        if rank == 0:
            with q.Simulator(pn, precision=prec, device=local_rank) as one:   # the same circuit unsharded, same GPU
                one.apply(pg)
                err = float(np.max(np.abs(got - one.state())))
        et = torch.tensor([err], dtype=torch.float64, device="cuda")
        dist.broadcast(et, 0)
        err = float(et.cpu()[0])
        parity = {"n": pn, "depth": pdepth, "seed": pseed, "what": "sharded run (default exchange flavour) vs the same circuit on one GPU, full state",
                  "exchanges": int(pst["swaps"]), "max_abs_err": err, "tol": tol, "ok": bool(err <= tol)}
        del got
        if not parity["ok"]:
            if rank == 0:
                print(json.dumps({"metric": "gates_per_sec", "value": None, "n_gpus": world, "parity": parity, "error": "sharded parity failed"}))
            dist.barrier(); dist.destroy_process_group()
            raise SystemExit(3)

    # workload: 34 q at every N (strong scaling); smaller only if the state does not fit
    n = args.qubits or 34
    m = None
    while m is None:
        try:
            m = measure(n, args.steps, args.warmup, True)
        except q.QsbError as e:
            if args.qubits or "Malloc" not in str(e) or n <= 30:
                raise
            n -= 1
    circ, sim, plan, pst = m["circ"], m["sim"], m["plan"], m["pst"]
    ms_per_step, value, wall_ms, xch_ms, clocks, roofline = (m[k] for k in ("ms_per_step", "value", "wall_ms", "xch_ms", "clocks", "roofline"))
    n_loc_amps = m["n_loc_amps"]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, sim)

    # ---- e2e: QASM text (host) -> parse -> plan (H2D) -> |0> -> execute -> result to host memory
    e2e = None
    if not args.no_e2e:
        text = circuits.to_qasm(circ, n)
        head = min(1 << 20, n_loc_amps)
        host = torch.empty(2 * head, dtype=torch.float64, pin_memory=True).numpy()
        e2e_steps = max(1, min(args.steps, 3))
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            nq, g2 = q.parse_qasm_string(text)
            sim.reset()
            p2 = sim.plan(g2)
            sim.execute(p2)
            norm, amax, pmax = sim.norm_argmax()              # D2H: per-block partial sums / maxima
            sim.shard_head(head, out=host)                    # D2H: the first 2^20 local amplitudes (fp64 pairs)
            p2.close()
        barrier()
        e2e_s = (time.perf_counter() - t0) / e2e_steps
        te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_s = float(te.cpu()[0])
        tn = torch.tensor([norm], dtype=torch.float64, device="cuda")     # per-rank partial of sum |a|^2
        if dist is not None:
            dist.all_reduce(tn, op=dist.ReduceOp.SUM)
        norm_total = float(tn.cpu()[0])
        if abs(norm_total - 1.0) > 1e-3:
            raise SystemExit(f"norm check failed after the e2e run: sum |a|^2 = {norm_total}")
        e2e = {"value": len(circ) / e2e_s, "unit": "gates/s",
               "h2d_bytes_per_step": int(len(text) + pst["passes"] * 4000),
               "d2h_bytes_per_step": int(head * 16 + 148 * 4 * 32), "seconds_per_step": e2e_s,
               "what": "qsb_parse_qasm_string + qsb_plan_create + qsb_reset + qsb_execute + qsb_norm_argmax + "
                       "first 2^20 local amplitudes to pinned host memory; pass descriptors travel as kernel parameters"}

    # ---- N = 1: the 30 q circuit, the size the single-GPU target is quoted on
    at_30q = None
    if world == 1 and n != 30 and not args.qubits and not args.no_30q:
        plan.close(); sim.close()
        m30 = measure(30, max(3, min(args.steps, 10)), 3, False)
        at_30q = {"workload": f"random_layered_30q_d{DEPTH}", "value": m30["value"], "unit": "gates/s",
                  "ms_per_step": m30["ms_per_step"], "passes": m30["pst"]["passes"], "rounds": m30["pst"]["rounds"],
                  "roofline": m30["roofline"]}
        plan, sim = m30["plan"], m30["sim"]
        # the same circuit with the fusion depth capped (more, lighter passes): the HBM-bound regime of the kernel
        if not args.cost_cap:
            plan.close(); sim.close()
            args.cost_cap = 12
            ms = measure(30, max(3, min(args.steps, 10)), 3, False)
            args.cost_cap = 0
            at_30q["shallow_fusion"] = {"cost_cap": 12, "value": ms["value"], "unit": "gates/s", "ms_per_step": ms["ms_per_step"],
                                        "passes": ms["pst"]["passes"], "rounds": ms["pst"]["rounds"], "roofline": ms["roofline"]}
            plan, sim = ms["plan"], ms["sim"]

    # ---- N = 1: every BASELINE.json configuration gets a driver-timed number in the same run (VERDICT r1, task 6)
    configs = e2e_full = reference_gpu = None
    if world == 1 and not args.qubits and not args.no_30q and not args.no_extras:
        plan.close(); sim.close()
        configs = {}
        for name, cn, cprec, cwl in (("random_layered_28q_f32", 28, q.F32, "layered"), ("qft_30q_f32", 30, q.F32, "qft"),
                                     ("qft_30q_f64", 30, q.F64, "qft"), ("random_layered_30q_f64", 30, q.F64, "layered"),
                                     ("random_layered_32q_f32", 32, q.F32, "layered")):
            try:
                mc = measure(cn, 3, 3, False, prec=cprec, workload=cwl)
            except q.QsbError as e:
                configs[name] = {"error": str(e)}
                continue
            configs[name] = {"ms_per_step": mc["ms_per_step"], "value": mc["value"], "unit": "gates/s", "source_gates": len(mc["circ"]),
                             "passes": mc["pst"]["passes"], "rounds": mc["pst"]["rounds"], "frac": mc["roofline"]["frac"],
                             "achieved_GBps": mc["roofline"]["achieved"], "dtype": "f32" if cprec == q.F32 else "f64", "steps": 3, "warmup": 3}
            mc["plan"].close(); mc["sim"].close()
        # ---- honest e2e at 30 q: QASM text in, the ENTIRE state (2^30 amplitudes, device dtype) out to pinned host memory,
        #      as the reference programs copy the whole state back (naive.cu:193-194, 4x4.cu:512-513)
        try:
            c30 = circuits.random_layered(30, DEPTH, SEED)
            text30 = circuits.to_qasm(c30, 30)
            host = torch.empty(2 << 30, dtype=torch.float32, pin_memory=True).numpy()
            s30 = make_sim(30, q.F32)
            secs, dl = [], []
            for _ in range(2):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                nq, g30 = q.parse_qasm_string(text30)
                s30.reset()
                p30 = s30.plan(g30)
                s30.execute(p30)
                t1 = time.perf_counter()
                s30.state_native(out=host)                      # qsb_download_native: double-buffered export + D2H
                t2 = time.perf_counter()
                p30.close()
                secs.append(t2 - t0); dl.append(t2 - t1)
            nrm = float(np.dot(host[: 1 << 24].astype(np.float64), host[: 1 << 24].astype(np.float64)))
            e2e_full = {"workload": f"random_layered_30q_d{DEPTH}", "value": len(c30) / min(secs), "unit": "gates/s", "seconds_per_step": min(secs),
                        "h2d_bytes_per_step": len(text30), "d2h_bytes_per_step": int(host.nbytes), "download_seconds": min(dl),
                        "download_GBps": host.nbytes / min(dl) / 1e9, "head_norm_check": nrm,
                        "what": "qsb_parse_qasm_string + qsb_plan_create + qsb_reset + qsb_execute + qsb_download_native of all 2^30 amplitudes (8 GiB, f32) into pinned host memory"}
            s30.close(); del host
        except Exception as e:   # e.g. not enough pinned host memory on the box
            e2e_full = {"error": str(e)}
        # ---- the reference's own fastest CUDA variant on this GPU (BASELINE.md section 3 "courtesy baseline")
        reference_gpu = run_reference_gpu(circuits)
        sim = make_sim(20); plan = sim.plan(q.gates_from_circuit(circuits.random_layered(20, 2, 1)))   # placeholders for the common close below

    line = None
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu:
            try:
                cpu, _ = reference_full_depth(n)
            except Exception as e:   # keep the bench line even if the checker binary is missing
                cpu = {"value": None, "unit": "gates/s", "cores": 1, "kind": "reference", "sample": f"unavailable: {e}"}
        line = {"metric": "gates_per_sec", "value": value, "unit": "gates/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32" if prec == q.F32 else "f64", "data": "synthetic",
                "config": {"workload": f"random_layered_{n}q_d{DEPTH}" if args.workload == "layered" else f"qft_{n}q_after_h_layer",
                           "qubits": n, "depth": DEPTH, "seed": SEED, "source_gates": len(circ), "passes": pst["passes"], "rounds": pst["rounds"], "swaps": pst["swaps"],
                           "l2": "inputs larger than L2 (state = %d MiB per GPU)" % (n_loc_amps * amp_bytes >> 20),
                           "parallelism": f"shard{world}" if world > 1 else "single"},
                "effective_gate_GBps": len(circ) * 2 * (1 << n) * amp_bytes / (ms_per_step * 1e-3) / 1e9,
                "wall_ms_per_step": wall_ms / args.steps, "exchange_ms_per_step": xch_ms / args.steps,
                "roofline": roofline, "at_30q": at_30q, "configs": configs, "e2e_full_30q": e2e_full, "reference_gpu": reference_gpu,
                "parity": parity, "cpu_baseline": cpu, "e2e": e2e,
                "gpu_launches": int(pst["kernel_launches"]) * args.steps, "clocks": clocks,
                "lib": q.lib.qsb_version().decode()}
        print(json.dumps(line))
    plan.close()
    sim.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--qubits", type=int, default=0)
    ap.add_argument("--precision", type=int, default=32, choices=[32, 64])
    ap.add_argument("--low-bits", type=int, default=0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-30q", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="N = 1: skip the per-config lines, the full-state e2e and the reference-GPU run")
    ap.add_argument("--no-lazy-diag", type=int, default=0, help="planner A/B: 2 = lazy diagonals on")
    ap.add_argument("--trim", type=int, default=0, help="planner A/B: k+1 = trim tail rounds with < k gates (1 = off)")
    ap.add_argument("--cost-cap", type=int, default=0, help="fusion-depth sweep: SM cost cap per pass in gate units")
    ap.add_argument("--workload", default="layered", choices=["layered", "qft"])
    ap.add_argument("--no-sink", type=int, default=0, help="planner A/B (qsb_options_t.reserved[6]): 1 = do not sink thread-level phases to later rounds, 2 = first-come tile choice (no hill climbing), 3 = no end-of-pass lane relocation, 4 = lane relocation only on conflict")
    ap.add_argument("--fused", type=int, default=0, help="multi-GPU A/B: exchange flavour, 0 = default (fused peer scatter; pipelined at 2 GPUs), 1 = fused peer scatter (direct: victims anywhere), 2 = NCCL all-to-all, 3 = pipelined copy-engine exchange, 4 = round-1 fused flavour")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--res4", type=int, default=0, help="planner A/B: qsb_options_t.reserved[4] (1 = vector-bit phases not deferred, 2 = no 2x2 products, 3 = no Hadamard-like slot form, 4 = no merged phase runs, 5 = h cx h stays as it is, 6 = CX -> controlled phase with an h on one side too)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a seeded sample of the state the last one "
                                                          "computed to DIR/state.npy and its logical indices to DIR/state_index.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
