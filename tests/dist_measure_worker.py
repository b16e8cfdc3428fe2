"""torchrun worker: marginals, measurement, collapse and reset of a sharded state (one rank per GPU) against numpy on
the gathered state, with qubit sets that include qubits on rank bits; then a second circuit on the same handles against
a single-GPU handle loaded with the projected state (the exchange buffers and peer mappings must survive a collapse)."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import gpu_quantum_simulator_b200 as q  # noqa: E402
from gpu_quantum_simulator_b200 import circuits, dist as qdist  # noqa: E402
from test_gpu_measure import marginal_np, probs_ld, project_np, rule  # noqa: E402


def same_on_every_rank(values):
    """values (float64 array) bit-identical on every rank"""
    t = torch.from_numpy(np.ascontiguousarray(values, dtype=np.float64).view(np.int64)).cuda()
    parts = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(parts, t)
    return all(torch.equal(parts[0], p) for p in parts)


def main():
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    for prec, tol in ((q.F32, 1e-5), (q.F64, 1e-12)):
        for flavour in (0, 2):          # qsb_options_t.reserved[5]: default exchange, NCCL all-to-all
            for n, seed in ((22, 3), (23, 4)):
                rng = np.random.default_rng(seed)
                circ1 = circuits.random_layered(n, depth=5, seed=seed)
                circ2 = circuits.random_layered(n, depth=3, seed=seed + 50)
                sim = q.Simulator(n, precision=prec, rank=rank, world_size=world, device=local, reserved=[0, 0, 0, 0, 0, flavour])
                qdist.init_comm(sim, dist)
                sim.apply(q.gates_from_circuit(circ1))
                perm, nloc = sim.layout()
                rq = [qb for qb in range(n) if perm[qb] >= nloc]
                lq = [qb for qb in range(n) if perm[qb] < nloc]
                low = [qb for qb in range(n) if perm[qb] == 0]
                sets = [[rq[0]], rq, rq[::-1] + lq[:2], [lq[0], rq[-1], lq[5]], low + [rq[-1]], rng.permutation(n)[:12].tolist(),
                        rng.permutation(n)[:20].tolist()]
                full = qdist.gather_state(sim, dist)
                p = probs_ld(full)
                for qs in sets:
                    got = sim.marginal_probabilities(qs)
                    assert same_on_every_rank(got), ("tables differ between ranks", qs)
                    err = float(np.max(np.abs(got - marginal_np(p, qs))))
                    assert err <= 1e-12, (n, prec, flavour, qs, err)
                # measurement with rank-bit qubits: every rank gets the same outcome
                qm = [lq[2], rq[0], lq[7]]
                table = sim.marginal_probabilities(qm)
                b, pb = sim.measure_qubits(qm, 0.37)
                assert same_on_every_rank(np.array([float(b), pb])), "outcomes differ between ranks"
                assert pb == table[b] and b == rule(table, 0.37)
                state = qdist.gather_state(sim, dist)
                want, _ = project_np(full, qm, b)
                assert np.max(np.abs(state - want)) <= tol, (n, prec, flavour, "measure")
                # collapse onto a non-zero outcome of a set that holds every rank-bit qubit
                qc = rq + [lq[3]]
                tc = sim.marginal_probabilities(qc)
                oc = int(np.flatnonzero(tc > 1e-9)[-1])
                pc = sim.collapse(qc, oc)
                assert pc == tc[oc] and same_on_every_rank(np.array([pc]))
                want, _ = project_np(state, qc, oc)
                state = qdist.gather_state(sim, dist)
                assert np.max(np.abs(state - want)) <= tol, (n, prec, flavour, "collapse")
                # reset of a qubit on a rank bit (X through the apply path)
                ob = sim.reset_qubits([rq[-1]], 0.5)
                m = sim.marginal_probabilities([rq[-1]])
                assert abs(m[0] - 1.0) <= tol and m[1] <= tol, m
                projected, _ = project_np(state, [rq[-1]], ob)
                state = qdist.gather_state(sim, dist)
                want = projected[np.arange(1 << n) ^ (ob << rq[-1])]
                assert np.max(np.abs(state - want)) <= 10 * tol, (n, prec, flavour, "reset")
                # a second circuit through the exchange paths after the collapses
                sim.apply(q.gates_from_circuit(circ2))
                after = qdist.gather_state(sim, dist)
                sim.close()
                if rank == 0:
                    with q.Simulator(n, precision=prec, device=local) as ref:
                        ref.set_state(state)
                        ref.apply(q.gates_from_circuit(circ2))
                        serr = float(np.max(np.abs(after - ref.state())))
                    assert serr <= 10 * tol, (n, prec, flavour, serr)
                    print(f"n={n} prec={prec} world={world} flavour={flavour} outcome={b} p={pb:.6f} second circuit err={serr:.2e}")
                dist.barrier()
    if rank == 0:
        print("sharded_measure_ok")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
