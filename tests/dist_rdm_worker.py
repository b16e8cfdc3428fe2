"""torchrun worker: reduced density matrices of a sharded state (one rank per GPU) against numpy on the gathered state,
with qubit sets that hold no rank qubit, one, all of them, rank qubits with a lane qubit, and k = 12 with rank qubits;
the results must be bit-identical on every rank.  Then a second circuit on the same handles against a single-GPU handle:
the partner shards went through the exchange buffer."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import gpu_quantum_simulator_b200 as q  # noqa: E402
from gpu_quantum_simulator_b200 import circuits, dist as qdist  # noqa: E402
from test_gpu_rdm import check_structure, rho_np  # noqa: E402


def same_on_every_rank(values):
    t = torch.from_numpy(np.ascontiguousarray(values).view(np.int64).reshape(-1)).cuda()
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
            n, seed = 22, 7
            rng = np.random.default_rng(seed)
            circ1 = circuits.random_layered(n, depth=5, seed=seed)
            circ2 = circuits.random_layered(n, depth=3, seed=seed + 50)
            sim = q.Simulator(n, precision=prec, rank=rank, world_size=world, device=local, reserved=[0, 0, 0, 0, 0, flavour])
            qdist.init_comm(sim, dist)
            sim.apply(q.gates_from_circuit(circ1))
            perm, nloc = sim.layout()
            rq = [qb for qb in range(n) if perm[qb] >= nloc]
            lq = [qb for qb in range(n) if perm[qb] < nloc]
            lane = [qb for qb in range(n) if perm[qb] in (0, 1)]
            sets = [lq[3:6], [rq[0]], rq, rq[::-1] + lane, [lq[0], rq[-1], lq[5]],
                    rq + rng.permutation(lq)[:12 - len(rq)].tolist()]
            full = qdist.gather_state(sim, dist)
            for qs in sets:
                got = sim.reduced_density_matrix(qs)
                assert same_on_every_rank(got), ("matrices differ between ranks", qs)
                check_structure(got, len(qs))
                err = float(np.max(np.abs(got - rho_np(full, qs))))
                assert err <= 1e-12, (n, prec, flavour, qs, err)
            sim.apply(q.gates_from_circuit(circ2))
            after = qdist.gather_state(sim, dist)
            sim.close()
            if rank == 0:
                with q.Simulator(n, precision=prec, device=local) as ref:
                    ref.set_state(full)
                    ref.apply(q.gates_from_circuit(circ2))
                    serr = float(np.max(np.abs(after - ref.state())))
                assert serr <= 10 * tol, (n, prec, flavour, serr)
                print(f"n={n} prec={prec} world={world} flavour={flavour} second circuit err={serr:.2e}")
            dist.barrier()
    if rank == 0:
        print("sharded_rdm_ok")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
