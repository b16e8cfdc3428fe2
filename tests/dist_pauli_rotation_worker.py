"""torchrun worker: Pauli rotations on a sharded state (one rank per GPU) against numpy on the gathered state, then a
second circuit on the same handles checked against the oracle (the partner shards fetched into the exchange buffer
must not disturb later executions)."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import helpers  # noqa: E402
import gpu_quantum_simulator_b200 as q  # noqa: E402
from gpu_quantum_simulator_b200 import circuits, dist as qdist  # noqa: E402
from test_gpu_pauli_rotation import rotate_np  # noqa: E402


def rotations_for(n, perm, nloc, rng):
    """Rank qubits alone, rank qubits with local qubits outside any tile, X on every qubit, then random ones."""
    rq = [qb for qb in range(n) if perm[qb] >= nloc]
    hi = sorted((qb for qb in range(n) if perm[qb] < nloc), key=lambda qb: -perm[qb])   # local, highest bits first
    out = [f"X{rq[0]}", f"Y{rq[-1]}", f"Z{rq[0]}", " ".join(f"X{qb}" for qb in rq), f"Z{rq[-1]} Z{hi[0]}",
           f"X{rq[0]} X{hi[0]}", f"Y{rq[-1]} Z{hi[1]} X{hi[2]}", f"X{rq[0]} X{hi[3]} Y{hi[-1]}",
           " ".join(f"X{k}" for k in range(n)), " ".join(f"{'XYZ'[k % 3]}{k}" for k in range(n))]
    for _ in range(60):
        qs = rng.choice(n, int(rng.integers(1, 5)), replace=False)
        out.append(" ".join(f"{'XYZ'[rng.integers(3)]}{k}" for k in qs))
    return out


def main():
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    for prec, tol in ((q.F32, 1e-5), (q.F64, 1e-12)):
        for flavour in (0, 2):          # qsb_options_t.reserved[5]: default exchange, NCCL all-to-all
            for n, seed in ((22, 3), (23, 4)):
                circ1 = circuits.random_layered(n, depth=5, seed=seed)
                circ2 = circuits.random_layered(n, depth=3, seed=seed + 50)
                sim = q.Simulator(n, precision=prec, rank=rank, world_size=world, device=local, reserved=[0, 0, 0, 0, 0, flavour])
                qdist.init_comm(sim, dist)
                sim.apply(q.gates_from_circuit(circ1))
                perm, nloc = sim.layout()
                rng = np.random.default_rng(seed)
                terms = rotations_for(n, perm, nloc, rng)
                th = rng.uniform(-np.pi, np.pi, size=len(terms))
                before = qdist.gather_state(sim, dist)
                sim.apply_pauli_rotations(terms, th)
                assert np.array_equal(sim.layout()[0], perm)
                got = qdist.gather_state(sim, dist)
                sim.apply(q.gates_from_circuit(circ2))
                after = qdist.gather_state(sim, dist)
                sim.close()
                if rank == 0:
                    want = rotate_np(before, terms, th, n)
                    err = float(np.max(np.abs(got - want)))
                    assert err <= tol, (n, prec, flavour, err)
                    # the second circuit, from the rotated state, against the oracle
                    ref = helpers.oracle_run_circuit(circ2, n, state=want)
                    serr = float(np.max(np.abs(after - ref)))
                    assert serr <= tol, (n, prec, flavour, serr)
                    sw = q.pauli_rotation_dry_run(n, terms, prec, world_size=world)
                    print(f"n={n} prec={prec} world={world} flavour={flavour} rotations={len(terms)} {sw} err={err:.2e} "
                          f"second circuit err={serr:.2e}")
    if rank == 0:
        print("sharded_pauli_rotation_ok")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
