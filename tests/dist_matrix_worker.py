"""torchrun worker: dense matrices on a sharded state (one rank per GPU) against numpy on the gathered state, then a second
circuit on the same handles checked against the oracle (the partner shards fetched into the exchange buffer must not
disturb later executions)."""
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
from test_gpu_matrix import apply_np, contraction, random_ops, unitary  # noqa: E402


def ops_for(n, perm, nloc, seed):
    """One rank target, two and three rank targets (world >= 4 / 8), rank-bit controls, then random ops."""
    rq = sorted((qb for qb in range(n) if perm[qb] >= nloc), key=lambda qb: perm[qb])
    hi = sorted((qb for qb in range(n) if perm[qb] < nloc), key=lambda qb: -perm[qb])   # local, highest bits first
    lo = hi[::-1]
    out = [(unitary(1, 1), [rq[0]]), (unitary(2, 2), [lo[0], rq[-1]]), (contraction(3, 3), [rq[0], hi[0], lo[1]]),
           (unitary(1, 4), [rq[0]]), (unitary(2, 5), [hi[1], hi[2]], [rq[-1]]),
           (unitary(2, 6), [rq[0], lo[2]], [hi[3], lo[3]]), (unitary(6, 7), [rq[-1]] + hi[:3] + lo[:2])]
    if len(rq) >= 2:
        out += [(unitary(2, 8), [rq[1], rq[0]]), (unitary(3, 9), [lo[0], rq[0], rq[1]], [hi[0]]),
                (unitary(1, 10), [lo[4]], [rq[0], rq[1]]), (unitary(2, 11), [rq[0], hi[1]], [rq[1]])]
    if len(rq) >= 3:
        out += [(unitary(3, 12), rq[:3]), (contraction(5, 13), [rq[2], lo[0], rq[0], hi[0], rq[1]], [lo[5]])]
    return out + random_ops(n, 20, seed)


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
                ops = ops_for(n, perm, nloc, seed)
                before = qdist.gather_state(sim, dist)
                sim.apply_matrices(ops)
                assert np.array_equal(sim.layout()[0], perm)
                got = qdist.gather_state(sim, dist)
                sim.apply(q.gates_from_circuit(circ2))
                after = qdist.gather_state(sim, dist)
                sim.close()
                if rank == 0:
                    want = apply_np(before, ops, n)
                    err = float(np.max(np.abs(got - want)))
                    assert err <= 3 * tol, (n, prec, flavour, err)
                    ref = helpers.oracle_run_circuit(circ2, n, state=want)
                    serr = float(np.max(np.abs(after - ref)))
                    assert serr <= 3 * tol, (n, prec, flavour, serr)
                    print(f"n={n} prec={prec} world={world} flavour={flavour} ops={len(ops)} err={err:.2e} "
                          f"second circuit err={serr:.2e}")
    if rank == 0:
        print("sharded_matrix_ok")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
