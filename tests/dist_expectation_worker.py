"""torchrun worker: expectation values of a sharded state (one rank per GPU) against numpy on the gathered state,
then a second circuit on the same handles checked against the oracle (the partner shards fetched into the exchange
buffer must not disturb later executions)."""
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
from test_gpu_expectation import expect_np  # noqa: E402


def terms_for(n, perm, nloc, rng):
    """X/Y on the qubits that sit on rank bits, Z on them, mixed strings, then random ones."""
    rq = [qb for qb in range(n) if perm[qb] >= nloc]
    lq = [qb for qb in range(n) if perm[qb] < nloc]
    out = ["", f"Z{rq[0]}", f"X{rq[0]}", f"Y{rq[-1]}", " ".join(f"X{qb}" for qb in rq), " ".join(f"Z{qb}" for qb in rq),
           f"X{rq[0]} Z{lq[0]}", f"Y{rq[0]} X{lq[0]} Z{lq[-1]}", f"Z{rq[-1]} X{lq[3]}", f"Z{rq[0]} Y{lq[-1]} X{lq[1]}",
           " ".join(f"{'XYZ'[k % 3]}{k}" for k in range(n))]
    for _ in range(40):
        qs = rng.choice(n, int(rng.integers(1, 5)), replace=False)
        out.append(" ".join(f"{'XYZ'[rng.integers(3)]}{k}" for k in qs))
    return out


def main():
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    worst = 0.0
    for prec, tol, tol_state in ((q.F32, 1e-6, 1e-5), (q.F64, 1e-12, 1e-12)):
        for flavour in (0, 2):          # qsb_options_t.reserved[5]: default exchange, NCCL all-to-all
            for n, seed in ((22, 3), (23, 4)):
                circ1 = circuits.random_layered(n, depth=5, seed=seed)
                circ2 = circuits.random_layered(n, depth=3, seed=seed + 50)
                sim = q.Simulator(n, precision=prec, rank=rank, world_size=world, device=local, reserved=[0, 0, 0, 0, 0, flavour])
                qdist.init_comm(sim, dist)
                sim.apply(q.gates_from_circuit(circ1))
                perm, nloc = sim.layout()
                terms = terms_for(n, perm, nloc, np.random.default_rng(seed))
                got = sim.expectation(terms)
                t = torch.from_numpy(got).cuda()
                parts = [torch.empty_like(t) for _ in range(world)]
                dist.all_gather(parts, t)
                assert all(torch.equal(parts[0], p) for p in parts), "ranks disagree"
                full = qdist.gather_state(sim, dist)
                sim.apply(q.gates_from_circuit(circ2))
                after = qdist.gather_state(sim, dist)
                sim.close()
                if rank == 0:
                    want = expect_np(full, terms, n)
                    err = float(np.max(np.abs(got - want)))
                    worst = max(worst, err / tol)
                    assert err <= tol, (n, prec, flavour, err, terms[int(np.argmax(np.abs(got - want)))])
                    ref = helpers.oracle_run_circuit(list(circ1) + list(circ2), n)
                    serr = float(np.max(np.abs(after - ref)))
                    assert serr <= tol_state, (n, prec, flavour, serr)
                    print(f"n={n} prec={prec} world={world} flavour={flavour} terms={len(terms)} err={err:.2e} second circuit err={serr:.2e}")
    if rank == 0:
        print(f"sharded_expectation_ok worst_err_over_tol={worst:.3f}")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
