"""torchrun worker: rotation gradients on a sharded state (one rank per GPU) against the numpy adjoint on the gathered
state, with rotations and observable terms on rank qubits; every rank must receive identical energy and gradient bits,
and a second circuit on the same handles must still match the oracle."""
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
from dist_pauli_rotation_worker import rotations_for  # noqa: E402
from test_gpu_rotation_gradient import adjoint_grad_np  # noqa: E402


def observable_for(n, perm, nloc, rng):
    rq = [qb for qb in range(n) if perm[qb] >= nloc]
    hi = sorted((qb for qb in range(n) if perm[qb] < nloc), key=lambda qb: -perm[qb])
    out = [f"Z{rq[0]}", f"X{rq[-1]}", f"Z{rq[0]} Z{hi[0]}", f"Y{rq[0]} X{hi[1]}", " ".join(f"X{qb}" for qb in rq),
           f"Z{hi[0]} Z{hi[2]}", "", " ".join(f"{'XYZ'[k % 3]}{k}" for k in range(n))]
    for _ in range(20):
        qs = rng.choice(n, int(rng.integers(1, 5)), replace=False)
        out.append(" ".join(f"{'XYZ'[rng.integers(3)]}{k}" for k in qs))
    return out, rng.normal(size=len(out))


def main():
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    for prec, rel in ((q.F32, 2e-4), (q.F64, 1e-10)):
        for flavour in (0, 2):          # qsb_options_t.reserved[5]: default exchange, NCCL all-to-all
            n, seed = 22, 3
            circ1 = circuits.random_layered(n, depth=5, seed=seed)
            circ2 = circuits.random_layered(n, depth=3, seed=seed + 50)
            sim = q.Simulator(n, precision=prec, rank=rank, world_size=world, device=local, reserved=[0, 0, 0, 0, 0, flavour])
            qdist.init_comm(sim, dist)
            sim.apply(q.gates_from_circuit(circ1))
            perm, nloc = sim.layout()
            rng = np.random.default_rng(seed)
            rots = rotations_for(n, perm, nloc, rng)[:40]
            th = rng.uniform(-np.pi, np.pi, size=len(rots))
            th[::4] = 0.0
            obs, coef = observable_for(n, perm, nloc, rng)
            before = qdist.gather_state(sim, dist)
            e, g = sim.rotation_gradient(rots, th, obs, coef)
            assert np.array_equal(sim.layout()[0], perm)
            got = qdist.gather_state(sim, dist)
            sim.apply(q.gates_from_circuit(circ2))
            after = qdist.gather_state(sim, dist)
            sim.close()
            bits = torch.from_numpy(np.concatenate([[e], g]).view(np.int64).copy()).cuda()
            every = [torch.empty_like(bits) for _ in range(world)]
            dist.all_gather(every, bits)
            assert all(torch.equal(every[0], b) for b in every), "ranks differ"
            if rank == 0:
                want_e, want_g, want_psi = adjoint_grad_np(before, rots, th, obs, coef, n)
                tol = rel * np.sum(np.abs(coef))
                gerr = float(np.max(np.abs(g - want_g)))
                assert gerr <= tol and abs(e - want_e) <= tol, (prec, flavour, gerr, e, want_e)
                serr = float(np.max(np.abs(got - want_psi)))
                assert serr <= (1e-5 if prec == q.F32 else 1e-12), serr
                ref = helpers.oracle_run_circuit(circ2, n, state=want_psi)
                assert float(np.max(np.abs(after - ref))) <= (1e-5 if prec == q.F32 else 1e-12)
                dr = q.rotation_gradient_dry_run(n, rots, obs, prec, world_size=world)
                print(f"n={n} prec={prec} world={world} flavour={flavour} rotations={len(rots)} {dr} grad err={gerr:.2e}")
    if rank == 0:
        print("sharded_rotation_gradient_ok")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
