"""torchrun worker: noise channels on a sharded state (one rank per GPU), on local and rank qubits.  Every rank must get
the same branches and probabilities bit for bit, and the gathered state must match a single-GPU handle run with the same
r on the same input state."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import gpu_quantum_simulator_b200 as q  # noqa: E402
from gpu_quantum_simulator_b200 import circuits, dist as qdist  # noqa: E402
from test_gpu_channels import stinespring  # noqa: E402


def channels_for(n, perm, nloc):
    rq = sorted((qb for qb in range(n) if perm[qb] >= nloc), key=lambda qb: perm[qb])
    lo = sorted((qb for qb in range(n) if perm[qb] < nloc), key=lambda qb: perm[qb])
    hi = lo[::-1]
    out = [(q.amplitude_damping(0.3), [k]) for k in lo[:6]]                        # local groups
    out += [(q.amplitude_damping(0.4), [rq[0]]), (q.depolarizing(0.5), [rq[-1]])]   # a group and a run on rank qubits
    out += [(stinespring(2, 3, 1), [hi[0], rq[0]]), (q.depolarizing(0.3, 2), [lo[1], hi[1]])]
    if len(rq) >= 2:
        out += [(stinespring(2, 4, 2), [rq[1], rq[0]]), (stinespring(3, 5, 3), [lo[0], rq[1], hi[2]])]
    out += [(q.phase_damping(0.5), [k]) for k in hi[:5]]
    return out


def main():
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    for prec, tol in ((q.F32, 1e-5), (q.F64, 1e-12)):
        for flavour in (0, 2):          # qsb_options_t.reserved[5]: default exchange, NCCL all-to-all
            for n, seed in ((22, 3), (23, 4)):
                circ = circuits.random_layered(n, depth=5, seed=seed)
                sim = q.Simulator(n, precision=prec, rank=rank, world_size=world, device=local, reserved=[0, 0, 0, 0, 0, flavour])
                qdist.init_comm(sim, dist)
                sim.apply(q.gates_from_circuit(circ))
                perm, nloc = sim.layout()
                chans = channels_for(n, perm, nloc)
                before = qdist.gather_state(sim, dist)
                b, p = sim.apply_channels(chans, seed=seed)
                assert np.array_equal(sim.layout()[0], perm)
                got = qdist.gather_state(sim, dist)
                sim.close()
                mine = torch.tensor(np.concatenate([b.astype(np.float64), p]), dtype=torch.float64, device="cuda")
                every = [torch.empty_like(mine) for _ in range(world)]
                dist.all_gather(every, mine)
                for other in every:
                    assert torch.equal(other, every[0]), "ranks disagree on branches or probabilities"
                if rank == 0:
                    with q.Simulator(n, precision=prec, device=local) as one:
                        one.set_state(before)
                        b1, p1 = one.apply_channels(chans, seed=seed)
                        want = one.state()
                    assert np.array_equal(b, b1), (b, b1)
                    assert np.allclose(p, p1, rtol=1e-5 if prec == q.F32 else 1e-10, atol=0), (p, p1)
                    err = float(np.max(np.abs(got - want)))
                    assert err <= 3 * tol, (n, prec, flavour, err)
                    print(f"n={n} prec={prec} world={world} flavour={flavour} channels={len(chans)} err={err:.2e}")
    if rank == 0:
        print("sharded_channel_ok")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
