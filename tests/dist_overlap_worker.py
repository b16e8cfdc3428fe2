"""torchrun worker: overlaps and copies of sharded states (one rank per GPU) against numpy on the gathered states, for
circuit layouts and crafted layouts whose rank qubits differ, in every precision pair and two exchange flavours; then a
second circuit on b checked against the oracle (partner shards received into b's exchange buffer must not disturb later
executions)."""
import os
import shutil
import sys
import tempfile

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import helpers  # noqa: E402
import gpu_quantum_simulator_b200 as q  # noqa: E402
from gpu_quantum_simulator_b200 import circuits, dist as qdist  # noqa: E402
from test_gpu_overlap import random_state, write_shard  # noqa: E402

N = 20


def same_on_every_rank(vals):
    t = torch.tensor(vals, dtype=torch.float64, device="cuda")
    parts = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(parts, t)
    return all(torch.equal(p, parts[0]) for p in parts)


def rank_set(sim):
    perm, nloc = sim.layout()
    return {qb for qb in range(sim.num_qubits) if perm[qb] >= nloc}


def crafted_layouts(g):
    """(name, perm_a, perm_b): d = 0 with the rank qubits in swapped positions, d = 1 with b's first rank qubit on a's
    lowest (lane) bit, and disjoint rank sets."""
    nloc = N - g
    ident = list(range(N))

    def swapped(pairs):
        p = list(ident)
        for x, y in pairs:
            p[x], p[y] = p[y], p[x]
        return p
    out = []
    if g >= 2:
        out.append(("d0 swapped", ident, swapped([(nloc, nloc + 1)])))
    out.append(("d1 lane", swapped([(3, 9)]), swapped([(0, nloc)])))
    out.append(("disjoint", ident, swapped([(i, nloc + i) for i in range(g)])))
    return out


def main():
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    g = world.bit_length() - 1
    tmp = tempfile.mkdtemp(prefix=f"qsb_overlap_{rank}_")
    differing = 0
    for pa, pb in ((q.F32, q.F32), (q.F32, q.F64), (q.F64, q.F32), (q.F64, q.F64)):
        tol = 1e-12 if pa == pb == q.F64 else 1e-5
        for flavour in (0, 2):          # qsb_options_t.reserved[5]: default exchange, NCCL all-to-all
            kw = dict(rank=rank, world_size=world, device=local, reserved=[0, 0, 0, 0, 0, flavour])
            cases = [("circuits", None, None)] + crafted_layouts(g)
            for name, perm_a, perm_b in cases:
                a = q.Simulator(N, precision=pa, **kw)
                b = q.Simulator(N, precision=pb, **kw)
                qdist.init_comm(a, dist)
                qdist.init_comm(b, dist)
                if perm_a is None:
                    a.apply(q.gates_from_circuit(circuits.random_layered(N, depth=6, seed=1)))
                    b.apply(q.gates_from_circuit(circuits.random_layered(N, depth=5, seed=2)))
                else:
                    x, y = random_state(N, 7), random_state(N, 8)
                    for s, perm, psi, tag in ((a, perm_a, x, "a"), (b, perm_b, 0.6 * x + 0.8 * y, "b")):
                        path = os.path.join(tmp, f"{tag}.qsb")
                        write_shard(path, N, s.precision, perm, psi, world=world, rank=rank)
                        s.load_state(path)
                if rank_set(a) != rank_set(b):
                    differing += 1
                xa, xb = qdist.gather_state(a, dist), qdist.gather_state(b, dist)
                raw_a, raw_b = a.shard_physical(), b.shard_physical()
                got, na, nb = a._inner(b)
                again = a._inner(b)
                assert again == (got, na, nb), name
                assert same_on_every_rank([got.real, got.imag, na, nb]), name
                want = np.vdot(xa, xb)
                scale = np.sqrt(np.vdot(xa, xa).real * np.vdot(xb, xb).real)
                assert abs(got - want) <= tol * scale, (name, pa, pb, flavour, got, want)
                assert abs(na - np.vdot(xa, xa).real) <= tol * na and abs(nb - np.vdot(xb, xb).real) <= tol * nb, name
                rev = b.overlap(a)
                assert abs(rev - np.conj(want)) <= tol * scale, name
                assert np.array_equal(a.shard_physical(), raw_a) and np.array_equal(b.shard_physical(), raw_b), name
                # a second circuit on b: its exchanges run through the buffer the call received partner shards into
                circ2 = circuits.random_layered(N, depth=3, seed=50)
                b.apply(q.gates_from_circuit(circ2))
                after = qdist.gather_state(b, dist)
                if rank == 0:
                    ref = helpers.oracle_run_circuit(circ2, N, state=xb)
                    serr = float(np.max(np.abs(after - ref)))
                    assert serr <= 3 * tol, (name, pa, pb, flavour, serr)
                if pa == pb:                                  # the copy, then the exact self overlap
                    b.copy_from(a)
                    assert np.array_equal(b.layout()[0], a.layout()[0])
                    assert np.array_equal(b.shard_physical(), a.shard_physical())
                    ov, n1, n2 = a._inner(b)
                    assert ov.imag == 0.0 and ov.real == n1 == n2, name
                    assert same_on_every_rank([ov.real, n1]), name
                if rank == 0:
                    print(f"{name}: prec {pa}/{pb} world={world} flavour={flavour} |d|={abs(got - want):.2e}")
                a.close()
                b.close()
    shutil.rmtree(tmp, ignore_errors=True)
    assert differing > 0, "no case had different rank qubits"
    if rank == 0:
        print("sharded_overlap_ok")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
