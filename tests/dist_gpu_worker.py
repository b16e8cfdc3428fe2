"""torchrun worker: sharded GPU run (one rank per GPU, NCCL exchanges) checked against the oracle."""
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


def check_sharded_readout(sim, got, n, rank, world, prec):
    """Collective sampler: every rank receives the same shots; each one is what the reference's search rule
    (first index with cdf != 0 and cdf >= r) gives on the CDF taken in rank-major physical order.  Then a
    per-rank shard dump / reload round trip."""
    seed, count = 17, 96
    shots = sim.measurement(count, seed=seed)
    perm, nloc = sim.layout()
    t = torch.from_numpy(shots.astype(np.int64)).cuda()
    parts = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(parts, t)
    assert all(torch.equal(parts[0], p) for p in parts)
    idx = np.arange(1 << n, dtype=np.uint64)
    phys = np.zeros_like(idx)
    for qb in range(n):
        phys |= ((idx >> np.uint64(qb)) & np.uint64(1)) << np.uint64(int(perm[qb]))
    p_phys = np.zeros(1 << n)
    p_phys[phys] = np.abs(got) ** 2
    cdf = np.cumsum(p_phys)
    L = helpers.oracle_lib()
    for k in range(count):
        r = q.sample_uniform(seed, k)
        want = int(L.oc_measure(cdf.ctypes.data, n, r))
        g_phys = int(phys[int(shots[k])])
        assert p_phys[g_phys] > 0.0
        if g_phys != want:
            assert abs(cdf[want] - r) < 1e-9 or abs(cdf[g_phys] - r) < 1e-9, (k, r, g_phys, want)
    try:                                   # the global CDF needs the other ranks' amplitudes: refused, not computed
        sim.compute_state_cumulative_distribution(0, 1)
        raise AssertionError("qsb_cdf accepted a sharded state")
    except q.QsbError as e:
        assert e.code == -1 and "qsb_sample" in str(e), e
    path = f"/tmp/qsb_shard_{os.getpid()}_{rank}.bin"
    before = sim.shard_physical().copy()
    sim.save_state(path)
    sim.reset()
    sim.load_state(path)
    os.unlink(path)
    assert np.array_equal(sim.shard_physical(), before)
    assert np.array_equal(sim.layout()[0], perm)
    if rank == 0:
        print(f"sharded readout ok: n={n} prec={prec} world={world} shots={count}")


def main():
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    worst = 0.0
    # exchange flavours (qsb_options_t.reserved[5]): 0 = default by world size, 1 = fused peer scatter, 2 = NCCL all-to-all,
    # 3 = pipelined copy-engine exchange, 4 = round-1 fused flavour (victims moved to the top local positions first)
    configs = ((q.F32, 1e-5, 0), (q.F64, 1e-12, 0), (q.F32, 1e-5, 1), (q.F64, 1e-12, 1), (q.F32, 1e-5, 2), (q.F32, 1e-5, 3), (q.F64, 1e-12, 3), (q.F32, 1e-5, 4))
    sizes = ((22, 8, 7), (23, 5, 8))
    if os.environ.get("QSB_DIST_QUICK"):       # readout-only run: default exchange flavour, one small circuit per precision
        configs, sizes = configs[:2], ((22, 5, 7),)
    for prec, tol, mode in configs:
        for n, depth, seed in sizes:
            circ = circuits.random_layered(n, depth=depth, seed=seed)
            sim = q.Simulator(n, precision=prec, rank=rank, world_size=world, device=local, reserved=[0, 0, 0, 0, 0, mode])
            qdist.init_comm(sim, dist)
            st = sim.apply(q.gates_from_circuit(circ))
            got = qdist.gather_state(sim, dist)
            if mode == 0:
                check_sharded_readout(sim, got, n, rank, world, prec)
            sim.close()
            if rank == 0:
                want = helpers.oracle_run_circuit(circ, n)
                err = float(np.max(np.abs(got - want)))
                worst = max(worst, err / tol)
                print(f"n={n} prec={prec} world={world} exchange_mode={mode} swaps={st['swaps']} passes={st['passes']} err={err:.3e}")
                assert st["swaps"] >= 1
                assert err <= tol, (n, prec, err)
    if rank == 0:
        print(f"sharded_gpu_ok worst_err_over_tol={worst:.3f}")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
