"""Multi-GPU parity (needs 2 GPUs, and 4 for the 4-rank case): the spatially decomposed VelocityVerlet run must reproduce
the single-GPU run of the same system (same kernels; only the order of the 24-byte momentum reduction differs)."""
import os
import socket

import numpy as np
import pytest

import mbhelpers as H
import mollyb200 as mb

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out_dir, n_steps, p2p):
    import torch
    import torch.distributed as dist
    os.environ["MOLLYB200_P2P"] = "1" if p2p else "0"
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sd = H.lj_fluid(16, seed=9, dtype=np.float64, temp=120.0)
    inter = (mb.LennardJones(cutoff=mb.ShiftedForceCutoff(1.0), use_neighbors=True),)
    atoms = mb.atoms_from_arrays(sd["mass"], sd["charge"], sd["sigma"], sd["eps"], np.float64)
    nf = mb.GPUNeighborFinder(dist_cutoff=1.15, n_steps=20)
    s = mb.System(atoms=atoms, coords=sd["coords"].copy(), boundary=mb.CubicBoundary(*sd["box"]),
                  velocities=sd["velocities"].copy(), pairwise_inters=inter, neighbor_finder=nf, dtype=np.float64, device=rank)
    s.engine()
    uid = [mb.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    mb.comm_init(s, uid[0], rank, world)
    mb.simulate(s, mb.VelocityVerlet(dt=0.002), n_steps)
    mb.simulate(s, mb.VelocityVerlet(dt=0.002), 15, init_step=n_steps)  # second call re-enters with a live list
    st = s.stats()
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"), x=s.coords, v=s.velocities,
             stats=np.array([st["n_rebuilds"], st["peer_transport"]]))
    s.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("world,p2p", [(2, True), (2, False), (4, True)])
def test_decomposed_matches_single_gpu(tmp_path, world, p2p):
    """p2p=True: halo exchange + momentum sum over NVLink peer memory (peer.cuh); False: the NCCL transport."""
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    n_steps = 45
    sd = H.lj_fluid(16, seed=9, dtype=np.float64, temp=120.0)
    inter = (mb.LennardJones(cutoff=mb.ShiftedForceCutoff(1.0), use_neighbors=True),)
    ref = H.make_system(sd, inter, np.float64, r_list=1.15, n_steps=20)
    mb.simulate(ref, mb.VelocityVerlet(dt=0.002), n_steps)
    mb.simulate(ref, mb.VelocityVerlet(dt=0.002), 15, init_step=n_steps)
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path), n_steps, p2p), nprocs=world, join=True)
    outs = [np.load(tmp_path / f"rank{r}.npz") for r in range(world)]
    for o in outs:
        d = o["x"] - ref.coords
        d -= sd["box"] * np.round(d / sd["box"])
        print(f"decomposed ({world} ranks, p2p requested {p2p}) vs single: dx", np.abs(d).max(), "dv",
              np.abs(o["v"] - ref.velocities).max(), "rebuilds / peer_transport", o["stats"])
        assert np.abs(d).max() < 1e-9 and np.abs(o["v"] - ref.velocities).max() < 1e-8
    for o in outs[1:]:  # every rank returns the same whole system, and all ranks took the same transport
        assert np.array_equal(outs[0]["x"], o["x"]) and np.array_equal(outs[0]["v"], o["v"])
        assert o["stats"][1] == outs[0]["stats"][1]
    if not p2p:
        assert outs[0]["stats"][1] == 0
    ref.close()
