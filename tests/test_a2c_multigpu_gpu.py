"""Two-rank data-parallel A2C (skipped on a one-GPU box): the replicas stay bit-identical with the gradient exchange fused into the
clip + RMSprop launch (peer memory) and with the NCCL all-reduce + tmla_rmsprop_clip_fused path."""
import os
import socket

import pytest
import torch

pytestmark = pytest.mark.gpu


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out, allreduce):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank),
                      TMLA_ALLREDUCE=allreduce)
    from three_mlagents_b200 import distributed as D
    from three_mlagents_b200.a2c import CudaA2C
    from three_mlagents_b200.vec_env import CudaVecEnv

    D.init_from_env("nccl", device_index=rank)
    N = 512
    first, _ = D.env_shard(rank, world, N)
    env = CudaVecEnv("ball3d", N, seed=3, device=rank, env_id_base=first)
    model = CudaA2C("MlpPolicy", env, seed=3, ent_coef=0.01, normalize_advantage=True)
    model.learn(world * N * 5 * 20)
    params = [torch.empty_like(model.params) for _ in range(world)]
    dist.all_gather(params, model.params)
    if rank == 0:
        out["params_equal"] = all(torch.equal(params[0], p) for p in params[1:])
        out["finite"] = bool(torch.isfinite(params[0]).all())
        out["updates"] = model.n_updates
        out["allreduce_impl"] = model.allreduce_impl
    dist.barrier()
    model.close()
    env.close()
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("impl", ["peer", "nccl"])
def test_two_rank_a2c_keeps_replicas_identical(impl):
    import torch.multiprocessing as mp

    world, port = 2, _free_port()
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_worker, args=(world, port, out, impl), nprocs=world, join=True)
        res = dict(out)
    assert res["params_equal"] and res["finite"] and res["updates"] == 20
    assert ("peer-memory" in res["allreduce_impl"]) == (impl == "peer")
