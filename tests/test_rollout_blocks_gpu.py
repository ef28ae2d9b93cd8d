"""Fused random-policy rollouts that start and end inside a 16-step action block.

The fast rollout kernel (n % 32 == 0) runs over the 16-step blocks of the action stream: a call whose step index is not a
multiple of 16 starts with a partial block, and one that ends early stops inside a block.  Consecutive calls of 5, 40, 23,
2 and 70 steps put both cases at every call boundary (the first call and the 2-step call end before the next block
begins), and the last call also crosses spare-refill windows.  Each call must give the actions, observations, rewards,
dones and final state of single steps.
"""
import numpy as np
import pytest
import torch

from oracle import envs_oracle as eo

pytestmark = pytest.mark.gpu

TASKS = ("basic", "ball3d", "gridworld", "push", "walljump", "brickbreak", "bicycle", "glider")
CALLS = (5, 40, 23, 2, 70)


@pytest.mark.parametrize("task", TASKS)
def test_unaligned_fused_rollouts_equal_single_steps(task):
    from three_mlagents_b200.vec_env import CudaVecEnv

    n, seed = 1024, 33
    d = eo.TASKS[task][0]
    fused, single = CudaVecEnv(task, n, seed=seed), CudaVecEnv(task, n, seed=seed)
    cur = single.reset_tensor().clone()
    ids = np.arange(n, dtype=np.uint64)
    t0 = 0
    for T in CALLS:
        obs = torch.empty((T, n, d), device="cuda")
        act = torch.empty((T, n), dtype=torch.int32, device="cuda")
        rew = torch.empty((T, n), device="cuda")
        done = torch.empty((T, n), dtype=torch.uint8, device="cuda")
        fused.rollout_random(T, obs, act, rew, done)
        assert fused.step_count == t0 + T
        for t in range(T):
            a = eo.random_actions(task, seed, ids, t0 + t)
            assert np.array_equal(act[t].cpu().numpy(), a), (t0, t)
            assert torch.equal(obs[t], cur), (t0, t)
            b = single.step_tensor(torch.from_numpy(a).cuda())
            assert torch.equal(rew[t].view(torch.int32), b["rew"].view(torch.int32)), (t0, t)
            assert torch.equal(done[t], b["done"]), (t0, t)
            cur = b["obs"].clone()
        assert fused.get_state().tobytes() == single.get_state().tobytes(), t0
        t0 += T
    fused.close(); single.close()
