"""Reference half of the planning-rollout tests (tests/test_gpu_plan.py, tests/test_plan_cpu.py): the return recurrence of
gpd_plan (include/gpd.h) restated in torch, one elementwise operation per line so that each is rounded in the tensors'
dtype as the kernel rounds it, and the replica of a source handle (E*S envs holding the repeated state)."""
import torch


def plan_returns(reward, done, gamma):
    """reward (K, ...) float, done (K, ...) bool (terminated | truncated) -> (returns, done_step) of shape (...).

    G = 0; w = 1; for k: if not ended: G = G + w * r_k; then ended if done_k, else w = w * gamma."""
    K = reward.shape[0]
    g = torch.tensor(gamma, dtype=reward.dtype, device=reward.device)
    G = torch.zeros_like(reward[0])
    w = torch.ones_like(reward[0])
    ended = torch.zeros(reward.shape[1:], dtype=torch.bool, device=reward.device)
    step = torch.full(reward.shape[1:], K, dtype=torch.int32, device=reward.device)
    for k in range(K):
        wr = w * reward[k]
        G = torch.where(ended, G, G + wr)
        ends = ~ended & done[k]
        step = torch.where(ends, torch.full_like(step, k), step)
        wg = w * g
        w = torch.where(ended | done[k], w, wg)
        ended = ended | done[k]
    return G, step
