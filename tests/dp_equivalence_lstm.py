"""Multi-GPU check of the LSTM agents (RecurrentContinuousPPO with RecurrentContinuousLSTMActorCriticNetwork) under env-sharded data
parallelism, launched by torchrun (one rank per GPU):

  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29541 \
      tests/dp_equivalence_lstm.py

As in the RecurrentPPO section of tests/dp_equivalence.py: with every rank holding the SAME device Pendulum-v1 rollout and the same
permutation, the DP update (rank-local permutations, global advantage statistics and loss means, NCCL gradient sum before the clip)
equals the single-GPU update on one copy and the replicas stay identical; train() with distinct shards keeps the replicas identical."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "diamond-ppo_b200")):
    sys.path.insert(0, p)


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from diamond import RecurrentContinuousPPO, RecurrentContinuousPPOConfig
    from diamond.envs import DeviceVectorEnv
    from diamond.recurrent import RecurrentContinuousLSTMActorCriticNetwork as Net
    n_r, t_r = 64, 32
    # advantage_norm off: duplicating the data changes the unbiased (n - 1) standard deviation, which is all that would distinguish
    # the two runs
    cfg = RecurrentContinuousPPOConfig(num_envs=n_r, rollout_steps=t_r, num_epochs=2, num_minibatches=4, verbose=False, seed=11,
                                       total_steps=n_r * t_r * 1000, advantage_norm=False)

    def agent(dp):
        a = RecurrentContinuousPPO(DeviceVectorEnv.factory("Pendulum-v1", seed=11), cfg, network_cls=Net, dp=dp)
        a.envs.desc.env_offset = 0                                     # replicated data: every rank simulates the same environments
        a.engine.env_offset = 0
        a.current_observations, _ = a.envs.reset(seed=11)
        a.prev_dones = np.zeros(n_r, dtype=bool)
        a.current_hx = torch.zeros(1, n_r, a.state_dim, device=a.device)
        return a

    ag = agent(True)
    init = {k: v.detach().clone() for k, v in ag.network.state_dict().items()}
    ro = ag.rollout()
    np.random.seed(5)
    ag.learn(ro)
    torch.cuda.synchronize()
    flat = ag.engine.P.clone(); ref = flat.clone(); dist.broadcast(ref, src=0)
    ok = bool(torch.equal(flat, ref)) and bool(torch.isfinite(flat).all())
    if rank == 0:
        single = agent(False)
        single.network.load_state_dict(init)
        ro1 = single.rollout()
        assert torch.equal(ro1.obs, ro.obs) and torch.equal(ro1.actions, ro.actions), "replicated rollouts differ"
        np.random.seed(5)
        single.learn(ro1)
        torch.cuda.synchronize()
        worst = max(float((p_ - q_).abs().max() / q_.abs().max().clamp_min(1e-12))
                    for (_, p_), (_, q_) in zip(ag.network.named_parameters(), single.network.named_parameters()))
        lerr = float((ag.last_losses - single.last_losses).abs().max())
        ok = ok and worst <= 2e-5 and lerr <= 2e-5
        print(f"dp{world} [LSTM RecurrentContinuousPPO, NCCL gradient sum] vs single on replicated data: max param err {worst:.2e}, "
              f"max loss err {lerr:.2e} -> {'OK' if ok else 'FAIL'}", flush=True)
    cfg_t = RecurrentContinuousPPOConfig(num_envs=n_r, rollout_steps=t_r, verbose=False, seed=13, gru_hidden_dim=64, total_steps=n_r * t_r * 4)
    ag = RecurrentContinuousPPO(DeviceVectorEnv.factory("Pendulum-v1", seed=13), cfg_t, network_cls=Net, dp=True)
    ag.train()
    torch.cuda.synchronize()
    flat = ag.engine.P.clone(); ref = flat.clone(); dist.broadcast(ref, src=0)
    st0 = ag.envs.state.clone()
    gathered = [torch.empty_like(st0) for _ in range(world)]
    dist.all_gather(gathered, st0)
    train_ok = (bool(torch.equal(flat, ref)) and bool(torch.isfinite(flat).all()) and bool(torch.isfinite(ag.last_losses).all())
                and all(not torch.equal(gathered[0], g_) for g_ in gathered[1:]))
    if rank == 0:
        print(f"dp{world} [LSTM RecurrentContinuousPPO, device envs, train()]: replicas identical, shards distinct, finite -> "
              f"{'OK' if train_ok else 'FAIL'}", flush=True)
    t = torch.tensor([int(ok and train_ok)], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    dist.destroy_process_group()
    if int(t) != 1:
        sys.exit(1)


if __name__ == "__main__":
    main()
