"""TEST / BASELINE INFRASTRUCTURE ONLY -- the UNMODIFIED reference learner (habitat_baselines classes imported through
oracle/ref_shim.py from the install under oracle/_ref/) wired up the way
`PPOTrainer._update_agent` drives it (habitat-baselines/habitat_baselines/rl/ppo/ppo_trainer.py:484-523):

    rollouts.compute_returns(next_value, use_gae, gamma, tau)   # common/rollout_storage.py:174-205
    updater.update(rollouts)                                    # rl/ppo/ppo.py:301-332 (DDPPO: rl/ddppo/algo/ddppo.py:110-157)

on `device="cpu"` (bench.py --impl reference / cpu_baseline) or `device="cuda"` with the reference's own settings for a
CUDA run (TF32 cuDNN convolutions = torch default, `cudnn.benchmark = True` as rl/ver/ver_trainer.py:379 sets it,
DistributedDataParallel + NCCL through DDPPO.init_distributed for world > 1) -- the north-star's "reference PyTorch-CUDA
DD-PPO" competitor.  Never imported by the product package."""
from __future__ import annotations

import numpy as np
import torch

from . import ref_shim

PPO_KW = dict(clip_param=0.2, value_loss_coef=0.5, entropy_coef=0.01, lr=2.5e-4, eps=1e-5, max_grad_norm=0.2,
              use_clipped_value_loss=True)


class ReferenceLearner:
    def __init__(self, T: int, N: int, H: int, W: int, device, hidden=512, layers=2, rnn_type="LSTM", ppo_epoch=2,
                 num_mini_batch=2, use_normalized_advantage=False, distributed=False, state_dict=None, seed=100,
                 backbone="resnet18", sensors="pointnav", n_actions=4, n_categories=21):
        import collections

        R = ref_shim.ref()
        self.R = R
        sp = R.spaces
        self.device = torch.device(device)
        od = collections.OrderedDict()
        od["rgb"] = sp.Box(0, 255, (H, W, 3), np.uint8)
        if sensors == "pointnav":      # BASELINE config #2
            od["depth"] = sp.Box(0, 1, (H, W, 1), np.float32)
            od["pointgoal_with_gps_compass"] = sp.Box(-1e9, 1e9, (2,), np.float32)
        elif sensors == "objectnav":   # config #3
            od["depth"] = sp.Box(0, 1, (H, W, 1), np.float32)
            od["semantic"] = sp.Box(0, 2 ** 30, (H, W, 1), np.int32)
            od["objectgoal"] = sp.Box(0, n_categories - 1, (1,), np.int64)
            od["compass"] = sp.Box(-np.pi, np.pi, (1,), np.float32)
            od["gps"] = sp.Box(-1e9, 1e9, (2,), np.float32)
        else:                          # config #4 (imagenav)
            od["imagegoal"] = sp.Box(0, 255, (H, W, 3), np.uint8)
            od["compass"] = sp.Box(-np.pi, np.pi, (1,), np.float32)
            od["gps"] = sp.Box(-1e9, 1e9, (2,), np.float32)
        obs_space = sp.Dict(od)
        act_space = sp.Discrete(n_actions)
        torch.manual_seed(seed)
        pol = R.PointNavResNetPolicy(obs_space, act_space, hidden_size=hidden, num_recurrent_layers=layers,
                                     rnn_type=rnn_type, resnet_baseplanes=32, backbone=backbone,
                                     normalize_visual_inputs=True)
        if state_dict is not None:
            pol.load_state_dict(state_dict)
        pol.to(self.device)
        pol.train()
        cls = R.DDPPO if distributed else R.PPO
        self.updater = cls(pol, ppo_epoch=ppo_epoch, num_mini_batch=num_mini_batch,
                           use_normalized_advantage=use_normalized_advantage, **PPO_KW)
        if distributed:
            self.updater.init_distributed(find_unused_params=False)
        self.policy = pol
        self.storage = R.RolloutStorage(T, N, obs_space, act_space, pol)
        self.storage.to(self.device)
        self.T, self.N = T, N
        self.next_value = None

    def load_rollout(self, buffers, next_value):
        """buffers: a mapping with the RolloutStorage layout [T+1, N, ...] (ours or the recipe's); copied in."""
        b = self.storage.buffers
        for k, v in buffers["observations"].items():
            b["observations"][k].copy_(v)
        for k in ("recurrent_hidden_states", "masks", "rewards", "value_preds", "returns", "action_log_probs", "actions",
                  "prev_actions"):
            b[k].copy_(buffers[k])
        self.next_value = next_value.to(self.device).clone()

    def step(self, gamma=0.99, tau=0.95):
        self.storage.current_rollout_step_idxs = [self.T]
        self.storage.compute_returns(self.next_value, True, gamma, tau)
        return self.updater.update(self.storage)


def cuda_settings():
    """What a CUDA run of the reference uses: torch defaults (cuDNN TF32 on, matmul fp32) + cudnn.benchmark."""
    torch.backends.cudnn.benchmark = True
    return {"cudnn.benchmark": True, "cudnn.allow_tf32": bool(torch.backends.cudnn.allow_tf32),
            "cuda.matmul.allow_tf32": bool(torch.backends.cuda.matmul.allow_tf32)}
