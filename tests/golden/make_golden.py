"""Generates tests/golden/*.pt by running the UNMODIFIED reference classes (installed under
oracle/_ref by build(), imported through oracle/ref_shim.py) on recipe inputs.  Run where the
reference is installed:

    python tests/golden/make_golden.py [case ...]

The fixtures hold only small outputs (losses, per-frame values, per-tensor gradient norms ...);
inputs and weights are regenerated from seeds by tests/golden/recipe.py.
"""
from __future__ import annotations

import collections
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from oracle import ref_shim  # noqa: E402
from recipe import recipe_state_dict, synthetic_rollout  # noqa: E402

CASES = {
    # name: (T, N, H, W, rnn_type, layers, ppo_epoch, num_mini_batch, use_normalized_advantage)
    "small128": dict(T=8, N=4, H=128, W=128, rnn="LSTM", layers=2, epochs=2, mb=2, norm_adv=False, seed=11),
    "full256": dict(T=4, N=2, H=256, W=256, rnn="LSTM", layers=2, epochs=1, mb=1, norm_adv=True, seed=12),
    # BASELINE config #2 at the rollout length the bench runs (T = 128): 16 envs, minibatch = 8 envs x 128 steps = 1024
    # frames of 256x256 RGB-D through the 2-layer LSTM (BPTT over 128 steps, ~1 reset per 100 steps)
    "bench128": dict(T=128, N=16, H=256, W=256, rnn="LSTM", layers=2, epochs=1, mb=2, norm_adv=False, seed=13,
                     p_done=0.01, grad_samples=64),
}
NEXT_CASES = {
    # BASELINE config #3: ObjectNav DD-PPO, ResNet50 RGB(-D) + semantic channel, GRU-512
    "r50_objectnav": dict(T=4, N=2, H=128, W=128, backbone="resnet50", rnn="GRU", layers=1, n_actions=6, n_categories=21,
                          imagegoal=False, seed=31),
    # BASELINE config #4: ImageNav DD-PPO, ResNeXt50 dual encoder (observation + goal image), LSTM-512
    "rx50_imagenav": dict(T=4, N=2, H=128, W=128, backbone="resneXt50", rnn="LSTM", layers=2, n_actions=4,
                          n_categories=0, imagegoal=True, seed=41),
}
PPO_KW = dict(clip_param=0.2, value_loss_coef=0.5, entropy_coef=0.01, lr=2.5e-4, eps=1e-5, max_grad_norm=0.2,
              use_clipped_value_loss=True)


def build_reference(R, c):
    sp = R.spaces
    obs_space = sp.Dict({
        "rgb": sp.Box(0, 255, (c["H"], c["W"], 3), np.uint8),
        "depth": sp.Box(0, 1, (c["H"], c["W"], 1), np.float32),
        "pointgoal_with_gps_compass": sp.Box(-1e9, 1e9, (2,), np.float32),
    })
    act_space = sp.Discrete(4)
    pol = R.PointNavResNetPolicy(obs_space, act_space, hidden_size=512, num_recurrent_layers=c["layers"],
                                 rnn_type=c["rnn"], resnet_baseplanes=32, backbone="resnet18",
                                 normalize_visual_inputs=True)
    shapes = {k: tuple(v.shape) for k, v in pol.state_dict().items()}
    pol.load_state_dict(recipe_state_dict(shapes, c["seed"]))
    return pol, obs_space, act_space, shapes


def fill_storage(R, pol, obs_space, act_space, c):
    st = R.RolloutStorage(c["T"], c["N"], obs_space, act_space, pol)
    bufs, next_value = synthetic_rollout(c["T"], c["N"], c["H"], c["W"], 4, pol.num_recurrent_layers, 512, c["seed"],
                                         p_done=c.get("p_done", 1 / 25))
    for k, v in bufs["observations"].items():
        st.buffers["observations"][k].copy_(v)
    for k in ("recurrent_hidden_states", "masks", "rewards", "value_preds", "returns", "action_log_probs",
              "actions", "prev_actions"):
        st.buffers[k].copy_(bufs[k])
    st.current_rollout_step_idxs = [c["T"]]
    return st, next_value


def _next_cases(R, only):
    """BASELINE configs #3 / #4 ("next" rows): ResNet50 + GRU with the ObjectNav sensors, ResNeXt50 dual encoder + LSTM."""
    from recipe import objectnav_rollout  # noqa: E402
    for name, c in NEXT_CASES.items():
        if only and name not in only and "next" not in only:
            continue
        sp = R.spaces
        H, W = c["H"], c["W"]
        od = collections.OrderedDict()
        od["rgb"] = sp.Box(0, 255, (H, W, 3), np.uint8)
        if c["imagegoal"]:
            od["imagegoal"] = sp.Box(0, 255, (H, W, 3), np.uint8)
        else:
            od["depth"] = sp.Box(0, 1, (H, W, 1), np.float32)
            od["semantic"] = sp.Box(0, 2 ** 30, (H, W, 1), np.int32)
            od["objectgoal"] = sp.Box(0, c["n_categories"] - 1, (1,), np.int64)
        od["compass"] = sp.Box(-np.pi, np.pi, (1,), np.float32)
        od["gps"] = sp.Box(-1e9, 1e9, (2,), np.float32)
        obs_space = sp.Dict(od)
        act_space = sp.Discrete(c["n_actions"])
        torch.manual_seed(c["seed"])
        pol = R.PointNavResNetPolicy(obs_space, act_space, hidden_size=512, num_recurrent_layers=c["layers"],
                                     rnn_type=c["rnn"], resnet_baseplanes=32, backbone=c["backbone"],
                                     normalize_visual_inputs=True)
        shapes = {k: tuple(v.shape) for k, v in pol.state_dict().items()}
        pol.load_state_dict(recipe_state_dict(shapes, c["seed"]))
        st = R.RolloutStorage(c["T"], c["N"], obs_space, act_space, pol)
        bufs, next_value = objectnav_rollout(c["T"], c["N"], H, W, c["n_actions"], pol.num_recurrent_layers, 512,
                                             c["seed"], c["n_categories"], c["imagegoal"])
        for k, v in bufs["observations"].items():
            st.buffers["observations"][k].copy_(v)
        for k in ("recurrent_hidden_states", "masks", "rewards", "value_preds", "returns", "action_log_probs",
                  "actions", "prev_actions"):
            st.buffers[k].copy_(bufs[k])
        st.current_rollout_step_idxs = [c["T"]]
        st.compute_returns(next_value, True, 0.99, 0.95)
        ppo = R.PPO(pol, ppo_epoch=1, num_mini_batch=1, use_normalized_advantage=False, **PPO_KW)
        adv = ppo.get_advantages(st)
        pol.train()
        torch.manual_seed(1000 + c["seed"])
        batch = next(iter(st.data_generator(adv, 1)))
        values, lp, ent, hid, _ = pol.evaluate_actions(batch["observations"], batch["recurrent_hidden_states"],
                                                       batch["prev_actions"], batch["masks"], batch["actions"],
                                                       batch["rnn_build_seq_info"])
        ratio = torch.exp(lp - batch["action_log_probs"])
        action_loss = -torch.min(batch["advantages"] * ratio, batch["advantages"] * torch.clamp(ratio, 0.8, 1.2))
        delta = values.detach() - batch["value_preds"]
        vv = torch.where(delta.abs() < 0.2, values, batch["value_preds"] + delta.clamp(-0.2, 0.2))
        value_loss = 0.5 * (vv - batch["returns"]) ** 2
        total = 0.5 * value_loss.mean() + action_loss.mean() - 0.01 * ent.mean()
        pol.zero_grad()
        total.backward()
        out = dict(case=c, shapes=shapes, visual_keys=list(pol.net.visual_encoder.visual_keys),
                   returns=st.buffers["returns"].clone(), advantages=adv.clone(), mb_env_inds_seed=1000 + c["seed"],
                   eval_values=values.detach(), eval_log_probs=lp.detach(), eval_entropy=ent.detach(),
                   eval_hidden=hid.detach(),
                   mb_losses=dict(value_loss=value_loss.mean().item(), action_loss=action_loss.mean().item(),
                                  dist_entropy=ent.mean().item(), total=total.item()),
                   grad_norms={k: p.grad.norm().item() for k, p in pol.named_parameters()},
                   n_params=sum(p.numel() for p in pol.parameters()))
        torch.save(out, os.path.join(HERE, f"{name}.pt"))
        print(name, out["mb_losses"], "params", out["n_params"], "tensors", len(shapes))



def _ppo_loss_case(R):
    """PPO._update_from_batch's loss section (rl/ppo/ppo.py:164-299) on random features through linear heads: the
    inputs, the head weights and the metrics the reference logs, for tests/test_oracle.py."""
    torch.manual_seed(0)
    B, A = 64, 4
    feats = torch.randn(B, 512)

    class FakeAC(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.lin = torch.nn.Linear(512, A)
            self.val = torch.nn.Linear(512, 1)

        def evaluate_actions(self, obs, h, pa, m, actions, info):
            dist = torch.distributions.Categorical(logits=self.lin(obs))
            return self.val(obs), dist.log_prob(actions.squeeze(-1)).unsqueeze(-1), dist.entropy().unsqueeze(-1), h, {}

        def policy_parameters(self):
            return self.parameters()

        def aux_loss_parameters(self):
            return {}

    ac = FakeAC()
    ppo = R.PPO(ac, clip_param=0.2, ppo_epoch=1, num_mini_batch=1, value_loss_coef=0.5, entropy_coef=0.01, lr=0.0,
                eps=1e-5, max_grad_norm=0.2, use_clipped_value_loss=True, use_normalized_advantage=False)
    batch = dict(observations=feats, recurrent_hidden_states=None, prev_actions=None, masks=None,
                 actions=torch.randint(0, A, (B, 1)), action_log_probs=torch.randn(B, 1) * 0.3 - 1.4,
                 advantages=torch.randn(B, 1), value_preds=torch.randn(B, 1) * 0.3, returns=torch.randn(B, 1))
    heads = {k: v.detach().clone() for k, v in ac.state_dict().items()}
    inputs = {k: v.clone() for k, v in batch.items() if torch.is_tensor(v)}
    metrics = collections.defaultdict(list)
    ppo._update_from_batch(batch, 0, None, metrics)
    out = dict(inputs=inputs, heads=heads, metrics={k: float(torch.as_tensor(v[0]).detach()) for k, v in metrics.items()})
    torch.save(out, os.path.join(HERE, "ppo_loss.pt"))
    print("ppo_loss", out["metrics"])


def main():
    R = ref_shim.ref()
    torch.set_num_threads(8)
    only = sys.argv[1:]
    if not only or "ppo_loss" in only:
        _ppo_loss_case(R)
        if only == ["ppo_loss"]:
            return
    for name, c in CASES.items():
        if only and name not in only:
            continue
        torch.manual_seed(c["seed"])
        pol, obs_space, act_space, shapes = build_reference(R, c)
        st, next_value = fill_storage(R, pol, obs_space, act_space, c)
        out = {"case": c, "shapes": shapes}
        # --- compute_returns + advantages (rollout_storage.py:174-205, ppo.py:139-157)
        st.compute_returns(next_value, True, 0.99, 0.95)
        out["returns"] = st.buffers["returns"].clone()
        out["value_preds_after"] = st.buffers["value_preds"].clone()
        ppo = R.PPO(pol, ppo_epoch=c["epochs"], num_mini_batch=c["mb"], use_normalized_advantage=c["norm_adv"], **PPO_KW)
        out["advantages"] = ppo.get_advantages(st).clone()
        ppo_nn = R.PPO(pol, ppo_epoch=1, num_mini_batch=1, use_normalized_advantage=not c["norm_adv"], **PPO_KW)
        out["advantages_other_mode"] = ppo_nn.get_advantages(st).clone()

        # --- actor path (rl/ppo/policy.py:322-357): eval-mode act(deterministic) / get_value on rollout step 1 (all envs)
        pol.eval()
        with torch.no_grad():
            o1 = {k: v[1] for k, v in st.buffers["observations"].items()}
            a = pol.act(o1, st.buffers["recurrent_hidden_states"][1], st.buffers["prev_actions"][1],
                        st.buffers["masks"][1], deterministic=True)
            feats, _, _ = pol.net(o1, st.buffers["recurrent_hidden_states"][1], st.buffers["prev_actions"][1],
                                  st.buffers["masks"][1])
            out["act"] = dict(values=a.values.clone(), actions=a.actions.clone(), action_log_probs=a.action_log_probs.clone(),
                              rnn_hidden_states=a.rnn_hidden_states.clone(),
                              logits=pol.action_distribution(feats).logits.clone(),
                              get_value=pol.get_value(o1, st.buffers["recurrent_hidden_states"][1],
                                                      st.buffers["prev_actions"][1], st.buffers["masks"][1]).clone())
        # --- one minibatch: evaluate_actions + loss + backward (no optimizer step)
        pol.train()
        torch.manual_seed(1000 + c["seed"])  # randperm of data_generator
        adv = ppo.get_advantages(st)
        batch = next(iter(st.data_generator(adv, c["mb"])))
        out["mb_env_inds_seed"] = 1000 + c["seed"]
        stats_before = {k: v.clone() for k, v in pol.state_dict().items() if "running_mean_and_var" in k}
        values, lp, ent, hid, _ = pol.evaluate_actions(batch["observations"], batch["recurrent_hidden_states"],
                                                       batch["prev_actions"], batch["masks"], batch["actions"],
                                                       batch["rnn_build_seq_info"])
        out["eval_values"], out["eval_log_probs"], out["eval_entropy"] = values.detach(), lp.detach(), ent.detach()
        out["eval_hidden"] = hid.detach()
        out["running_stats_after_one_forward"] = {k: v.clone() for k, v in pol.state_dict().items()
                                                  if "running_mean_and_var" in k}
        ratio = torch.exp(lp - batch["action_log_probs"])
        s1 = batch["advantages"] * ratio
        s2 = batch["advantages"] * torch.clamp(ratio, 0.8, 1.2)
        action_loss = -torch.min(s1, s2)
        delta = values.detach() - batch["value_preds"]
        vclip = batch["value_preds"] + delta.clamp(-0.2, 0.2)
        vv = torch.where(delta.abs() < 0.2, values, vclip)
        value_loss = 0.5 * (vv - batch["returns"]) ** 2
        total = 0.5 * value_loss.mean() + action_loss.mean() - 0.01 * ent.mean()
        pol.zero_grad()
        total.backward()
        out["mb_losses"] = dict(value_loss=value_loss.mean().item(), action_loss=action_loss.mean().item(),
                                dist_entropy=ent.mean().item(), total=total.item())
        out["grad_norms"] = {k: p.grad.norm().item() for k, p in pol.named_parameters()}
        ns = c.get("grad_samples", 16)
        out["grad_samples"] = {k: p.grad.flatten()[:: max(1, p.numel() // ns)][:ns].clone()
                               for k, p in pol.named_parameters()}
        # restore running stats so update() starts from the recipe state
        pol.load_state_dict({**pol.state_dict(), **stats_before})
        pol.zero_grad()

        # --- full PPO.update (ppo.py:301-332)
        torch.manual_seed(2000 + c["seed"])
        metrics = ppo.update(st)
        out["update_metrics"] = metrics
        out["param_norms_after_update"] = {k: v.float().norm().item() for k, v in pol.state_dict().items()}
        out["param_samples_after_update"] = {k: v.flatten()[:: max(1, v.numel() // 16)][:16].clone()
                                             for k, v in pol.state_dict().items()}
        torch.save(out, os.path.join(HERE, f"{name}.pt"))
        print(name, "losses", out["mb_losses"], "update", {k: round(v, 6) for k, v in metrics.items()})

    if only and all(o == "next" or o in NEXT_CASES for o in only):
        return _next_cases(R, only)
    # --- BASELINE config #1: PointNavBaselinePolicy (SimpleCNN depth-only 128x128 + GRU), num_envs = 2
    c = dict(T=8, N=2, H=128, W=128, seed=21, mb=1)
    sp = R.spaces
    obs_space = sp.Dict({"depth": sp.Box(0, 1, (c["H"], c["W"], 1), np.float32),
                         "pointgoal_with_gps_compass": sp.Box(-1e9, 1e9, (2,), np.float32)})
    pol = R.PointNavBaselinePolicy(obs_space, sp.Discrete(4), hidden_size=512)
    shapes = {k: tuple(v.shape) for k, v in pol.state_dict().items()}
    pol.load_state_dict(recipe_state_dict(shapes, c["seed"]))
    st = R.RolloutStorage(c["T"], c["N"], obs_space, sp.Discrete(4), pol)
    bufs, next_value = synthetic_rollout(c["T"], c["N"], c["H"], c["W"], 4, 1, 512, c["seed"], rgb=False)
    for k, v in bufs["observations"].items():
        st.buffers["observations"][k].copy_(v)
    for k in ("recurrent_hidden_states", "masks", "rewards", "value_preds", "returns", "action_log_probs", "actions",
              "prev_actions"):
        st.buffers[k].copy_(bufs[k])
    st.current_rollout_step_idxs = [c["T"]]
    st.compute_returns(next_value, True, 0.99, 0.95)
    ppo = R.PPO(pol, ppo_epoch=1, num_mini_batch=1, use_normalized_advantage=False, **PPO_KW)
    adv = ppo.get_advantages(st)
    torch.manual_seed(1000 + c["seed"])
    batch = next(iter(st.data_generator(adv, 1)))
    values, lp, ent, hid, _ = pol.evaluate_actions(batch["observations"], batch["recurrent_hidden_states"],
                                                   batch["prev_actions"], batch["masks"], batch["actions"],
                                                   batch["rnn_build_seq_info"])
    ratio = torch.exp(lp - batch["action_log_probs"])
    action_loss = -torch.min(batch["advantages"] * ratio, batch["advantages"] * torch.clamp(ratio, 0.8, 1.2))
    delta = values.detach() - batch["value_preds"]
    vv = torch.where(delta.abs() < 0.2, values, batch["value_preds"] + delta.clamp(-0.2, 0.2))
    value_loss = 0.5 * (vv - batch["returns"]) ** 2
    total = 0.5 * value_loss.mean() + action_loss.mean() - 0.01 * ent.mean()
    pol.zero_grad()
    total.backward()
    out = dict(case=c, shapes=shapes, returns=st.buffers["returns"].clone(), advantages=adv.clone(),
               value_preds_after=st.buffers["value_preds"].clone(), mb_env_inds_seed=1000 + c["seed"],
               eval_values=values.detach(), eval_log_probs=lp.detach(), eval_entropy=ent.detach(), eval_hidden=hid.detach(),
               mb_losses=dict(value_loss=value_loss.mean().item(), action_loss=action_loss.mean().item(),
                              dist_entropy=ent.mean().item(), total=total.item()),
               grad_norms={k: p.grad.norm().item() for k, p in pol.named_parameters()})
    pol.zero_grad()
    torch.manual_seed(2000 + c["seed"])
    out["update_metrics"] = ppo.update(st)
    torch.save(out, os.path.join(HERE, "baseline_cnn.pt"))
    print("baseline_cnn", out["mb_losses"], {k: round(v, 6) for k, v in out["update_metrics"].items()})

    _next_cases(R, only)

    # --- RNN packed-sequence semantics (test/test_rnn_state_encoder.py) golden
    torch.manual_seed(3)
    enc = R.build_rnn_state_encoder(32, 32, rnn_type="LSTM", num_layers=2)
    T, N = 13, 5
    masks = torch.rand(T * N, 1) > (1 / 25)
    x = torch.randn(T * N, 32)
    hidden = torch.randn(N, 4, 32)
    info = R.build_rnn_build_seq_info(device=torch.device("cpu"),
                                      build_fn_result=R.build_pack_info_from_dones(
                                          torch.logical_not(masks).view(T, N).numpy()))
    with torch.no_grad():
        y, h = enc(x, hidden, masks, info)
    torch.save(dict(state_dict=enc.state_dict(), x=x, masks=masks, hidden=hidden, out=y, hidden_out=h, T=T, N=N),
               os.path.join(HERE, "rnn_lstm.pt"))
    print("rnn golden saved")


if __name__ == "__main__":
    main()
