"""Runs on the GPU box: how far is the REFERENCE's own CUDA path (cuDNN TF32 convolutions, torch defaults) from its
fp32 CPU path?  Same minibatch as tests/golden/bench128.pt (T=128 x 8 envs = 1024 frames of 256x256 RGB-D), unmodified
reference classes from oracle/_ref, per-tensor gradient cosine / norm ratio of device=cuda vs device=cpu.
Writes gpurun_out/ref_cuda_precision.json -- the yardstick the hb200 precision bars are read against."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from helpers import gather_minibatch, load_golden, minibatch_env_inds, recipe_state_dict, synthetic_rollout  # noqa: E402
from oracle import ref_shim  # noqa: E402


def run(R, G, device, allow_tf32=True):
    c = G["case"]
    sp = R.spaces
    obs_space = sp.Dict({"rgb": sp.Box(0, 255, (c["H"], c["W"], 3), np.uint8),
                         "depth": sp.Box(0, 1, (c["H"], c["W"], 1), np.float32),
                         "pointgoal_with_gps_compass": sp.Box(-1e9, 1e9, (2,), np.float32)})
    pol = R.PointNavResNetPolicy(obs_space, sp.Discrete(4), hidden_size=512, num_recurrent_layers=c["layers"],
                                 rnn_type=c["rnn"], resnet_baseplanes=32, backbone="resnet18", normalize_visual_inputs=True)
    pol.load_state_dict(recipe_state_dict(G["shapes"], c["seed"]))
    pol.to(device).train()
    torch.backends.cudnn.allow_tf32 = allow_tf32
    bufs, _ = synthetic_rollout(c["T"], c["N"], c["H"], c["W"], 4, 2 * c["layers"], 512, c["seed"], p_done=c.get("p_done", 1 / 25))
    bufs["value_preds"], bufs["returns"] = G["value_preds_after"].clone(), G["returns"].clone()
    inds = minibatch_env_inds(G["mb_env_inds_seed"], c["N"], c["mb"])[0]
    b = gather_minibatch(bufs, G["advantages"], inds, c["T"])
    mv = lambda t: t.to(device)  # noqa: E731
    obs = {k: mv(v) for k, v in b["observations"].items()}
    info = R.build_rnn_build_seq_info(device=torch.device(device), build_fn_result=R.build_pack_info_from_dones(
        torch.logical_not(b["masks"]).view(c["T"], -1).numpy()))
    values, lp, ent, hid, _ = pol.evaluate_actions(obs, mv(b["recurrent_hidden_states"]), mv(b["prev_actions"]),
                                                   mv(b["masks"]), mv(b["actions"]), info)
    ratio = torch.exp(lp - mv(b["action_log_probs"]))
    adv = mv(b["advantages"])
    action_loss = -torch.min(adv * ratio, adv * torch.clamp(ratio, 0.8, 1.2))
    delta = values.detach() - mv(b["value_preds"])
    vv = torch.where(delta.abs() < 0.2, values, mv(b["value_preds"]) + delta.clamp(-0.2, 0.2))
    value_loss = 0.5 * (vv - mv(b["returns"])) ** 2
    total = 0.5 * value_loss.mean() + action_loss.mean() - 0.01 * ent.mean()
    pol.zero_grad()
    total.backward()
    return ({k: p.grad.detach().cpu() for k, p in pol.named_parameters()},
            dict(value_loss=value_loss.mean().item(), action_loss=action_loss.mean().item(), dist_entropy=ent.mean().item()),
            values.detach().cpu())


def main():
    name = sys.argv[1] if len(sys.argv) > 1 else "bench128"
    G = load_golden(name)
    R = ref_shim.ref()
    torch.set_num_threads(min(32, len(os.sched_getaffinity(0))))
    g_cpu, l_cpu, v_cpu = run(R, G, "cpu")
    out = {"case": name, "losses_cpu": l_cpu, "golden_losses": G["mb_losses"]}
    for tag, tf32 in (("cuda_tf32_default", True), ("cuda_fp32_convs", False)):
        g, l, v = run(R, G, "cuda", tf32)
        rows = []
        for k in g_cpu:
            a, r = g[k].flatten().double(), g_cpu[k].flatten().double()
            rows.append((float(a @ r / (a.norm() * r.norm() + 1e-30)), float(a.norm() / (r.norm() + 1e-30)), k))
        rows.sort()
        enc = [x for x in rows if "visual_encoder" in x[2]]
        out[tag] = {"losses": l, "values_max_abs_diff": float((v - v_cpu).abs().max()),
                    "worst_cos": rows[:6], "min_cos_encoder": min(x[0] for x in enc),
                    "median_cos_encoder": sorted(x[0] for x in enc)[len(enc) // 2],
                    "max_norm_dev_encoder": max(abs(x[1] - 1) for x in enc)}
        print(tag, json.dumps(out[tag])[:600])
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump(out, open(os.path.join(ROOT, "gpurun_out", "ref_cuda_precision.json"), "w"), indent=1)


if __name__ == "__main__":
    main()
