#!/usr/bin/env python
"""bench.py -- DD-PPO learner frames/sec on BASELINE.json config #2:
PointNav DD-PPO, ResNet18 (baseplanes 32, GroupNorm 16) RGB-D 256x256, LSTM-512 x 2,
num_envs = 64 per rank, T = 128, ppo_epoch = 2, num_mini_batch = 2, synthetic observations.

One "step" = one learner iteration on a full rollout: RolloutStorage.compute_returns (GAE) +
PPO.update (2 epochs x 2 minibatches of 4096 frames: forward, backward, [all-reduce], clip,
Adam), each timed step from the same policy and optimizer state.  value = world * T * N / t_step  (the reference's perf/fps definition,
habitat-baselines/habitat_baselines/rl/ppo/ppo_trainer.py:595-598, learner part).

    python bench.py --gpus 1 --steps K --warmup W           # this repo's sm_100a path
    python bench.py --impl reference ...                     # the UNMODIFIED reference classes (oracle/_ref) on the CPU
    python bench.py --impl torch_cuda ...                    # ... and on CUDA (TF32 cuDNN, cudnn.benchmark; DDP + NCCL at N > 1)
    torchrun --nproc-per-node N bench.py --gpus N ...        # one rank per GPU, NCCL

Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

_PPO = dict(clip_param=0.2, value_loss_coef=0.5, entropy_coef=0.01, lr=2.5e-4, eps=1e-5, max_grad_norm=0.2, gamma=0.99, tau=0.95)
# BASELINE.json configs[1..3]; config 2 is the headline (the default), 3 / 4 are selected with --config
WORKLOADS = {
    2: dict(cfg=dict(T=128, N=64, H=256, W=256, hidden=512, layers=2, rnn="LSTM", backbone="resnet18", ppo_epoch=2,
                     num_mini_batch=2, sensors="pointnav", n_actions=4, **_PPO),
            metric="DD-PPO learner frames/sec (ResNet18 RGB-D 256x256)",
            text="BASELINE configs[1]: PointNav DD-PPO ResNet18 RGB-D 256x256, LSTM-512x2, 64 envs/rank, T=128, 2 epochs x 2 "
                 "minibatches (4096 frames each), synthetic obs"),
    3: dict(cfg=dict(T=64, N=32, H=256, W=256, hidden=512, layers=1, rnn="GRU", backbone="resnet50", ppo_epoch=4,
                     num_mini_batch=2, sensors="objectnav", n_actions=6, n_categories=21, **_PPO),
            metric="DD-PPO learner frames/sec (ResNet50 RGB-D + semantic 256x256, ObjectNav)",
            text="BASELINE configs[2]: ObjectNav DD-PPO ResNet50 RGB-D + int32 semantic channel 256x256, objectgoal / compass "
                 "/ gps embeddings, GRU-512, 32 envs/rank, T=64, 4 epochs x 2 minibatches (1024 frames each), synthetic obs"),
    4: dict(cfg=dict(T=64, N=32, H=256, W=256, hidden=512, layers=2, rnn="LSTM", backbone="resneXt50", ppo_epoch=4,
                     num_mini_batch=2, sensors="imagenav", n_actions=4, **_PPO),
            metric="DD-PPO learner frames/sec (ResNeXt50 dual encoder RGB 256x256, ImageNav)",
            text="BASELINE configs[3]: ImageNav DD-PPO ResNeXt50 dual encoder (observation + goal image) RGB 256x256, compass "
                 "/ gps embeddings, LSTM-512x2, 32 envs/rank, T=64, 4 epochs x 2 minibatches (1024 frames each), synthetic obs"),
}
CONFIG_ID = 2
CFG = WORKLOADS[2]["cfg"]
METRIC = WORKLOADS[2]["metric"]


def select_workload(config_id: int) -> None:
    global CONFIG_ID, CFG, METRIC
    CONFIG_ID, CFG, METRIC = config_id, WORKLOADS[config_id]["cfg"], WORKLOADS[config_id]["metric"]


def make_spaces():
    from habitat_lab_b200 import synthetic as syn
    if CFG["sensors"] == "pointnav":
        return syn.pointnav_spaces(CFG["H"], CFG["W"], CFG["n_actions"])
    if CFG["sensors"] == "objectnav":
        return syn.objectnav_spaces(CFG["H"], CFG["W"], CFG["n_actions"], CFG["n_categories"])
    return syn.imagenav_spaces(CFG["H"], CFG["W"], CFG["n_actions"])


def make_policy(hb, obs_space, act_space):
    return hb.PointNavResNetPolicy(obs_space, act_space, hidden_size=CFG["hidden"], num_recurrent_layers=CFG["layers"],
                                   rnn_type=CFG["rnn"], resnet_baseplanes=32, backbone=CFG["backbone"],
                                   normalize_visual_inputs=True)


def fill(st, seed, obs_space):
    from habitat_lab_b200.synthetic import fill_rollout_
    if CFG["sensors"] == "pointnav":
        return fill_rollout_(st, seed=seed)
    return fill_rollout_(st, seed=seed, observation_space=obs_space, n_actions=CFG["n_actions"])
# algorithmic work per frame of config #2 (SURVEY.md section 8d / DESIGN.md)
CONV_FWD_GFLOP = 0.3376
CONV_TRAIN_GFLOP = 0.9614  # config #2: fwd + dgrad + wgrad, no dgrad for conv1 (SURVEY 8d); other configs: from the engine


def conv_train_gflop_per_frame(policy):
    """algorithmic conv FLOPs of one training frame-pass (fwd + dgrad + wgrad, no dgrad for the stems), all encoders"""
    tot = 0.0
    for eng in policy._engines.values():
        for c in eng.convs:
            f = 2.0 * c.out_hw[0] * c.out_hw[1] * c.co * (c.ci_real // c.conv_groups) * c.k * c.k
            tot += f * (2 if c is eng.stem else 3)
    return tot * 1e-9


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], bf16=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower() == "active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
# reference arm: the reference's CPU learner (oracle port) on the host cores
# ---------------------------------------------------------------------------------------------
def _cpu_threads():
    """Threads for the CPU learner: all host cores the reference's op-level parallelism can use.  Beyond ~32
    threads torch's intra-op pools only add contention on these small convolutions (measured: 128 threads
    is >100x slower than 16 on the GPU box), so the count is capped and reported as `cores`."""
    return max(1, min(len(os.sched_getaffinity(0)), 32))


CPU_SAMPLE = dict(T=128, N=4)   # bounded CPU sample: the config's rollout length, 4 of its envs per iteration (~4 s each)
if os.environ.get("HB200_CPU_SAMPLE"):   # "T,N": the contract test shrinks the sample, the wording below follows
    CPU_SAMPLE = dict(zip(("T", "N"), (int(v) for v in os.environ["HB200_CPU_SAMPLE"].split(","))))


def _recipe_rollout(T, N, seed=5):
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from recipe import objectnav_rollout, synthetic_rollout
    layers_h = CFG["layers"] * (2 if CFG["rnn"] == "LSTM" else 1)
    if CFG["sensors"] == "pointnav":
        return synthetic_rollout(T, N, CFG["H"], CFG["W"], 4, layers_h, CFG["hidden"], seed, p_done=1.0 / 250.0)
    return objectnav_rollout(T, N, CFG["H"], CFG["W"], CFG["n_actions"], layers_h, CFG["hidden"], seed,
                             CFG.get("n_categories", 0), CFG["sensors"] == "imagenav")


def _ref_kwargs():
    return dict(hidden=CFG["hidden"], layers=CFG["layers"], rnn_type=CFG["rnn"], backbone=CFG["backbone"],
                sensors=CFG["sensors"], n_actions=CFG["n_actions"], n_categories=CFG.get("n_categories", 0),
                ppo_epoch=CFG["ppo_epoch"], num_mini_batch=CFG["num_mini_batch"])


def _make_cpu_learner(T=CPU_SAMPLE["T"], N=CPU_SAMPLE["N"]):
    """The UNMODIFIED reference (oracle/_ref through the import shim): RolloutStorage.compute_returns
    + PPO.update on device="cpu" -- the reference's own CPU PPO path."""
    from oracle.ref_learner import ReferenceLearner

    learner = ReferenceLearner(T, N, CFG["H"], CFG["W"], "cpu", **_ref_kwargs())
    bufs, next_value = _recipe_rollout(T, N)
    learner.load_rollout(bufs, next_value)
    return learner.step, T * N


def _cpu_sample_text(threads):
    return (f"learner iteration(s) of T={CPU_SAMPLE['T']} x N={CPU_SAMPLE['N']} frames ({CFG['H']}x{CFG['W']}, config "
            f"#{CONFIG_ID} sensors and policy; the config has T={CFG['T']}, N={CFG['N']} envs per rank; {CFG['ppo_epoch']} epochs x {CFG['num_mini_batch']} minibatches of "
            f"{CPU_SAMPLE['T'] * CPU_SAMPLE['N'] // CFG['num_mini_batch']} frames), unmodified reference classes on "
            f"device=cpu, {threads} threads")


def _cpu_learner_sample(threads, updates):
    torch.set_num_threads(threads)
    step, frames = _make_cpu_learner()
    step()  # warm-up
    t0 = time.perf_counter()
    for _ in range(updates):
        step()
    dt = time.perf_counter() - t0
    return updates * frames / dt, f"{updates} " + _cpu_sample_text(threads) + f" after 1 warm-up, {dt:.1f} s"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = _cpu_threads()
    torch.set_num_threads(threads)
    step, frames = _make_cpu_learner()
    for _ in range(max(1, args.warmup)):
        step()
    ms = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        step()
        ms.append((time.perf_counter() - t0) * 1e3)
    v = frames * len(ms) / (sum(ms) * 1e-3)
    sample = "each step = 1 " + _cpu_sample_text(threads)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": max(1, args.warmup), "ms_per_step": sum(ms) / len(ms),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": _config(args.gpus),
            "cpu_baseline": {"value": v, "unit": "frames/s", "cores": threads, "kind": "reference", "sample": sample},
            "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(line)


# ---------------------------------------------------------------------------------------------
# the competitor: the unmodified reference on CUDA (TF32 cuDNN, cudnn.benchmark, DDP + NCCL)
# ---------------------------------------------------------------------------------------------
def torch_cuda_measure(dev, world, rollout_buffers, next_value, steps, warmup, seed):
    """frames/s of the reference's own PyTorch-CUDA DD-PPO learner on config #2 (same T, N, minibatching, same
    synthetic rollout tensors as the hb200 arm), CUDA events, barrier both sides, max over ranks."""
    from oracle.ref_learner import ReferenceLearner, cuda_settings

    settings = cuda_settings()
    T, N = CFG["T"], CFG["N"]
    learner = ReferenceLearner(T, N, CFG["H"], CFG["W"], dev, distributed=world > 1, seed=seed, **_ref_kwargs())
    learner.load_rollout(rollout_buffers, next_value)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, warmup)):
        learner.step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = None
    for _ in range(steps):
        out = learner.step()
    e1.record()
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
    ms = ms.item()
    peak_gb = torch.cuda.max_memory_allocated(dev) / 2 ** 30
    del learner
    torch.cuda.empty_cache()
    return {"value": world * T * N * steps / (ms * 1e-3), "unit": "frames/s", "ms_per_step": ms / steps, "steps": steps,
            "warmup": max(3, warmup), "n_gpus": world, "kind": "reference (unmodified habitat_baselines classes, device=cuda)",
            "settings": settings, "parallelism": "DistributedDataParallel + NCCL (DDPPO.init_distributed)" if world > 1 else "single process",
            "peak_mem_gb": round(peak_gb, 1), "learner_metrics": {k: round(float(v), 6) for k, v in (out or {}).items()}}


def run_torch_cuda(args):
    """bench.py --impl torch_cuda: the competitor arm alone, launched like the hb200 arm (torchrun for N > 1)."""
    import habitat_lab_b200 as hb
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=dev)
    T, N = CFG["T"], CFG["N"]
    obs_space, act_space = make_spaces()

    class _Shape:   # RolloutStorage only reads these two attributes of the policy
        num_recurrent_layers, recurrent_hidden_size = CFG["layers"] * (2 if CFG["rnn"] == "LSTM" else 1), CFG["hidden"]

    st = hb.RolloutStorage(T, N, obs_space, act_space, _Shape())
    st.to(dev)
    next_value = fill(st, 100 + rank * N, obs_space)
    res = torch_cuda_measure(dev, world, st.buffers, next_value, args.steps, args.warmup, seed=100)
    if rank == 0:
        line = {"impl": "torch_cuda", "metric": METRIC, "value": res["value"], "unit": "frames/s", "n_gpus": world,
                "steps": args.steps, "warmup": res["warmup"], "ms_per_step": res["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "tf32 convs / fp32", "data": "synthetic",
                "config": _config(world), "torch_cuda": res}
        _emit(line)
    if world > 1:
        torch.distributed.destroy_process_group()


def _config(n):
    return {"workload": WORKLOADS[CONFIG_ID]["text"],
            "num_envs_per_rank": CFG["N"], "rollout_steps": CFG["T"], "frames_per_step_per_rank": CFG["T"] * CFG["N"],
            "parallelism": f"dp{n}", "l2_policy": "inputs (3.8 GB of observations per rank) far exceed the 126 MB L2"}


# ---------------------------------------------------------------------------------------------
# hb200 arm
# ---------------------------------------------------------------------------------------------
class LearnerState:
    """What one learner step reads besides the rollout: the policy's parameters and buffers (RunningMeanAndVar), the
    Adam moments and step count, and the CPU generator that data_generator's minibatch split draws from.  The timed steps
    each start from the state captured before warm-up, so they compute from the same inputs in every run: the gradient
    kernels accumulate with atomics, and a state carried from step to step would drift apart between runs by far more
    than one step's rounding."""

    def __init__(self, policy, optimizer):
        self.policy, self.opt = policy, optimizer
        flat = optimizer._bind()
        self.params = flat["params"].clone()
        self.buffers = [b.detach().clone() for b in policy.buffers()]
        self.m, self.v, self.step = optimizer._m.clone(), optimizer._v.clone(), optimizer._step
        self.rng = torch.get_rng_state()

    @torch.no_grad()
    def restore(self):
        self.opt._bind()["params"].copy_(self.params)
        for b, s in zip(self.policy.buffers(), self.buffers):
            b.copy_(s)
        self.opt._m.copy_(self.m)
        self.opt._v.copy_(self.v)
        self.opt._step = self.step
        for st in self.opt.state.values():
            st["step"].fill_(float(self.step))
        self.policy.mark_weights_changed()
        torch.set_rng_state(self.rng)


def run_hb200(args):
    import habitat_lab_b200 as hb
    from habitat_lab_b200 import ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hb200 path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        # NCCL_DEBUG is left exactly as the launcher set it (the driver reads the communicator's rank count from the
        # INFO log); main() points fd 1 at stderr, so whatever NCCL prints cannot reach the JSON line
        dist.init_process_group("nccl", device_id=dev)
    lib = hb.load()
    T, N = CFG["T"], CFG["N"]
    torch.manual_seed(100 + rank * N)  # habitat.seed=100, ppo_trainer.py:207-215
    obs_space, act_space = make_spaces()
    policy = make_policy(hb, obs_space, act_space).to(dev)
    cls = hb.DDPPO if world > 1 else hb.PPO
    ppo = cls(policy, clip_param=CFG["clip_param"], ppo_epoch=CFG["ppo_epoch"], num_mini_batch=CFG["num_mini_batch"],
              value_loss_coef=CFG["value_loss_coef"], entropy_coef=CFG["entropy_coef"], lr=CFG["lr"], eps=CFG["eps"],
              max_grad_norm=CFG["max_grad_norm"], use_clipped_value_loss=True, use_normalized_advantage=False)
    if world > 1:
        ppo.init_distributed(find_unused_params=False)
    policy.train()
    st = hb.RolloutStorage(T, N, obs_space, act_space, policy)
    st.to(dev)
    next_value = fill(st, 100 + rank * N, obs_space)

    def learner_step():
        st.current_rollout_step_idxs = [T]
        st.compute_returns(next_value, True, CFG["gamma"], CFG["tau"])
        return ppo.update(st)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, before_each=None):
        """device time of `steps` calls of fn; with before_each, the sum over the calls alone (what before_each
        enqueues between them is not counted)"""
        barrier()
        n_ev = steps if before_each is not None else 1
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_ev)]
        out = None
        if before_each is None:
            ev[0][0].record()
            for _ in range(steps):
                out = fn()
            ev[0][1].record()
        else:
            for e0, e1 in ev:
                before_each()
                e0.record()
                out = fn()
                e1.record()
        barrier()
        ms = torch.tensor([sum(e0.elapsed_time(e1) for e0, e1 in ev)], device=dev)
        if world > 1:
            torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
        return ms.item(), out

    start = LearnerState(policy, ppo.optimizer)   # every timed step starts from here
    for _ in range(max(args.warmup, 3)):
        learner_step()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = lib.hb200_launch_count()
    ms, metrics = timed(learner_step, args.steps, before_each=start.restore)
    launches = lib.hb200_launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:   # before the e2e leg below trains the policy further
        dump_outputs(args.dump_outputs, metrics, st.buffers["returns"], policy)
    frames = world * T * N * args.steps
    value = frames / (ms * 1e-3)
    cross_rank = cross_rank_equality(policy, dev, world) if world > 1 else None

    # ---- e2e: same iteration through the public API with HOST inputs: every step's rollout (observations and
    # scalars) is copied from pinned host memory and the metrics dict goes back to the host, all inside the timed
    # region.  The copies run on a copy stream into the second of two device rollout storages while the learner
    # works on the first (a double-buffered input pipeline): step k+1's H2D overlaps step k's update; the first
    # step's copy is fully exposed.  Exactly `steps` copies of 3.86 GB happen between the two timing events.
    keys = ("rewards", "masks", "actions", "prev_actions", "action_log_probs", "value_preds", "recurrent_hidden_states")
    host = {}
    h2d = 0
    for k, v in list(st.buffers["observations"].items()) + [(k, st.buffers[k]) for k in keys]:
        host[k] = torch.empty(v.shape, dtype=v.dtype, pin_memory=True)
        host[k].copy_(v)
        h2d += v.numel() * v.element_size()
    nv_host = next_value.cpu().pin_memory()
    h2d += nv_host.numel() * 4
    st_b = hb.RolloutStorage(T, N, obs_space, act_space, policy)
    st_b.to(dev)
    slots = [dict(st=st, nv=torch.empty_like(next_value), ready=torch.cuda.Event(), free=torch.cuda.Event()),
             dict(st=st_b, nv=torch.empty_like(next_value), ready=torch.cuda.Event(), free=torch.cuda.Event())]
    copy_stream = torch.cuda.Stream(device=dev)

    def h2d_async(slot):
        copy_stream.wait_event(slot["free"])          # the learner has finished with this storage
        with torch.cuda.stream(copy_stream):
            for k in slot["st"].buffers["observations"]:
                slot["st"].buffers["observations"][k].copy_(host[k], non_blocking=True)
            for k in keys:
                slot["st"].buffers[k].copy_(host[k], non_blocking=True)
            slot["nv"].copy_(nv_host, non_blocking=True)
            slot["ready"].record(copy_stream)

    def e2e_run(steps):
        for sl in slots:
            sl["free"].record()
        h2d_async(slots[0])
        out = None
        for i in range(steps):
            sl = slots[i % 2]
            if i + 1 < steps:
                h2d_async(slots[(i + 1) % 2])
            torch.cuda.current_stream().wait_event(sl["ready"])
            sl["st"].current_rollout_step_idxs = [T]
            sl["st"].compute_returns(sl["nv"], True, CFG["gamma"], CFG["tau"])
            out = ppo.update(sl["st"])   # returns python floats: one D2H read of the metric vector per step
            sl["free"].record()
        return out

    e2e_run(2)
    e2e_steps = max(1, args.steps)
    ms_e2e, _ = timed(lambda: e2e_run(e2e_steps), 1)
    e2e_value = world * T * N * e2e_steps / (ms_e2e * 1e-3)

    # ---- the competitor, in the same process group right after the hb200 measurement: the UNMODIFIED reference on
    # CUDA (TF32 cuDNN convs, cudnn.benchmark, DDP + NCCL for world > 1) on the same synthetic rollout tensors
    torch_cuda = None
    if not args.no_torch_cuda:
        del st_b, slots, host
        torch.cuda.empty_cache()
        try:
            torch_cuda = torch_cuda_measure(dev, world, st.buffers, next_value, args.steps, args.warmup, seed=100)
            torch_cuda["hb200_over_torch_cuda"] = value / torch_cuda["value"]
            torch_cuda["hb200_e2e_over_torch_cuda"] = e2e_value / torch_cuda["value"]
        except Exception as e:   # e.g. oracle/_ref not installed: report, never lose the hb200 line
            torch_cuda = {"unavailable": repr(e)[:300]}
    line = None
    if rank == 0:
        peaks = _peaks()
        roof = kernel_roofline(hb, ops, policy, st, dev, peaks)
        hbm_roofs = hbm_kernel_rooflines(hb, ops, dev, peaks) if world == 1 else None
        cores = _cpu_threads()
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            try:
                fps, sample = _cpu_learner_sample(cores, updates=2)   # ~15-30 s of host work
                cpu = {"value": fps, "unit": "frames/s", "cores": cores, "kind": "reference", "sample": sample}
            except Exception as e:
                cpu = {"unavailable": repr(e)[:300]}
        # ---- informational: the actor half of the loop (SURVEY 8f row 1, "next"): T sequential act() calls at batch N
        # on the same synthetic observations (eager and CUDA-graph replay), so that learner-only and learner+actor
        # frames/s can be read side by side.  Measured last and fully guarded: it can never cost the bench line.
        actor = None
        if world == 1:
            try:
                ob = st.buffers["observations"]
                hid0 = st.buffers["recurrent_hidden_states"][0].clone()

                def rollout(step_fn):
                    h = hid0
                    for t in range(T):
                        out = step_fn({k: v[t] for k, v in ob.items()}, h, st.buffers["prev_actions"][t],
                                      st.buffers["masks"][t])
                        h = out.rnn_hidden_states
                    return h

                with torch.no_grad():
                    rollout(policy.act)
                    ms_eager, _ = timed(lambda: rollout(policy.act), 2)
                ms_eager /= 2
                actor = {"ms_per_rollout_eager": ms_eager, "steps": T, "batch": N}
                ms_best = ms_eager
                try:
                    ga = hb.GraphedActor(policy, {k: v[0] for k, v in ob.items()}, hid0, st.buffers["prev_actions"][0],
                                         st.buffers["masks"][0])
                    rollout(ga)
                    ms_graph, _ = timed(lambda: rollout(ga), 2)
                    actor["ms_per_rollout_cuda_graph"] = ms_graph / 2
                    ms_best = min(ms_best, ms_graph / 2)
                except Exception as e:
                    actor["cuda_graph_error"] = repr(e)[:200]
                actor["frames_per_s_learner_plus_actor"] = T * N / ((ms / args.steps + ms_best) * 1e-3)
                actor["note"] = ("act() at batch 64 is launch-bound (~100 small kernels per step; weight images cached "
                                 "across calls); GraphedActor replays the captured step")
            except Exception as e:
                actor = {"error": repr(e)[:200]}
        line = {"metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": _config(world),
                "clocks": clocks, "gpu_launches": int(launches),
                "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": int(h2d),
                        "d2h_bytes_per_step": 14 * 4, "ms_per_step": ms_e2e / e2e_steps, "steps": e2e_steps,
                        "h2d": "pinned host -> device on a copy stream, double-buffered across steps; first copy exposed"},
                "roofline": roof, "hbm_kernel_rooflines": hbm_roofs, "cpu_baseline": cpu, "actor": actor,
                "torch_cuda_baseline": torch_cuda, "cross_rank_equality": cross_rank,
                "conv_tensor_frac_of_step": (world * T * N * CFG["ppo_epoch"] * conv_train_gflop_per_frame(policy) * 1e-3 * args.steps)
                / (ms * 1e-3) / (peaks["bf16_sustained"] * world),
                "learner_metrics": {k: round(float(v), 6) for k, v in metrics.items()}}
        _emit(line)
    if world > 1:
        torch.distributed.destroy_process_group()


# ---------------------------------------------------------------------------------------------
# BASELINE configs[4]: PPO.update minibatch sweep -- GAE-scan HBM GB/s + conv tensor-pipe fraction vs the reference
# ---------------------------------------------------------------------------------------------
def run_sweep(args):
    """frames per rollout in {1k, 4k, 16k, 64k, 256k} = T=128 x N in {8, 32, 128, 512, 2048} envs (SURVEY 8d).
    Per size: (a) the fused GAE + advantage kernel on the [T+1, N] scalars -- time, algorithmic GB/s (17 B per element) and
    the reference's `RolloutStorage.compute_returns` python loop on the same CUDA tensors; (b) one PPO minibatch
    (frames / 2, forward + loss + backward + clip/Adam) through hb200 and through the unmodified reference on CUDA:
    ms, frames/s, algorithmic conv TFLOP/s and its fraction of the measured bf16 peak.  Minibatches above 16384
    frames are not materialised (their rollout alone is 30-120 GB): the 64k / 256k rows repeat the 16k-frame pass, which
    is what a larger minibatch is to these kernels (same tiles, more of them); the reference arm stops where its
    autograd graph no longer fits next to it (8192 frames = 100 GB)."""
    import habitat_lab_b200 as hb
    from habitat_lab_b200 import ops

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    hb.load()
    peaks = _peaks()
    obs_space, act_space = make_spaces()
    T = CFG["T"]
    rows = []

    def ev_ms(fn, reps):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    ref_ok = True
    for N in (8, 32, 128, 512, 2048):
        frames = T * N
        row = {"frames": frames, "envs": N}
        # ---- (a) GAE + advantages
        g = torch.Generator(device=dev).manual_seed(N)
        rewards = torch.randn(T + 1, N, 1, device=dev, generator=g)
        values = torch.randn(T + 1, N, 1, device=dev, generator=g)
        masks = torch.rand(T + 1, N, 1, device=dev, generator=g) > 0.004
        nv = torch.randn(N, device=dev, generator=g)
        returns, adv = torch.empty_like(rewards), torch.empty_like(rewards)
        stats = torch.zeros(4, dtype=torch.float64, device=dev)
        ms = ev_ms(lambda: ops.gae_adv(rewards, values, masks, nv, returns, adv, stats, T, 0.99, 0.95, True, 1), 50)
        by = 17.0 * (T + 1) * N
        row["gae"] = {"ms": ms, "gbs": by / ms * 1e-6, "frac_hbm": by / ms * 1e-6 / peaks["hbm"],
                      "note": "launch-latency bound below ~1 MB (17 B x (T+1) x N = %.2f MB)" % (by * 1e-6)}

        def ref_gae():   # rollout_storage.py:174-205 on the same CUDA tensors
            vp = values.clone()
            vp[T] = nv.view(-1, 1)
            gae = 0
            for step in reversed(range(T)):
                delta = rewards[step] + 0.99 * vp[step + 1] * masks[step + 1] - vp[step]
                gae = delta + 0.99 * 0.95 * gae * masks[step + 1]
                returns[step] = gae + vp[step]
        row["gae"]["torch_cuda_ms"] = ev_ms(ref_gae, 3)
        del rewards, values, masks, returns, adv
        # ---- (b) one minibatch through the learner
        mb_frames = min(frames // 2, 16384)
        n_env_mb = mb_frames // T
        row["minibatch_frames"] = frames // 2
        row["materialised_minibatch_frames"] = mb_frames
        policy = make_policy(hb, obs_space, act_space).to(dev)
        policy.train()
        ppo = hb.PPO(policy, clip_param=CFG["clip_param"], ppo_epoch=1, num_mini_batch=1, value_loss_coef=CFG["value_loss_coef"],
                     entropy_coef=CFG["entropy_coef"], lr=CFG["lr"], eps=CFG["eps"], max_grad_norm=CFG["max_grad_norm"],
                     use_clipped_value_loss=True, use_normalized_advantage=False)
        st = hb.RolloutStorage(T, n_env_mb, obs_space, act_space, policy)
        st.to(dev)
        nvv = fill(st, 100 + N, obs_space)

        def step():
            st.current_rollout_step_idxs = [T]
            st.compute_returns(nvv, True, CFG["gamma"], CFG["tau"])
            return ppo.update(st)

        for _ in range(2):
            step()
        ms = ev_ms(step, 3)
        gf = conv_train_gflop_per_frame(policy) * mb_frames
        row["hb200"] = {"ms_per_minibatch": ms, "frames_per_s": mb_frames / ms * 1e3, "conv_tflops": gf / ms,
                        "conv_frac_of_bf16_peak": gf / ms / peaks["bf16_sustained"]}
        bufs, nv_keep = st.buffers, nvv
        del policy, ppo
        torch.cuda.empty_cache()
        if ref_ok and mb_frames <= 8192:
            try:
                from oracle.ref_learner import ReferenceLearner, cuda_settings
                cuda_settings()
                kw = _ref_kwargs()
                kw.update(ppo_epoch=1, num_mini_batch=1)
                learner = ReferenceLearner(T, n_env_mb, CFG["H"], CFG["W"], dev, seed=100, **kw)
                learner.load_rollout(bufs, nv_keep)
                for _ in range(2):
                    learner.step()
                ms_r = ev_ms(learner.step, 3)
                row["torch_cuda"] = {"ms_per_minibatch": ms_r, "frames_per_s": mb_frames / ms_r * 1e3,
                                     "conv_tflops": gf / ms_r, "hb200_over_torch_cuda": ms_r / ms}
                del learner
            except Exception as e:   # out of memory at the large sizes: stop trying
                row["torch_cuda"] = {"unavailable": repr(e)[:200]}
                ref_ok = False
        del st, bufs
        torch.cuda.empty_cache()
        rows.append(row)
        print("sweep", json.dumps(row), file=sys.stderr, flush=True)
    _emit({"metric": "PPO.update minibatch sweep (BASELINE configs[4])", "unit": "per-size table", "n_gpus": 1,
           "config": {"workload": "T=128 x N in {8,32,128,512,2048} envs of config #%d; minibatch = frames / 2" % CONFIG_ID},
           "peaks": {"hbm_gbs": peaks["hbm"], "bf16_tflops_sustained": peaks["bf16_sustained"], "source": peaks["src"]},
           "rows": rows, "data": "synthetic"})



DUMP_MAX_ELEMS = 12 << 20   # per array: 48 MB of float32, so that one policy state plus the small outputs stay under 64 MB


def dump_outputs(out_dir, metrics, returns, policy):
    """What the last timed learner step produced, for comparing two builds output for output: every learner metric
    PPO.update returned (`metric_<key>.npy`, float64), the GAE returns left in the rollout storage (`returns.npy`) and
    every floating-point tensor of the updated policy's state_dict, flattened and concatenated in state_dict order
    (`policy_state.npy`, float32).  An array above DUMP_MAX_ELEMS is replaced by the elements at a fixed, seeded set of
    positions (`<name>_sample.npy`), the same positions for the same array size.  Every timed step starts from the same
    state (LearnerState), so two runs with the same arguments differ only by the rounding of the atomic gradient sums."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    arrays = {f"metric_{k}": np.float64(v) for k, v in metrics.items()}
    arrays["returns"] = returns.detach().float().cpu().numpy()
    state = [t.detach().float().flatten() for t in policy.state_dict().values() if t.is_floating_point()]
    arrays["policy_state"] = torch.cat(state).cpu().numpy()
    for name, a in arrays.items():
        if a.size > DUMP_MAX_ELEMS:
            idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))
            name, a = f"{name}_sample", a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def cross_rank_equality(policy, dev, world):
    """After the timed optimizer steps every rank must hold bit-identical parameters and RunningMeanAndVar buffers
    (what DDP guarantees for the reference, test/test_ddppo_reduce.py:111-118): rank 0's copies are broadcast and
    compared byte for byte on every rank, the verdict is reduced with MIN."""
    import torch.distributed as dist

    flat = policy.flatten_parameters_()
    tensors = [("flat_params", flat["params"])] + [(n, b) for n, b in policy.named_buffers()]
    out = {}
    for name, t in tensors:
        ref = t.detach().clone()
        dist.broadcast(ref, src=0)
        ok = torch.tensor([1 if torch.equal(ref, t.detach()) else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        out[name.split(".")[-1] if name != "flat_params" else name] = bool(ok.item())
    out["all_equal"] = all(out.values())
    out["world"] = world
    return out


def _ncu_traffic():
    """DRAM bytes per launch of the most frequent conv kernel, from the committed `ncu --set full` capture of this
    round (profiles/*_ncu_traffic.json; offline measurement, not taken during the bench run)."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu_traffic.json")))
    if not files:
        return None
    with open(files[-1]) as f:
        t = json.load(f)
    return {"kernel": t["kernel"], "dram_bytes_per_launch": t["traffic_bytes_per_launch"],
            "algorithmic_bytes_per_launch": 2.0 * 2 * 4096 * 32 * 32 * 32, "source": t["source"]}


def kernel_roofline(hb, ops, policy, st, dev, peaks):
    """Live CUDA-event timing of the dominant kernel family (the tcgen05 implicit-GEMM convolutions)
    on the real config-#2 minibatch buffers: algorithmic FLOPs of every conv launch of one
    minibatch pass (forward + dgrad + wgrad) / the summed launch durations."""
    eng = policy._engine_()
    B = CFG["T"] * CFG["N"] // CFG["num_mini_batch"]
    ws = eng._ws.get((B, True))
    if ws is None:
        return None
    idx = {id(c): i for i, c in enumerate(eng.convs)}

    def t_ms(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    inputs = {id(eng.stem): ws["x0"]}
    x = ws["x1"]
    for j, (convs, cd) in enumerate(eng.blocks):
        for i, c in enumerate(convs):
            inputs[id(c)] = x if i == 0 else ws[f"a{j}_{i - 1}"]
        if cd is not None:
            inputs[id(cd)] = x
        x = ws[f"o{j}"]
    inputs[id(eng.comp)] = x
    per = {"fwd": [0.0, 0.0], "dgrad": [0.0, 0.0], "wgrad": [0.0, 0.0]}
    detail = []
    sol = [0.0, 0.0]
    for c in eng.convs:
        i = idx[id(c)]
        s = c.shape(B)
        flop = 2.0 * B * c.out_hw[0] * c.out_hw[1] * c.co * (c.ci_real // c.conv_groups) * c.k * c.k
        xin, y = inputs[id(c)], ws[f"y{i}"]
        stats = ws[f"st{i}"]
        fused_into = None
        if getattr(c, "s2_pair", None) is not None:
            # stride-2 block entry: ONE launch serves this 3x3 conv and the block's 1x1 downsample conv (conv_s2.cu);
            # its time is booked here, the downsample row below carries only its FLOPs (and its own weight gradient)
            d = c.s2_pair
            kd = idx[id(d)]
            yd, std = ws[f"y{kd}"], ws[f"st{kd}"]
            tf = t_ms(lambda: ops.conv_s2_fwd(xin, c.wh, y, yd, B, c.in_hw[0], c.in_hw[1], c.ci, c.co, d.co,
                                              stats_a=stats, groups_a=c.groups, stats_b=std, groups_b=d.groups))
            if c.dw_s2 is not None:
                tw = t_ms(lambda: ops.conv_s2_wgrad(xin, y, c.dw_s2, B, c.in_hw[0], c.in_hw[1], c.ci, c.co))
            else:
                tw = t_ms(lambda: ops.conv_wgrad(xin, y, c.dw_acc, s))
        elif getattr(c, "s2_main", None) is not None:
            fused_into = c.s2_main
            tf = 0.0
            tw = t_ms(lambda: ops.conv_wgrad(xin, y, c.dw_acc, s))
        elif c.stem_s2d:
            tf = t_ms(lambda: ops.conv_halo(xin, c.wh, y, B, c.out_hw[0], c.out_hw[1], 16, c.co, 4, 0, gn_stats=stats, gn_groups=c.groups))
            tw = t_ms(lambda: ops.conv_halo_wgrad(xin, y, c.dw_acc, B, c.out_hw[0], c.out_hw[1], 16, c.co, 4))
        elif c.halo:
            tf = t_ms(lambda: ops.conv_halo(xin, c.wh, y, B, c.in_hw[0], c.in_hw[1], c.ci, c.co, 3, 0, gn_stats=stats, gn_groups=c.groups))
            tw = t_ms(lambda: ops.conv_halo_wgrad(xin, y, c.dw_acc, B, c.in_hw[0], c.in_hw[1], c.ci, c.co, 3))
        else:
            tf = t_ms(lambda: ops.conv_fwd(xin, c.wp, y, s, stats, c.groups))
            if getattr(c, "halo_w", False):
                tw = t_ms(lambda: ops.conv_halo_wgrad(xin, y, c.dw_acc, B, c.in_hw[0], c.in_hw[1], c.ci, c.co, 3))
            else:
                tw = t_ms(lambda: ops.conv_wgrad(xin, y, c.dw_acc, s))
        per["fwd"][0] += flop; per["fwd"][1] += tf
        per["wgrad"][0] += flop; per["wgrad"][1] += tw
        td = None
        if c is not eng.stem:
            dx = ws["g0"][: xin.numel()].view_as(xin)
            if getattr(c, "s2_pair", None) is not None:
                d = c.s2_pair
                yd = ws[f"y{idx[id(d)]}"]
                td = t_ms(lambda: ops.conv_s2_dgrad(y, yd, c.wht, dx, B, c.in_hw[0], c.in_hw[1], c.ci, c.co, d.co))
            elif fused_into is not None:
                td = 0.0
            else:
                td = t_ms(lambda: eng._dgrad(c, y, dx, B))
            per["dgrad"][0] += flop; per["dgrad"][1] += td
        # speed of light of each launch: max(tensor time, HBM time of reading both operands / writing the result once)
        nbytes = 2.0 * (xin.numel() + y.numel())
        t_sol = max(flop / (peaks["bf16"] * 1e12), nbytes / (peaks["hbm"] * 1e9)) * 1e3
        bound = "tensor" if flop / (peaks["bf16"] * 1e12) > nbytes / (peaks["hbm"] * 1e9) else "hbm"
        sol[0] += t_sol * (2 if td is None else 3)
        sol[1] += tf + tw + (td or 0.0)
        detail.append({"conv": f"{c.ci_real}->{c.co} k{c.k}s{c.stride} @{c.in_hw[0]}"
                               + (" (fwd / dgrad fused into the 3x3 stride-2 launch)" if fused_into is not None else ""),
                       "gflop": flop * 1e-9,
                       "mbytes": nbytes * 1e-6, "bound": bound, "sol_ms": t_sol,
                       "fwd_ms": tf, "dgrad_ms": td, "wgrad_ms": tw})
    flops = sum(v[0] for v in per.values())
    ms = sum(v[1] for v in per.values())
    achieved = flops / (ms * 1e-3) * 1e-12
    return {"kernel": "conv_halo_ws_kernel / conv_s2_*_kernel / conv_igemm_kernel / conv_*wgrad_kernel (tcgen05, all 21 convs of "
                      "one 4096-frame minibatch pass, forward + dgrad + wgrad)",
            "bound": "tensor", "achieved": achieved, "peak": peaks["bf16"], "unit": "TFLOP/s",
            "frac": achieved / peaks["bf16"], "peak_source": peaks["src"] + " (burst: kernels timed alone)",
            "traffic": _ncu_traffic(),
            "speed_of_light": {"note": "per launch max(FLOPs / bf16 peak, (input + output bytes) / HBM peak): the 32- and "
                                       "64-channel layers are HBM-bound, not tensor-bound", "sol_ms": sol[0],
                               "measured_ms": sol[1], "frac": sol[0] / sol[1] if sol[1] else None},
            "by_pass": {k: {"tflops": (v[0] / (v[1] * 1e-3) * 1e-12) if v[1] else None, "ms": v[1]} for k, v in per.items()},
            "per_layer": detail}


def hbm_kernel_rooflines(hb, ops, dev, peaks):
    """HBM-bound kernels timed alone on batched instances >> L2 (the config-#2 sizes of GAE / loss / Adam are
    launch-latency bound: 8192 x 17 B), CUDA events, an L2-sized scratch write between repetitions."""
    out = {}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def t_ms(fn, reps=5):
        fn()
        ts = []
        for _ in range(reps):
            flush.fill_(1)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return sorted(ts)[len(ts) // 2]

    # GAE + advantages: T = 128, N = 655,360 envs -> 17 B x (T+1) x N = 1.44 GB
    T, N = 128, 655360
    g = torch.Generator(device=dev).manual_seed(1)
    rewards = torch.randn(T + 1, N, 1, device=dev, generator=g)
    values = torch.randn(T + 1, N, 1, device=dev, generator=g)
    masks = torch.rand(T + 1, N, 1, device=dev, generator=g) > 0.004
    nv = torch.randn(N, device=dev, generator=g)
    returns, adv = torch.empty_like(rewards), torch.empty_like(rewards)
    stats = torch.zeros(4, dtype=torch.float64, device=dev)
    ms = t_ms(lambda: ops.gae_adv(rewards, values, masks, nv, returns, adv, stats, T, 0.99, 0.95, True, 1))
    by = 17.0 * (T + 1) * N
    out["gae_adv"] = {"workload": f"T={T} x N={N} (batched: cfg #2 is 8192 elements = launch bound)", "bytes": by,
                      "ms": ms, "achieved": by / ms * 1e-6, "peak": peaks["hbm"], "unit": "GB/s",
                      "frac": by / ms * 1e-6 / peaks["hbm"]}
    del rewards, values, masks, returns, adv
    # clip + Adam on 64 x the policy's parameter count: 32 B/param
    n = 8481125 * 16
    bufs = [torch.randn(n, device=dev) * 0.01 for _ in range(2)] + [torch.zeros(n, device=dev) for _ in range(2)]
    ws, gn = ops.clip_adam_workspace(n, dev), torch.zeros(1, device=dev)
    ms = t_ms(lambda: ops.clip_adam(bufs[0], bufs[1], bufs[2], bufs[3], 2.5e-4, (0.9, 0.999), 1e-5, 0.0, 0.2, 1.0, 1, gn, ws))
    by = 32.0 * n
    out["clip_adam"] = {"workload": f"{n} params (16 x cfg #2)", "bytes": by, "ms": ms, "achieved": by / ms * 1e-6,
                        "peak": peaks["hbm"], "unit": "GB/s", "frac": by / ms * 1e-6 / peaks["hbm"]}
    del bufs
    # heads + PPO loss fwd+bwd: B = 1M frames, H = 512: features in + d_features out = 4096 B/frame
    B, H, A = 1 << 20, 512, 4
    feats = torch.randn(B, H, device=dev)
    o = dict(values=torch.empty(B, device=dev), log_probs=torch.empty(B, device=dev), entropy=torch.empty(B, device=dev),
             d_features=torch.empty(B, H, device=dev), d_w_act=torch.empty(A, H, device=dev), d_b_act=torch.empty(A, device=dev),
             d_w_val=torch.empty(H, device=dev), d_b_val=torch.empty(1, device=dev), metrics=torch.empty(12, device=dev))
    small = [torch.randn(B, device=dev) for _ in range(4)]
    acts = torch.randint(0, A, (B,), device=dev)
    w_a, b_a, w_v, b_v = torch.randn(A, H, device=dev) * 0.01, torch.zeros(A, device=dev), torch.randn(1, H, device=dev) * 0.05, torch.zeros(1, device=dev)
    wsl = ops.ppo_loss_workspace(B, H, A, dev)
    ms = t_ms(lambda: ops.ppo_loss(feats, w_a, b_a, w_v, b_v, acts, small[0], small[1], small[2], small[3], 0.2, 0.5, 0.01,
                                   True, True, o, wsl))
    by = (2 * H * 4 + 64 + 2 * H * 4) * float(B)  # features read twice (loss + head-weight gradient) + d_features + scalars
    out["ppo_loss_fwd_bwd"] = {"workload": f"B={B} frames, H=512, A=4", "bytes": by, "ms": ms, "achieved": by / ms * 1e-6,
                               "peak": peaks["hbm"], "unit": "GB/s", "frac": by / ms * 1e-6 / peaks["hbm"]}
    return out


_REAL_STDOUT = None


def _emit(line) -> None:
    """The one JSON line of the contract, written to the process's ORIGINAL stdout (see main)."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    # stdout must carry exactly one JSON line, but libraries print there too (NCCL's "NCCL version ..." banner comes out
    # on stdout whatever NCCL_DEBUG says): point fd 1 at stderr for the whole run and keep the real stdout for _emit.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="hb200", choices=["hb200", "reference", "torch_cuda"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4],
                    help="BASELINE.json configs[N-1]; 2 (the headline metric) is the default")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-torch-cuda", action="store_true", help="skip the reference PyTorch-CUDA competitor leg")
    ap.add_argument("--sweep", action="store_true", help="BASELINE configs[4]: minibatch-size sweep (1 GPU), one JSON line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed learner step computed as DIR/<name>.npy (hb200 arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.sweep or args.impl != "hb200"):
        ap.error("--dump-outputs applies to the hb200 arm only")
    select_workload(args.config)
    if args.sweep:
        return run_sweep(args)
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "torch_cuda":
        run_torch_cuda(args)
    else:
        run_hb200(args)


if __name__ == "__main__":
    main()
