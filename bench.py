#!/usr/bin/env python
"""bench.py -- env-steps/sec of the PHC hot path (fused obs+reward+PPO) on N B200s of one node.

    python bench.py --gpus 1 --steps 5 --warmup 3                (N > 1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference ...                         (the reference algorithm's CPU port on the host cores)

One "step" = one PPO epoch of the BASELINE.json configuration `4096 envs, 1xB200: fused obs+reward+GAE+PPO on synthetic
24-body SMPL rigid-body state` PER GPU (weak scaling: every rank owns 4096 envs):
  32 rollout steps x [ simulator snapshot -> fused env step kernel (MotionLib query, self/task obs, reward, reset, AMP
  obs) -> masked reset path -> obs normalise -> actor + critic forward -> Gaussian sample -> critic on next obs ]
  + discriminator reward over 32x4096 AMP windows + GAE + advantage normalisation
  + 6 mini-epochs x 8 minibatches of 16384: actor/critic/disc forward + backward (incl. gradient penalty), one NCCL
    all-reduce of the flat gradient bucket, global-norm clip, Adam           (phc/data/cfg/learning/im.yaml)
=> 131072 env-steps per step per GPU.  Networks: im.yaml sizes (934->1024->512->69/1, disc 1960->1024->512->1), fp32
(3xTF32 tensor-core emulation), random init; simulator state and motion clips are seeded synthetic data (one 60-300
frame clip per env, ~1 GB of frame tables per GPU, so frames come from HBM, not L2).

Printed JSON (one line, rank 0): see the driver contract in the task statement; `roofline` is the fused env-step
kernel against the measured HBM copy bandwidth, `cpu_baseline` the oracle port timed on this host's cores.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

NUM_ENVS = 4096
MAX_CPU_THREADS = 64                    # threads of the CPU arm: batches this small stop scaling (and start thrashing) beyond that
HORIZON = 32
ALGO_BYTES_PER_ENV_STEP = 9384          # SURVEY.md section 8(d): core algorithmic bytes of the fused obs+reward kernel, J=24
METRIC = "env-steps/sec (fused obs+reward+PPO) at 4096 envs/GPU"


_T0 = time.perf_counter()


def note(msg: str) -> None:
    """Progress line on stderr (stdout carries exactly one JSON line)."""
    print(f"[bench {time.perf_counter() - _T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="phc_b200", choices=["phc_b200", "reference"])
    ap.add_argument("--num-envs", type=int, default=NUM_ENVS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-points", action="store_true", help="skip the 16384 / 65536-env points of the env-step roofline")
    ap.add_argument("--workload", default="smpl", choices=sorted(WORKLOADS), help="configuration of the headline numbers (default: the one the metric is quoted on)")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary configurations (H1, PNN big nets) reported as extra_configs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed epochs, write what the last one computed to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "phc_b200":
        ap.error("--dump-outputs needs --impl phc_b200")
    return args


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------------------------
# clocks sampling during the timed region
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if val.strip().lower() == "active":
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [s for s in sm if s > 0.5 * max(sm)] or sm
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------
# the reference algorithm on the CPU (oracle port) -- cpu_baseline and --impl reference
# ----------------------------------------------------------------------------------------------------------------
def cpu_epoch_estimate(num_envs: int, rollout_steps: int = 1, minibatches: int = 1, rollout_envs: int = 0, mb_rows: int = 0):
    """Time a bounded SAMPLE of one epoch with the torch-CPU oracle (the reference's algorithm, all host threads) and
    scale it to a whole epoch: 32 x rollout step + GAE/adv + 48 x minibatch update.  rollout_envs / mb_rows shrink the sample
    (envs of the sampled rollout step, rows of the sampled minibatch); both parts are per-row work and are scaled linearly to
    num_envs envs / 16384 rows."""
    full_envs = num_envs
    if rollout_envs and rollout_envs < num_envs:
        num_envs = rollout_envs
    from oracle import phc_oracle as O
    from oracle import ppo_oracle as PO
    from phc_b200 import synthetic as syn
    import math
    cores = min(os.cpu_count() or 1, MAX_CPU_THREADS)
    torch.set_num_threads(cores)
    torch._C._jit_set_profiling_mode(False)          # as phc/env/tasks/base_task.py:95-96
    torch._C._jit_set_profiling_executor(False)
    n_clips = min(num_envs, 512)                       # CPU sample: fewer clips (table size does not change the arithmetic)
    m = syn.make_motions(n_clips, seed=0)
    st = syn.make_env_state(m, num_envs, seed=0)
    tab = O.MotionTables(m.gts, m.grs, m.lrs, m.gvs, m.gavs, m.dvs, m.lengths, m.num_frames, m.dts, m.length_starts)
    cfg = O.StepConfig(key_bodies=syn.SMPL_KEY_BODIES, reset_bodies=syn.SMPL_RESET_BODIES, dof_subset=torch.tensor(syn.SMPL_DOF_SUBSET))
    obs_dim, act, amp = 934, 69, 1960
    g = torch.Generator().manual_seed(0)
    sd = {"a2c_network.sigma": torch.full((act,), -2.9)}

    def stack(prefix, head, i, o):
        d = i
        for k, u in enumerate((1024, 512)):
            sd[f"a2c_network.{prefix}.{2 * k}.weight"] = (torch.rand(u, d, generator=g) * 2 - 1) / math.sqrt(d)
            sd[f"a2c_network.{prefix}.{2 * k}.bias"] = torch.zeros(u)
            d = u
        sd[f"a2c_network.{head}.weight"] = (torch.rand(o, d, generator=g) * 2 - 1) / math.sqrt(d)
        sd[f"a2c_network.{head}.bias"] = torch.zeros(o)
    stack("actor_mlp", "mu", obs_dim, act); stack("critic_mlp", "value", obs_dim, 1); stack("_disc_mlp", "_disc_logits", amp, 1)
    aw, ab = PO.stack_params(sd, "actor_mlp", "mu", 2)
    cw, cb = PO.stack_params(sd, "critic_mlp", "value", 2)
    mean, var = torch.zeros(obs_dim, dtype=torch.float64), torch.ones(obs_dim, dtype=torch.float64)

    def rollout_step():
        out = O.env_step(tab, cfg, st.body_state, st.dof_state, st.dof_force, st.progress, st.motion_ids, st.start_times,
                         st.start_offsets, st.global_offset, st.amp_hist)
        x = O.rms_normalize(out["obs"], mean, var)
        with torch.no_grad():
            mu = O.mlp_forward(x, aw, ab)
            O.mlp_forward(x, cw, cb)
            O.mlp_forward(x, cw, cb)                    # second critic pass on the next observation (amp_agent.py:354)
            a = mu + math.exp(-2.9) * torch.randn_like(mu)
            O.gaussian_neglogp(a, mu, torch.full_like(mu, math.exp(-2.9)), torch.full_like(mu, -2.9))
        return out

    rollout_step()                                      # warm-up (jit / thread pool)
    t0 = time.perf_counter()
    for _ in range(rollout_steps):
        rollout_step()
    t_roll = (time.perf_counter() - t0) / rollout_steps * (full_envs / num_envs)
    sampled_envs, num_envs = num_envs, full_envs

    fd, v, r, nv = syn.make_rollout(num_envs, HORIZON, seed=0)
    t0 = time.perf_counter()
    adv = O.gae(fd, v, r, nv, 0.99, 0.95)
    O.normalize_advantages((adv + v).reshape(-1, 1), v.reshape(-1, 1))
    t_gae = time.perf_counter() - t0

    B_full = min(16384, HORIZON * num_envs)
    B = min(B_full, mb_rows) if mb_rows else B_full
    Bd = max(1, B // 4)
    gen = torch.Generator().manual_seed(1)
    rn = lambda *s: torch.randn(*s, generator=gen)
    batch = dict(obs_n=rn(B, obs_dim), actions=rn(B, act) * 0.1, old_neglogp=rn(B) * 0.1 + 60, advantages=rn(B),
                 old_mu=rn(B, act) * 0.1, old_sigma=torch.full((B, act), math.exp(-2.9)), returns=rn(B, 1),
                 amp_agent=rn(Bd, amp), amp_replay=rn(Bd, amp), amp_demo=rn(Bd, amp))
    pcfg = dict(e_clip=0.2, critic_coef=5.0, entropy_coef=0.0, bounds_loss_coef=10.0, disc_coef=5.0, disc_logit_reg=0.01,
                disc_grad_penalty=5.0, disc_weight_decay=0.0001, grad_norm=50.0, learning_rate=2e-5, truncate_grads=True)
    t0 = time.perf_counter()
    for _ in range(minibatches):
        PO.minibatch_update(sd, batch, pcfg)
    t_mb = (time.perf_counter() - t0) / minibatches * (B_full / B)
    n_mb = 6 * (HORIZON * num_envs // B_full)
    t_epoch = HORIZON * t_roll + t_gae + n_mb * t_mb
    return dict(t_epoch=t_epoch, t_rollout_step=t_roll, t_gae=t_gae, t_minibatch=t_mb, cores=cores,
                sample=f"{rollout_steps} rollout step(s) of {sampled_envs} envs (env step + actor/critic, x{full_envs / sampled_envs:g}) + GAE(32x{num_envs}) + "
                       f"{minibatches} of {n_mb} minibatch updates on {B} of {B_full} rows (x{B_full / B:g}), scaled to one epoch of {full_envs} envs; "
                       f"torch {torch.__version__} CPU, {cores} threads")


CPU_SAMPLE_ENVS = 4096      # FIXED sample of the CPU arm (never adapted to the host's speed): envs of the sampled rollout step ...
CPU_SAMPLE_ROWS = 4096      # ... and rows of the sampled minibatch update (x4 -> the 16384-row minibatch)


def workload_string(num_envs: int) -> str:
    return (f"PPO epoch: {num_envs} envs/GPU x 32 steps, SMPL 24 bodies, obs 934, AMP 10x196, im.yaml nets "
            f"(1024-512), minibatch 16384 x 6 mini-epochs, one synthetic clip per env")


_cpu_warm = False


def cpu_epoch_sample(num_envs: int, repeats: int = 3):
    """The CPU arm's measurement, identical for `cpu_baseline` and `--impl reference`: after one untimed warm-up of the same
    size (thread pool, TorchScript specialisation, autograd's first pass), `repeats` timed samples of [one rollout step of
    4096 envs + GAE/advantages of the whole 32 x 4096 rollout + one minibatch update on 4096 rows]; per-part medians are
    scaled to one epoch (32 rollout steps, 48 minibatch updates of 16384 rows).  The sample size never depends on how fast
    the host is (round-1 verdict: a budget-gated sample made this number move 30x between runs)."""
    global _cpu_warm
    n_roll, rows = min(CPU_SAMPLE_ENVS, num_envs), CPU_SAMPLE_ROWS
    if not _cpu_warm:
        cpu_epoch_estimate(num_envs, rollout_steps=1, minibatches=1, rollout_envs=n_roll, mb_rows=rows)
        _cpu_warm = True
    parts = [cpu_epoch_estimate(num_envs, rollout_steps=1, minibatches=1, rollout_envs=n_roll, mb_rows=rows) for _ in range(repeats)]
    med = lambda k: statistics.median(p[k] for p in parts)
    est = dict(parts[0])
    est.update(t_rollout_step=med("t_rollout_step"), t_gae=med("t_gae"), t_minibatch=med("t_minibatch"))
    n_mb = 6 * (HORIZON * num_envs // min(16384, HORIZON * num_envs))
    est["t_epoch"] = HORIZON * est["t_rollout_step"] + est["t_gae"] + n_mb * est["t_minibatch"]
    est["sample"] = f"median of {repeats} x [" + parts[0]["sample"] + "]"
    est["breakdown_s"] = {"rollout_step_4096_envs (env step + get_motion_state + actor/critic)": est["t_rollout_step"],
                          "gae_and_adv_norm_32x4096": est["t_gae"], "minibatch_update_16384_rows": est["t_minibatch"]}
    return est


def run_reference_arm(args):
    """--impl reference: every step is ONE fixed sample (see cpu_epoch_sample) scaled to an epoch; value = median over the
    timed steps.  The reference itself cannot run on the GPU box (no /root/reference there, Isaac Gym / rl_games absent
    everywhere): this is the oracle port of its algorithm (BASELINE.md section 2 says why)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t_all = []
    est = None
    for i in range(args.warmup + args.steps):
        est = cpu_epoch_sample(args.num_envs, repeats=1)
        if i >= args.warmup:
            t_all.append(est["t_epoch"])
    t = statistics.median(t_all)
    value = HORIZON * args.num_envs / t
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(args.num_envs),
                       "note": "CPU port of the reference algorithm (oracle/), rank 0 only; each step is the fixed sample below scaled to one epoch"},
            "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": est["cores"], "kind": "port",
                             "sample": est["sample"].replace("median of 1 x ", f"median of {args.steps} x "), "breakdown_s": est["breakdown_s"]},
            "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
# the B200 arm
# ----------------------------------------------------------------------------------------------------------------
WORKLOADS = {
    # BASELINE.json configs[1]: the configuration the metric is quoted on (and what the driver's default run measures)
    "smpl": dict(desc="SMPL 24 bodies, obs 934, AMP 10x196, im.yaml nets (1024-512)", envs=NUM_ENVS, algo_bytes=ALGO_BYTES_PER_ENV_STEP,
                 kernel="phc::fast::env_step_fast_kernel"),
    # configs[4]: Unitree H1, 20 bodies + 3 extend bodies in the reward, 19 hinge dofs, obs 778, AMP 10x63 (env_im_h1_phc.yaml, unitree_h1.yaml)
    "h1": dict(desc="Unitree H1 20 bodies + 3 extend bodies, 19 hinge dofs, obs 778, AMP 10x63, im.yaml nets (1024-512)", envs=4096, algo_bytes=7528,
               kernel="phc::env_step_kernel<1, 0, false, false> (run-time body count)"),
    # configs[3]: PHC+ progressive network, 4 primitive columns of im_pnn_big.yaml nets (6 hidden layers, SiLU), 8192 envs
    "pnn_big": dict(desc="SMPL 24 bodies, amp_pnn network: 4 primitive columns (training column 0) of 2048-1536-1024-1024-512-512 SiLU, disc 1024-512 ReLU "
                         "(im_pnn_big.yaml)", envs=8192, algo_bytes=ALGO_BYTES_PER_ENV_STEP, kernel="phc::fast::env_step_fast_kernel"),
}


def build_agent(num_envs: int, device, rank: int, world: int, host_bank: bool, workload: str = "smpl"):
    from phc_b200 import synthetic as syn
    from phc_b200.env.humanoid_im import HumanoidIm, RLGPUEnv
    from phc_b200.learning.amp_agent import AMPAgent
    cfg = {"multi_gpu": world > 1, "seed": 0, "device": str(device)}
    if workload == "h1":
        motion = syn.make_robot_motions(num_envs, seed=rank)
    else:
        motion = syn.make_motions(num_envs, seed=rank)                   # one clip per env, seed + rank (run_hydra.py:121)
    if workload.startswith("pnn_big"):
        if workload == "pnn_big_tf32":
            cfg["mlp_precision"] = "tf32"
        cfg["network"] = {"name": "amp_pnn", "num_prim": 4, "training_prim": 0, "mlp": {"units": [2048, 1536, 1024, 1024, 512, 512], "activation": "silu"},
                          "disc": {"units": [1024, 512], "activation": "relu"}}
    task = HumanoidIm({"env": {"num_envs": num_envs}, "motion_data": motion, "seed": rank, "host_sim_bank": host_bank},
                      device_type="cuda", device_id=device.index)
    cfg["vec_env"] = RLGPUEnv(task)
    agent = AMPAgent("bench", cfg)
    agent.obs = agent.env_reset()
    agent._init_amp_demo_buf()
    return agent, task


def timed_epochs(agent, steps: int, warmup: int, world: int, read_result: bool):
    for _ in range(warmup):
        agent.train_epoch()
        if read_result:
            agent.train_result_dict()
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    lib = agent._lib
    l0 = lib.phc_launch_count()
    ev0.record()
    for _ in range(steps):
        out = agent.train_epoch()
        if read_result:
            agent.train_result_dict()            # device->host read of the epoch's last losses (e2e mode)
    ev1.record()
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    ms = ev0.elapsed_time(ev1)
    launches = lib.phc_launch_count() - l0
    if world > 1:
        t = torch.tensor([ms], device=agent.device)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = float(t.item())
    return ms / steps, launches, out


DUMP_BYTES = 64 * 1000 * 1000


def dump_outputs(agent, epoch_out, out_dir: str) -> None:
    """--dump-outputs: what the last timed epoch returned (train_epoch's tensors, the last minibatch's losses) and what it left to
    its caller (network parameters, normaliser statistics), one float32 / float64 array per file.  The inputs are seeded, so two
    builds run with the same arguments can be compared file by file.  Between two runs of the same build the environment outputs
    are bit-identical; the learner's atomically accumulated reductions differ in the last bits, which 3 + 5 epochs of training
    grow to ~1e-4 relative in losses and weights (B200, 1000 W power limit).  The files share DUMP_BYTES smallest first; an array
    larger than its share is replaced by a fixed sample of its flattened elements (the same seeded indices in every run)."""
    import numpy as np
    arrays = {f"epoch.{k}": v for k, v in epoch_out.items() if torch.is_tensor(v)}
    arrays.update({f"loss.{k}": torch.tensor(v, dtype=torch.float64) for k, v in agent.train_result_dict().items()})
    arrays.update({f"model.{k}": v for k, v in agent.model.state_dict().items()})
    for name, sd in agent.get_stats_weights().items():
        arrays.update({f"stats.{name}.{k}": v for k, v in sd.items()})
    arrays = {k: v.detach().to("cpu", torch.float64 if v.dtype == torch.float64 else torch.float32) for k, v in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    budget, left = DUMP_BYTES, len(arrays)
    for name in sorted(arrays, key=lambda k: arrays[k].numel() * arrays[k].element_size()):
        t = arrays[name]
        keep = (budget // left - 128) // t.element_size()          # 128 bytes: the .npy header
        if t.numel() > keep:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:keep].sort().values
            t = t.reshape(-1)[idx]
        path = os.path.join(out_dir, name + ".npy")
        np.save(path, t.numpy())
        budget, left = budget - os.path.getsize(path), left - 1


def env_kernel_roofline(task, peak_gbs: float, peak_src: str, iters: int = 40, algo_bytes: int = ALGO_BYTES_PER_ENV_STEP,
                         kernel: str = "phc::fast::env_step_fast_kernel"):
    """Average duration of the fused env-step kernel with inputs coming from HBM (L2 flushed by a 256 MB write before every
    launch), CUDA events on the launching stream.  Two measurements:
      * `kernel_us` (used for `achieved`): K x [flush, kernel] and K x [flush] are each bracketed by ONE event pair and the
        difference is divided by K -- the per-event-pair overhead (a few microseconds, comparable to the kernel itself)
        cancels, the launch rate is what the GPU front end sustains back to back, as in the rollout.  The flush is a plain torch
        fill_; the env step is launched the way the product always launches it (programmatic stream serialisation, the kernel
        waits on griddepcontrol.wait before its first global-memory access);
      * `kernel_us_event_pair`: the median of K single launches each inside its own event pair (includes that overhead)."""
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=task.device)
    times = []
    for i in range(iters + 5):
        task.sim.simulate(None)
        flush.fill_(float(i))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        task._plan.run()
        e1.record()
        torch.cuda.synchronize()
        if i >= 5:
            times.append(e0.elapsed_time(e1) * 1e-3)
    t_pair = statistics.median(times)

    def batch(with_kernel: bool) -> float:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for i in range(iters):
            flush.fill_(float(i))
            if with_kernel:
                task._plan.run()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3
    diffs = []
    for _ in range(5):
        t_f = batch(False)
        t_fk = batch(True)
        diffs.append((t_fk - t_f) / iters)
    t = statistics.median(diffs)
    sane = 0.2 * t_pair < t < t_pair             # the differential estimate must be sane; otherwise report the conservative one
    if not sane:
        t = t_pair
    N = task.num_envs
    traffic = None            # DRAM bytes per launch from the committed ncu --set full capture of this kernel at this size
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "env_step_traffic.json")))
        if int(tj.get("num_envs", -1)) == N:
            traffic = int(tj["dram_bytes_per_launch"])
    except Exception:
        traffic = None
    achieved = algo_bytes * N / t / 1e9
    # what the launch really moves per env at J=24: inputs 1248 (state) + 1248 (cached reference pose of the reward time)
    # + 2 x 1248 (observation bracket) + 552 + 276 (dof) + 56 (scalars, env_motion); outputs 3744 (obs row incl. 8 pad bytes)
    # + 40 (reward/reset) + 784 (AMP ring slot) + 1248 (pose cache for the next step = the ref_* buffers)
    actual = 1248 + 1248 + 2 * 1248 + 552 + 276 + 56 + 3744 + 40 + 784 + 1248
    return {"bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs, "traffic": traffic,
            "kernel": kernel, "kernel_us": t * 1e6, "kernel_us_event_pair": t_pair * 1e6,
            "kernel_us_differential_raw": statistics.median(diffs) * 1e6, "differential_used": sane,
            "frac_event_pair": algo_bytes * N / t_pair / 1e9 / peak_gbs,
            "algorithmic_bytes_per_launch": algo_bytes * N,
            "bytes_moved_per_launch_incl_amp_slot_and_pose_cache": actual * N, "achieved_incl_extras_gbs": actual * N / t / 1e9,
            "peak_source": peak_src,
            "timing": "L2 flushed (torch fill_ of 256 MB) before each launch; kernel_us = (%d x [flush, kernel] - %d x [flush]) / %d, one "
                      "CUDA-event pair per batch, median of 5; the env step is a programmatic-dependent launch as everywhere in the product "
                      "(PHC_ENV_PDL=0 gives the plain stream-ordered launch: +2.4 us at 4096 envs, profiles/ab_env_r2.log); "
                      "kernel_us_event_pair = median of %d single launches, one event pair each" % (iters, iters, iters, iters)}


def measured_peak_tf32():
    """Dense TF32 tensor peak to hold the 3xTF32 GEMMs against: MEASURED_PEAKS.json has no TF32 entry, so half of the measured
    cuBLAS bf16 rate (kind::tf32 issues at half the kind::f16 rate: tcgen05 K = 8 vs 16 per instruction at the same cycle cost).
    The sustained figure, because the GEMMs run back to back inside a long step (B200_PROFILING.md)."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return 0.5 * float(j["bf16_tflops_sustained"]), "0.5 x measured bf16_tflops_sustained (MEASURED_PEAKS.json); burst would be 0.5 x %.0f" % float(j["bf16_tflops"])
        except Exception:
            pass
    return 0.5 * 1400.0, "0.5 x fallback 1.4 PFLOP/s sustained bf16 (B200_PROFILING.md)"


def gemm_roofline(agent, iters: int = 20):
    """Tensor-pipe roofline of the learner's dominant kernel (phc::tc5::smem_split::gemm_tc5s_kernel): the three grouped
    forward launches of one minibatch (layer 1 / layer 2 / heads of actor + critic at 16384 rows and discriminator at 12288
    rows) and the grouped backward launches, timed back to back with CUDA events on the launching stream.  achieved = 3 x
    algorithmic fp32 FLOPs (3xTF32: three tensor-core products per fp32 product) / time."""
    eng, net = agent.engine, agent.model
    if eng.backend != "tc5s":
        return None
    x, xa, Bd = agent._x_mb, agent._amp_mb, agent._amp_minibatch_size
    stacks = [(net.actor, x, agent._ws_actor), (net.critic, x, agent._ws_critic), (net.disc, xa, agent._ws_disc)]
    depth = max(len(st.layers) for st, _, _ in stacks)
    bwd = []
    for k in range(depth):
        descs = []
        for st, xin, ws in stacks:
            li = len(st.layers) - 1 - k
            if li >= 0:
                descs += [d for d in eng.bwd_descs(st, li, xin, ws) if d is not None]
        bwd.append(descs)

    def timed(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        f0 = eng.gemm_flops
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        sec = e0.elapsed_time(e1) * 1e-3 / iters
        return sec, (eng.gemm_flops - f0) / iters

    t_f, fl_f = timed(lambda: eng.forward_group(stacks))
    t_b, fl_b = timed(lambda: [eng.run_group(d) for d in bwd])
    net.grads.zero_()
    peak, src = measured_peak_tf32()
    passes = 1.0 if eng.precision == "tf32" else 3.0          # tensor-core products per fp32 product
    ach = passes * (fl_f + fl_b) / (t_f + t_b) / 1e12
    return {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
            "kernel": "phc::tc5::smem_split::gemm_tc5s_kernel (grouped forward + backward launches of one minibatch)",
            "forward_us": t_f * 1e6, "forward_tflops": passes * fl_f / t_f / 1e12, "backward_us": t_b * 1e6,
            "backward_tflops": passes * fl_b / t_b / 1e12, "tensor_products_per_fp32_product": passes, "algorithmic_fp32_flops_per_minibatch": fl_f + fl_b,
            "fp32_equivalent_tflops": (fl_f + fl_b) / (t_f + t_b) / 1e12, "peak_source": src,
            "timing": "%d x [3 forward launches] and %d x [3 backward launches] of the bench minibatch, one CUDA-event pair each; operands (2.1 GB experience "
                      "buffer aside) are the minibatch workspaces, ~0.5 GB, larger than L2" % (iters, iters)}


def env_roofline_points(device, rank, peak_gbs, peak_src, sizes=(16384, 65536)):
    """The same fused env-step kernel at larger batches (several waves: launch ramp and tail amortised), 4096 clips shared by the envs."""
    from phc_b200 import synthetic as syn
    from phc_b200.env.humanoid_im import HumanoidIm
    pts = []
    motion = syn.make_motions(4096, seed=rank)
    for n in sizes:
        try:
            task = HumanoidIm({"env": {"num_envs": n}, "motion_data": motion, "seed": rank}, device_type="cuda", device_id=device.index)
            task.reset()
            for _ in range(3):
                task.step(None)
            r = env_kernel_roofline(task, peak_gbs, peak_src, iters=20)
            pts.append({"num_envs": n, "kernel_us": r["kernel_us"], "achieved": r["achieved"], "frac": r["frac"]})
            del task
            torch.cuda.empty_cache()
        except Exception as e:          # diagnostic extra: never fails the bench line
            pts.append({"num_envs": n, "error": str(e)[:200]})
    return pts


def run_extra_config(name: str, device, rank: int, world: int, peak_gbs: float, peak_src: str, steps: int = 2, warmup: int = 3):
    """One of the other BASELINE.json configurations, measured the same way as the headline (device-resident simulator snapshots,
    CUDA events around `steps` epochs after `warmup`) and reported inside the same JSON line (`extra_configs`)."""
    w = WORKLOADS[name]
    try:
        agent, task = build_agent(w["envs"], device, rank, world, host_bank=False, workload=name)
        ms, launches, _ = timed_epochs(agent, steps, warmup, world, read_result=False)
        out = {"workload": f"PPO epoch: {w['envs']} envs/GPU x 32 steps, {w['desc']}, minibatch 16384 x 6 mini-epochs", "num_envs_per_gpu": w["envs"],
               "value": HORIZON * w["envs"] * world / (ms * 1e-3), "unit": "env-steps/s", "ms_per_step": ms, "steps": steps, "warmup": warmup,
               "gpu_launches": int(launches), "dtype": "tf32 single pass (MLPs), f32 elsewhere" if name.endswith("_tf32") else "f32"}
        if rank == 0:
            r = env_kernel_roofline(task, peak_gbs, peak_src, iters=20, algo_bytes=w["algo_bytes"], kernel=w["kernel"])
            out["roofline"] = {k: r[k] for k in ("bound", "achieved", "peak", "unit", "frac", "kernel", "kernel_us", "algorithmic_bytes_per_launch")}
            g = gemm_roofline(agent, iters=5)
            if g is not None:
                out["roofline_gemm"] = {k: g[k] for k in ("bound", "achieved", "peak", "unit", "frac", "forward_us", "backward_us")}
        del agent, task
        torch.cuda.empty_cache()
        return out
    except Exception as e:          # a secondary measurement never fails the headline line
        torch.cuda.empty_cache()
        return {"workload": name, "error": f"{type(e).__name__}: {e}"[:300]}


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; phc_b200 has no CPU path (use --impl reference for the CPU port)")
    device = torch.device(f"cuda:{local}")
    torch.cuda.set_device(device)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.distributed.init_process_group("nccl", device_id=device)
    # the library __graft_entry__.build() left in the tree; the bench itself compiles nothing (the tree may be read-only)
    from phc_b200 import _lib
    if _lib.load().phc_compiled_sm() != 100:
        raise SystemExit(f"bench.py: {_lib.LIB_PATH} was not compiled for sm_100a")

    # the synthetic data is seeded; this seeds what the run draws from torch's global generators (reset times, action noise,
    # minibatch order), so the same arguments give the same inputs in every run
    torch.manual_seed(rank)
    sampler = ClockSampler(local)
    note("building agent (device-resident simulator snapshots)")
    wl = WORKLOADS[args.workload]
    if args.workload != "smpl" and args.num_envs == NUM_ENVS:
        args.num_envs = wl["envs"]
    agent, task = build_agent(args.num_envs, device, rank, world, host_bank=False, workload=args.workload)
    note("agent built; timed epochs")
    if rank == 0:
        sampler.start()
    sec_per_step, launches, last_epoch = timed_epochs(agent, args.steps, args.warmup, world, read_result=False)
    clocks = sampler.stop() if rank == 0 else None
    note(f"value arm done: {sec_per_step:.1f} ms/epoch")
    if args.dump_outputs and rank == 0:
        dump_outputs(agent, last_epoch, args.dump_outputs)
        note(f"outputs of the last timed epoch written to {args.dump_outputs}")
    if os.environ.get("PHC_PHASE_TIMING", "0") == "1" and rank == 0:       # diagnostic only: CUDA-event phase breakdown of one epoch
        agent.timer.report()
        agent.train_epoch()
        rep = agent.timer.report()
        print(json.dumps({"phase_ms": {k: round(v, 3) for k, v in sorted(rep.items(), key=lambda kv: -kv[1])}, "sum_ms": round(sum(rep.values()), 2)}), file=sys.stderr, flush=True)
    env_steps = HORIZON * args.num_envs * world
    value = env_steps / (sec_per_step * 1e-3)

    peak, peak_src = measured_peak_gbs()
    roof = env_kernel_roofline(task, peak, peak_src, algo_bytes=wl["algo_bytes"], kernel=wl["kernel"]) if rank == 0 else None
    note("roofline kernel timed")
    roof_gemm = gemm_roofline(agent) if rank == 0 else None
    note("gemm roofline timed")
    if world > 1:
        torch.distributed.barrier()
    del agent, task
    torch.cuda.empty_cache()
    if roof is not None and not args.no_points:
        roof["points"] = [{"num_envs": args.num_envs, "kernel_us": roof["kernel_us"], "achieved": roof["achieved"], "frac": roof["frac"]}] + \
            env_roofline_points(device, rank, peak, peak_src)
        note("roofline points timed")

    e2e = None
    if not args.no_e2e:
        agent2, task2 = build_agent(args.num_envs, device, rank, world, host_bank=True, workload=args.workload)
        note("e2e agent built (pinned host snapshots)")
        ms2, _, _ = timed_epochs(agent2, max(1, args.steps), max(3, args.warmup) if args.warmup >= 3 else args.warmup, world, read_result=True)
        e2e = {"value": env_steps / (ms2 * 1e-3), "unit": "env-steps/s", "ms_per_step": ms2,
               "h2d_bytes_per_step": HORIZON * task2.sim.h2d_bytes_per_step, "d2h_bytes_per_step": 16 * 4,
               "note": "simulator state (rigid bodies, dof state, dof forces) copied from pinned host memory every env step; epoch losses read back"}
        del agent2, task2
        torch.cuda.empty_cache()
        note(f"e2e arm done: {ms2:.1f} ms/epoch")

    extras = []
    if not args.no_extras and args.workload == "smpl":
        # the other BASELINE.json configurations: H1 (configs[4]) and the PNN big nets at 8192 envs (configs[3]) on one GPU; at 8 ranks the
        # 16384-envs-over-8 split of configs[2] (2048 envs per rank instead of the weak-scaling 4096)
        WORKLOADS["pnn_big_tf32"] = dict(WORKLOADS["pnn_big"], desc=WORKLOADS["pnn_big"]["desc"] + "; MLP GEMMs in the opt-in single-pass TF32 mode "
                                         "(bf16-class: 8-bit exponent, 10-bit mantissa, fp32 accumulate) instead of 3xTF32")
        names = ["h1", "pnn_big", "pnn_big_tf32"] if world == 1 else []
        for nm in names:
            extras.append(run_extra_config(nm, device, rank, world, peak, peak_src))
            note(f"extra config {nm} done")
        if world == 8:
            WORKLOADS["smpl_2048"] = dict(WORKLOADS["smpl"], envs=2048, desc=WORKLOADS["smpl"]["desc"] + " -- 16384 envs sharded over 8 GPUs (BASELINE configs[2])")
            extras.append(run_extra_config("smpl_2048", device, rank, world, peak, peak_src))

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            est = cpu_epoch_sample(args.num_envs, repeats=3)
            note(f"cpu baseline sample done: {est['t_epoch']:.1f} s/epoch estimated on {est['cores']} threads")
            cpu = {"value": HORIZON * args.num_envs / est["t_epoch"], "unit": "env-steps/s", "cores": est["cores"], "kind": "port",
                   "sample": est["sample"], "ms_per_step": 1e3 * est["t_epoch"], "breakdown_s": est["breakdown_s"]}
        line = {"metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": sec_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": workload_string(args.num_envs) if args.workload == "smpl" else f"PPO epoch: {args.num_envs} envs/GPU x 32 steps, {wl['desc']}, minibatch 16384 x 6 mini-epochs",
                           "parallelism": f"dp{world} (env shards, 1 NCCL all-reduce per minibatch)",
                           "arithmetic": "fp32 throughout (the reference trains with mixed_precision: False): env kernels fp32, MLP GEMMs 3xTF32 on tcgen05 with fp32 accumulation",
                           "l2": "inputs larger than L2: 2.1 GB experience buffer + ~1 GB frame tables per epoch; the roofline kernel is timed with an explicit L2 flush"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roof, "roofline_gemm": roof_gemm, "cpu_baseline": cpu, "extra_configs": extras}
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
