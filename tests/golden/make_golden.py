"""Generate the golden vectors that pin oracle/phc_oracle.py (and through it the CUDA path).

Runs ONLY in the build container (needs /root/reference): imports the UNMODIFIED reference through
ref_shim.py, drives its real code on seeded synthetic inputs and stores inputs + outputs as .npz:

  python tests/golden/make_golden.py            # rewrites tests/golden/*.npz

What is executed on the reference side (no restatement involved):
  quat.npz     phc/utils/torch_utils.py + isaacgym_torch_utils.py functions
  motion.npz   MotionLibBase.get_motion_state / _calc_frame_blend (phc/utils/motion_lib_base.py:437-559)
  envstep.npz  HumanoidIm._compute_reward / _compute_reset / _compute_observations and
               HumanoidAMP._update_hist_amp_obs / _compute_amp_observations / build_amp_obs_demo, called as bound
               methods of an instance created with object.__new__ (no Isaac Gym) -- humanoid_im.py:694-948,
               :1117-1190, humanoid_amp.py:253-284,:662-707
  mcp.npz      PNN.__init__/forward/load_actor/freeze_pnn (phc/learning/pnn.py), load_pnn / load_mcp_mlp
               (phc/learning/network_loader.py:11-73) and HumanoidImMCP.step (phc/env/tasks/humanoid_im_mcp.py:56-90) with the
               three simulator hooks replaced by recorders
  h1.npz       the hinge-joint robot path (humanoid_type 'h1'): MotionLibReal.get_motion_state (phc/utils/motion_lib_real.py:236-361),
               HumanoidIm._compute_reward with the extend bodies (humanoid_im.py:916-923), _compute_reset, _compute_observations,
               build_amp_observations_robot through _compute_amp_observations / build_amp_obs_demo
  learn.npz    CommonAgent.discount_values/_calc_advs/_actor_loss/_critic_loss/bound_loss,
               AMPAgent._disc_loss/_calc_disc_rewards/_combine_rewards, RunningMeanStd.forward
  load.npz     MotionLibSMPL.load_motion_with_skeleton (phc/utils/motion_lib_smpl.py:101-180): heading randomisation, poselib FK,
               gaussian-filtered velocities, compute_motion_dof_vels -- the loader
  getup.npz    env_im_getup_mcp.yaml: zero_out_far + cycle_motion through _compute_reward / _compute_reset / _compute_observations
  fut.npz      fut_tracks with 3 future samples (the [B, T, J*24] layout of compute_imitation_observations_v6)
  reset.npz    HumanoidAMP._init_amp_obs_ref, MotionLibBase.sample_time_interval
  g1.npz, smplx.npz   the h1.npz / envstep.npz recipes at the shipped shapes beyond 32 bodies (Unitree G1 38 + 1, SMPL-X 52)
  replay.npz   ReplayBuffer.store / sample (phc/learning/replay_buffer.py)
  dropin_signatures.json   positional parameters of the HumanoidIm / AMPAgent methods the drop-in mirrors line up with

  python tests/golden/make_golden.py load getup      # regenerate selected files only
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)

import ref_shim  # noqa: E402

ref_shim.install()
torch.set_num_threads(1)

from phc_b200 import synthetic as syn  # noqa: E402


def npify(d):
    out = {}
    for k, v in d.items():
        if torch.is_tensor(v):
            out[k] = v.detach().cpu().numpy()
        else:
            out[k] = np.asarray(v)
    return out


def save(name, d):
    path = os.path.join(HERE, name)
    np.savez_compressed(path, **npify(d))
    print(f"wrote {path}: {os.path.getsize(path) / 1024:.1f} KiB, {len(d)} arrays")


# ------------------------------------------------------------------------------------------------
def gen_quat():
    import phc.utils.torch_utils as tu
    g = torch.Generator().manual_seed(7)
    n = 512
    a = torch.nn.functional.normalize(torch.randn(n, 4, generator=g), dim=-1)
    b = torch.nn.functional.normalize(torch.randn(n, 4, generator=g), dim=-1)
    # near-identity / exactly-equal / antipodal cases
    b[:32] = a[:32]
    b[32:64] = -a[32:64]
    small = torch.nn.functional.normalize(torch.cat((torch.randn(64, 3, generator=g) * 1e-3, torch.ones(64, 1)), -1), dim=-1)
    b[64:128] = tu.quat_mul(a[64:128], small)
    v = torch.randn(n, 3, generator=g)
    t = torch.rand(n, 1, generator=g)
    t[:8] = 0.0
    t[8:16] = 1.0
    e = torch.randn(n, 3, generator=g)
    e[:8] = 0.0
    e[8:16] *= 1e-6
    e[16:32] *= 4.0          # angles beyond pi -> wrap
    ang, axis = tu.quat_to_angle_axis(a)
    ang_s, axis_s = tu.quat_to_angle_axis(small)
    d = dict(a=a, b=b, v=v, t=t, e=e, small=small,
             quat_mul=tu.quat_mul(a, b), quat_conjugate=tu.quat_conjugate(a), my_quat_rotate=tu.my_quat_rotate(a, v),
             quat_to_tan_norm=tu.quat_to_tan_norm(a), angle=ang, axis=axis, angle_small=ang_s, axis_small=axis_s,
             quat_to_exp_map=tu.quat_to_exp_map(a), exp_map_to_quat=tu.exp_map_to_quat(e), slerp=tu.slerp(a, b, t),
             calc_heading=tu.calc_heading(a), calc_heading_quat=tu.calc_heading_quat(a),
             calc_heading_quat_inv=tu.calc_heading_quat_inv(a))
    from phc.env.tasks.humanoid import remove_base_rot
    d["remove_base_rot"] = remove_base_rot(a)
    save("quat.npz", d)


# ------------------------------------------------------------------------------------------------
def make_ref_motion_lib(m: syn.MotionData):
    from phc.utils.motion_lib_base import MotionLibBase
    lib = object.__new__(MotionLibBase)
    lib._device = torch.device("cpu")
    lib.gts, lib.grs, lib.lrs, lib.gvs, lib.gavs, lib.dvs = m.gts, m.grs, m.lrs, m.gvs, m.gavs, m.dvs
    lib._motion_lengths, lib._motion_num_frames, lib._motion_dt = m.lengths, m.num_frames, m.dts
    lib.length_starts = m.length_starts
    lib.num_bodies = m.num_bodies
    F = m.gts.shape[0]
    lib._motion_aa = torch.zeros(F, 72)
    lib._motion_bodies = torch.zeros(m.num_motions, 17)
    lib._motion_limb_weights = torch.zeros(m.num_motions, 10)
    lib._motion_fps = 1.0 / m.dts
    return lib


def motion_tables_dict(m: syn.MotionData, prefix="tab_"):
    return {prefix + f: getattr(m, f) for f in m.__dataclass_fields__}


def gen_motion():
    m = syn.make_motions(6, seed=3, min_frames=20, max_frames=40)
    lib = make_ref_motion_lib(m)
    g = torch.Generator().manual_seed(11)
    n = 96
    ids = torch.randint(0, m.num_motions, (n,), generator=g)
    ln = m.lengths[ids]
    times = torch.rand(n, generator=g) * ln
    times[:8] = -0.05 * torch.arange(8)                 # negative (history before clip start)
    times[8:16] = ln[8:16] + 0.03 * torch.arange(8)     # at/after the clip end
    times[16:32] = ((torch.rand(16, generator=g) * ln[16:32]) / (1 / 30)).long() * (1 / 30)  # on the frame grid
    offset = torch.randn(n, 3, generator=g)
    i0, i1, bl = lib._calc_frame_blend(times, ln, m.num_frames[ids], m.dts[ids])
    res = lib.get_motion_state(ids, times, offset=offset)
    res_no = lib.get_motion_state(ids, times)
    d = dict(ids=ids, times=times, offset=offset, idx0=i0, idx1=i1, blend=bl, **motion_tables_dict(m))
    for k in ("root_pos", "root_rot", "dof_pos", "root_vel", "root_ang_vel", "dof_vel", "rg_pos", "rb_rot", "body_vel", "body_ang_vel"):
        d["out_" + k] = res[k]
    d["out_noffset_rg_pos"] = res_no["rg_pos"]
    save("motion.npz", d)


# ------------------------------------------------------------------------------------------------
def build_ref_env(m: syn.MotionData, st: syn.EnvState, power_coef=0.0005, upright=True, local_root_obs=True,
                  im_eval=False):
    """A HumanoidIm instance without Isaac Gym: every attribute the post-physics methods read is set by hand."""
    from phc.env.tasks.humanoid_im import HumanoidIm
    from phc.utils.flags import flags
    flags.test, flags.im_eval, flags.real_traj, flags.no_collision_check = False, im_eval, False, False
    N, J = st.body_state.shape[0], st.body_state.shape[1]
    D = (J - 1) * 3
    env = object.__new__(HumanoidIm)
    env.device = torch.device("cpu")
    env.num_envs = N
    env.num_bodies = J
    env.dt = 1.0 / 30.0
    body = st.body_state.clone()
    env._rigid_body_state_reshaped = body
    env._rigid_body_pos, env._rigid_body_rot = body[..., 0:3], body[..., 3:7]
    env._rigid_body_vel, env._rigid_body_ang_vel = body[..., 7:10], body[..., 10:13]
    dof = st.dof_state.clone()
    env._dof_pos, env._dof_vel = dof[..., 0], dof[..., 1]
    env.dof_force_tensor = st.dof_force.clone()
    env.progress_buf = st.progress.clone()
    env.reset_buf = torch.zeros(N, dtype=torch.long)
    env._terminate_buf = torch.zeros(N, dtype=torch.long)
    env.rew_buf = torch.zeros(N)
    env._motion_start_times = st.start_times.clone()
    env._motion_start_times_offset = st.start_offsets.clone()
    env._sampled_motion_ids = st.motion_ids.clone()
    env._global_offset = st.global_offset.clone()
    env.ref_motion_cache = {}
    env._motion_lib = make_ref_motion_lib(m)
    env.humanoid_type = "smpl"
    env.zero_out_far = False
    env.zero_out_far_train = False
    env._full_body_reward = True
    env.reward_specs = {"k_pos": 100, "k_rot": 10, "k_vel": 0.1, "k_ang_vel": 0.1, "w_pos": 0.5, "w_rot": 0.3, "w_vel": 0.1, "w_ang_vel": 0.1}
    env.power_reward = True
    env.power_coefficient = power_coef
    env.max_episode_length = 300
    env.cycle_motion = False
    env._reset_bodies_id = torch.tensor(syn.SMPL_RESET_BODIES)
    env._track_bodies_id = torch.arange(J)
    env._occl_training = False
    env._contact_forces = torch.zeros(N, J, 3)
    env._contact_body_ids = torch.tensor([7, 3, 8, 4])
    env._enable_early_termination = True
    env._termination_distances = torch.full((J,), 0.25)
    env.strict_eval = False
    env._cycle_counter = torch.zeros(N, dtype=torch.int)
    # observation side
    env.self_obs_v, env.obs_v = 1, 6
    env._local_root_obs, env._root_height_obs, env._has_upright_start = local_root_obs, True, upright
    env._has_shape_obs, env._has_limb_weight_obs = False, False
    env.humanoid_shapes = torch.zeros(N, 17)
    env.humanoid_limb_and_weights = torch.zeros(N, 10)
    env._enable_task_obs = True
    env._enable_hist_obs = False
    env.add_obs_noise = False
    env._fut_tracks = False
    env._fut_tracks_dropout = False
    env._num_traj_samples = 1
    env._dof_names = syn.SMPL_BODY_NAMES[1:]
    env.self_obs_buf = torch.zeros(N, 1 + J * 15 - 3)
    env.obs_buf = torch.zeros(N, 1 + J * 15 - 3 + J * 24)
    env.ref_body_pos = torch.zeros(N, J, 3)
    env.ref_body_vel = torch.zeros(N, J, 3)
    env.ref_body_rot = torch.zeros(N, J, 4)
    env.ref_body_pos_subset = torch.zeros(N, J, 3)
    env.ref_dof_pos = torch.zeros(N, D)
    # AMP side
    S, A = st.amp_hist.shape[1], st.amp_hist.shape[2]
    env._num_amp_obs_steps, env._num_amp_obs_per_step = S, A
    env._amp_obs_buf = st.amp_hist.clone()
    env._curr_amp_obs_buf = env._amp_obs_buf[:, 0]
    env._hist_amp_obs_buf = env._amp_obs_buf[:, 1:]
    env._key_body_ids = torch.tensor(syn.SMPL_KEY_BODIES)
    env.dof_subset = torch.tensor(syn.SMPL_DOF_SUBSET)
    env.amp_obs_v = 1
    env._amp_root_height_obs = True
    env._has_dof_subset = True
    env._has_shape_obs_disc, env._has_limb_weight_obs_disc = False, False
    env._add_amp_input_noise = False
    env.extras = {}
    return env


def run_ref_step(env):
    """The body of Humanoid.post_physics_step (humanoid.py:1634-1650) + HumanoidAMP.post_physics_step
    (humanoid_amp.py:194-210) minus the simulator refresh; progress_buf is already incremented in the inputs."""
    env._compute_reward(None)
    env._compute_reset()
    env._compute_observations()
    # HumanoidAMP._update_hist_amp_obs (humanoid_amp.py:662-670) first tries `hist[:] = buf[:, 0:S-1]` where hist
    # aliases buf[:, 1:]; the torch the reference targets rejects that partial overlap and the method falls back to
    # its `except:` branch (`.clone()` first = a true shift by one slot).  torch 2.11 on CPU raises nothing and
    # smears slot 0 over the whole window instead, so the golden executes the fallback statement (:667) directly.
    S = env._num_amp_obs_steps
    env._hist_amp_obs_buf[:] = env._amp_obs_buf[:, 0:(S - 1)].clone()
    env._compute_amp_observations()
    return dict(obs=env.obs_buf.clone(), rew=env.rew_buf.clone(), reward_raw=env.reward_raw.clone(),
                reset=env.reset_buf.clone(), terminate=env._terminate_buf.clone(),
                amp_obs_buf=env._amp_obs_buf.clone(), ref_body_pos=env.ref_body_pos.clone(),
                ref_body_rot=env.ref_body_rot.clone(), ref_body_vel=env.ref_body_vel.clone(),
                ref_dof_pos=env.ref_dof_pos.clone(), self_obs=env.self_obs_buf.clone())


def gen_envstep():
    m = syn.make_motions(32, seed=1, min_frames=12, max_frames=24)   # one clip per env (humanoid_im.py:1121 compares [N] with [M])
    cases = {}
    # case A: the shipped config (frame-grid start times, no offset)
    stA = syn.make_env_state(m, 32, seed=0, max_progress=20)
    # case B: generic blend values + global offset
    stB = syn.make_env_state(m, 32, seed=1, max_progress=20, with_offset=True, blend_jitter=True)
    for tag, st, kw in (("A", stA, {}), ("B", stB, {}), ("C", stA, dict(upright=False, local_root_obs=False)),
                        ("D", stB, dict(im_eval=True))):
        env = build_ref_env(m, st, **kw)
        out = run_ref_step(env)
        for k, v in out.items():
            cases[f"{tag}_out_{k}"] = v
        if tag in ("A", "B"):
            for f in st.__dataclass_fields__:
                cases[f"{tag}_in_{f}"] = getattr(st, f)
    # AMP demo observation (build_amp_obs_demo) and history init (_init_amp_obs_ref arithmetic) on the reference motion
    env = build_ref_env(m, stA)
    g = torch.Generator().manual_seed(5)
    ids = torch.randint(0, m.num_motions, (24,), generator=g)
    t0 = torch.rand(24, generator=g) * m.lengths[ids]
    t0[:4] = 0.1                                         # history reaches before the clip start (negative times)
    env.ref_motion_cache = {}
    demo = env.build_amp_obs_demo(ids, t0).view(24, env._num_amp_obs_steps, -1)
    cases["demo_ids"], cases["demo_t0"], cases["demo_out"] = ids, t0, demo
    cases.update(motion_tables_dict(m))
    save("envstep.npz", cases)


def gen_vr():
    """env_vr.yaml (trackBodies = reset_bodies = Head + both hands, humanoid_im.py:64-66) with the subset reward (full_body_reward:
    False, :926-935) and the shape / limb-weight columns of robot/smpl_humanoid_shape.yaml (humanoid.py:2043-2047) [E]; the same subset
    with the full-body reward [F]; occlusion training on the full body (:797-804 in the observation, :1180-1181 in the reset test --
    random_occlu_idx is indexed by BODY id there, so the reference only supports it with every body tracked) [G]; all through the
    real _compute_reward / _compute_reset / _compute_observations."""
    N = 24
    m = syn.make_motions(N, seed=6, min_frames=12, max_frames=24)
    st = syn.make_env_state(m, N, seed=5, max_progress=20, with_offset=True, blend_jitter=True)
    track = [syn.SMPL_BODY_NAMES.index(n) for n in ("Head", "L_Hand", "R_Hand")]
    g = torch.Generator().manual_seed(8)
    cases = {}
    for tag, subset, subset_reward, occl, shape in (("E", True, True, False, True), ("F", True, False, False, False), ("G", False, False, True, False)):
        env = build_ref_env(m, st)
        J = env.num_bodies
        K = len(track) if subset else J
        if subset:
            env._track_bodies_id = torch.tensor(track)
            env._reset_bodies_id = torch.tensor(track)
        env._full_body_reward = not subset_reward
        env.ref_body_pos_subset = torch.zeros(N, K, 3)
        ns = nl = 0
        if shape:
            env._has_shape_obs, env._has_limb_weight_obs = True, True
            env.humanoid_shapes = torch.randn(N, 17, generator=g)
            env.humanoid_limb_and_weights = torch.randn(N, 10, generator=g)
            ns, nl = 11, 10          # the observation takes humanoid_shapes[:, :-6] (humanoid.py:1469): gender + 10 betas
            cases[f"{tag}_shape"], cases[f"{tag}_limb"] = env.humanoid_shapes, env.humanoid_limb_and_weights
        if occl:
            env._occl_training = True
            env.random_occlu_idx = torch.rand(N, K, generator=g) < 0.4
            env.random_occlu_idx[:, 0] = False
            cases[f"{tag}_occlusion"] = env.random_occlu_idx
        env.self_obs_buf = torch.zeros(N, 1 + J * 15 - 3 + ns + nl)
        env.obs_buf = torch.zeros(N, 1 + J * 15 - 3 + ns + nl + K * 24)
        out = run_ref_step(env)
        for k, v in out.items():
            cases[f"{tag}_out_{k}"] = v
    for f in st.__dataclass_fields__:
        cases[f"in_{f}"] = getattr(st, f)
    cases["track"] = torch.tensor(track)
    cases.update(motion_tables_dict(m))
    save("vr.npz", cases)


# ------------------------------------------------------------------------------------------------
def gen_learn():
    import phc.learning.common_agent as ca
    import phc.learning.amp_agent as aa
    from phc.utils.running_mean_std import RunningMeanStd
    T, N = 16, 24
    fd, val, rew, nval = syn.make_rollout(N, T, seed=0)
    agent = types.SimpleNamespace(horizon_length=T, gamma=0.99, tau=0.95, normalize_advantage=True, bounds_loss_coef=10)
    adv = ca.CommonAgent.discount_values(agent, fd, val, rew, nval)
    ret = adv + val
    flat = lambda x: x.transpose(0, 1).reshape(T * N, -1)      # a2c_common.swap_and_flatten01
    advn = ca.CommonAgent._calc_advs(agent, {"returns": flat(ret), "values": flat(val)})
    g = torch.Generator().manual_seed(21)
    B, A = 64, 69
    old_nlp, nlp = torch.randn(B, generator=g) * 0.3 + 60, torch.randn(B, generator=g) * 0.3 + 60
    advb = torch.randn(B, generator=g)
    a_info = ca.CommonAgent._actor_loss(agent, old_nlp, nlp, advb, 0.2)
    v, r = torch.randn(B, 1, generator=g), torch.randn(B, 1, generator=g)
    c_info = ca.CommonAgent._critic_loss(agent, v, v * 0.9, 0.2, r, False)
    mu = torch.randn(B, A, generator=g) * 1.5
    b_loss = ca.CommonAgent.bound_loss(agent, mu)

    # discriminator loss on a tiny real MLP (amp_agent.py:732-789)
    torch.manual_seed(3)
    din = 40
    disc_mlp = torch.nn.Sequential(torch.nn.Linear(din, 32), torch.nn.ReLU(), torch.nn.Linear(32, 16), torch.nn.ReLU())
    disc_logits = torch.nn.Linear(16, 1)
    torch.nn.init.uniform_(disc_logits.weight, -1.0, 1.0)
    net = types.SimpleNamespace(
        get_disc_logit_weights=lambda: torch.flatten(disc_logits.weight),
        get_disc_weights=lambda: [torch.flatten(mm.weight) for mm in disc_mlp if isinstance(mm, torch.nn.Linear)] + [torch.flatten(disc_logits.weight)])
    dagent = types.SimpleNamespace(model=types.SimpleNamespace(a2c_network=net), _disc_logit_reg=0.01, _disc_grad_penalty=5,
                                   _disc_weight_decay=0.0001)
    for nm in ("_disc_loss_neg", "_disc_loss_pos", "_compute_disc_acc"):
        setattr(dagent, nm, types.MethodType(getattr(aa.AMPAgent, nm), dagent))
    x_agent = torch.randn(48, din, generator=g)
    x_demo = torch.randn(24, din, generator=g).requires_grad_(True)
    la = disc_logits(disc_mlp(x_agent))
    ld = disc_logits(disc_mlp(x_demo))
    dinfo = aa.AMPAgent._disc_loss(dagent, la, ld, x_demo)
    params = list(disc_mlp.parameters()) + list(disc_logits.parameters())
    grads = torch.autograd.grad(dinfo["disc_loss"], params)
    ragent = types.SimpleNamespace(ppo_device="cpu", _disc_reward_scale=2, _norm_disc_reward=lambda: False,
                                   _eval_disc=lambda x: disc_logits(disc_mlp(x)), _task_reward_w=0.5, _disc_reward_w=0.5)
    dr = aa.AMPAgent._calc_disc_rewards(ragent, x_agent)
    comb = aa.AMPAgent._combine_rewards(ragent, torch.ones(48, 1) * 0.7, {"disc_rewards": dr})

    # running mean/std: normalise + update in train mode, then the un-normalise path
    rms = RunningMeanStd((12,))
    rms.train()
    xs = [torch.randn(32, 12, generator=g) * 3 + 1 for _ in range(3)]
    ys = [rms(x) for x in xs]
    rms.eval()
    yu = rms(xs[0][:, :12] * 0.1, unnorm=True)

    d = dict(gae_fdones=fd, gae_values=val, gae_rewards=rew, gae_next_values=nval, gae_adv=adv, adv_norm=advn,
             al_old=old_nlp, al_new=nlp, al_adv=advb, al_out=a_info["actor_loss"], cl_v=v * 0.9, cl_r=r,
             cl_out=c_info["critic_loss"], bl_mu=mu, bl_out=b_loss,
             d_w1=disc_mlp[0].weight, d_b1=disc_mlp[0].bias, d_w2=disc_mlp[2].weight, d_b2=disc_mlp[2].bias,
             d_w3=disc_logits.weight, d_b3=disc_logits.bias, d_x_agent=x_agent, d_x_demo=x_demo,
             d_loss=dinfo["disc_loss"], d_gp=dinfo["disc_grad_penalty"], d_logit_loss=dinfo["disc_logit_loss"],
             d_agent_acc=dinfo["disc_agent_acc"], d_demo_acc=dinfo["disc_demo_acc"],
             d_reward=dr, d_combined=comb,
             rms_x0=xs[0], rms_x1=xs[1], rms_x2=xs[2], rms_y0=ys[0], rms_y1=ys[1], rms_y2=ys[2],
             rms_mean=rms.running_mean, rms_var=rms.running_var, rms_count=rms.count, rms_unnorm=yu)
    for i, gr in enumerate(grads):
        d[f"d_grad{i}"] = gr
    save("learn.npz", d)


def gen_mcp():
    from phc.learning.pnn import PNN
    from phc.learning.network_loader import load_pnn, load_mcp_mlp
    from phc.env.tasks.humanoid_im_mcp import HumanoidImMCP
    torch.manual_seed(23)
    obs_dim, units, act_dim, K, N = 40, [48, 32], 12, 3, 64
    d = dict(obs_dim=np.int64(obs_dim), units=np.array(units), act_dim=np.int64(act_dim), num_prim=np.int64(K))
    mlp_args = {'input_size': obs_dim, 'units': units, 'activation': "relu", 'dense_func': torch.nn.Linear}
    pnn = PNN(mlp_args, output_size=act_dim, numCols=K, has_lateral=False)
    with torch.no_grad():
        for p in pnn.parameters():                         # PNN's default init leaves biases at their Linear defaults; spread them
            p.add_(0.05 * torch.randn_like(p))
    # a single-policy checkpoint folded into column 1 by the reference's own loader (pnn.py:53-60)
    single = {"a2c_network.actor_mlp.0.weight": torch.randn(units[0], obs_dim) * 0.2, "a2c_network.actor_mlp.0.bias": torch.randn(units[0]) * 0.1,
              "a2c_network.actor_mlp.2.weight": torch.randn(units[1], units[0]) * 0.2, "a2c_network.actor_mlp.2.bias": torch.randn(units[1]) * 0.1,
              "a2c_network.mu.weight": torch.randn(act_dim, units[1]) * 0.2, "a2c_network.mu.bias": torch.randn(act_dim) * 0.1}
    pnn.load_actor({"model": single}, idx=1)
    for k, v in single.items():
        d["single/" + k] = v
    sd = {"a2c_network.pnn." + k: v.clone() for k, v in pnn.state_dict().items()}
    sd["a2c_network.mu.bias"] = torch.zeros(act_dim)       # load_pnn reads the action width from this key
    for k, v in sd.items():
        d["model/" + k] = v
    x = torch.randn(N, obs_dim)
    d["x"] = x
    with torch.no_grad():
        for k in range(K):
            _, a = pnn(x, idx=k)
            d[f"col{k}"] = a
        _, allc = pnn(x)
        d["all"] = torch.stack(allc, dim=0)
    # freeze_pnn(idx): which parameters stay trainable when training column idx (pnn.py:45-51)
    pnn.freeze_pnn(1)
    d["trainable_after_freeze1"] = np.array([int(p.requires_grad) for _, p in pnn.named_parameters()])
    d["param_names"] = np.array([n for n, _ in pnn.named_parameters()])

    # HumanoidImMCP.step with recorders for the simulator hooks
    rms = {"running_mean": torch.randn(obs_dim, dtype=torch.float64) * 0.3, "running_var": torch.rand(obs_dim, dtype=torch.float64) + 0.2}
    ck = {"model": sd, "running_mean_std": rms}
    env = object.__new__(HumanoidImMCP)
    env.device = torch.device("cpu")
    env.num_prim, env.has_pnn, env.mlp_bypass = K, True, False
    env.pnn = load_pnn(ck, num_prim=K, has_lateral=False, activation="relu", device="cpu")
    env.running_mean, env.running_var = rms["running_mean"], rms["running_var"]
    env.obs_buf = torch.randn(N, obs_dim) * 2.5            # wide enough that the +-5 clamp bites on some entries
    got = {}
    env.pre_physics_step = lambda a: got.__setitem__("actions", a.clone())
    env._physics_step = lambda: None
    env.post_physics_step = lambda: None
    env.dr_randomizations = {}
    # the primitives' outputs inside step are recorded too: the mixing is pinned bit for bit on them, independent of the
    # host's CPU matmul rounding
    pnn_forward = env.pnn.forward

    def recording_forward(x, idx=-1):
        out = pnn_forward(x, idx)
        got["prim"] = torch.stack(out[1], dim=0)
        return out
    env.pnn.forward = recording_forward
    weights = torch.relu(torch.randn(N, K))                # composer output ends in a ReLU
    d["rms_mean"], d["rms_var"], d["obs_buf"], d["weights"] = rms["running_mean"], rms["running_var"], env.obs_buf, weights
    for disc in (False, True):
        env.discrete_mcp = disc
        env.step(weights)
        d["actions_discrete" if disc else "actions"] = got["actions"]
        d["step_prim"] = got["prim"]

    # composer (amp_network_mcp_builder.py:57-63) rebuilt by the reference's own loader: ReLU after the last Linear
    comp = {"a2c_network.composer.0.weight": torch.randn(units[0], obs_dim) * 0.2, "a2c_network.composer.0.bias": torch.randn(units[0]) * 0.1,
            "a2c_network.composer.2.weight": torch.randn(units[1], units[0]) * 0.2, "a2c_network.composer.2.bias": torch.randn(units[1]) * 0.1,
            "a2c_network.composer.4.weight": torch.randn(K, units[1]) * 0.3, "a2c_network.composer.4.bias": torch.randn(K) * 0.1}
    mlp = load_mcp_mlp({"model": comp}, activation="relu", device="cpu", mlp_name="composer")
    for k, v in comp.items():
        d["composer/" + k] = v
    with torch.no_grad():
        d["composer_out"] = mlp(x)
        # im_mcp_big.yaml: activation silu, ending_act true -> SiLU after the last Linear as well
        d["composer_out_silu"] = load_mcp_mlp({"model": comp}, activation="silu", device="cpu", mlp_name="composer")(x)
    save("mcp.npz", d)


def make_ref_robot_lib(m):
    from phc.utils.motion_lib_real import MotionLibReal
    J = m.num_bodies
    lib = object.__new__(MotionLibReal)
    lib._device = torch.device("cpu")
    lib.gts, lib.grs, lib.gvs, lib.gavs = (t[:, :J].contiguous() for t in (m.gts_t, m.grs_t, m.gvs_t, m.gavs_t))
    lib.gts_t, lib.grs_t, lib.gvs_t, lib.gavs_t = m.gts_t, m.grs_t, m.gvs_t, m.gavs_t
    lib.dof_pos, lib.dvs = m.dof_pos, m.dvs
    lib._motion_lengths, lib._motion_num_frames, lib._motion_dt = m.lengths, m.num_frames, m.dts
    lib.length_starts = m.length_starts
    lib.num_bodies = J
    lib._get_num_bodies = lambda: J
    F = m.gts_t.shape[0]
    lib._motion_aa = torch.zeros(F, 72)
    lib._motion_bodies = torch.zeros(m.num_motions, 17)
    lib._motion_limb_weights = torch.zeros(m.num_motions, 10)
    lib._motion_fps = 1.0 / m.dts
    return lib


def _gen_robot(name, m, ext_parents, ext_pos, key_bodies, n_env=24):
    """Hinge-joint robot goldens (h1.npz / g1.npz): MotionLibReal.get_motion_state, the HumanoidIm step with extend bodies,
    build_amp_observations_robot through _compute_amp_observations / build_amp_obs_demo."""
    J, D, E = m.num_bodies, m.num_dofs, m.num_ext
    lib = make_ref_robot_lib(m)
    d = {"tab_" + f: getattr(m, f) for f in ("gts_t", "grs_t", "gvs_t", "gavs_t", "dof_pos", "dvs", "lengths", "num_frames", "dts", "length_starts")}
    d["ext_parents"], d["ext_pos"], d["key_bodies"] = np.array(ext_parents), np.array(ext_pos, dtype=np.float32), np.array(key_bodies)
    # --- MotionLibReal.get_motion_state
    g = torch.Generator().manual_seed(31)
    n = 64
    ids = torch.randint(0, m.num_motions, (n,), generator=g)
    ln = m.lengths[ids]
    times = torch.rand(n, generator=g) * ln
    times[:6] = -0.05 * torch.arange(6)
    times[6:12] = ln[6:12] + 0.03 * torch.arange(6)
    offset = torch.randn(n, 3, generator=g)
    res = lib.get_motion_state(ids, times, offset=offset)
    d.update(ms_ids=ids, ms_times=times, ms_offset=offset)
    for k in ("root_pos", "root_rot", "dof_pos", "root_vel", "root_ang_vel", "dof_vel", "rg_pos", "rb_rot", "body_vel", "body_ang_vel",
              "rg_pos_t", "rg_rot_t", "body_vel_t", "body_ang_vel_t"):
        d["ms_out_" + k] = res[k]
    # --- env step (two cases: frame-grid starts; generic blend + global offset)
    A = 13 + 2 * D + 3 * len(key_bodies)
    for tag, kw in (("A", {}), ("B", dict(with_offset=True, blend_jitter=True))):
        st = syn.make_robot_env_state(m, n_env, seed=4, amp_dim=A, max_progress=20, **kw)
        base = syn.MotionData(gts=lib.gts, grs=lib.grs, lrs=lib.grs, gvs=lib.gvs, gavs=lib.gavs, dvs=torch.zeros(1), lengths=m.lengths,
                              num_frames=m.num_frames, dts=m.dts, length_starts=m.length_starts)
        env = build_ref_env(base, st)
        env._motion_lib = lib
        env.humanoid_type = name
        env.extend_body_parent_ids = torch.tensor(ext_parents)
        env.extend_body_pos_in_parent = torch.tensor(ext_pos).repeat(env.num_envs, 1, 1)
        env.num_extend_bodies = E
        env._reset_bodies_id = torch.arange(J)
        env._key_body_ids = torch.tensor(key_bodies)
        env.dof_subset, env._has_dof_subset = None, False
        env._dof_names = [f"d{i}" for i in range(D)]
        env._contact_body_ids = torch.tensor([5, 10])
        env.ref_dof_pos = torch.zeros(env.num_envs, D)
        out = run_ref_step(env)
        for k, v in out.items():
            d[f"{tag}_out_{k}"] = v
        for f in st.__dataclass_fields__:
            d[f"{tag}_in_{f}"] = getattr(st, f)
    # --- AMP demo observation of the reference motion
    ids = torch.randint(0, m.num_motions, (16,), generator=g)
    t0 = torch.rand(16, generator=g) * m.lengths[ids]
    t0[:3] = 0.1
    env.ref_motion_cache = {}
    d["demo_ids"], d["demo_t0"] = ids, t0
    d["demo_out"] = env.build_amp_obs_demo(ids, t0).view(16, env._num_amp_obs_steps, -1)
    save(name + ".npz", d)


def gen_h1():
    m = syn.make_robot_motions(24, seed=2, min_frames=12, max_frames=24)
    _gen_robot("h1", m, syn.H1_EXT_PARENTS, syn.H1_EXT_POS, syn.H1_KEY_BODIES)


def gen_g1():
    """Unitree G1 shapes (phc/data/cfg/robot/unitree_g1.yaml: 38 bodies, 37 hinge dofs, one extend body 0.4 m above the pelvis):
    more than 32 bodies incl. the extend body -- the case the fused step kernel does not take yet (oracle pinned ahead of it)."""
    m = syn.make_robot_motions(12, seed=6, num_bodies=syn.G1_NUM_BODIES, num_dofs=syn.G1_NUM_DOFS, ext_parents=syn.G1_EXT_PARENTS,
                               ext_pos=syn.G1_EXT_POS, min_frames=12, max_frames=20)
    _gen_robot("g1", m, syn.G1_EXT_PARENTS, syn.G1_EXT_POS, syn.G1_KEY_BODIES, n_env=12)


def gen_smplx():
    """SMPL-X shapes (phc/data/cfg/robot/smplx_humanoid.yaml: 52 bodies, spherical joints) through the same HumanoidIm methods as
    envstep.npz -- more than 32 bodies, not taken by the fused step kernel yet (oracle pinned ahead of it)."""
    J = 52
    m = syn.make_motions(8, seed=13, num_bodies=J, min_frames=12, max_frames=20)
    A = 1 + 12 + 9 * (J - 1) + 3 * 4
    st = syn.make_env_state(m, 8, seed=13, amp_dim=A, max_progress=16, with_offset=True, blend_jitter=True)
    env = build_ref_env(m, st)
    env.humanoid_type = "smplx"
    env._reset_bodies_id = torch.arange(J)
    env._key_body_ids = torch.tensor(syn.SMPLX_KEY_BODIES)
    # Humanoid always holds a (possibly empty) tensor here (humanoid.py:413,:435); `None` would switch on the in-place zeroing of
    # four SMPL joints in _compute_amp_observations (humanoid_amp.py:676-679), which no shipped configuration reaches
    env.dof_subset, env._has_dof_subset = torch.tensor([]).long(), False
    env._dof_names = [f"j{i}" for i in range(1, J)]
    out = run_ref_step(env)
    d = {f"out_{k}": v for k, v in out.items()}
    for f in st.__dataclass_fields__:
        d[f"in_{f}"] = getattr(st, f)
    d.update(motion_tables_dict(m))
    save("smplx.npz", d)


# ------------------------------------------------------------------------------------------------
def gen_fut():
    """env.fut_tracks: True with numTrajSamples 3, trajSampleTimestepInv 10 -- the T = 3 future reference samples of
    _compute_task_obs (humanoid_im.py:743-749) through compute_imitation_observations_v6 ([B, T, J*24] layout, :1308-1358), and the
    save_buffer branch that keeps sample 0 (:856-861).  The fused kernel's T_MAX = 4 instantiation."""
    m = syn.make_motions(24, seed=21, min_frames=30, max_frames=50)
    st = syn.make_env_state(m, 24, seed=21, max_progress=25, with_offset=True, blend_jitter=True)
    env = build_ref_env(m, st)
    J = st.body_state.shape[1]
    env._fut_tracks, env._num_traj_samples, env._traj_sample_timestep = True, 3, 1 / 10
    env.obs_buf = torch.zeros(env.num_envs, 1 + J * 15 - 3 + 3 * J * 24)
    out = run_ref_step(env)
    d = {f"out_{k}": v for k, v in out.items()}
    for f in st.__dataclass_fields__:
        d[f"in_{f}"] = getattr(st, f)
    d.update(motion_tables_dict(m))
    save("fut.npz", d)


# ------------------------------------------------------------------------------------------------
def gen_reset():
    """Reset-path pieces with the real methods: HumanoidAMP._init_amp_obs_ref (humanoid_amp.py:575-603: history slots 1..S-1 =
    AMP observations of the reference motion at t0 - k dt) and MotionLibBase.sample_time_interval (motion_lib_base.py:414-423)
    with the uniform numbers it draws recorded as the `phase` input."""
    m = syn.make_motions(16, seed=8, min_frames=12, max_frames=30)
    st = syn.make_env_state(m, 16, seed=8, max_progress=10)
    env = build_ref_env(m, st)
    g = torch.Generator().manual_seed(3)
    env_ids = torch.tensor([0, 3, 4, 9, 15])
    ids = st.motion_ids[env_ids]
    t0 = torch.rand(5, generator=g) * m.lengths[ids]
    t0[0] = 0.0                                          # history entirely before the clip start
    before = env._hist_amp_obs_buf.clone()
    env._init_amp_obs_ref(env_ids, ids, t0)
    d = dict(env_ids=env_ids, motion_ids=ids, t0=t0, hist_before=before, hist_after=env._hist_amp_obs_buf.clone())
    torch.manual_seed(41)
    phase = torch.rand(ids.shape)
    torch.manual_seed(41)
    env._motion_lib._device = torch.device("cpu")
    d["phase"], d["sampled_times"] = phase, env._motion_lib.sample_time_interval(ids)
    d.update(motion_tables_dict(m))
    save("reset.npz", d)


# ------------------------------------------------------------------------------------------------
def gen_getup(J=24, name="getup.npz", seed=4):
    """env_im_getup_mcp.yaml (the configuration HumanoidImMCP trains in): zero_out_far + cycle_motion, zero_out_far_train False.
    The real HumanoidIm._compute_reward (:873-948), _compute_reset (:1117-1190 incl. the clip wrap-around :1123-1146) and
    _compute_observations (zero_out_far overwrites :783-796).  The uniform numbers sample_time_interval draws for the wrapping
    envs are reproduced by re-seeding torch's generator and stored as the `cycle_phase` input."""
    N = 48 if J == 24 else 24
    m = syn.make_motions(N, seed=seed, num_bodies=J, min_frames=16, max_frames=40)
    A = 196 if J == 24 else 1 + 12 + 9 * (J - 1) + 3 * 4
    st = syn.make_env_state(m, N, seed=2, amp_dim=A, max_progress=20, with_offset=True)
    g = torch.Generator().manual_seed(9)
    # the simulated state was generated around reference + global_offset: moving the offset moves the reference away
    st.global_offset[0:10, :2] += torch.randn(10, 2, generator=g) * 4.0        # far: beyond far_distance for most
    st.global_offset[10:20, :2] += torch.randn(10, 2, generator=g) * 0.8       # between close and far
    st.global_offset[20:24, :2] += torch.randn(4, 2, generator=g) * 0.15       # around the 0.25 m transition
    cc_in = torch.tensor([0, 0, 0, 1, 2, 7], dtype=torch.int)[torch.randint(0, 6, (N,), generator=g)]
    point_goal = torch.rand(N, generator=g) * 6
    env = build_ref_env(m, st)
    if J != 24:          # SMPL-X shapes (env_im_x_getup_mcp.yaml), set up as in gen_smplx
        env.humanoid_type = "smplx"
        env._reset_bodies_id = torch.arange(J)
        env._key_body_ids = torch.tensor(syn.SMPLX_KEY_BODIES)
        env.dof_subset, env._has_dof_subset = torch.tensor([]).long(), False
        env._dof_names = [f"j{i}" for i in range(1, J)]
    env.zero_out_far, env.zero_out_far_train, env.cycle_motion, env.cycle_motion_xp = True, False, True, False
    env.close_distance, env.far_distance = 0.25, 3
    env.max_episode_length = 15
    env._cycle_counter = torch.clamp_min(cc_in - 1, 0)             # pre_physics_step ran _update_cycle_count (:1076-1079)
    env._point_goal = point_goal.clone()
    env._humanoid_root_states = env._rigid_body_state_reshaped[:, 0, :]
    env._motion_lib._device = torch.device("cpu")
    # the wrapping envs, as _compute_reset will find them, and the numbers it will draw for them
    t_now = st.progress * env.dt + st.start_times + st.start_offsets
    wrap = t_now >= m.lengths[st.motion_ids]
    torch.manual_seed(77)
    phase = torch.zeros(N)
    phase[wrap] = torch.rand(int(wrap.sum()))
    env._compute_reward(None)
    torch.manual_seed(77)
    env._compute_reset()
    env._compute_observations()
    S = env._num_amp_obs_steps
    env._hist_amp_obs_buf[:] = env._amp_obs_buf[:, 0:(S - 1)].clone()
    env._compute_amp_observations()
    d = dict(in_cycle_counter=cc_in, in_point_goal=point_goal, in_cycle_phase=phase, in_wrap=wrap,
             out_obs=env.obs_buf, out_rew=env.rew_buf, out_reward_raw=env.reward_raw, out_reset=env.reset_buf,
             out_terminate=env._terminate_buf, out_amp_obs_buf=env._amp_obs_buf, out_ref_body_pos=env.ref_body_pos,
             out_ref_body_rot=env.ref_body_rot, out_ref_body_vel=env.ref_body_vel, out_start_times=env._motion_start_times,
             out_start_offsets=env._motion_start_times_offset, out_global_offset=env._global_offset,
             out_cycle_counter=env._cycle_counter, out_point_goal=env._point_goal)
    for f in st.__dataclass_fields__:
        d[f"in_{f}"] = getattr(st, f)
    d.update(motion_tables_dict(m))
    print("getup golden: wrapping envs", int(wrap.sum()), "far (reward)", int((d["out_reward_raw"][:, 1] == 0).sum()),
          "resets", int(env.reset_buf.sum()))
    save(name, d)


def gen_getup_smplx():
    """The getup configuration at SMPL-X shapes (env_im_x_getup_mcp.yaml: 52 bodies, zero_out_far + cycle_motion)."""
    gen_getup(J=52, name="getup_smplx.npz", seed=14)


# ------------------------------------------------------------------------------------------------
def gen_load():
    """MotionLibSMPL.load_motion_with_skeleton (phc/utils/motion_lib_smpl.py:101-180) executed UNMODIFIED on synthetic
    clips in the on-disk format ({pose_quat_global [T,J,4], root_trans_offset [T,3], pose_aa, fps}): heading randomisation
    (scipy), SkeletonState.from_rotation_and_root_translation(is_local=False), SkeletonMotion.from_skeleton_state (FK +
    gaussian-filtered finite differences, poselib skeleton3d.py:1000-1121) and compute_motion_dof_vels
    (motion_lib_base.py:47-70).  The heading angle of clip f is pi*(2u-1) with u the f-th np.random.random() after
    np.random.seed(0) (pid 0 seeds with randint(5000)*0) -- recorded here as an input."""
    from poselib.poselib.skeleton.skeleton3d import SkeletonTree, SkeletonState
    import phc.utils.motion_lib_smpl as mls
    from phc.utils.motion_lib_smpl import MotionLibSMPL
    # smpl_sim (unpinned git dependency, absent here) supplies to_torch: tensor -> itself, ndarray -> torch.from_numpy
    mls.to_torch = lambda x: x if torch.is_tensor(x) else torch.from_numpy(np.asarray(x))
    from phc.utils import flags as flags_mod
    flags = flags_mod.flags
    flags.im_eval, flags.test, flags.real_traj = False, False, False
    J = 24
    g = torch.Generator().manual_seed(5)
    frames = [2, 3, 9, 17, 18, 45]                    # shorter than / equal to / longer than the 17-tap filter window
    fps_list = [30, 30, 30, 60, 30, 30]
    parents = torch.tensor(syn.SMPL_PARENTS)
    base_off = torch.tensor(syn._SMPL_OFFSETS, dtype=torch.float64)
    trees, clips = [], []
    for F, fps in zip(frames, fps_list):
        scale = 0.8 + 0.4 * torch.rand(J, 1, generator=g, dtype=torch.float64)     # per-clip body shape: own bone lengths
        off = base_off * scale
        tree = SkeletonTree([f"b{j}" for j in range(J)], parents, off)
        walk = torch.cumsum(torch.randn(F, J, 3, generator=g, dtype=torch.float64) * 0.08, 0) + torch.randn(1, J, 3, generator=g, dtype=torch.float64) * 0.5
        ang = walk.norm(dim=-1, keepdim=True).clamp(min=1e-12)
        lr = torch.cat([walk / ang * torch.sin(ang / 2), torch.cos(ang / 2)], -1)
        if F >= 9:
            lr[4, 7] = lr[3, 7]                       # a joint that does not move between two frames (zero angle branch)
        trans = torch.cumsum(torch.randn(F, 3, generator=g, dtype=torch.float64) * 0.03, 0) + torch.tensor([0.3, -0.2, 0.9], dtype=torch.float64)
        st = SkeletonState.from_rotation_and_root_translation(tree, lr, trans, is_local=True)
        gq = st.global_rotation.clone()
        if F >= 9:
            gq[5] = -gq[5]                            # on-disk quaternions carry arbitrary signs
        clips.append({"pose_quat_global": gq.numpy().copy(), "root_trans_offset": trans.clone(),
                      "pose_aa": np.zeros((F, J * 3)), "fps": fps})
        trees.append(tree)
    cfg = types.SimpleNamespace(max_length=-1, fix_height=0, multi_thread=False)
    np.random.seed(0)
    heading = np.array([np.pi * (2 * np.random.random() - 1.0) for _ in frames])
    shape_params = [torch.zeros(17) for _ in frames]
    res = MotionLibSMPL.load_motion_with_skeleton(np.arange(len(frames)), clips, trees, shape_params, None, cfg, None, 0)
    d = dict(parents=parents, heading=heading, num_frames=np.array(frames), fps=np.array(fps_list, dtype=np.float64),
             offsets=torch.stack([t.local_translation.double() for t in trees]),
             pose_quat_global=np.concatenate([c["pose_quat_global"] for c in clips]),
             root_trans=torch.cat([c["root_trans_offset"] for c in clips]))
    ms = [res[i][1] for i in range(len(frames))]
    d["gts"] = torch.cat([m.global_translation for m in ms]).float()
    d["grs"] = torch.cat([m.global_rotation for m in ms]).float()
    d["lrs"] = torch.cat([m.local_rotation for m in ms]).float()
    d["gvs"] = torch.cat([m.global_velocity for m in ms]).float()
    d["gavs"] = torch.cat([m.global_angular_velocity for m in ms]).float()
    d["dvs"] = torch.cat([m.dof_vels for m in ms]).float()
    save("load.npz", d)


# ------------------------------------------------------------------------------------------------
def gen_replay():
    """ReplayBuffer (phc/learning/replay_buffer.py): circular store, the pre-fill `% head` rule, the permutation refresh.  The
    buffer draws its permutations from the global generator seeded with 5; the stored rows come from their own generator."""
    from phc.learning.replay_buffer import ReplayBuffer
    from tests.test_replay_buffer_cpu import SAMPLE_SIZES, STORE_SIZES
    size, width = 50, 7
    torch.manual_seed(5)
    ref = ReplayBuffer(size, "cpu")
    g = torch.Generator().manual_seed(1)
    d = dict(size=np.int64(size))
    for step, n in enumerate(STORE_SIZES):
        rows = torch.randn(n, width, generator=g)
        ref.store({"amp_obs": rows})
        d[f"rows{step}"], d[f"total{step}"], d[f"data{step}"] = rows, np.int64(ref.get_total_count()), ref._data_buf["amp_obs"].clone()
        for k in SAMPLE_SIZES:
            d[f"sample{step}_{k}"] = ref.sample(k)["amp_obs"]
    save("replay.npz", d)


def gen_dropin():
    """Positional parameters (name, required) of the HumanoidIm / AMPAgent methods the mirrors must accept the same way."""
    import importlib
    import inspect
    import json
    from tests.test_dropin_surface import SIGNATURE_METHODS
    classes = {"HumanoidIm": importlib.import_module("phc.env.tasks.humanoid_im").HumanoidIm,
               "AMPAgent": importlib.import_module("phc.learning.amp_agent").AMPAgent}
    out = {}
    for cname, names in SIGNATURE_METHODS.items():
        cls = classes[cname]
        out[cname] = {}
        for n in names:
            assert any(n in vars(b) for b in cls.__mro__), f"reference lacks {cname}.{n}"
            out[cname][n] = [[p.name, p.default is p.empty] for p in inspect.signature(getattr(cls, n)).parameters.values()
                             if p.kind in (p.POSITIONAL_ONLY, p.POSITIONAL_OR_KEYWORD)]
    path = os.path.join(HERE, "dropin_signatures.json")
    with open(path, "w") as f:               # one line per method
        f.write("{\n" + ",\n".join(f' "{c}": {{\n' + ",\n".join(f'  "{n}": {json.dumps(v)}' for n, v in m.items()) + "\n }"
                                   for c, m in out.items()) + "\n}\n")
    print(f"wrote {path}")


if __name__ == "__main__":
    if len(sys.argv) > 1:
        for name in sys.argv[1:]:
            globals()["gen_" + name]()
        sys.exit(0)
    gen_mcp()
    gen_h1()
    gen_quat()
    gen_motion()
    gen_envstep()
    gen_learn()
    gen_load()
    gen_getup()
    gen_fut()
    gen_replay()
    gen_dropin()
    gen_reset()
    gen_g1()
    gen_smplx()
    gen_getup_smplx()
    gen_vr()
