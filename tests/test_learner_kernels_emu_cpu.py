"""The learner's non-GEMM kernels on the CPU (phc_b200/csrc/ppo_scalars.cu and ppo_update.cu, verbatim): block-level emulation
(tests/emu/: every thread of a block is a std::thread, __syncthreads = a block barrier, `__shared__` = function-local statics,
atomicAdd = a lock) against the unmodified reference where it has the function (tests/golden/learn.npz: discount_values,
_calc_advs, RunningMeanStd, _calc_disc_rewards / _combine_rewards; mcp.npz: HumanoidImMCP's mixing), against autograd of the
pinned loss functions for the gradient kernels, and against torch for the rl_games pieces (Gaussian head, clip + Adam).  The
tensor-core GEMMs are the one part of the learner that cannot be emulated this way."""
import ctypes as C
import os
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "emu"))

from tests.helpers import close, load      # noqa: E402

P = C.c_void_p


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    import shutil
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    import build_emu
    lib = C.CDLL(build_emu.build_scalars(str(tmp_path_factory.mktemp("semu"))))
    lib.emu_gae.argtypes = [P, P, P, P, C.c_int32, C.c_int64, C.c_float, C.c_float, P, P]
    lib.emu_adv_norm.argtypes = [P, P, C.c_int64, C.c_int32, P, P]
    return lib


def test_gae_and_adv_norm_vs_reference_golden(emu):
    g = load("learn.npz")
    fd, v, r, nv = (g[k].float().contiguous() for k in ("gae_fdones", "gae_values", "gae_rewards", "gae_next_values"))
    T, N = int(fd.shape[0]), int(fd.shape[1])
    adv, ret = torch.zeros(T, N), torch.zeros(T, N)
    assert emu.emu_gae(fd.data_ptr(), v.data_ptr(), r.data_ptr(), nv.data_ptr(), T, N, 0.99, 0.95, adv.data_ptr(), ret.data_ptr()) == 0
    close(adv.view_as(g["gae_adv"]), g["gae_adv"], rtol=1e-5, atol=5e-6, what="discount_values")
    close(ret, adv + v.view(T, N), what="returns = advs + values")
    flat = lambda t: t.reshape(T, N).transpose(0, 1).reshape(-1).contiguous()
    rets, vals = flat(ret), flat(v)
    out = torch.zeros(T * N)
    ws = torch.zeros(2 * 296, dtype=torch.float64)
    emu.emu_adv_norm(rets.data_ptr(), vals.data_ptr(), T * N, 1, out.data_ptr(), ws.data_ptr())
    close(out, g["adv_norm"].reshape(-1), rtol=1e-4, atol=1e-5, what="_calc_advs")


def test_gae_long_horizon_chunks(emu):
    """T > 32 walks the time axis in chunks of 32 with a carried A_{t+1}; N not a multiple of the 32-env tile."""
    from oracle import phc_oracle as O
    g = torch.Generator().manual_seed(0)
    T, N = 75, 45
    fd = (torch.rand(T, N, generator=g) < 0.05).float()
    v, r, nv = torch.randn(T, N, generator=g), torch.randn(T, N, generator=g), torch.randn(T, N, generator=g)
    adv = torch.zeros(T, N)
    emu.emu_gae(fd.data_ptr(), v.data_ptr(), r.data_ptr(), nv.data_ptr(), T, N, 0.99, 0.95, adv.data_ptr(), None)
    u = lambda t: t.unsqueeze(-1)
    close(adv, O.gae(fd, u(v), u(r), u(nv), 0.99, 0.95).view(T, N), rtol=1e-5, atol=5e-6, what="gae T=75")


# ---- ppo_update.cu: RunningMeanStd, discriminator reward, Gaussian head ----------------------------------------------
@pytest.fixture(scope="module")
def upd(tmp_path_factory):
    import shutil
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    import build_emu
    lib = C.CDLL(build_emu.build_update(str(tmp_path_factory.mktemp("uemu"))))
    lib.emu_rms_apply.argtypes = [P, C.c_int64, C.c_int64, C.c_int32, P, P, C.c_float, C.c_int32, P, C.c_int64, P]
    lib.emu_rms_update.argtypes = [P, C.c_int64, C.c_int64, C.c_int32, P, P, P, P, P]
    lib.emu_rms_apply_update_vec.argtypes = [P, C.c_int64, C.c_int64, C.c_int32, P, P, C.c_float, P, C.c_int64, P, P, P, P, P, C.c_int32, C.c_int32, C.c_int32]
    lib.emu_disc_reward.argtypes = [P, C.c_int64, P, C.c_int64, C.c_float, C.c_float, C.c_float, P, P]
    lib.emu_gaussian_sample.argtypes = [P, C.c_int64, P, P, C.c_int64, C.c_int32, P, P, P, P]
    return lib


def test_running_mean_std_kernels_vs_reference_golden(upd):
    """RunningMeanStd.forward in train mode over three batches (normalise with the current stats, then fold the batch in), the
    final fp64 statistics and the un-normalise direction: phc/utils/running_mean_std.py through tests/golden/learn.npz."""
    g = load("learn.npz")
    d = 12
    mean, var, cnt = torch.zeros(d, dtype=torch.float64), torch.ones(d, dtype=torch.float64), torch.ones((), dtype=torch.float64)
    acc = torch.zeros(2 * d, dtype=torch.float64)
    for i in range(3):
        x = g[f"rms_x{i}"].float().contiguous()
        y = torch.zeros_like(x)
        upd.emu_rms_apply(x.data_ptr(), d, x.shape[0], d, mean.data_ptr(), var.data_ptr(), 1e-5, 0, y.data_ptr(), d, None)
        close(y, g[f"rms_y{i}"], what=f"rms_y{i}")
        upd.emu_rms_update(x.data_ptr(), d, x.shape[0], d, mean.data_ptr(), var.data_ptr(), cnt.data_ptr(), acc.data_ptr(), None)
    # the reference takes the batch mean / var in float32 (input.mean / input.var) before the float64 merge; the kernel
    # accumulates the moments in float64 throughout, so the statistics agree to float32 rounding of the batch moments
    close(mean, g["rms_mean"], rtol=1e-6, atol=1e-7, what="running_mean")
    close(var, g["rms_var"], rtol=1e-6, atol=1e-7, what="running_var")
    close(cnt, g["rms_count"], what="count")
    x = (g["rms_x0"] * 0.1).float().contiguous()
    y = torch.zeros_like(x)
    upd.emu_rms_apply(x.data_ptr(), d, x.shape[0], d, mean.data_ptr(), var.data_ptr(), 1e-5, 1, y.data_ptr(), d, None)
    close(y, g["rms_unnorm"], what="unnorm")
    # row-gathered form (index-composed minibatches): rows 5, 0, 31 of batch 1
    idx = torch.tensor([5, 0, 31], dtype=torch.int64)
    x1 = g["rms_x1"].float().contiguous()
    yg = torch.zeros(3, d)
    upd.emu_rms_apply(x1.data_ptr(), d, 3, d, mean.data_ptr(), var.data_ptr(), 1e-5, 0, yg.data_ptr(), d, idx.data_ptr())
    yf = torch.zeros_like(x1)
    upd.emu_rms_apply(x1.data_ptr(), d, x1.shape[0], d, mean.data_ptr(), var.data_ptr(), 1e-5, 0, yf.data_ptr(), d, None)
    assert torch.equal(yg, yf[idx])


@pytest.mark.parametrize("V,d,ld", [(4, 70, 72), (2, 70, 70), (4, 130, 132), (2, 5, 6)])
def test_vectorised_normalise_and_moments_equal_the_scalar_kernels(upd, V, d, ld):
    """rms_apply_vec_kernel (V columns per lane, gathered rows, fp64 moments through shared memory) against rms_apply_kernel +
    rms_moments_kernel: the normalised rows bit for bit (ragged last vector, pad columns untouched), the merged statistics to fp64
    rounding; both the apply-only and the apply + update form."""
    g = torch.Generator().manual_seed(V * 100 + d)
    n_src, n = 90, 77
    x = torch.zeros(n_src, ld)
    x[:, :d] = torch.randn(n_src, d, generator=g) * 3 + 1
    idx = torch.randint(0, n_src, (n,), generator=g)
    mean_a, var_a = torch.randn(d, generator=g).double(), (torch.rand(d, generator=g) + 0.5).double()
    ys, yv, yv2 = torch.zeros(n, ld), torch.full((n, ld), 9.0), torch.full((n, ld), 9.0)
    upd.emu_rms_apply(x.data_ptr(), ld, n, d, mean_a.data_ptr(), var_a.data_ptr(), 1e-5, 0, ys.data_ptr(), ld, idx.data_ptr())
    st = [(torch.full((d,), 0.3, dtype=torch.float64), torch.full((d,), 1.7, dtype=torch.float64), torch.full((), 50.0, dtype=torch.float64)) for _ in range(2)]
    acc = torch.zeros(2 * d, dtype=torch.float64)
    upd.emu_rms_update(x.data_ptr(), ld, n, d, st[0][0].data_ptr(), st[0][1].data_ptr(), st[0][2].data_ptr(), acc.data_ptr(), idx.data_ptr())
    upd.emu_rms_apply_update_vec(x.data_ptr(), ld, n, d, mean_a.data_ptr(), var_a.data_ptr(), 1e-5, yv.data_ptr(), ld, idx.data_ptr(),
                                 st[1][0].data_ptr(), st[1][1].data_ptr(), st[1][2].data_ptr(), acc.data_ptr(), V, 32, 1)
    assert torch.equal(yv[:, :d], ys[:, :d]) and bool((yv[:, d:] == 9.0).all())
    close(st[1][0], st[0][0], rtol=1e-13, atol=1e-13, what="mean")
    close(st[1][1], st[0][1], rtol=1e-12, atol=1e-13, what="var")
    assert float(st[1][2]) == float(st[0][2]) == 50.0 + n
    upd.emu_rms_apply_update_vec(x.data_ptr(), ld, n, d, mean_a.data_ptr(), var_a.data_ptr(), 1e-5, yv2.data_ptr(), ld, idx.data_ptr(),
                                 None, None, None, acc.data_ptr(), V, 64, 0)
    assert torch.equal(yv2[:, :d], ys[:, :d]) and bool((yv2[:, d:] == 9.0).all())


def test_disc_reward_kernel_vs_reference_golden(upd):
    """AMPAgent._calc_disc_rewards + _combine_rewards (amp_agent.py:848-878) on the golden discriminator logits."""
    from oracle import phc_oracle as O
    g = load("learn.npz")
    logits = O.mlp_forward(g["d_x_agent"], [g["d_w1"], g["d_w2"], g["d_w3"]], [g["d_b1"], g["d_b2"], g["d_b3"]]).float().contiguous()
    n = logits.shape[0]
    task = torch.full((n,), 0.7)
    dr, comb = torch.zeros(n), torch.zeros(n)
    upd.emu_disc_reward(logits.data_ptr(), 1, task.data_ptr(), n, 2.0, 0.5, 0.5, dr.data_ptr(), comb.data_ptr())
    close(dr.view(n, 1), g["d_reward"], what="disc reward")
    close(comb.view(n, 1), g["d_combined"], what="combined reward")


def test_gaussian_head_kernel_self_pinned(upd):
    """rl_games' ModelA2CContinuousLogStd (absent from the reference tree): action = mu + sigma * eps, neglogp; against
    torch.distributions.Normal like the oracle's own pin."""
    gen = torch.Generator().manual_seed(2)
    n, A = 37, 69
    mu, noise = torch.randn(n, A, generator=gen), torch.randn(n, A, generator=gen)
    logstd = torch.full((A,), -2.9)
    act, nlp, mus, sig = torch.zeros(n, A), torch.zeros(n), torch.zeros(n, A), torch.zeros(n, A)
    upd.emu_gaussian_sample(mu.data_ptr(), A, logstd.data_ptr(), noise.data_ptr(), n, A, act.data_ptr(), nlp.data_ptr(), mus.data_ptr(), sig.data_ptr())
    close(act, mu + logstd.exp() * noise, what="actions")
    ref = -torch.distributions.Normal(mu, logstd.exp().expand_as(mu)).log_prob(act).sum(-1)
    close(nlp, ref, rtol=1e-5, atol=1e-4, what="neglogp")
    assert torch.equal(mus, mu) and torch.allclose(sig, logstd.exp().expand_as(mu))


def _bind_more(upd):
    upd.emu_ppo_actor_grad.argtypes = [P, C.c_int64, P, P, P, P, P, P, C.c_int64, C.c_int32, C.c_float, C.c_float, C.c_float, P, C.c_int64, P]
    upd.emu_ppo_critic_grad.argtypes = [P, C.c_int64, P, C.c_int64, C.c_float, C.c_float, P, C.c_int64, P]
    upd.emu_disc_logit_grad.argtypes = [P, C.c_int64, C.c_int64, C.c_int64, C.c_float, P, C.c_int64, P]
    upd.emu_clip_adam.argtypes = [P, P, P, P, C.c_int64, P, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int64]
    upd.emu_mcp_combine.argtypes = [P, C.c_int64, P, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, P, C.c_int64]
    return upd


def test_ppo_loss_gradient_kernels_vs_autograd_of_the_pinned_losses(upd):
    """phc_ppo_actor_grad / phc_ppo_critic_grad / phc_disc_logit_grad against autograd of the oracle's loss functions (which
    tests/test_oracle_golden.py pins to CommonAgent._actor_loss / _critic_loss / bound_loss and AMPAgent._disc_loss): the
    gradients the kernels hand to the GEMM chain and the statistics they accumulate."""
    from oracle import phc_oracle as O
    upd = _bind_more(upd)
    gen = torch.Generator().manual_seed(4)
    n, A = 77, 69
    mu = (torch.randn(n, A, generator=gen) * 0.7).requires_grad_(True)           # some |mu| > 1: the bound loss is active
    logstd = torch.full((A,), -2.9)
    sigma = logstd.exp().expand(n, A)
    old_mu = mu.detach() + 0.02 * torch.randn(n, A, generator=gen)
    actions = old_mu + sigma * torch.randn(n, A, generator=gen)
    old_nlp = O.gaussian_neglogp(actions, old_mu, sigma, logstd.expand(n, A))
    adv = torch.randn(n, generator=gen)
    e_clip, bound_coef = 0.2, 10.0
    nlp = O.gaussian_neglogp(actions, mu, sigma, logstd.expand(n, A))
    a_loss, b_loss = O.actor_loss(old_nlp, nlp, adv, e_clip), O.bound_loss(mu)
    (a_loss.mean() + bound_coef * b_loss.mean()).backward()
    dmu, stats = torch.zeros(n, A), torch.zeros(16)
    c = lambda t: t.detach().float().contiguous()
    mu_c, act_c, onlp_c, adv_c, omu_c, osig_c = c(mu), c(actions), c(old_nlp), c(adv), c(old_mu), c(sigma)
    upd.emu_ppo_actor_grad(mu_c.data_ptr(), A, logstd.data_ptr(), act_c.data_ptr(), onlp_c.data_ptr(), adv_c.data_ptr(), omu_c.data_ptr(),
                           osig_c.data_ptr(), n, A, e_clip, bound_coef, 1.0 / n, dmu.data_ptr(), A, stats.data_ptr())
    close(dmu, mu.grad, rtol=2e-4, atol=1e-6, what="d loss / d mu")
    close(stats[0], a_loss.sum().detach(), rtol=1e-4, atol=1e-4, what="sum actor loss")
    close(stats[1], b_loss.sum().detach(), rtol=1e-4, atol=1e-5, what="sum bound loss")
    close(stats[3] / n, O.policy_kl(mu.detach(), sigma, old_mu, sigma), rtol=1e-3, atol=1e-5, what="kl")
    # critic
    v = torch.randn(n, 1, generator=gen).requires_grad_(True)
    ret = torch.randn(n, 1, generator=gen)
    (5.0 * O.critic_loss(v, ret).mean()).backward()
    dv = torch.zeros(n, 1)
    v_c, r_c = c(v), c(ret.reshape(-1))
    upd.emu_ppo_critic_grad(v_c.data_ptr(), 1, r_c.data_ptr(), n, 5.0, 1.0 / n, dv.data_ptr(), 1, stats.data_ptr())
    close(dv, v.grad, rtol=1e-5, atol=1e-7, what="d loss / d value")
    close(stats[5], O.critic_loss(v, ret).sum().detach(), rtol=1e-5, atol=1e-5, what="sum critic loss")
    # discriminator prediction loss: 0.5 * (BCE(agent+replay, 0) + BCE(demo, 1)) (amp_agent.py:737-743)
    na, nd = 48, 24
    logit = (torch.randn(na + nd, 1, generator=gen) * 2).requires_grad_(True)
    bce = torch.nn.functional.binary_cross_entropy_with_logits
    loss = 0.5 * (bce(logit[:na], torch.zeros(na, 1)) + bce(logit[na:], torch.ones(nd, 1)))
    (5.0 * loss).backward()
    dl = torch.zeros(na + nd, 1)
    l_c = c(logit)
    upd.emu_disc_logit_grad(l_c.data_ptr(), 1, na, nd, 5.0, dl.data_ptr(), 1, stats.data_ptr())
    close(dl, logit.grad, rtol=1e-5, atol=1e-7, what="d loss / d logit")
    close(0.5 * (stats[6] / na + stats[7] / nd), loss.detach(), rtol=1e-5, atol=1e-6, what="disc prediction loss")
    assert int(stats[8]) == int((logit[:na] < 0).sum()) and int(stats[9]) == int((logit[na:] > 0).sum())


def test_clip_and_adam_kernels_vs_torch(upd):
    """torch.nn.utils.clip_grad_norm_(50) + torch.optim.Adam(lr, eps 1e-8) over three steps (amp_agent.py:670-679)."""
    upd = _bind_more(upd)
    gen = torch.Generator().manual_seed(6)
    n = 5000
    p0 = torch.randn(n, generator=gen)
    ref = torch.nn.Parameter(p0.clone())
    opt = torch.optim.Adam([ref], lr=2e-3, eps=1e-8)
    p, m, v = p0.clone(), torch.zeros(n), torch.zeros(n)
    sumsq = torch.zeros(1, dtype=torch.float64)
    for step in range(1, 4):
        g = torch.randn(n, generator=gen) * (3.0 if step == 2 else 0.3)      # step 2 is clipped (norm ~212 > 50)
        ref.grad = g.clone()
        torch.nn.utils.clip_grad_norm_([ref], 50.0)
        opt.step()
        upd.emu_clip_adam(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), n, sumsq.data_ptr(), 1.0, 50.0, 2e-3, 0.9, 0.999, 1e-8, step)
        close(p, ref.detach(), rtol=1e-5, atol=1e-6, what=f"parameters after step {step}")


def test_mcp_combine_kernel_vs_reference_golden(upd):
    """HumanoidImMCP.step's mixing (humanoid_im_mcp.py:64-82, golden from the real class): bit-exact in both modes on the
    primitives' outputs the reference computed inside step (the oracle's PNN reproduces them up to CPU matmul rounding)."""
    import numpy as np
    from oracle import mcp_oracle as mo
    upd = _bind_more(upd)
    z = np.load(os.path.join(HERE, "golden", "mcp.npz"))
    sd = {k[len("model/"):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("model/")}
    K = int(z["num_prim"])
    mean, var = torch.from_numpy(z["rms_mean"]).float(), torch.from_numpy(z["rms_var"]).float()
    cur = torch.clamp((torch.from_numpy(z["obs_buf"]) - mean) / torch.sqrt(var + 1e-05), -5.0, 5.0)
    prim = torch.from_numpy(z["step_prim"]).contiguous()                         # [K, n, A]: the primitives' outputs
    close(torch.stack(mo.pnn_forward(sd, cur, K), dim=0), prim, rtol=1e-5, atol=1e-6, what="PNN columns")
    n, A = prim.shape[1], prim.shape[2]
    w = torch.from_numpy(z["weights"]).float().contiguous()
    for discrete, key in ((0, "actions"), (1, "actions_discrete")):
        out = torch.zeros(n, A)
        upd.emu_mcp_combine(w.data_ptr(), K, prim.data_ptr(), A, n * A, n, K, A, discrete, out.data_ptr(), A)
        assert torch.equal(out, torch.from_numpy(z[key])), key
