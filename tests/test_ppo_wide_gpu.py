"""The on-device PPO at input widths other than the reference's 487 (PPOConfig.num_obs): the bf16 cast of the observation
rows at ragged widths, the fp32 rollout and minibatch updates on a terrain env with the height scan (674 columns) against
the plain-torch restatement of the reference's rl_games fork (oracle/ppo_oracle.py), the packed bf16 networks against
fp32 autograd at that width, the trainer's width checks, checkpoints, and training end to end on curriculum terrain."""
import ctypes as C
import dataclasses
import math

import numpy as np
import pytest
import torch

from oracle import ppo_oracle as PO

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
W = 674


def terrain_env(N, **terrain):
    from isaacgymdyros_b200 import DyrosDynamicWalk, default_cfg
    cfg = default_cfg(N)
    cfg["env"]["terrain"] = {"curriculum": True, "measure_heights": True, "seed": 2, **terrain}
    return DyrosDynamicWalk(cfg, DEV, use_cuda_graph=False)


def make_trainer(N=64, H=16, mb=256, **kw):
    from isaacgymdyros_b200.ppo import PPOConfig, PPOTrainer
    env = terrain_env(N)
    assert env.num_obs == W
    return env, PPOTrainer(env, PPOConfig(horizon_length=H, minibatch_size=mb, num_obs=W, **kw))


@pytest.mark.parametrize("width", [487, 488, 489, 674, 1511])
def test_cast_obs_at_ragged_widths(width):
    """dyros_ppo_cast_obs directly: bf16 rows of width K0 = round_up(W, 8), bit for bit torch's rounding, zero padding
    (written by the kernel: both stores start as 0xFFFF), and the same row at e*H + step of the rollout store."""
    from isaacgymdyros_b200 import native
    lib = native.load()
    N, H, step = 37, 5, 3
    K0 = (width + 7) // 8 * 8
    g = torch.Generator(device=DEV).manual_seed(width)
    obs = torch.randn(N, width, device=DEV, generator=g) * 3
    x_step = torch.full((N, K0), -1, dtype=torch.int16, device=DEV).view(torch.bfloat16)
    x_roll = torch.full((N * H, K0), -1, dtype=torch.int16, device=DEV).view(torch.bfloat16)
    st = torch.tensor([step], dtype=torch.int32, device=DEV)
    pb = native.DyrosPpoBuffers()
    pb.N, pb.H, pb.step, pb.obs_dim = N, H, st.data_ptr(), width
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    native.check(lib.dyros_ppo_cast_obs(C.byref(pb), C.c_void_p(obs.data_ptr()), C.c_void_p(x_step.data_ptr()),
                                        C.c_void_p(x_roll.data_ptr()), s), "cast_obs")
    torch.cuda.synchronize()
    bits = lambda t: t.view(torch.int16)
    assert torch.equal(bits(x_step[:, :width]), bits(obs.bfloat16()))
    assert int(bits(x_step[:, width:]).abs().sum()) == 0
    rows = torch.arange(N, device=DEV) * H + step
    assert torch.equal(bits(x_roll[rows]), bits(x_step))
    others = torch.ones(N * H, dtype=torch.bool, device=DEV)
    others[rows] = False
    assert bool((bits(x_roll[others]) == -1).all())                 # no other row of the store is touched
    pb.obs_dim = -1
    with pytest.raises(native.DyrosError, match="obs_dim < 0"):
        native.check(lib.dyros_ppo_cast_obs(C.byref(pb), C.c_void_p(obs.data_ptr()), C.c_void_p(x_step.data_ptr()), None, s), "cast_obs")


def test_fp32_rollout_on_terrain_with_height_scan_matches_oracle():
    N, H = 64, 16
    env, tr = make_trainer(N=N, H=H, mixed_precision="fp32", use_cuda_graph=False)
    g = torch.Generator(device=DEV); g.manual_seed(0)
    z = torch.randn(H, N, 13, device=DEV, generator=g)
    tr.inject_normal = z.contiguous()
    env.progress_buf[::7] = 7999                                    # time-outs: the value bootstrap (test_ppo_gpu.py)
    obs_seen, done_seen, rew_seen, to_seen, val_seen, mu_seen = [], [], [], [], [], []
    for n in range(H):
        obs_seen.append(env.obs_buf.clone()); done_seen.append(env.reset_buf.clone())
        with torch.no_grad():
            mu, v = tr.net.forward(env.obs_buf)
        mu_seen.append(mu.clone()); val_seen.append(v.clone())
        tr._rollout_step()
        rew_seen.append(env.rew_buf.clone()); to_seen.append(env.timeout_buf.clone())
    torch.cuda.synchronize()
    b = tr.buf
    tm = lambda t: t.transpose(0, 1)
    obs = torch.stack(obs_seen)
    heights = obs[..., 487:]
    assert obs.shape[-1] == W and bool((heights != 0).any()) and heights.unique().numel() > 10   # a 487-wide copy would fail
    assert torch.equal(tm(b["obs"]), obs)
    logstd = tr.net.logstd
    mu_s, val_s = torch.stack(mu_seen), torch.stack(val_seen)
    act = mu_s + torch.exp(logstd) * z
    assert torch.equal(tm(b["dones"]), (torch.stack(done_seen) != 0).float())
    assert torch.allclose(tm(b["actions"]), act, rtol=1e-6, atol=1e-7)
    assert torch.allclose(tm(b["neglogp"]), PO.neglogp(act, mu_s, logstd), rtol=1e-5, atol=1e-5)
    shaped = torch.stack(rew_seen) + 0.99 * val_s * (torch.stack(to_seen) != 0).float()
    assert torch.allclose(tm(b["rewards"]), shaped, rtol=1e-6, atol=1e-7)
    assert int((torch.stack(to_seen) != 0).sum()) > 0
    with torch.no_grad():
        _, last_v = tr.net.forward(env.obs_buf)
    from isaacgymdyros_b200 import native
    native.check(tr.lib.dyros_ppo_gae(C.byref(tr.pb), tr._p(last_v.contiguous()), tr._p(env.reset_buf), tr._stream), "gae")
    torch.cuda.synchronize()
    want = PO.discount_values((env.reset_buf != 0).float(), last_v, tm(b["dones"]), tm(b["values"]), tm(b["rewards"]), 0.99, 0.95)
    assert torch.allclose(tm(b["advantages"]), want, rtol=1e-5, atol=1e-6)
    assert torch.allclose(b["returns"], b["advantages"] + b["values"], rtol=1e-6, atol=1e-7)
    env.close()


def fill_synthetic(tr, seed):
    g = torch.Generator(device=DEV); g.manual_seed(seed)
    r = lambda *s: torch.randn(*s, device=DEV, generator=g)
    b, N, H = tr.buf, tr.N, tr.H
    if tr.packed is None:
        b["obs"].copy_(r(N, H, W))
    b["mus"].copy_(0.3 * r(N, H, 13))
    b["actions"].copy_(b["mus"] + 0.12 * r(N, H, 13))
    b["neglogp"].copy_(PO.neglogp(b["actions"], b["mus"], tr.net.logstd) + 0.3 * r(N, H))
    b["values"].copy_(r(N, H)); b["returns"].copy_(b["values"] + r(N, H)); b["advantages"].copy_(b["returns"] - b["values"])
    tr._prepare()
    return r


def oracle_batch(tr, r0, mb):
    b, NH = tr.buf, tr.N * tr.H
    f = lambda k, *s: b[k].reshape(NH, *s)[r0:r0 + mb].clone()
    return {"actions": f("actions", 13), "old_neglogp": f("neglogp"), "advantages": tr.adv_norm.reshape(NH)[r0:r0 + mb].clone(),
            "returns": f("returns"), "old_mu": f("mus", 13)}


@pytest.mark.parametrize("graph", [False, True])
def test_minibatch_updates_at_674_track_the_oracle_fp32(graph):
    """test_ppo_gpu.py's test_minibatch_updates_track_the_oracle_fp32 at W = 674: the actor with the same tolerances, the
    critic with an absolute one of 1 % of its Adam step (lr 5e-4). Adam divides by sqrt(v), so a rounding-level difference
    in a small gradient moves a parameter by a fraction of the rate: measured on one B200, 62 of the critic's 238,849
    entries (hidden layer 1 and its bias) were up to 2.5e-6 past the actor's tolerance, every actor entry within it."""
    from isaacgymdyros_b200.ppo import FlatActorCritic
    env, tr = make_trainer(mixed_precision="fp32", mini_epochs=2, use_cuda_graph=graph)
    fill_synthetic(tr, seed=2)
    flat0 = tr.net.flat.clone()
    onet = FlatActorCritic(DEV, tr.cfg)
    onet.flat.copy_(flat0)
    params = [p for wb in onet.layers.values() for p in wb]
    actor_p = [p for k, wb in onet.layers.items() if k.startswith("actor") or k == "mu" for p in wb]
    critic_p = [p for k, wb in onet.layers.items() if k.startswith("critic") or k == "value" for p in wb]
    oa, oc = torch.optim.Adam(actor_p, lr=1e-5, eps=1e-8), torch.optim.Adam(critic_p, lr=5e-4, eps=1e-8)
    old_mu = tr.buf["mus"].reshape(-1, 13).clone()
    logs, step = [], 0
    for ep in range(2):
        for i in range(tr.num_minibatches):
            r0, mb = i * 256, 256
            batch = oracle_batch(tr, r0, mb)
            batch["old_mu"] = old_mu[r0:r0 + mb].clone()
            mu, v = onet.forward(tr.buf["obs"].reshape(-1, W)[r0:r0 + mb])
            loss, a_loss, c_loss, kl, cf = PO.total_loss(mu, v, onet.logstd, batch, 0.2, 0.5)
            for p in params:
                p.grad = None
            loss.backward()
            torch.nn.utils.clip_grad_norm_(actor_p, 0.5)
            oa.step(); oc.step()
            step += 1
            for gp in oa.param_groups:
                gp["lr"] = PO.linear_lr(step, 1e-5, 3e-6, 5000)
            old_mu[r0:r0 + mb] = mu.detach()
            logs.append((a_loss.item(), c_loss.item(), kl.item(), cf.item()))
    tr.update()
    torch.cuda.synchronize()
    na = tr.net.n_actor
    assert torch.allclose(tr.net.flat[:na], onet.flat[:na], rtol=1e-4, atol=2e-7)
    assert torch.allclose(tr.net.flat[na:], onet.flat[na:], rtol=1e-4, atol=5e-6)
    assert float((tr.net.flat - flat0).abs().max()) > 1e-5
    w0 = tr.net.layers["actor_mlp.0"][0]
    assert float((w0[:, 487:] - flat0[:256 * W].view(256, W)[:, 487:]).abs().max()) > 0   # the height columns' weights train
    got = (tr.stats / (2 * tr.num_minibatches)).tolist()
    for x, y in zip(got, np.mean(np.array(logs), axis=0)):
        assert x == pytest.approx(y, rel=1e-3, abs=1e-6)
    assert torch.allclose(tr.buf["mus"].reshape(-1, 13), old_mu, rtol=1e-4, atol=1e-6)
    env.close()


def test_packed_bf16_networks_at_674_match_the_fp32_networks():
    """test_ppo_gpu.py's test_packed_bf16_networks_match_the_fp32_networks at W = 674 (K0 = 680), same tolerances and
    reasoning: identical bf16-representable weights, so what differs is the bf16 rounding of the activations."""
    from isaacgymdyros_b200 import native
    from isaacgymdyros_b200.ppo import FlatActorCritic
    env, tr = make_trainer()
    pk = tr.packed
    assert pk.K0 == 680 and tuple(pk.w0.shape) == (2, 256, 680) and tuple(tr.x_roll.shape) == (64 * 16, 680)
    assert pk.desc.inputs == W and tr.pb.obs_dim == W
    r = fill_synthetic(tr, seed=9)
    tr.net.flat.copy_((tr.net.flat * 30 + 0.02 * r(tr.net.n)).to(torch.bfloat16).float())
    pk.pack()
    torch.cuda.synchronize()
    assert float(pk.w0[:, :, W:].float().abs().max()) == 0.0
    mb, r0 = 256, 512
    tr.x_roll[:, :W] = r(tr.N * tr.H, W).to(torch.bfloat16); tr.x_roll[:, W:] = 0
    batch = oracle_batch(tr, r0, mb)
    onet = FlatActorCritic(DEV, dataclasses.replace(tr.cfg, mixed_precision="fp32"))
    onet.flat.copy_(tr.net.flat)
    mu, v = onet.forward(tr.x_roll[r0:r0 + mb, :W].float())
    loss, a_loss, c_loss, kl, cf = PO.total_loss(mu, v, onet.logstd, batch, 0.2, 0.5)
    onet.grad.zero_()
    loss.backward()
    x = tr.x_roll[r0:r0 + mb]
    out = pk.forward(x)
    mu_p, v_p = pk.mu_value(out)
    scale = lambda t: float(t.abs().max())
    assert float((mu_p - mu).abs().max()) < 2e-2 * scale(mu) and float((v_p - v).abs().max()) < 2e-2 * scale(v)
    tr.stats.zero_()
    native.check(tr.lib.dyros_ppo_loss_grad_packed(C.byref(tr.pb), r0, mb, tr._p(out), tr._p(pk.bh), tr._p(tr.net.logstd), tr._p(tr.adv_norm),
                                                   tr._p(pk._buffers(mb)["dout"]), tr._p(pk.gbh), tr._p(tr.stats), tr._stream), "loss_grad_packed")
    pk.backward(x)
    pk.unpack_grads()
    torch.cuda.synchronize()
    assert float(pk.gw0[:, :, W:].float().abs().max()) == 0.0
    for name, (w, bias) in onet.layers.items():
        gw, gb = tr.net.layers[name][0].grad, tr.net.layers[name][1].grad
        for got, want, what in ((gw, w.grad, "weight"), (gb, bias.grad, "bias")):
            err = float((got - want).abs().max())
            cos = float((got * want).sum() / (got.norm() * want.norm() + 1e-30))
            assert err < 0.2 * scale(want) + 1e-12, (name, what, err, scale(want))
            assert cos > 0.997, (name, what, cos)
    for x_, y_ in zip(tr.stats.tolist(), (a_loss.item(), c_loss.item(), kl.item(), cf.item())):
        assert x_ == pytest.approx(y_, rel=5e-2, abs=2e-3)
    # the fused optimiser (n_actor from DyrosPpoNet.inputs) against dyros_ppo_adam on the flat buffers
    grad = tr.net.grad.clone().mul_(100.0)
    ref = {k: t.clone() for k, t in (("p", tr.net.flat), ("m", tr.net.exp_avg), ("v", tr.net.exp_avg_sq))}
    lr2, st2, n2 = tr.lr.clone(), tr.opt_step.clone(), torch.zeros(1, device=DEV)
    native.check(tr.lib.dyros_ppo_adam(tr._p(ref["p"]), tr._p(grad), tr._p(ref["m"]), tr._p(ref["v"]), tr.net.n_actor, tr.net.n, 0.5, 0.5,
                                       tr._p(n2), tr._p(lr2), tr._p(st2), 0.9, 0.999, 1e-8, 1e-5, 3e-6, 5000, tr._stream), "adam")
    tr.net.grad.copy_(grad)
    tr.norm2.zero_()                                                 # norm_done = 0: the kernel measures the actor's norm itself
    native.check(tr.lib.dyros_ppo_adam_packed(C.byref(pk.desc), tr._p(tr.net.flat), tr._p(tr.net.grad), tr._p(tr.net.exp_avg),
                                              tr._p(tr.net.exp_avg_sq), 0.5, 0.5, 0, tr._p(tr.norm2), tr._p(tr.lr), tr._p(tr.opt_step),
                                              0.9, 0.999, 1e-8, 1e-5, 3e-6, 5000, tr._stream), "adam_packed")
    torch.cuda.synchronize()
    assert torch.allclose(tr.net.flat, ref["p"], rtol=1e-6, atol=1e-9) and torch.allclose(tr.net.exp_avg_sq, ref["v"], rtol=1e-5, atol=1e-12)
    assert float((tr.net.flat - ref["p"]).abs().max()) < 1e-8
    for net, name in ((0, "actor_mlp.0"), (1, "critic_mlp.0")):
        w0 = tr.net.layers[name][0].detach()
        assert torch.equal(pk.w0[net, :, :W].float(), w0.to(torch.bfloat16).float())
    assert float(pk.w0[:, :, W:].float().abs().max()) == 0.0
    env.close()


def test_trainer_width_checks():
    from isaacgymdyros_b200 import DyrosDynamicWalk, default_cfg
    from isaacgymdyros_b200.ppo import PPOConfig, PPOTrainer
    wide = terrain_env(64)
    with pytest.raises(ValueError, match=r"height scan.*PPOConfig\(num_obs=674\)"):
        PPOTrainer(wide, PPOConfig(horizon_length=8, minibatch_size=256))
    plane = DyrosDynamicWalk(default_cfg(64), DEV, use_cuda_graph=False)
    with pytest.raises(ValueError, match="PPOConfig.num_obs = 674 .* this env has 487"):
        PPOTrainer(plane, PPOConfig(horizon_length=8, minibatch_size=256, num_obs=W))
    wide.close(); plane.close()


def test_checkpoint_round_trip_at_674(tmp_path):
    from isaacgymdyros_b200 import DyrosDynamicWalk, default_cfg
    from isaacgymdyros_b200.ppo import PPOConfig, PPOTrainer
    env, tr = make_trainer(H=8)
    out = tr.train_epoch()
    assert 0 <= out["terrain_level"] < env.terrain_origins.shape[0]                     # [0, num_rows)
    path = tr.save(str(tmp_path / "ckpt"))
    sd = torch.load(path, map_location="cpu", weights_only=False)
    assert tuple(sd["model"]["a2c_network.actor_mlp.0.weight"].shape) == (256, W)
    env2, tr2 = make_trainer(H=8)
    tr2.net.flat.add_(1.0)
    tr2.restore(path)
    for a, b in ((tr.net.flat, tr2.net.flat), (tr.net.exp_avg, tr2.net.exp_avg), (tr.net.exp_avg_sq, tr2.net.exp_avg_sq),
                 (tr.net.logstd, tr2.net.logstd), (tr.packed.w0, tr2.packed.w0), (tr.packed.bh, tr2.packed.bh)):
        assert torch.equal(a, b)
    assert int(tr2.opt_step.item()) == int(tr.opt_step.item()) > 0 and tr2.epoch == 1
    files = tr.dump_weights_txt(str(tmp_path / "result"))
    assert np.loadtxt(str(tmp_path / "result" / "a2c_network_actor_mlp_0_weight.txt")).shape == (256, W) and len(files) == 13
    plane = DyrosDynamicWalk(default_cfg(64), DEV, use_cuda_graph=False)
    narrow = PPOTrainer(plane, PPOConfig(horizon_length=8, minibatch_size=256))
    p487 = narrow.save(str(tmp_path / "narrow"))
    with pytest.raises(ValueError, match=r"actor_mlp\.0\.weight: shape \(256, 487\), expected \(256, 674\)"):
        tr2.restore(p487)
    env.close(); env2.close(); plane.close()


def test_on_device_ppo_learns_on_curriculum_terrain_with_height_scan():
    """4096 envs on the generated terrain (curriculum, initial levels 0..5) with the height scan, the packed bf16 networks
    at W = 674 and CUDA graphs, the reference's hyper-parameters: 60 epochs = 31 M env-steps. Measured on one B200
    (1000 W), this test's run: mean episode length 107.9 at epoch 1, 391.7 at epoch 60 (3.6x), mean reward 99.4 -> 402.0,
    the mean terrain level 1.74 -> 0.0. Envs that fall early walk less than half their commanded distance, so the
    curriculum moves them down, and by epoch 20 every env is on level 0: the curriculum is exercised downward only, and
    the longer episodes are learned on the easiest level. profiles/ppo_terrain.md has the 200-epoch curve. The threshold
    is 1.5x."""
    from isaacgymdyros_b200.ppo import PPOConfig, PPOTrainer
    env = terrain_env(4096)
    tr = PPOTrainer(env, PPOConfig(num_obs=W))
    outs = [tr.train_epoch() for _ in range(60)]
    first, last = outs[0], outs[-1]
    print("terrain learning:", [(round(o["mean_length"], 1), round(o["mean_reward"], 1), round(o["terrain_level"], 3))
                                for o in outs[::10] + [last]])
    for o in outs:
        assert all(math.isfinite(v) for v in o.values()), o
        assert 0.0 <= o["terrain_level"] < env.terrain_origins.shape[0]                 # [0, num_rows)
    assert first["episodes"] > 1000, first
    assert last["mean_length"] > 1.5 * first["mean_length"], (first, last)
    for t in (env.obs_buf, env.core.sim_t["root_states"], env.core.sim_t["dof_state"]):
        assert bool(torch.isfinite(t).all())
    env.close()
