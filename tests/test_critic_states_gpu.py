"""Critic states on the B200: the kernels' state rows against tests/critic_states_oracle.py (fused and staged, the plane
and the generated curriculum terrain, ragged N), fused against staged bit for bit, the prefix against obs_buf, an env
with states against the same env without them, the asymmetric packed bf16 and fp32 PPO paths at (Wa, Wc) = (487, 705),
the trainer's refusals and checkpoints, and a learning run of a blind actor with a privileged critic."""
import ctypes as C
import dataclasses
import math

import numpy as np
import pytest
import torch

from isaacgymdyros_b200.core import CoreConfig, DyrosCore, TerrainCurriculum
from isaacgymdyros_b200.terrain import TerrainConfig, generate
from oracle import ppo_oracle as PO
from oracle import task_oracle as O
from tests import critic_states_oracle as CS
from tests import height_scan_oracle as H
from tests.test_height_scan_gpu import POINTS, load_wide, oracle_state, staged
from tests.test_task_parity_gpu import inject_noise, read_state

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
f32 = np.float32
WA, WC = 487, 705


@pytest.fixture(scope="module")
def terrain():
    return generate(TerrainConfig(seed=11))


def make_cores(N, terrain, rng, variants, ground="curriculum"):
    """One core per variant (critic_states, heights_in_obs, scan), loaded with the same oracle state. On the curriculum
    terrain with DR (friction and PD-gain tables, redrawn on reset) and pushes; on the plane without either table."""
    cores = []
    for cs, hio, scan in variants:
        if ground == "curriculum":
            hf, origins = terrain
            L, T = origins.shape[:2]
            r = np.random.default_rng(99)
            levels, types = r.integers(0, L, N).astype(np.int32), np.floor(np.arange(N) / (N / T)).astype(np.int32)
            cfg = CoreConfig(heightfield=hf, with_rb_force_tensors=True, height_scan=POINTS if scan else None,
                             terrain_curriculum=TerrainCurriculum(origins, types, levels, 4.0, 16.0), randomize=True,
                             perturb=True, dr_friction_range=(0.5, 1.5), dr_pd_gain_range=(0.8, 1.2),
                             critic_states=cs, critic_heights_in_obs=hio)
        else:
            cfg = CoreConfig(with_rb_force_tensors=True, height_scan=POINTS if scan else None, critic_states=cs,
                             critic_heights_in_obs=hio)
        cores.append(DyrosCore(N, DEV, cfg))
    s, _c = oracle_state(N, rng)
    s["progress_buf"][::3] = 7999  # time-outs at the first step
    jump = torch.tensor(rng.uniform(-3, 3, (N, 2)).astype(f32), device=DEV)
    fr = torch.tensor(rng.uniform(0.5, 1.5, N).astype(f32), device=DEV)
    pd = torch.tensor(rng.uniform(0.8, 1.2, (N, 2)).astype(f32), device=DEV)
    for core in cores:
        load_wide(core, s)
        if ground == "curriculum":
            core.sim_t["root_states"][:, 0:3] = core.task_t["env_origins"] + torch.tensor([0.0, 0.0, 0.93], device=DEV)
            core.sim_t["root_states"][:, 0:2] += jump
            core.sim_t["contact_friction"].copy_(fr)
            core.task_t["pd_gain_scale"].copy_(pd)
            core.task_t["perturb_start"].fill_(1)
            t = core.task_t                                  # every other env in the middle of a push
            t["pert_on"][::2] = 1
            t["perturbation_count"][::2] = 0
            t["pert_duration"][::2] = 1000
            t["magnitude"][::2] = 150.0
            t["phase"][::2] = 0.7
    return cores


def expected_states(core):
    """The oracle's state row from the core's own buffers after a step."""
    torch.cuda.synchronize()
    t, s, N = core.task_t, core.sim_t, core.N
    cfg = core.cfg
    lf, rf = core.tables.body_names.index(cfg.left_foot), core.tables.body_names.index(cfg.right_foot)
    cpu = lambda x: x.cpu().numpy()
    root = cpu(s["root_states"])
    fr = cpu(s["contact_friction"]) if "contact_friction" in s else cfg.friction
    pd = cpu(t["pd_gain_scale"]) if "pd_gain_scale" in t else None
    priv = CS.privileged(root, cpu(s["net_contact_force"]).reshape(N, 38, 3), lf, rf, cpu(t["push_force"]),
                         cpu(t["motor_constant_scale"]), cpu(t["total_mass"]), core.nominal_mass, fr, pd, cpu(t["epi_len"]))
    hc = H.obs_columns(root, cpu(t["measured_heights"])) if "measured_heights" in t else None
    return CS.state_rows(cpu(t["obs_buf"]), hc, priv)


def step_both(cores, rng, paths):
    N = cores[0].N
    noise = O.draw_noise(N, 2, rng)
    actions = torch.tensor(rng.uniform(-1, 1, (N, 13)).astype(f32), device=DEV)
    for core, path in zip(cores, paths):
        inject_noise(core, noise)
        if path == "fused":
            core.step(actions)
            core.compact_resets()
        else:
            staged(core, actions)


@pytest.mark.parametrize("N", [1, 33, 1025, 4096])
@pytest.mark.parametrize("ground", ["plane", "curriculum"])
@pytest.mark.parametrize("path", ["fused", "staged"])
def test_state_row_matches_oracle(terrain, path, ground, N):
    rng = np.random.default_rng(N + (7 if ground == "plane" else 0))
    scan = ground == "curriculum"
    (core,) = make_cores(N, terrain, rng, [(True, False, scan)], ground)
    S = 487 + (187 if scan else 0) + 31
    assert tuple(core.task_t["states_buf"].shape) == (N, S) and core.obs_width == 487
    starts = pushes = 0
    for t in range(6):
        step_both([core], rng, [path])
        want = expected_states(core)
        got = core.task_t["states_buf"].cpu().numpy()
        assert np.array_equal(got, want), f"step {t}: {int((got != want).sum())} entries differ, first at " \
                                          f"{np.argwhere(got != want)[:3].tolist()}"
        assert np.isfinite(got).all() and np.abs(got[:, S - 31:]).max() <= 5
        starts += int((core.task_t["epi_len"] == 0).sum())
        pushes += int((core.task_t["push_force"] != 0).any(1).sum())
    if N >= 33:
        assert starts > 0
        if ground == "curriculum":
            assert pushes > 0
    core.close()


@pytest.mark.parametrize("hio", [False, True])
def test_fused_equals_staged_with_states(terrain, hio):
    N = 257
    rng = np.random.default_rng(5)
    a, b = make_cores(N, terrain, rng, [(True, hio, True), (True, hio, True)])
    for t in range(5):
        step_both([a, b], rng, ["fused", "staged"])
        torch.cuda.synchronize()
        ga, gb = read_state(a), read_state(b)
        for g in (ga, gb):
            g["contact_forces_pre"] = g["contact_forces_pre"].reshape(N, 38, 3)[:, [8, 16]]
        assert ga["states_buf"].shape == (N, 705) and ga["obs_buf"].shape == (N, 674 if hio else 487)
        for k in ga:
            assert np.array_equal(ga[k], gb[k], equal_nan=True), f"step {t}: {k} differs between fused and staged"
    a.close(); b.close()


def test_prefix_and_no_side_effects(terrain):
    """Blind (heights in the state row only), perceptive (heights in both) and no states, same inputs: every buffer but
    obs_buf / states_buf equal bit for bit, the prefix equal to obs_buf, and the blind obs_buf the first 487 columns of
    the 674-wide rows."""
    N = 512
    rng = np.random.default_rng(6)
    blind, seeing, off = make_cores(N, terrain, rng, [(True, False, True), (True, True, True), (False, False, True)])
    g = torch.Generator(device=DEV).manual_seed(1)
    resets = 0
    for t in range(40):
        actions = torch.rand(N, 13, device=DEV, generator=g) * 2 - 1
        for c in (blind, seeing, off):
            c.step(actions)
        torch.cuda.synchronize()
        resets += int(off.task_t["reset_buf"].sum())
        gb, gs, go = read_state(blind), read_state(seeing), read_state(off)
        sb, ss = gb.pop("states_buf"), gs.pop("states_buf")
        ob, os_, oo = gb.pop("obs_buf"), gs.pop("obs_buf"), go.pop("obs_buf")
        assert ob.shape == (N, 487) and os_.shape == (N, 674) and oo.shape == (N, 674)
        assert np.array_equal(os_, oo) and np.array_equal(ob, oo[:, :487])
        assert np.array_equal(sb[:, :487], ob) and np.array_equal(ss[:, :674], os_)
        assert np.array_equal(sb, ss)
        assert gb.keys() == go.keys() == gs.keys()
        for k in go:
            assert np.array_equal(gb[k], go[k], equal_nan=True), f"step {t}: {k} differs with blind states on"
            assert np.array_equal(gs[k], go[k], equal_nan=True), f"step {t}: {k} differs with states on"
    assert resets > 0
    assert blind.step_launches() == off.step_launches() == 3
    blind.close(); seeing.close(); off.close()


# ------------------------------------------------------------------ DyrosDynamicWalk and the PPO paths
def terrain_env(N, critic=True, graph=False, **terrain):
    from isaacgymdyros_b200 import DyrosDynamicWalk, default_cfg
    cfg = default_cfg(N)
    cfg["env"]["terrain"] = {"curriculum": True, "measure_heights": True, "seed": 2, **terrain}
    if critic is not None:
        cfg["env"]["criticStates"] = critic
    return DyrosDynamicWalk(cfg, DEV, use_cuda_graph=graph)


def make_trainer(N=64, H=16, mb=256, **kw):
    from isaacgymdyros_b200.ppo import PPOConfig, PPOTrainer
    env = terrain_env(N)
    assert (env.num_obs, env.num_states) == (WA, WC)
    return env, PPOTrainer(env, PPOConfig(horizon_length=H, minibatch_size=mb, num_states=WC, **kw))


def test_dynamic_walk_with_critic_states():
    N = 1024
    env = terrain_env(N, graph=True)
    assert env.critic_states and env.state_space.shape == (WC,) and env.observation_space.shape == (WA,)
    assert env.states_buf.data_ptr() == env.core.task_t["states_buf"].data_ptr()
    g = torch.Generator(device=DEV).manual_seed(0)
    for i in range(10):
        obs, _rew, _reset, _extras = env.step(torch.rand(N, 13, device=DEV, generator=g) * 2 - 1)
        assert obs["obs"].shape == (N, WA) and obs["states"].shape == (N, WC)
        assert torch.equal(obs["states"][:, :WA], obs["obs"]) and bool(torch.isfinite(obs["states"]).all())
    assert "states" in env.reset() and "states" in env.reset_done()[0]
    with pytest.raises(RuntimeError, match="no critic states"):
        env.step_async(torch.zeros(N, 13, device=DEV))
    plain = terrain_env(64, critic=None)
    assert "states" not in plain.step(torch.zeros(64, 13, device=DEV))[0] and "states" not in plain.reset()
    env.close(); plain.close()


def fill_synthetic(tr, seed):
    g = torch.Generator(device=DEV); g.manual_seed(seed)
    r = lambda *s: torch.randn(*s, device=DEV, generator=g)
    b, N, H = tr.buf, tr.N, tr.H
    if tr.packed is None:
        b["obs"].copy_(r(N, H, WC))
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


def test_packed_bf16_asymmetric_matches_fp32():
    """The packed path at (487, 705), K0 = 712, against fp32 autograd on identical weights (the tolerances of
    test_ppo_wide_gpu.py's packed test); the actor's W0 columns 487..711 zero after pack and after fused Adam steps."""
    from isaacgymdyros_b200 import native
    from isaacgymdyros_b200.ppo import FlatActorCritic
    env, tr = make_trainer()
    pk = tr.packed
    assert pk.K0 == 712 and tuple(pk.w0.shape) == (2, 256, 712) and tuple(tr.x_roll.shape) == (64 * 16, 712)
    assert pk.desc.inputs == WA and pk.critic_inputs == WC and tr.pb.obs_dim == WC
    r = fill_synthetic(tr, seed=9)
    tr.net.flat.copy_((tr.net.flat * 30 + 0.02 * r(tr.net.n)).to(torch.bfloat16).float())
    pk.pack()
    torch.cuda.synchronize()
    assert float(pk.w0[0, :, WA:].float().abs().max()) == 0.0 and float(pk.w0[1, :, WC:].float().abs().max()) == 0.0
    mb, r0 = 256, 512
    tr.x_roll[:, :WC] = r(tr.N * tr.H, WC).to(torch.bfloat16); tr.x_roll[:, WC:] = 0
    batch = oracle_batch(tr, r0, mb)
    onet = FlatActorCritic(DEV, dataclasses.replace(tr.cfg, mixed_precision="fp32"))
    onet.flat.copy_(tr.net.flat)
    mu, v = onet.forward(tr.x_roll[r0:r0 + mb, :WC].float())
    loss, a_loss, c_loss, kl, cf = PO.total_loss(mu, v, onet.logstd, batch, 0.2, 0.5)
    onet.grad.zero_()
    loss.backward()
    mu, v = mu.detach(), v.detach()
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
    for name, (w, bias) in onet.layers.items():
        gw, gb = tr.net.layers[name][0].grad, tr.net.layers[name][1].grad
        assert gw.shape == w.grad.shape
        for got, want, what in ((gw, w.grad, "weight"), (gb, bias.grad, "bias")):
            err = float((got - want).abs().max())
            cos = float((got * want).sum() / (got.norm() * want.norm() + 1e-30))
            assert err < 0.2 * scale(want) + 1e-12, (name, what, err, scale(want))
            assert cos > 0.997, (name, what, cos)
    for x_, y_ in zip(tr.stats.tolist(), (a_loss.item(), c_loss.item(), kl.item(), cf.item())):
        assert x_ == pytest.approx(y_, rel=5e-2, abs=2e-3)
    # the fused optimiser against dyros_ppo_adam on the flat buffers, three steps; the actor's padding stays zero
    for it in range(3):
        grad = tr.net.grad.clone().mul_(100.0 * (it + 1))
        ref = {k: t.clone() for k, t in (("p", tr.net.flat), ("m", tr.net.exp_avg), ("v", tr.net.exp_avg_sq))}
        lr2, st2, n2 = tr.lr.clone(), tr.opt_step.clone(), torch.zeros(1, device=DEV)
        native.check(tr.lib.dyros_ppo_adam(tr._p(ref["p"]), tr._p(grad), tr._p(ref["m"]), tr._p(ref["v"]), tr.net.n_actor, tr.net.n, 0.5,
                                           0.5, tr._p(n2), tr._p(lr2), tr._p(st2), 0.9, 0.999, 1e-8, 1e-5, 3e-6, 5000, tr._stream), "adam")
        tr.net.grad.copy_(grad)
        tr.norm2.zero_()
        native.check(tr.lib.dyros_ppo_adam_packed_ac(C.byref(pk.desc), WC, tr._p(tr.net.flat), tr._p(tr.net.grad), tr._p(tr.net.exp_avg),
                                                     tr._p(tr.net.exp_avg_sq), 0.5, 0.5, 0, tr._p(tr.norm2), tr._p(tr.lr),
                                                     tr._p(tr.opt_step), 0.9, 0.999, 1e-8, 1e-5, 3e-6, 5000, tr._stream), "adam_packed")
        torch.cuda.synchronize()
        assert float((tr.net.flat - ref["p"]).abs().max()) < 1e-8
        for net, name, w in ((0, "actor_mlp.0", WA), (1, "critic_mlp.0", WC)):
            w0 = tr.net.layers[name][0].detach()
            assert w0.shape == (256, w)
            assert torch.equal(pk.w0[net, :, :w].float(), w0.to(torch.bfloat16).float())
        assert float(pk.w0[0, :, WA:].float().abs().max()) == 0.0 and float(pk.w0[1, :, WC:].float().abs().max()) == 0.0
    env.close()


def test_deployable_actor_reads_the_observation_row_alone(tmp_path):
    """The packed actor's mu from the state rows against an fp64 numpy forward of the dumped actor_mlp / mu weights on
    obs_buf alone (the robot-side controller's computation), within the packed-vs-fp32 tolerance."""
    env, tr = make_trainer(H=8)
    tr.train_epoch()
    # weights of a trained scale, bf16-representable (as in the packed test): what differs is the activations' rounding
    tr.net.flat.copy_((tr.net.flat * 30).to(torch.bfloat16).float())
    tr.packed.pack()
    tr._cast_obs(False)
    mu_p, _ = tr.packed.mu_value(tr.packed.forward(tr.x_step))
    torch.cuda.synchronize()
    tr.dump_weights_txt(str(tmp_path))
    L = lambda n: np.loadtxt(str(tmp_path / (n + ".txt")), ndmin=1)
    w0, b0 = L("a2c_network_actor_mlp_0_weight"), L("a2c_network_actor_mlp_0_bias")
    w1, b1 = L("a2c_network_actor_mlp_2_weight"), L("a2c_network_actor_mlp_2_bias")
    wm, bm = L("a2c_network_mu_weight"), L("a2c_network_mu_bias")
    assert w0.shape == (256, WA)
    obs = env.obs_buf.double().cpu().numpy()
    assert obs.shape[1] == WA
    h = np.maximum(obs @ w0.T + b0, 0)
    h = np.maximum(h @ w1.T + b1, 0)
    mu = h @ wm.T + bm
    got = mu_p.double().cpu().numpy()
    assert np.abs(got - mu).max() < 2e-2 * np.abs(mu).max(), np.abs(got - mu).max()
    env.close()


@pytest.mark.parametrize("graph", [False, True])
def test_minibatch_updates_at_487_705_track_the_oracle_fp32(graph):
    """test_ppo_wide_gpu.py's fp32 update test with an asymmetric critic: the actor reads the first 487 columns of each
    stored state row (its master W0 is 256 x 487), the critic all 705; same tolerances."""
    from isaacgymdyros_b200.ppo import FlatActorCritic
    env, tr = make_trainer(mixed_precision="fp32", mini_epochs=2, use_cuda_graph=graph)
    assert tr.buf["obs"].shape == (64, 16, WC) and tr.net.layers["actor_mlp.0"][0].shape == (256, WA)
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
            rows = tr.buf["obs"].reshape(-1, WC)[r0:r0 + mb]
            mu = onet._mlp(rows[:, :WA], "actor_mlp", "mu")
            v = onet._mlp(rows, "critic_mlp", "value").squeeze(-1)
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
    assert na == 194061
    assert torch.allclose(tr.net.flat[:na], onet.flat[:na], rtol=1e-4, atol=2e-7)
    assert torch.allclose(tr.net.flat[na:], onet.flat[na:], rtol=1e-4, atol=5e-6)
    w0 = tr.net.layers["critic_mlp.0"][0]
    assert float((w0[:, WA:] - flat0[na:na + 256 * WC].view(256, WC)[:, WA:]).abs().max()) > 0   # privileged columns train
    got = (tr.stats / (2 * tr.num_minibatches)).tolist()
    for x, y in zip(got, np.mean(np.array(logs), axis=0)):
        assert x == pytest.approx(y, rel=1e-3, abs=1e-6)
    env.close()


def test_trainer_refusals_checkpoint_and_bootstrap(tmp_path):
    from isaacgymdyros_b200 import DyrosDynamicWalk, default_cfg
    from isaacgymdyros_b200.ppo import PPOConfig, PPOTrainer
    plain = terrain_env(64, critic=None)
    with pytest.raises(ValueError, match=r"no kernel-written critic states.*PPOConfig\(num_states=env.num_states\)"):
        PPOTrainer(plain, PPOConfig(horizon_length=8, minibatch_size=256, num_obs=674, num_states=WC))
    cfg = default_cfg(64)
    cfg["env"]["criticStates"] = True
    plane = DyrosDynamicWalk(cfg, DEV, use_cuda_graph=False)
    assert plane.num_states == 518
    with pytest.raises(ValueError, match=r"rows of 518.*PPOConfig\(num_states=env.num_states\)"):
        PPOTrainer(plane, PPOConfig(horizon_length=8, minibatch_size=256, num_states=WC))
    env, tr = make_trainer(H=8)
    with pytest.raises(ValueError, match="rows of 705"):
        PPOTrainer(env, PPOConfig(horizon_length=8, minibatch_size=256, num_states=518))
    # the bootstrap value reads the state row: GAE's last value is the critic's on states_buf
    tr.rollout()
    tr._cast_obs(False)
    torch.cuda.synchronize()
    assert torch.equal(tr.x_step[:, :WC], env.states_buf.to(torch.bfloat16))
    tr.update()
    tr.epoch = 1
    path = tr.save(str(tmp_path / "ckpt"))
    sd = torch.load(path, map_location="cpu", weights_only=False)
    assert tuple(sd["model"]["a2c_network.actor_mlp.0.weight"].shape) == (256, WA)
    assert tuple(sd["model"]["a2c_network.critic_mlp.0.weight"].shape) == (256, WC)
    env2, tr2 = make_trainer(H=8)
    tr2.net.flat.add_(1.0)
    tr2.restore(path)
    for a, b in ((tr.net.flat, tr2.net.flat), (tr.net.exp_avg, tr2.net.exp_avg), (tr.packed.w0, tr2.packed.w0)):
        assert torch.equal(a, b)
    assert float(tr2.packed.w0[0, :, WA:].float().abs().max()) == 0.0
    files = tr.dump_weights_txt(str(tmp_path / "result"))
    assert np.loadtxt(str(tmp_path / "result" / "a2c_network_actor_mlp_0_weight.txt")).shape == (256, WA) and len(files) == 13
    narrow = PPOTrainer(plane, PPOConfig(horizon_length=8, minibatch_size=256))
    with pytest.raises(ValueError, match=r"critic_mlp\.0\.weight: shape \(256, 487\), expected \(256, 705\)"):
        tr2.restore(narrow.save(str(tmp_path / "narrow")))
    env.close(); env2.close(); plain.close(); plane.close()


def test_blind_actor_with_privileged_critic_learns_on_curriculum_terrain():
    """4096 envs on the generated curriculum terrain with the height scan in the critic's state row only: a 487-input
    actor and a 705-input critic, packed bf16, CUDA graphs, the reference's hyper-parameters, 60 epochs. The criterion
    of the perceptive terrain test: mean episode length more than 1.5x epoch 1's by epoch 60."""
    from isaacgymdyros_b200.ppo import PPOConfig, PPOTrainer
    env = terrain_env(4096, graph=True)
    tr = PPOTrainer(env, PPOConfig(num_states=env.num_states))
    outs = [tr.train_epoch() for _ in range(60)]
    first, last = outs[0], outs[-1]
    print("blind-actor terrain learning:", [(round(o["mean_length"], 1), round(o["mean_reward"], 1), round(o["terrain_level"], 3))
                                            for o in outs[::10] + [last]])
    for o in outs:
        assert all(math.isfinite(v) for v in o.values()), o
    assert first["episodes"] > 1000, first
    assert last["mean_length"] > 1.5 * first["mean_length"], (first, last)
    for t in (env.obs_buf, env.states_buf, env.core.sim_t["root_states"]):
        assert bool(torch.isfinite(t).all())
    env.close()
