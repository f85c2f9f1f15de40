"""Critic states on the CPU: the cfg["env"]["criticStates"] plumbing and its refusals, the oracle
(tests/critic_states_oracle.py) against hand-built known answers, the new C struct against gcc, the asymmetric critic's
layer shapes and parameter counts at (Wa, Wc) = (487, 705), the rl_games checkpoint at those widths, and the refusals of
the PPO trainer and of the *_ac entry points that need no GPU."""
import ctypes
import os
import shutil
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest
import torch
from torch import nn

from isaacgymdyros_b200 import native
from isaacgymdyros_b200.ppo import FlatActorCritic, PPOConfig, PPOTrainer, layer_shapes
from tests import critic_states_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32
WA, WC = 487, 705


def walk_cfg(critic=None, **terrain):
    from isaacgymdyros_b200 import default_cfg
    cfg = default_cfg(64)
    if terrain:
        cfg["env"]["terrain"] = dict(num_rows=2, num_cols=2, terrain_length=4.0, terrain_width=4.0, border_size=2.0, **terrain)
    if critic is not None:
        cfg["env"]["criticStates"] = critic
    return cfg


# ------------------------------------------------------------------ cfg plumbing
def test_widths():
    from isaacgymdyros_b200.tasks.dyros_dynamic_walk import core_config_from_cfg, num_observations, num_states
    cases = [(walk_cfg(True), 487, 518, False),                                             # the plane
             (walk_cfg(True, measure_heights=True), 487, 705, False),                        # blind actor
             (walk_cfg({"heights_in_obs": True}, measure_heights=True), 674, 705, True),     # perceptive actor
             (walk_cfg({}, measure_heights=True), 487, 705, False),
             (walk_cfg({"heights_in_obs": False}, measure_heights=True), 487, 705, False),
             (walk_cfg(True, mesh_type="plane", measure_heights=True), 487, 705, False)]
    for cfg, nobs, nst, hio in cases:
        assert (num_observations(cfg), num_states(cfg)) == (nobs, nst)
        c = core_config_from_cfg(cfg, torch.Generator().manual_seed(0))
        assert c.critic_states and c.critic_heights_in_obs == hio
    # off: absent or False, and numStates as today
    for cfg in (walk_cfg(), walk_cfg(False), walk_cfg(False, measure_heights=True), walk_cfg(None)):
        assert num_states(cfg) == 0
        assert not core_config_from_cfg(cfg, torch.Generator().manual_seed(0)).critic_states
    cfg = walk_cfg(measure_heights=True)
    assert num_observations(cfg) == 674
    cfg["env"]["numStates"] = 12
    assert num_states(cfg) == 12                                                             # (VecTask's own buffer)


def test_refusals():
    from isaacgymdyros_b200.tasks.dyros_dynamic_walk import DyrosDynamicWalk, core_config_from_cfg
    with pytest.raises(ValueError, match="heights_in_obs needs a height scan"):
        core_config_from_cfg(walk_cfg({"heights_in_obs": True}))
    with pytest.raises(ValueError, match="heights_in_obs needs a height scan"):
        core_config_from_cfg(walk_cfg({"heights_in_obs": True}, measure_heights=False))
    for bad in ("yes", 1, {"heights": True}, {"heights_in_obs": 1}, [True]):
        with pytest.raises(ValueError, match="criticStates"):
            core_config_from_cfg(walk_cfg(bad, measure_heights=True))
    # a given numStates that disagrees (refused before any device is touched)
    cfg = walk_cfg(True, measure_heights=True)
    cfg["env"]["numStates"] = 518
    with pytest.raises(ValueError, match="numStates.*705"):
        DyrosDynamicWalk(cfg, sim_device="cuda:0")
    cfg = walk_cfg(True, measure_heights=True)
    cfg["env"]["numStates"] = 705
    if not torch.cuda.is_available():  # (agreeing: passes the check, then needs the device)
        with pytest.raises(Exception) as e:
            DyrosDynamicWalk(cfg, sim_device="cuda:0")
        assert "numStates" not in str(e.value)


# ------------------------------------------------------------------ oracle
def test_oracle_known_answers():
    n = 3
    root = np.zeros((n, 13), f32)
    root[:, 7:10] = [[1.0, -2.0, 0.5], [3.0, 0.0, 0.0], [-0.25, 0.0, 0.0]]
    root[:, 10:13] = [[4.0, -8.0, 30.0], [0.0, 0.0, 0.0], [0.0, 0.0, 0.0]]
    ncf = np.zeros((n, 38, 3), f32)
    lf, rf = 7, 13
    ncf[:, lf] = [[100.0, -200.0, 900.0], [0.0, 0.0, 7000.0], [1.0, 1.0, 1.0]]
    ncf[:, rf] = [[0.0, 0.0, 400.0], [0.0, 0.0, -9000.0], [2.0, 2.0, 2.0]]
    ncf[:, 0] = 1e6                                                                  # (not a foot: never read)
    push = np.array([[50.0, -100.0, 0.0], [1000.0, 0.0, 0.0], [5.0, 5.0, 0.0]], f32)
    mcs = np.full((n, 12), 1.0, f32)
    mcs[0] = np.linspace(0.8, 1.2, 12)
    mass = np.array([104.48, 52.24, 1e6], f32)
    epi = np.array([3.0, 10.0, 0.0], f32)
    pd = np.array([[0.9, 1.1], [1.0, 1.0], [np.nan, 20.0]], f32)
    v = O.privileged(root, ncf, lf, rf, push, mcs, mass, 104.48, 1.0, pd, epi)
    assert v.shape == (3, 31) and v.dtype == f32
    np.testing.assert_array_equal(v[0, 0:6], f32([2.0, -4.0, 1.0, 1.0, -2.0, 5.0]))          # 30 * 0.25 = 7.5 -> 5
    np.testing.assert_array_equal(v[1, 0:3], f32([5.0, 0.0, 0.0]))                          # 6 -> clipped
    np.testing.assert_allclose(v[0, 6:12], [0.1, -0.2, 0.9, 0.0, 0.0, 0.4], rtol=1e-6)
    np.testing.assert_allclose(v[1, 6:12], [0.0, 0.0, 5.0, 0.0, 0.0, -5.0])                 # 7 and -9 -> clipped
    np.testing.assert_allclose(v[0, 12:15], [0.5, -1.0, 0.0], rtol=1e-6)
    assert v[1, 12] == 5.0                                                                  # 10 -> clipped
    # episode start (epi_len == 0): contact-force and push columns are 0, the others are not
    np.testing.assert_array_equal(v[2, 6:15], np.zeros(9, f32))
    assert v[2, 0] == f32(-0.5)
    np.testing.assert_allclose(v[0, 15:27], np.linspace(0.8, 1.2, 12) - 1, atol=1e-6)
    assert v[0, 27] == 0.0 and v[1, 27] == f32(-0.5) and v[2, 27] == 5.0                    # mass ratio, clipped
    np.testing.assert_array_equal(v[:, 28], np.zeros(3, f32))                               # friction 1.0 of the sim
    np.testing.assert_allclose(v[0, 29:31], [-0.1, 0.1], atol=1e-6)
    assert v[2, 29] == -5.0 and v[2, 30] == 5.0                                             # NaN -> -5 (fminf / fmaxf)
    assert np.all(np.isfinite(v))
    # a friction table, no PD-gain table
    v2 = O.privileged(root, ncf, lf, rf, push, mcs, mass, 104.48, np.array([0.5, 1.0, 9.0], f32), None, epi)
    np.testing.assert_array_equal(v2[:, 28], f32([-0.5, 0.0, 5.0]))
    np.testing.assert_array_equal(v2[:, 29:31], np.zeros((3, 2), f32))
    # row layout: 487 | P | 31
    obs = np.arange(3 * 674, dtype=f32).reshape(3, 674)
    rows = O.state_rows(obs, obs[:, 487:], v)
    assert rows.shape == (3, 705)
    np.testing.assert_array_equal(rows[:, :674], obs)
    np.testing.assert_array_equal(rows[:, 674:], v)
    assert O.state_rows(obs[:, :487], None, v).shape == (3, 518)


# ------------------------------------------------------------------ C ABI
def test_struct_layout_matches_the_header(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    names = [n for n, _ in native.DyrosCriticStates._fields_]
    prints = ['printf("size %zu\\n", sizeof(DyrosCriticStates));']
    prints += [f'printf("{n} %zu\\n", offsetof(DyrosCriticStates, {n}));' for n in names]
    src = tmp_path / "s.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "dyros_b200.h"\nint main(void) {\n' + "\n".join(prints)
                   + "\nreturn 0; }\n")
    subprocess.check_call(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(tmp_path / "s")])
    got = dict(line.rsplit(" ", 1) for line in subprocess.check_output([str(tmp_path / "s")], text=True).splitlines())
    assert int(got["size"]) == ctypes.sizeof(native.DyrosCriticStates) == 16
    for n in names:
        assert int(got[n]) == getattr(native.DyrosCriticStates, n).offset, n
    # the PPO structs keep their layouts: the critic's width travels as an argument of the *_ac entry points
    assert ctypes.sizeof(native.DyrosPpoNet) == 104 and native.DyrosPpoBuffers._fields_[-1][0] == "obs_dim"


def test_entry_points_exported_and_refusing():
    lib = native.load()
    syms = native.header_symbols()
    for s in ("dyros_task_set_critic_states", "dyros_ppo_pack_params_ac", "dyros_ppo_unpack_grads_ac",
              "dyros_ppo_adam_packed_ac", "dyros_ppo_unpack_grads_peers_ac"):
        assert s in syms and s in native.SIGNATURES
    assert lib.dyros_task_set_critic_states(None, None) != 0 and b"task is NULL" in lib.dyros_last_error()
    # a critic narrower than the actor, or a negative width, is refused before anything is launched
    net = native.DyrosPpoNet()
    net.hidden, net.inputs = 256, WA
    for k in ("w0", "b0", "w1", "b1", "wh", "bh", "gw0", "gw1", "gwh", "gb0", "gb1", "gbh"):
        setattr(net, k, 256)  # (never dereferenced: the width check comes first)
    for bad in (486, -1, 100):
        assert lib.dyros_ppo_pack_params_ac(ctypes.byref(net), bad, ctypes.c_void_p(256), None) != 0
        assert b"critic_inputs" in lib.dyros_last_error()
        assert lib.dyros_ppo_unpack_grads_ac(ctypes.byref(net), bad, ctypes.c_void_p(256), None, None) != 0
        assert b"critic_inputs" in lib.dyros_last_error()


# ------------------------------------------------------------------ networks and checkpoints
def test_layer_shapes_and_parameter_counts_at_487_705():
    actor, critic = layer_shapes((256, 256), WA, WC)
    assert actor == [("actor_mlp.0", 256, WA), ("actor_mlp.1", 256, 256), ("mu", 13, 256)]
    assert critic == [("critic_mlp.0", 256, WC), ("critic_mlp.1", 256, 256), ("value", 1, 256)]
    assert layer_shapes((256, 256), WA, 0) == layer_shapes((256, 256), WA)          # 0: the critic reads the obs row
    net = FlatActorCritic("cpu", PPOConfig(num_states=WC))
    assert net.n_actor == 256 * WA + 256 + 65536 + 256 + 13 * 256 + 13 == 194061
    assert net.n - net.n_actor == 256 * WC + 256 + 65536 + 256 + 256 + 1 == 246785
    assert net.layers["actor_mlp.0"][0].shape == (256, WA) and net.layers["critic_mlp.0"][0].shape == (256, WC)
    assert net.critic_inputs == WC
    with pytest.raises(ValueError, match="num_states = 400 < num_obs = 487"):
        FlatActorCritic("cpu", PPOConfig(num_states=400))
    # the actor reads the first num_obs columns of a state row; the critic all of them
    g = torch.Generator().manual_seed(1)
    net.flat.copy_(torch.randn(net.n, generator=g) * 0.05)
    rows = torch.randn(5, WC, generator=g)
    mu, v = net.forward(rows)
    mu0 = net._mlp(rows[:, :WA], "actor_mlp", "mu")
    assert torch.equal(mu, mu0)
    rows2 = rows.clone()
    rows2[:, WA:] += 1.0
    mu2, v2 = net.forward(rows2)
    assert torch.equal(mu2, mu) and not torch.equal(v2, v)


class RefA2CNetwork(nn.Module):  # A2CBuilder.Network for `separate: True`, fixed sigma, actor width wa, critic width wc
    def __init__(self, wa, wc):
        super().__init__()
        mlp = lambda w: nn.Sequential(nn.Linear(w, 256), nn.ELU(), nn.Linear(256, 256), nn.ELU())
        self.actor_cnn, self.critic_cnn = nn.Sequential(), nn.Sequential()
        self.actor_mlp, self.critic_mlp = mlp(wa), mlp(wc)
        self.value = nn.Linear(256, 1)
        self.mu = nn.Linear(256, 13)
        self.sigma = nn.Parameter(torch.zeros(13), requires_grad=False)


class RefModel(nn.Module):
    def __init__(self, wa, wc):
        super().__init__()
        self.a2c_network = RefA2CNetwork(wa, wc)


def test_checkpoint_format_at_487_705():
    net = FlatActorCritic("cpu", PPOConfig(num_states=WC))
    g = torch.Generator().manual_seed(0)
    net.flat.copy_(torch.randn(net.n, generator=g))
    sd = net.model_state_dict()
    assert tuple(sd["a2c_network.actor_mlp.0.weight"].shape) == (256, WA)
    assert tuple(sd["a2c_network.critic_mlp.0.weight"].shape) == (256, WC)
    ref = RefModel(WA, WC)
    assert list(sd.keys()) == list(ref.state_dict().keys())
    ref.load_state_dict(sd, strict=True)
    assert torch.equal(ref.a2c_network.critic_mlp[0].weight, net.layers["critic_mlp.0"][0])
    assert torch.equal(ref.a2c_network.actor_mlp[0].weight, net.layers["actor_mlp.0"][0])
    back = FlatActorCritic("cpu", PPOConfig(num_states=WC))
    back.load_model_state_dict(ref.state_dict())
    assert torch.equal(back.flat, net.flat)
    # a checkpoint of either other width fails on that shape
    with pytest.raises(ValueError, match=r"critic_mlp\.0\.weight: shape \(256, 487\), expected \(256, 705\)"):
        back.load_model_state_dict(FlatActorCritic("cpu", PPOConfig()).model_state_dict())
    with pytest.raises(ValueError, match=r"actor_mlp\.0\.weight: shape \(256, 674\), expected \(256, 487\)"):
        back.load_model_state_dict(FlatActorCritic("cpu", PPOConfig(num_obs=674, num_states=WC)).model_state_dict())


def test_trainer_refusals_without_a_gpu():
    plain = SimpleNamespace(num_obs=WA, num_envs=8, device="cpu", num_states=0)
    with pytest.raises(ValueError, match=r"no kernel-written critic states.*PPOConfig\(num_states=env.num_states\)"):
        PPOTrainer(plain, PPOConfig(num_states=WC))
    vectask = SimpleNamespace(num_obs=WA, num_envs=8, device="cpu", num_states=WC)  # a zero states_buf of VecTask
    with pytest.raises(ValueError, match="no kernel-written critic states"):
        PPOTrainer(vectask, PPOConfig(num_states=WC))
    wide = SimpleNamespace(num_obs=WA, num_envs=8, device="cpu", num_states=WC, critic_states=True)
    with pytest.raises(ValueError, match=r"rows of 705.*PPOConfig\(num_states=env.num_states\)"):
        PPOTrainer(wide, PPOConfig(num_states=518))
    plane = SimpleNamespace(num_obs=WA, num_envs=8, device="cpu", num_states=518, critic_states=True)
    with pytest.raises(ValueError, match="rows of 518"):
        PPOTrainer(plane, PPOConfig(num_states=WC))
