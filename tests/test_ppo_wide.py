"""The on-device PPO at an input width other than the reference's 487 (PPOConfig.num_obs; 674 = 487 + the 187 points of
the default height scan): the C structs that carry the width against their ctypes mirrors, the networks' parameter
counts and shapes, and the rl_games checkpoint format at that width (the 487 format is pinned in test_ppo_formats.py)."""
import ctypes
import os
import shutil
import subprocess

import pytest
import torch
from torch import nn

from isaacgymdyros_b200 import native
from isaacgymdyros_b200.ppo import FlatActorCritic, PPOConfig, layer_shapes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W = 674


def test_ppo_struct_layouts_match_the_header(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    fields = {"DyrosPpoBuffers": [n for n, _ in native.DyrosPpoBuffers._fields_],
              "DyrosPpoNet": [n for n, _ in native.DyrosPpoNet._fields_]}
    assert fields["DyrosPpoBuffers"][-1] == "obs_dim" and fields["DyrosPpoNet"][:2] == ["hidden", "inputs"]
    prints = []
    for s, names in fields.items():
        prints.append(f'printf("{s} %zu\\n", sizeof({s}));')
        prints += [f'printf("{s}.{n} %zu\\n", offsetof({s}, {n}));' for n in names]
    src = tmp_path / "s.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "dyros_b200.h"\nint main(void) {\n' + "\n".join(prints)
                   + "\nreturn 0; }\n")
    subprocess.check_call(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(tmp_path / "s")])
    got = dict(line.rsplit(" ", 1) for line in subprocess.check_output([str(tmp_path / "s")], text=True).splitlines())
    for s, names in fields.items():
        ct = getattr(native, s)
        assert int(got[s]) == ctypes.sizeof(ct), s
        for n in names:
            assert int(got[f"{s}.{n}"]) == getattr(ct, n).offset, (s, n)
    # `inputs` sits in the padding before the first pointer: the struct kept its size and every other offset
    assert ctypes.sizeof(native.DyrosPpoNet) == 8 + 12 * 8 and native.DyrosPpoNet.inputs.offset == 4
    assert native.DyrosPpoNet.w0.offset == 8
    # zero-initialised (what ctypes does) means the reference's width
    assert native.DyrosPpoBuffers().obs_dim == 0 and native.DyrosPpoNet().inputs == 0


def test_parameter_counts_and_layer_shapes_at_674():
    actor, critic = layer_shapes((256, 256), W)
    assert actor == [("actor_mlp.0", 256, W), ("actor_mlp.1", 256, 256), ("mu", 13, 256)]
    assert critic == [("critic_mlp.0", 256, W), ("critic_mlp.1", 256, 256), ("value", 1, 256)]
    net = FlatActorCritic("cpu", PPOConfig(num_obs=W))
    assert net.n_actor == 256 * W + 256 + 65536 + 256 + 13 * 256 + 13 == 241933
    assert net.n - net.n_actor == 256 * W + 256 + 65536 + 256 + 1 * 256 + 1 == 238849
    w, b = net.layers["actor_mlp.0"]
    assert w.shape == (256, W) and net.layers["critic_mlp.0"][0].shape == (256, W) and b.shape == (256,)
    assert layer_shapes() == layer_shapes((256, 256), 487)                   # the default is the reference's width


class RefA2CNetwork(nn.Module):  # A2CBuilder.Network for `separate: True`, fixed sigma, at input width W
    def __init__(self, w):
        super().__init__()
        mlp = lambda: nn.Sequential(nn.Linear(w, 256), nn.ELU(), nn.Linear(256, 256), nn.ELU())
        self.actor_cnn, self.critic_cnn = nn.Sequential(), nn.Sequential()
        self.actor_mlp, self.critic_mlp = mlp(), mlp()
        self.value = nn.Linear(256, 1)
        self.mu = nn.Linear(256, 13)
        self.sigma = nn.Parameter(torch.zeros(13), requires_grad=False)


class RefModel(nn.Module):
    def __init__(self, w):
        super().__init__()
        self.a2c_network = RefA2CNetwork(w)


def test_checkpoint_format_at_674():
    net = FlatActorCritic("cpu", PPOConfig(num_obs=W))
    g = torch.Generator().manual_seed(0)
    net.flat.copy_(torch.randn(net.n, generator=g))
    net.exp_avg.copy_(torch.randn(net.n, generator=g)); net.exp_avg_sq.copy_(torch.rand(net.n, generator=g))
    ref = RefModel(W)
    sd = net.model_state_dict()
    assert tuple(sd["a2c_network.actor_mlp.0.weight"].shape) == (256, W)
    assert list(sd.keys()) == list(ref.state_dict().keys())
    ref.load_state_dict(sd, strict=True)
    assert torch.equal(ref.a2c_network.critic_mlp[0].weight, net.layers["critic_mlp.0"][0])
    a = list(ref.a2c_network.actor_mlp.parameters()) + list(ref.a2c_network.mu.parameters())
    c = list(ref.a2c_network.critic_mlp.parameters()) + list(ref.a2c_network.value.parameters())
    oa, oc = torch.optim.Adam(a, lr=1e-5, eps=1e-8), torch.optim.Adam(c, lr=5e-4, eps=1e-8)
    oa.load_state_dict(net.optimizer_state_dict(True, 3, 9e-6))
    oc.load_state_dict(net.optimizer_state_dict(False, 3, 5e-4))
    p0 = ref.a2c_network.actor_mlp[0].weight
    assert torch.equal(oa.state[p0]["exp_avg"], net.exp_avg[:256 * W].view(256, W))
    back = FlatActorCritic("cpu", PPOConfig(num_obs=W))
    back.load_model_state_dict(ref.state_dict())
    assert back.load_optimizer_state_dict(True, oa.state_dict()) == 3 and back.load_optimizer_state_dict(False, oc.state_dict()) == 3
    for x, y in ((back.flat, net.flat), (back.exp_avg, net.exp_avg), (back.exp_avg_sq, net.exp_avg_sq)):
        assert torch.equal(x, y)


def test_a_487_checkpoint_does_not_load_into_a_674_net():
    sd = FlatActorCritic("cpu", PPOConfig()).model_state_dict()
    wide = FlatActorCritic("cpu", PPOConfig(num_obs=W))
    with pytest.raises(ValueError, match=r"actor_mlp\.0\.weight: shape \(256, 487\), expected \(256, 674\)"):
        wide.load_model_state_dict(sd)
