"""On-device PPO around the env step (SURVEY 8f-1, BASELINE configs[4]): the rollout / update loop of the reference's
rl_games fork -- learning/rl_games_custom/a2c_common_dyros.py (A2C: play_steps 629-703, discount_values 485-500,
prepare_dataset 921-969, train_epoch 837-918), a2c_continuous_seperate.py (AG: calc_gradients 108-227, the two Adam
optimisers 50-54), models_dyros.py (MD), network_builder_dyros.py, cfg/train/DyrosDynamicWalkPPO.yaml (PPO) -- with
nothing leaving the GPU: the policy reads the env's observation buffer in place, actions go to the env step in place,
the rollout buffers, GAE, the loss gradient and both optimisers are kernels of libdyros_b200.so (csrc/ppo_kernels.cu),
one rollout step and one minibatch update are each ONE CUDA graph, and with several ranks the only traffic is one NCCL
all-reduce of the flat 1.54 MB gradient bucket per minibatch (AG:161-203) plus a few scalars per epoch.

The two W-256-256-{13,1} MLPs are library GEMMs (torch / cuBLAS); parameters, gradients and Adam moments live in flat
fp32 buffers. W = PPOConfig.num_obs, the env's observation width: the reference's 487, or 674 with the default height scan
(terrain measure_heights). Both networks see the whole row, unless PPOConfig.num_states asks for an asymmetric critic:
the critic then reads the env's critic state row (num_states = Wc columns, DESIGN.md section 4, "Critic states"), whose
first num_obs columns are the observation row, and the actor reads those first num_obs columns only. Two network
paths:
  * `mixed_precision="bf16"` (default; the reference trains under fp16 autocast + GradScaler, PPO:59): `PackedNets` --
    actor and critic as ONE batch-2 problem in GEMM layout (bf16 weights, input width padded to K0 = round_up(W, 8):
    487 -> 488, 674 -> 680; with critic states W = Wc, 705 -> 712, and the actor's W0 is zero past its num_obs
    columns), 8 batched
    GEMMs per minibatch with hand-written backward and the library's own kernels in between (csrc/ppo_kernels.cu,
    "packed bf16 path"): 21 launches per minibatch instead of 79;
  * `mixed_precision="fp32"`: torch autograd on views of the flat buffers (what the tests pin against the oracle)."""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import Dict, Optional

import torch
import torch.nn.functional as F

from . import native

NOBS, NA = 487, 13


@dataclass
class PPOConfig:
    """cfg/train/DyrosDynamicWalkPPO.yaml (PPO:28-97)."""
    horizon_length: int = 128
    minibatch_size: int = 4096
    mini_epochs: int = 5
    gamma: float = 0.99
    tau: float = 0.95
    learning_rate: float = 1e-5
    learning_rate_min: float = 3e-6
    critic_learning_rate: float = 5e-4      # AG:54
    lr_schedule: str = "linear"
    max_epochs: int = 5000
    e_clip: float = 0.2
    critic_coef: float = 0.5
    grad_norm: float = 0.5
    truncate_grads: bool = True
    normalize_advantage: bool = True
    value_bootstrap: bool = True
    reward_scale: float = 1.0
    units: tuple = (256, 256)
    init_gain: float = 0.01                 # orthogonal_initializer gain, PPO:37-38
    sigma_init: float = -2.302585           # PPO:21-23
    sigma_last: float = -2.9957             # PPO:24-26
    mixed_precision: str = "bf16"           # "bf16" | "fp32"
    grad_sync: str = "peer"                 # world > 1, bf16 path: "peer" = sum over peer-mapped buffers inside the optimiser's
                                            # kernels (NVLink); "peer2" = the same as reduce-scatter + all-gather;
                                            # "nccl" = one all-reduce call per minibatch (AG:161-173)
    seed: int = 42
    use_cuda_graph: bool = True
    graph_span: str = "mini_epoch"          # one CUDA graph per "minibatch" update, or one for all minibatches of a "mini_epoch"
    num_obs: int = NOBS                     # input width of both networks = the env's num_obs (network_builder_dyros.py
                                            # takes it from the observation space); 674 with the default height scan
    num_states: int = 0                     # > 0: asymmetric critic, whose input is the env's critic state row of this
                                            # width (= env.num_states, criticStates); 0: the critic reads the observation row


def layer_shapes(units=(256, 256), num_obs=NOBS, num_states=0):
    """(name, out, in) of the actor and the critic (network_builder_dyros.py:129-216, `separate: True`); the critic's
    input width is num_states if > 0 (asymmetric critic), else num_obs."""
    dims = [num_obs] + list(units)
    cdims = [num_states or num_obs] + list(units)
    actor = [(f"actor_mlp.{i}", dims[i + 1], dims[i]) for i in range(len(units))] + [("mu", NA, dims[-1])]
    critic = [(f"critic_mlp.{i}", cdims[i + 1], cdims[i]) for i in range(len(units))] + [("value", 1, cdims[-1])]
    return actor, critic


class FlatActorCritic:
    """Parameters, gradients and Adam moments of both networks in flat fp32 buffers: [0, n_actor) actor, then critic.
    The layer tensors are views (the flat gradient buffer is what the all-reduce and the optimiser kernel see)."""

    def __init__(self, device, cfg: PPOConfig):
        self.cfg, self.device = cfg, torch.device(device)
        if cfg.num_states and cfg.num_states < cfg.num_obs:
            raise ValueError(f"PPOConfig.num_states = {cfg.num_states} < num_obs = {cfg.num_obs}: a critic state row starts "
                             "with the observation row")
        actor, critic = layer_shapes(cfg.units, cfg.num_obs, cfg.num_states)
        self.critic_inputs = cfg.num_states or cfg.num_obs
        self.n_actor = sum(o * i + o for _, o, i in actor)
        self.n = self.n_actor + sum(o * i + o for _, o, i in critic)
        self.flat = torch.zeros(self.n, device=device)
        self.grad = torch.zeros(self.n, device=device)
        self.exp_avg = torch.zeros(self.n, device=device)
        self.exp_avg_sq = torch.zeros(self.n, device=device)
        self.layers: Dict[str, tuple] = {}
        off = 0
        gen = torch.Generator(device="cpu")
        gen.manual_seed(cfg.seed)
        for name, o, i in actor + critic:
            w = torch.nn.Parameter(torch.empty(0, device=device))
            w.data = self.flat[off:off + o * i].view(o, i)
            w.grad = self.grad[off:off + o * i].view(o, i)
            init = torch.empty(o, i)
            torch.nn.init.orthogonal_(init, gain=cfg.init_gain, generator=gen)  # every nn.Linear, network_builder_dyros.py:113-118
            w.data.copy_(init)
            off += o * i
            b = torch.nn.Parameter(torch.empty(0, device=device))
            b.data = self.flat[off:off + o]
            b.grad = self.grad[off:off + o]  # zeros (network_builder_dyros.py:117-118)
            off += o
            self.layers[name] = (w, b)
        assert off == self.n
        # fixed, non-trainable log-std (network_builder_dyros.py:103; PPO:27 fixed_sigma), scheduled by update_action_noise
        self.logstd = torch.full((NA,), cfg.sigma_init, device=device)
        self.n_hidden = len(cfg.units)

    def update_action_noise(self, progress_remaining: float):
        """MD:64-70."""
        b = 2 * progress_remaining - 1 if progress_remaining > 0.5 else 0.0
        self.logstd.fill_(self.cfg.sigma_init * b + self.cfg.sigma_last * (1 - b))

    # ------------------------------------------------------------------ on-disk formats of the reference (SURVEY 8f-4)
    # model.state_dict() of ModelA2CContinuousLogStdDYROS.Network (models_dyros.py:17-20) around the A2CBuilder network
    # (network_builder_dyros.py:78-97): `a2c_network.sigma`, then the Linear layers of the two nn.Sequential MLPs
    # (Linear, activation, Linear, activation: indices 0 and 2), then `value`, then `mu`.
    def _named(self):
        out = []
        for prefix, head in (("actor_mlp", None), ("critic_mlp", None), (None, "value"), (None, "mu")):
            if prefix:
                for i in range(self.n_hidden):
                    out.append((f"a2c_network.{prefix}.{2 * i}", self.layers[f"{prefix}.{i}"]))
            else:
                out.append((f"a2c_network.{head}", self.layers[head]))
        return out

    def model_state_dict(self) -> "collections.OrderedDict":
        import collections
        sd = collections.OrderedDict()
        sd["a2c_network.sigma"] = self.logstd.detach().clone().cpu()
        for name, (w, b) in self._named():
            sd[name + ".weight"] = w.detach().clone().cpu()
            sd[name + ".bias"] = b.detach().clone().cpu()
        return sd

    def load_model_state_dict(self, sd) -> None:
        want = self.model_state_dict()
        if set(sd.keys()) != set(want.keys()):
            raise KeyError(f"model state dict: unexpected {sorted(set(sd) - set(want))}, missing {sorted(set(want) - set(sd))}")
        for k, v in sd.items():
            if tuple(v.shape) != tuple(want[k].shape):
                raise ValueError(f"{k}: shape {tuple(v.shape)}, expected {tuple(want[k].shape)}")
        with torch.no_grad():
            self.logstd.copy_(sd["a2c_network.sigma"])
            for name, (w, b) in self._named():
                w.copy_(sd[name + ".weight"])
                b.copy_(sd[name + ".bias"])

    def _optimizer_params(self, actor: bool):
        """Parameter order of optimizer_actor / optimizer_critic (AG:50-54): the MLP's parameters, then the head's."""
        names = ([f"actor_mlp.{i}" for i in range(self.n_hidden)] + ["mu"]) if actor else \
                ([f"critic_mlp.{i}" for i in range(self.n_hidden)] + ["value"])
        return [p for n in names for p in self.layers[n]]

    def _moment_views(self, p: torch.Tensor):
        off = (p.data_ptr() - self.flat.data_ptr()) // 4
        return self.exp_avg[off:off + p.numel()].view(p.shape), self.exp_avg_sq[off:off + p.numel()].view(p.shape)

    def optimizer_state_dict(self, actor: bool, step: int, lr: float) -> dict:
        """torch.optim.Adam.state_dict() of the fork's optimizer_actor / optimizer_critic."""
        params = self._optimizer_params(actor)
        state = {}
        for i, p in enumerate(params):
            m, v = self._moment_views(p)
            if step > 0:
                state[i] = {"step": torch.tensor(float(step)), "exp_avg": m.detach().clone().cpu(), "exp_avg_sq": v.detach().clone().cpu()}
        group = {"lr": lr, "betas": (0.9, 0.999), "eps": 1e-08, "weight_decay": 0.0, "amsgrad": False, "maximize": False,
                 "foreach": None, "capturable": False, "differentiable": False, "fused": None, "decoupled_weight_decay": False,
                 "params": list(range(len(params)))}
        return {"state": state, "param_groups": [group]}

    def load_optimizer_state_dict(self, actor: bool, sd: dict) -> int:
        params = self._optimizer_params(actor)
        step = 0
        with torch.no_grad():
            for i, p in enumerate(params):
                m, v = self._moment_views(p)
                st = sd["state"].get(i)
                if st is None:
                    m.zero_(); v.zero_()
                    continue
                m.copy_(st["exp_avg"]); v.copy_(st["exp_avg_sq"])
                step = int(float(st["step"]))
        return step

    def _mlp(self, x, prefix, head):
        for i in range(self.n_hidden):
            w, b = self.layers[f"{prefix}.{i}"]
            x = F.relu(F.linear(x, w, b))
        w, b = self.layers[head]
        return F.linear(x, w, b)

    def forward(self, obs):
        """mu (B,13), value (B) -- `mu_activation: None`, value head linear (PPO:17-18). With an asymmetric critic `obs`
        is a batch of critic state rows: the actor takes their first num_obs columns."""
        amp = self.cfg.mixed_precision == "bf16"
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp and obs.is_cuda):
            mu = self._mlp(obs[..., :self.cfg.num_obs] if obs.shape[-1] != self.cfg.num_obs else obs, "actor_mlp", "mu")
            v = self._mlp(obs, "critic_mlp", "value")
        return mu, v.squeeze(-1)


class PackedNets:
    """bf16 compute copies of the flat master parameters in GEMM layout (include/dyros_b200.h DyrosPpoNet) and the
    forward / backward of both networks as batch-2 GEMMs. Activations of the last `forward` are kept for `backward`.
    K0 = round_up(Wc, 8) is the padded input width of W0 and of the bf16 input rows, Wc the critic's input width
    (num_states, or num_obs): columns num_obs.. of the actor's W0 and Wc.. of the critic's and of the rows are zero."""
    HEAD = 16

    def __init__(self, net: FlatActorCritic, lib):
        if len(net.cfg.units) != 2 or net.cfg.units[0] != net.cfg.units[1] or net.cfg.units[0] % 8:
            raise ValueError("the packed path holds two hidden layers of equal width (a multiple of 8), PPO:28-35")
        self.net, self.lib, dev = net, lib, net.device
        Hd = self.hidden = net.cfg.units[0]
        self.critic_inputs = net.cfg.num_states  # (0: the actor's width; the *_ac entry points take it)
        self.K0 = (net.critic_inputs + 7) // 8 * 8
        zb = lambda *s: torch.zeros(*s, dtype=torch.bfloat16, device=dev)
        zf = lambda *s: torch.zeros(*s, dtype=torch.float32, device=dev)
        self.w0, self.w1, self.wh = zb(2, Hd, self.K0), zb(2, Hd, Hd), zb(2, self.HEAD, Hd)
        self.b0, self.b1, self.bh = zf(2, Hd), zf(2, Hd), zf(2, self.HEAD)
        self.gw0, self.gw1, self.gwh = zb(2, Hd, self.K0), zb(2, Hd, Hd), zb(2, self.HEAD, Hd)
        self.gb0, self.gb1, self.gbh = zf(2, Hd), zf(2, Hd), zf(2, self.HEAD)
        d = native.DyrosPpoNet()
        d.hidden, d.inputs = Hd, net.cfg.num_obs
        for k in ("w0", "b0", "w1", "b1", "wh", "bh", "gw0", "gw1", "gwh", "gb0", "gb1", "gbh"):
            setattr(d, k, getattr(self, k).data_ptr())
        self.desc = d
        self._act = {}   # rows -> (h0, h1, out, dout, t1, t0) work buffers
        self.pack()

    @property
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.net.device).cuda_stream)

    def pack(self):
        native.check(self.lib.dyros_ppo_pack_params_ac(C.byref(self.desc), self.critic_inputs, C.c_void_p(self.net.flat.data_ptr()),
                                                       self._stream), "pack")

    def unpack_grads(self, norm2: Optional[torch.Tensor] = None):
        native.check(self.lib.dyros_ppo_unpack_grads_ac(C.byref(self.desc), self.critic_inputs, C.c_void_p(self.net.grad.data_ptr()),
                                                     C.c_void_p(norm2.data_ptr()) if norm2 is not None else None, self._stream), "unpack")

    def _buffers(self, rows: int):
        b = self._act.get(rows)
        if b is None:
            dev, Hd = self.net.device, self.hidden
            zb = lambda *s: torch.empty(*s, dtype=torch.bfloat16, device=dev)
            b = {"h0": zb(2, rows, Hd), "h1": zb(2, rows, Hd), "out": zb(2, rows, self.HEAD), "dout": zb(2, rows, self.HEAD),
                 "d1": zb(2, rows, Hd), "d0": zb(2, rows, Hd)}
            self._act[rows] = b
        return b

    def forward(self, x: torch.Tensor):
        """x (rows, K0) bf16 -> head output (2, rows, 16) bf16 WITHOUT the head bias (the consumers add `bh`)."""
        rows = x.shape[0]
        b, s, lib = self._buffers(rows), self._stream, self.lib
        xe = x.unsqueeze(0).expand(2, rows, self.K0)
        torch.bmm(xe, self.w0.transpose(1, 2), out=b["h0"])
        native.check(lib.dyros_ppo_bias_relu(C.c_void_p(b["h0"].data_ptr()), C.c_void_p(self.b0.data_ptr()), rows, self.hidden, s), "bias_relu")
        torch.bmm(b["h0"], self.w1.transpose(1, 2), out=b["h1"])
        native.check(lib.dyros_ppo_bias_relu(C.c_void_p(b["h1"].data_ptr()), C.c_void_p(self.b1.data_ptr()), rows, self.hidden, s), "bias_relu")
        torch.bmm(b["h1"], self.wh.transpose(1, 2), out=b["out"])
        return b["out"]

    def backward(self, x: torch.Tensor):
        """Given `dout` (filled by dyros_ppo_loss_grad_packed for the rows of the last forward): all weight gradients
        (bf16, GEMM layout) and bias gradients (fp32, accumulated)."""
        rows = x.shape[0]
        b, s, lib = self._buffers(rows), self._stream, self.lib
        xe = x.unsqueeze(0).expand(2, rows, self.K0)
        torch.bmm(b["dout"].transpose(1, 2), b["h1"], out=self.gwh)                       # (2,16,H)
        torch.bmm(b["dout"], self.wh, out=b["d1"])                                        # (2,rows,H)
        native.check(lib.dyros_ppo_relu_bwd(C.c_void_p(b["d1"].data_ptr()), C.c_void_p(b["h1"].data_ptr()),
                                            C.c_void_p(self.gb1.data_ptr()), rows, self.hidden, s), "relu_bwd")
        torch.bmm(b["d1"].transpose(1, 2), b["h0"], out=self.gw1)                         # (2,H,H)
        torch.bmm(b["d1"], self.w1, out=b["d0"])
        native.check(lib.dyros_ppo_relu_bwd(C.c_void_p(b["d0"].data_ptr()), C.c_void_p(b["h0"].data_ptr()),
                                            C.c_void_p(self.gb0.data_ptr()), rows, self.hidden, s), "relu_bwd")
        torch.bmm(b["d0"].transpose(1, 2), xe, out=self.gw0)                              # (2,H,K0)

    def mu_value(self, out: torch.Tensor):
        """fp32 (rows,13) mu and (rows) value of a head output (tests, the bootstrap value of the last observation)."""
        return out[0, :, :NA].float() + self.bh[0, :NA], out[1, :, 0].float() + self.bh[1, 0]


class _DevMem:
    """A raw device allocation seen by torch (CUDA array interface)."""

    def __init__(self, ptr: int, nfloats: int):
        self.__cuda_array_interface__ = {"shape": (nfloats,), "typestr": "<f4", "data": (ptr, False), "version": 3}


class PeerGrads:
    """Every rank's two flat gradient buffers and flag words mapped into every rank (CUDA IPC, one node): the plumbing of
    include/dyros_b200.h DyrosPpoPeers. The exchange itself is dyros_ppo_reduce_peers."""

    def __init__(self, n: int, device, rank: int, world: int):
        import torch.distributed as dist
        if not 2 <= world <= 8:
            raise ValueError("peer-memory gradient exchange: 2..8 ranks on one node")
        self.lib = native.load()
        self.stride = (n + 3) // 4 * 4
        nfl = 4 * self.stride + 32                                   # [G0 | G1 | S0 | S1 | 8 + 8 flag words | 2 partial norms + pad]
        with torch.cuda.device(device):
            ptr, handle = C.c_void_p(), C.create_string_buffer(64)
            native.check(self.lib.dyros_peer_alloc(C.c_size_t(4 * nfl), C.byref(ptr), handle), "dyros_peer_alloc")
            self._own = ptr.value
            handles = [None] * world
            dist.all_gather_object(handles, handle.raw)
            self.ptrs, self._opened = [], []
            for r in range(world):
                if r == rank:
                    self.ptrs.append(self._own)
                    continue
                p = C.c_void_p()
                native.check(self.lib.dyros_peer_open(handles[r], C.byref(p)), "dyros_peer_open")
                self._opened.append(p.value)
                self.ptrs.append(p.value)
            self.local = torch.as_tensor(_DevMem(self._own, nfl), device=device)   # this rank's block, for tests and tools
        self.epoch = torch.zeros(8, dtype=torch.int32, device=device)              # [epoch, pad, pad, pad | 4 scratch words]
        d = native.DyrosPpoPeers()
        d.world, d.rank, d.stride = world, rank, self.stride
        for r, base in enumerate(self.ptrs):
            d.grad[r][0], d.grad[r][1] = base, base + 4 * self.stride
            d.sum[r][0], d.sum[r][1] = base + 8 * self.stride, base + 12 * self.stride
            d.flags[r] = base + 16 * self.stride
            d.flags2[r] = base + 16 * self.stride + 32
            d.pnorm[r] = base + 16 * self.stride + 64
        d.epoch, d.ticket = self.epoch.data_ptr(), self.epoch.data_ptr() + 16
        self.desc = d
        torch.cuda.synchronize(device)
        dist.barrier()   # every rank has mapped every (zeroed) buffer before anybody publishes

    def close(self):
        """After a barrier of the caller's: unmaps the peers' blocks and frees this rank's."""
        for p in self._opened:
            self.lib.dyros_peer_close(C.c_void_p(p))
        self._opened = []
        if self._own:
            self.lib.dyros_peer_free(C.c_void_p(self._own))
            self._own = 0


class PPOTrainer:
    def __init__(self, env, cfg: Optional[PPOConfig] = None, rank: int = 0, world: int = 1):
        cfg = cfg or PPOConfig()
        if env.num_obs != cfg.num_obs:
            raise ValueError(f"PPOTrainer: the networks take PPOConfig.num_obs = {cfg.num_obs} observation columns; this env "
                             f"has {env.num_obs} (a height scan, terrain measure_heights, adds its heights to each row). "
                             f"Train it with PPOConfig(num_obs={env.num_obs})")
        if cfg.num_states and (not getattr(env, "critic_states", False) or env.num_states != cfg.num_states):
            has = getattr(env, "critic_states", False)
            raise ValueError(f"PPOTrainer: the critic takes PPOConfig.num_states = {cfg.num_states} state columns; this env "
                             + (f"has critic state rows of {env.num_states}. " if has else
                                "has no kernel-written critic states (set cfg['env']['criticStates']). ")
                             + "Train it with PPOConfig(num_states=env.num_states)")
        self.env, self.cfg = env, cfg
        self.rank, self.world = rank, world
        self.lib = native.load()
        c, dev = self.cfg, env.device
        N, H = env.num_envs, c.horizon_length
        self.N, self.H = N, H
        if (N * H) % c.minibatch_size:
            raise ValueError("num_envs * horizon_length must be a multiple of minibatch_size (A2C:192)")
        self.num_minibatches = N * H // c.minibatch_size
        self.net = FlatActorCritic(dev, c)
        if world > 1:  # hvd.setup_algo: rank 0's parameters everywhere (A2C:980-981)
            import torch.distributed as dist
            dist.broadcast(self.net.flat, 0)
        z = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt, device=dev)
        self.packed: Optional[PackedNets] = PackedNets(self.net, self.lib) if c.mixed_precision == "bf16" else None
        if c.grad_sync not in ("peer", "peer2", "nccl"):
            raise ValueError("grad_sync: 'peer', 'peer2' or 'nccl'")
        self.peers: Optional[PeerGrads] = (PeerGrads(self.net.n, dev, rank, world)
                                           if world > 1 and self.packed is not None and c.grad_sync in ("peer", "peer2") else None)
        if self.packed is not None:  # the rollout's observations are kept as the bf16 rows the GEMMs read (N*H x K0)
            self.x_step = z(N, self.packed.K0, dt=torch.bfloat16)  # (rows of the critic's width: both nets read them)
            self.x_roll = z(N * H, self.packed.K0, dt=torch.bfloat16)
        self.W = self.net.critic_inputs  # columns of a stored input row: the state row with an asymmetric critic
        self.buf = {"obs": z(N, H, self.W) if self.packed is None else z(1), "actions": z(N, H, NA), "mus": z(N, H, NA), "neglogp": z(N, H), "values": z(N, H),
                    "rewards": z(N, H), "dones": z(N, H), "advantages": z(N, H), "returns": z(N, H), "cur_reward": z(N),
                    "cur_length": z(N), "ep_stats": z(3), "step": z(1, dt=torch.int32), "global_step": z(1, dt=torch.int64)}
        pb = native.DyrosPpoBuffers()
        pb.N, pb.H, pb.gamma, pb.tau, pb.e_clip, pb.critic_coef = N, H, c.gamma, c.tau, c.e_clip, c.critic_coef
        pb.reward_scale, pb.value_bootstrap, pb.seed = c.reward_scale, int(c.value_bootstrap), c.seed + 7919 * (rank + 1)
        pb.obs_dim = self.W
        for k, t in self.buf.items():
            setattr(pb, k, t.data_ptr())
        self.pb = pb
        self.actions = z(N, NA)
        self.adv_norm = z(N, H)
        self.mb_dmu, self.mb_dv = z(c.minibatch_size, NA), z(c.minibatch_size)
        self.stats = z(4)
        self.norm2 = z(1)
        self.lr = torch.tensor([c.learning_rate, c.critic_learning_rate], device=dev)
        self.opt_step = z(1, dt=torch.int32)
        self.inject_normal: Optional[torch.Tensor] = None  # (H,N,13) test hook
        self.epoch = 0
        self._g_rollout: Optional[torch.cuda.CUDAGraph] = None
        self._g_update: Dict[int, torch.cuda.CUDAGraph] = {}
        self._static_out: Dict[int, tuple] = {}

    # ------------------------------------------------------------------ plumbing
    @property
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.env.device).cuda_stream)

    def _p(self, t):
        return C.c_void_p(t.data_ptr()) if t is not None else None

    # ------------------------------------------------------------------ rollout (A2C:629-703)
    @property
    def _input_rows(self) -> torch.Tensor:
        """What the networks read: the env's critic state rows with an asymmetric critic, else its observation rows."""
        return self.env.states_buf if self.cfg.num_states else self.env.obs_buf

    def _cast_obs(self, into_rollout: bool):
        native.check(self.lib.dyros_ppo_cast_obs(C.byref(self.pb), self._p(self._input_rows), self._p(self.x_step),
                                                 self._p(self.x_roll) if into_rollout else None, self._stream), "dyros_ppo_cast_obs")

    def _rollout_step_packed(self):
        env, pk = self.env, self.packed
        self._cast_obs(True)
        out = pk.forward(self.x_step)
        native.check(self.lib.dyros_ppo_act_packed(C.byref(self.pb), self._p(out), self._p(pk.bh), self._p(self.net.logstd),
                                                   self._p(env.reset_buf), self._p(self.actions), self._p(self.inject_normal),
                                                   self._stream), "dyros_ppo_act_packed")
        env.core.step(self.actions)
        native.check(self.lib.dyros_ppo_reward(C.byref(self.pb), self._p(env.rew_buf), self._p(env.timeout_buf),
                                               self._p(env.reset_buf), self._stream), "dyros_ppo_reward")

    def _rollout_step(self):
        if self.packed is not None:
            return self._rollout_step_packed()
        env = self.env
        with torch.no_grad():
            mu, v = self.net.forward(self._input_rows)
            mu, v = mu.float().contiguous(), v.float().contiguous()
        native.check(self.lib.dyros_ppo_act(C.byref(self.pb), self._p(mu), self._p(v), self._p(self.net.logstd), self._p(self._input_rows),
                                            self._p(env.reset_buf), self._p(self.actions), self._p(self.inject_normal),
                                            self._stream), "dyros_ppo_act")
        env.core.step(self.actions)  # VecTask.step: 3 launches, reads `actions` in place
        native.check(self.lib.dyros_ppo_reward(C.byref(self.pb), self._p(env.rew_buf), self._p(env.timeout_buf),
                                               self._p(env.reset_buf), self._stream), "dyros_ppo_reward")

    def rollout(self):
        """horizon_length env steps + GAE; everything stays on the device."""
        if self.cfg.use_cuda_graph and self._g_rollout is None:
            self._rollout_step()  # warm-up (cuBLAS workspaces, lazy init) outside the capture
            torch.cuda.synchronize()
            self.buf["step"].zero_()
            side = torch.cuda.Stream(device=self.env.device)
            side.wait_stream(torch.cuda.current_stream())
            g = torch.cuda.CUDAGraph()
            self._rollout_span = self.H if self.cfg.graph_span == "mini_epoch" else 1   # steps per replay
            with torch.cuda.graph(g, stream=side):
                for _ in range(self._rollout_span):
                    self._rollout_step()
            self._g_rollout = g
            self.buf["step"].zero_()  # (capturing executes nothing; the warm-up step is an extra, unrecorded env step)
        if self._g_rollout is not None:
            for _ in range(self.H // self._rollout_span):
                self._g_rollout.replay()
        else:
            for _ in range(self.H):
                self._rollout_step()
        with torch.no_grad():                                # get_values(self.obs), A2C:686
            if self.packed is not None:
                self._cast_obs(False)
                last_v = self.packed.mu_value(self.packed.forward(self.x_step))[1].contiguous()
            else:
                _, last_v = self.net.forward(self._input_rows)
                last_v = last_v.float().contiguous()
        native.check(self.lib.dyros_ppo_gae(C.byref(self.pb), self._p(last_v), self._p(self.env.reset_buf), self._stream), "dyros_ppo_gae")

    # ------------------------------------------------------------------ update (A2C:921-969, A2C:862-903, AG:108-227)
    def _prepare(self):
        adv = self.buf["advantages"]
        if self.cfg.normalize_advantage:  # A2C:943-944 (torch.std: unbiased)
            self.adv_norm.copy_((adv - adv.mean()) / (adv.std() + 1e-8))
        else:
            self.adv_norm.copy_(adv)

    def _optimiser_step(self):
        c, n = self.cfg, self.net
        if self.world > 1:  # optimizer.synchronize(): one all-reduce of the flat bucket (AG:161-173)
            import torch.distributed as dist
            dist.all_reduce(n.grad)
        native.check(self.lib.dyros_ppo_adam(self._p(n.flat), self._p(n.grad), self._p(n.exp_avg), self._p(n.exp_avg_sq), n.n_actor, n.n,
                                             1.0 / self.world, c.grad_norm if c.truncate_grads else 0.0, self._p(self.norm2),
                                             self._p(self.lr), self._p(self.opt_step), 0.9, 0.999, 1e-8, c.learning_rate,
                                             c.learning_rate_min, c.max_epochs if c.lr_schedule == "linear" else 0,
                                             self._stream), "dyros_ppo_adam")

    def _minibatch_packed(self, i: int):
        pk, mb = self.packed, self.cfg.minibatch_size
        r0 = i * mb
        x = self.x_roll[r0:r0 + mb]
        out = pk.forward(x)
        native.check(self.lib.dyros_ppo_loss_grad_packed(C.byref(self.pb), r0, mb, self._p(out), self._p(pk.bh), self._p(self.net.logstd),
                                                         self._p(self.adv_norm), self._p(pk._buffers(mb)["dout"]), self._p(pk.gbh),
                                                         self._p(self.stats), self._stream), "dyros_ppo_loss_grad_packed")
        pk.backward(x)
        c, n, single = self.cfg, self.net, self.world == 1
        clip = c.grad_norm if c.truncate_grads else 0.0
        norm_done = True
        if single:
            pk.unpack_grads(self.norm2 if clip > 0 else None)   # (the norm reduction rides along)
        elif self.peers is not None:  # optimizer.synchronize() (AG:161-173) over peer memory: publish, wait, sum in rank order
            native.check(self.lib.dyros_ppo_unpack_grads_peers_ac(C.byref(pk.desc), pk.critic_inputs, C.byref(self.peers.desc),
                                                                  self._stream), "unpack_peers")
            if c.grad_sync == "peer2":
                native.check(self.lib.dyros_ppo_reduce_scatter_peers(C.byref(self.peers.desc), self._p(n.grad), n.n, n.n_actor,
                                                                     self._stream), "reduce_scatter_peers")
                native.check(self.lib.dyros_ppo_all_gather_peers(C.byref(self.peers.desc), self._p(n.grad), n.n,
                                                                 self._p(self.norm2) if clip > 0 else None, self._stream), "all_gather_peers")
            else:
                native.check(self.lib.dyros_ppo_reduce_peers(C.byref(self.peers.desc), self._p(n.grad), n.n, n.n_actor,
                                                             self._p(self.norm2) if clip > 0 else None, self._stream), "reduce_peers")
        else:  # ... or as one NCCL all-reduce of the flat bucket
            import torch.distributed as dist
            pk.unpack_grads(None)
            dist.all_reduce(n.grad)
            norm_done = False
        native.check(self.lib.dyros_ppo_adam_packed_ac(C.byref(pk.desc), pk.critic_inputs, self._p(n.flat), self._p(n.grad), self._p(n.exp_avg),
                                                       self._p(n.exp_avg_sq), 1.0 / self.world, clip, int(norm_done), self._p(self.norm2),
                                                       self._p(self.lr), self._p(self.opt_step), 0.9, 0.999, 1e-8, c.learning_rate,
                                                       c.learning_rate_min, c.max_epochs if c.lr_schedule == "linear" else 0,
                                                       self._stream), "dyros_ppo_adam_packed")

    def _minibatch(self, i: int):
        if self.packed is not None:
            return self._minibatch_packed(i)
        c, mb = self.cfg, self.cfg.minibatch_size
        r0 = i * mb
        obs = self.buf["obs"].view(self.N * self.H, self.W)[r0:r0 + mb]
        mu, v = self.net.forward(obs)
        mu32, v32 = mu.float().contiguous(), v.float().contiguous()
        native.check(self.lib.dyros_ppo_loss_grad(C.byref(self.pb), r0, mb, self._p(mu32), self._p(v32), self._p(self.net.logstd),
                                                  self._p(self.adv_norm), self._p(self.mb_dmu), self._p(self.mb_dv),
                                                  self._p(self.stats), self._stream), "dyros_ppo_loss_grad")
        self.net.grad.zero_()
        torch.autograd.backward([mu, v], [self.mb_dmu.to(mu.dtype), self.mb_dv.to(v.dtype)])
        self._optimiser_step()
        # dataset.update_mu_sigma (A2C:884): later mini-epochs measure the KL against this pass
        self.buf["mus"].view(self.N * self.H, NA)[r0:r0 + mb].copy_(mu32.detach())

    def update(self):
        self._prepare()
        self.stats.zero_()
        whole = self.cfg.use_cuda_graph and self.cfg.graph_span == "mini_epoch"
        for _ in range(self.cfg.mini_epochs):
            for i in ([-1] if whole else range(self.num_minibatches)):
                if not self.cfg.use_cuda_graph:
                    self._minibatch(i)
                    continue
                g = self._g_update.get(i)
                if g is None:
                    if not self._g_update:  # one eager pass first (autograd / cuBLAS / NCCL lazy init), undone below
                        i0 = max(i, 0)
                        snap = [t.clone() for t in (self.net.flat, self.net.exp_avg, self.net.exp_avg_sq, self.opt_step, self.lr,
                                                    self.stats, self.buf["mus"])]
                        self._minibatch(i0)
                        torch.cuda.synchronize()
                        for t, s in zip((self.net.flat, self.net.exp_avg, self.net.exp_avg_sq, self.opt_step, self.lr, self.stats,
                                         self.buf["mus"]), snap):
                            t.copy_(s)
                        if self.packed is not None:
                            self.packed.pack()
                    side = torch.cuda.Stream(device=self.env.device)
                    side.wait_stream(torch.cuda.current_stream())
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=side):
                        for k in (range(self.num_minibatches) if whole else [i]):
                            self._minibatch(k)
                    self._g_update[i] = g
                g.replay()

    # ------------------------------------------------------------------ checkpoints (A2C:550-585, AG:97-103) and the
    # deployment weight dump of the play path (torch_runner_dyros.py:140-150)
    def state_dict(self) -> dict:
        n = self.net
        step = int(self.opt_step.item())
        return {"model": n.model_state_dict(), "epoch": self.epoch,
                "optimizer_actor": n.optimizer_state_dict(True, step, float(self.lr[0].item())),
                "optimizer_critic": n.optimizer_state_dict(False, step, float(self.lr[1].item())),
                "frame": self.epoch * self.N * self.H * self.world, "last_mean_rewards": -100500, "env_state": None}

    def load_state_dict(self, state: dict) -> None:
        n = self.net
        n.load_model_state_dict(state["model"])
        step = max(n.load_optimizer_state_dict(True, state["optimizer_actor"]), n.load_optimizer_state_dict(False, state["optimizer_critic"]))
        self.opt_step.fill_(step)
        self.lr[0] = float(state["optimizer_actor"]["param_groups"][0]["lr"])
        self.lr[1] = float(state["optimizer_critic"]["param_groups"][0]["lr"])
        self.epoch = int(state.get("epoch", 0))
        if self.packed is not None:
            self.packed.pack()

    def save(self, fn: str) -> str:
        """agent.save(fn) (AG:97-99): rl_games' torch_ext.save_checkpoint appends '.pth'."""
        path = fn + ".pth"
        torch.save(self.state_dict(), path)
        return path

    def restore(self, fn: str) -> None:
        self.load_state_dict(torch.load(fn if fn.endswith(".pth") else fn + ".pth", map_location="cpu", weights_only=False))

    def dump_weights_txt(self, out_dir: str = "./result") -> list:
        """torch_runner_dyros.py:143-147: one np.savetxt file per entry of model.state_dict(), dots replaced by underscores
        (what the robot-side controller reads)."""
        import os
        import numpy as np
        os.makedirs(out_dir, exist_ok=True)
        files = []
        for name, param in self.net.model_state_dict().items():
            path = os.path.join(out_dir, name.replace(".", "_") + ".txt")
            np.savetxt(path, param.numpy())
            files.append(path)
        return files

    def train_epoch(self) -> Dict[str, float]:
        """One epoch of ContinuousA2CBase.train (A2C:983-1008): noise schedule, rollout, update. One device->host read.
        With a terrain curriculum, "terrain_level" is the envs' mean level at the end of the rollout (legged_gym's
        episode log), averaged over ranks."""
        c = self.cfg
        self.epoch += 1
        self.net.update_action_noise((c.max_epochs - self.epoch) / c.max_epochs)  # A2C:985
        self.buf["ep_stats"].zero_()
        self.rollout()
        self.update()
        k = c.mini_epochs * self.num_minibatches
        level = getattr(self.env, "terrain_level_mean", None)
        out = torch.cat([self.stats / k, self.buf["ep_stats"], self.lr[:1]] + ([level.reshape(1)] if level is not None else []))
        if self.world > 1:
            import torch.distributed as dist
            s = out.clone()
            dist.all_reduce(s)
            out = s / self.world
            out[4:7] = s[4:7]
        a_loss, c_loss, kl, clip_frac, ep_r, ep_l, ep_n, lr, *rest = out.tolist()
        res = {"a_loss": a_loss, "c_loss": c_loss, "kl": kl, "clip_frac": clip_frac, "lr": lr,
               "mean_reward": ep_r / max(ep_n, 1.0), "mean_length": ep_l / max(ep_n, 1.0), "episodes": ep_n,
               "frames": self.N * self.H * self.world}
        if rest:
            res["terrain_level"] = rest[0]
        return res
