"""DyrosDynamicWalk with the reference's VecTask API, running on the sm_100a kernels.

Mirrors python/IsaacGymEnvs/isaacgymenvs/tasks/dyros_dynamic_walk.py (T) and tasks/base/vec_task.py (VT):
same constructor signature, `step` / `reset` / `reset_idx` / `reset_done` / `zero_actions`, the properties rl_games
reads (VT:129-152, utils/rlgames_utils.py:157-186) and the same `extras` keys ("time_outs", "stacked_rewards",
"reward_names"; T:415-428, VT:336). One `step` is one CUDA-graph replay of dyros_task_step; nothing in it
synchronises the host.
"""
from __future__ import annotations

from typing import Any, Dict, Optional

import numpy as np
import torch

from .. import terrain as terrain_gen
from ..core import NOBS, NPRIV, CoreConfig, DyrosCore, HeightField, TerrainCurriculum
from ..native import DyrosError
from .spaces import Box

REWARD_NAMES = ["mimic_body_orientation_reward", "qpos_regulation", "qvel_regulation", "contact_force_penalty",
                "torque_regulation", "torque_diff_regulation", "body_vel_reward", "qacc_regulation",
                "foot_contact_reward", "contact_force_diff_regulation", "double_support_force_diff_regulation",
                "force_thres_penalty", "force_diff_thres_penalty", "force_ref_reward", "perturbation"]  # T:922-925, T:423


def default_cfg(num_envs: int = 4096, randomize: bool = True, perturbation: bool = True,
                friction_range=None, pd_gain_range=None) -> Dict[str, Any]:
    """The values of cfg/task/DyrosDynamicWalk.yaml (+ cfg/config.yaml defaults) as the plain dict VecTask receives.
    `friction_range` / `pd_gain_range` switch on the optional randomisations of BASELINE configs[3] (friction as in the
    yaml's commented-out block, CFG:89-96: [0.7, 1.3] scaling)."""
    cfg = _default_cfg(num_envs, randomize, perturbation)
    hum = cfg["task"]["randomization_params"]["actor_params"]["humanoid"]
    if friction_range is not None:
        hum["rigid_shape_properties"] = {"friction": {"range": list(friction_range), "operation": "scaling", "distribution": "uniform"}}
    if pd_gain_range is not None:
        hum["pd_gains"] = {"range": list(pd_gain_range), "operation": "scaling", "distribution": "uniform"}
    return cfg


def _default_cfg(num_envs: int, randomize: bool, perturbation: bool) -> Dict[str, Any]:
    return {
        "name": "DyrosDynamicWalk", "physics_engine": "physx",
        "env": {"numEnvs": num_envs, "envSpacing": 5, "episodeLength": 32, "enableDebugVis": False,
                "controlFrequencyInv": 2, "clipActions": 1.0, "NumSingleStepObs": 37, "NumAction": 13,
                "perturbation": perturbation, "NumHis": 10, "NumSkip": 2, "initialHieght": 0.93, "deathCost": 0.0,
                "terminationHeight": 0.6, "asset": {"assetFileName": "mjcf/dyros_tocabi/xml/dyros_tocabi.xml"}},
        "sim": {"dt": 0.002, "substeps": 1, "up_axis": "z", "use_gpu_pipeline": True, "gravity": [0.0, 0.0, -9.81],
                "physx": {"num_threads": 4, "solver_type": 1, "use_gpu": True, "num_position_iterations": 4,
                          "num_velocity_iterations": 1, "contact_offset": 0.002, "rest_offset": 0.0,
                          "bounce_threshold_velocity": 0.04, "max_depenetration_velocity": 10.0,
                          "contact_collection": 1}},
        "task": {"randomize": randomize, "randomization_params": {
            "frequency": 1, "actor_params": {"humanoid": {
                "rigid_body_properties": {"mass": {"range": [0.8, 1.2], "operation": "scaling",
                                                   "distribution": "uniform", "setup_only": True}},
                "dof_properties": {"damping": {"range": [0.0, 2.9], "operation": "additive", "distribution": "uniform"},
                                   "armature": {"range": [0.8, 1.2], "operation": "scaling", "distribution": "uniform"}}}}}},
    }


def height_scan_points(cfg: Dict[str, Any]) -> Optional[np.ndarray]:
    """(P, 2) points of the height scan that cfg["env"]["terrain"] asks for (measure_heights), or None."""
    tr = cfg["env"].get("terrain")
    return None if tr is None else terrain_gen.height_points(terrain_gen.TerrainConfig.from_dict(tr))


def critic_states(cfg: Dict[str, Any]) -> Optional[bool]:
    """cfg["env"]["criticStates"] (ours, not a key of the reference's yaml; DESIGN.md section 4, "Critic states"):
    None = off (absent or False); otherwise whether the heights of a height scan go into the observation row as well
    (True: `{"heights_in_obs": True}`; False: `True`, the heights go into the state row only)."""
    v = cfg["env"].get("criticStates", False)
    if v is False or v is None:
        return None
    if v is True:
        return False
    if isinstance(v, dict) and set(v) <= {"heights_in_obs"} and isinstance(v.get("heights_in_obs", False), bool):
        hio = bool(v.get("heights_in_obs", False))
        if hio and height_scan_points(cfg) is None:
            raise ValueError('cfg["env"]["criticStates"]: heights_in_obs needs a height scan (terrain measure_heights)')
        return hio
    raise ValueError(f'cfg["env"]["criticStates"]: False, True or {{"heights_in_obs": bool}} (got {v!r})')


def num_observations(cfg: Dict[str, Any]) -> int:
    """Columns of an observation row: the reference's 487 (T:36-44), plus P heights with measure_heights (unless
    critic states take the heights alone)."""
    p = height_scan_points(cfg)
    cs = critic_states(cfg)
    return NOBS + (0 if p is None or cs is False else len(p))


def num_states(cfg: Dict[str, Any]) -> int:
    """Columns of a critic state row: 487 + P + 31 with criticStates, else cfg["env"]["numStates"] (default 0)."""
    if critic_states(cfg) is None:
        return cfg["env"].get("numStates", 0)
    p = height_scan_points(cfg)
    return NOBS + (0 if p is None else len(p)) + NPRIV


def core_config_from_cfg(cfg: Dict[str, Any], generator: Optional[torch.Generator] = None) -> CoreConfig:
    """`generator` draws the envs' initial terrain levels when cfg["env"]["terrain"] is set (default: a CPU generator
    seeded with 0)."""
    env, sim, task = cfg["env"], cfg["sim"], cfg.get("task", {})
    px = sim.get("physx", {})
    c = CoreConfig(dt=sim["dt"], substeps=sim.get("substeps", 1), control_freq_inv=env.get("controlFrequencyInv", 1),
                   episode_length_s=env["episodeLength"], gravity=tuple(sim.get("gravity", (0, 0, -9.81))),
                   contact_offset=px.get("contact_offset", 0.002),
                   max_depenetration_velocity=px.get("max_depenetration_velocity", 10.0),
                   num_position_iterations=px.get("num_position_iterations", 4),
                   num_velocity_iterations=px.get("num_velocity_iterations", 1),
                   death_cost=env.get("deathCost", 0.0), initial_height=env.get("initialHieght", 0.93),
                   env_spacing=env.get("envSpacing", 5), perturb=env.get("perturbation", False),
                   randomize=task.get("randomize", False),
                   # (not a key of the reference's yaml: the reference always creates the actor with collision filter 0,
                   # T:354; `selfCollision: False` drops the self-collision pass, e.g. to time the step without it)
                   self_collision=env.get("selfCollision", True),
                   physics_program=env.get("physicsProgram", "roles"))  # (ours too: DESIGN.md section 4, "Two programs")
    # (not a key of the reference's yaml either: the reference's terrain code, T:203-270, builds the field and calls
    # gym.add_heightfield; here the field comes with the cfg. DESIGN.md section 4, "Ground")
    hf = env.get("heightfield")
    if hf is not None:
        c.heightfield = HeightField(np.asarray(hf["samples"]), float(hf["row_scale"]), float(hf["column_scale"]),
                                    float(hf["vertical_scale"]), tuple(hf.get("origin", (0.0, 0.0, 0.0))),
                                    friction=hf.get("friction"), env_origins=hf.get("env_origins"))
    # (not a key of the reference's yaml either: its TerrainCfg, terrain_cfg.py:2-21, switched on. DESIGN.md section 4,
    # "Curriculum")
    tr = env.get("terrain")
    if tr is not None:
        tcfg = terrain_gen.TerrainConfig.from_dict(tr)
        if tcfg.mesh_type in ("plane", "none"):
            pass  # the plane z = 0, as without the key
        elif hf is not None:
            raise DyrosError('cfg["env"]: give either "heightfield" or "terrain", not both')
        else:
            _terrain_config(c, tcfg, int(env["numEnvs"]), generator)
        c.height_scan = terrain_gen.height_points(tcfg)  # (any ground, the plane too)
    cs = critic_states(cfg)
    if cs is not None:
        c.critic_states, c.critic_heights_in_obs = True, cs
    ap = task.get("randomization_params", {}).get("actor_params", {}).get("humanoid", {})
    dp = ap.get("dof_properties", {})
    if "damping" in dp:
        c.dr_damping_range = tuple(dp["damping"]["range"])
    if "armature" in dp:
        c.dr_armature_range = tuple(dp["armature"]["range"])
    rb = ap.get("rigid_body_properties", {})
    if "mass" in rb:
        c.dr_mass_range = tuple(rb["mass"]["range"])
    # optional (commented out in the reference's yaml, CFG:89-96; named by BASELINE configs[3]): per-env friction of the
    # ground contacts and per-env scales of the upper-body PD gains, re-drawn on reset like damping / armature
    fr = ap.get("rigid_shape_properties", {}).get("friction")
    if fr is not None:
        c.dr_friction_range = tuple(fr["range"])
    pg = ap.get("pd_gains")
    if pg is not None:
        c.dr_pd_gain_range = tuple(pg["range"])
    return c


def _terrain_config(c: CoreConfig, tcfg: "terrain_gen.TerrainConfig", n: int, generator: Optional[torch.Generator]):
    """The generated field and the envs' sub-terrains (legged_gym's _get_env_origins): env e gets type
    floor(e / (N / num_cols)) and a random initial level, in [0, max_init_terrain_level] with the curriculum, in
    [0, num_rows) without."""
    field, origins = terrain_gen.generate(tcfg)
    g = generator if generator is not None else torch.Generator().manual_seed(0)
    top = min(tcfg.max_init_terrain_level, tcfg.num_rows - 1) if tcfg.curriculum else tcfg.num_rows - 1
    levels = torch.randint(0, top + 1, (n,), device=g.device, generator=g).cpu().numpy().astype(np.int32)
    types = np.floor(np.arange(n) / (n / tcfg.num_cols)).astype(np.int32)
    c.heightfield = field
    c.terrain_curriculum = TerrainCurriculum(origins, types, levels, move_up_distance=tcfg.terrain_length / 2,
                                             move_down_scale=c.episode_length_s * 0.5, curriculum=tcfg.curriculum)


class DyrosDynamicWalk:
    def __init__(self, cfg: Dict[str, Any], sim_device: str = "cuda:0", graphics_device_id: int = -1,
                 headless: bool = True, seed: int = 42, rank: int = 0, use_cuda_graph: bool = True):
        self.cfg = cfg
        env = cfg["env"]
        # T:36-44
        self.num_single_step_obs, self.num_action = env["NumSingleStepObs"], env["NumAction"]
        self.num_obs_his, self.num_obs_skip = env["NumHis"], env["NumSkip"]
        env["numObservations"] = (self.num_single_step_obs + self.num_action) * (self.num_obs_his - 1) + self.num_single_step_obs
        env["numActions"] = self.num_action
        if (self.num_single_step_obs, self.num_action, self.num_obs_his, self.num_obs_skip) != (37, 13, 10, 2):
            raise ValueError("the fused observation kernel is specialised to 37/13/10/2 (DyrosDynamicWalk.yaml:15-20)")
        env["numObservations"] = num_observations(cfg)  # + the measured heights (legged_gym's measure_heights)
        self.critic_states = critic_states(cfg) is not None  # kernel-written privileged rows in states_buf
        if self.critic_states:
            ns = num_states(cfg)
            if "numStates" in env and env["numStates"] != ns:
                raise ValueError(f'cfg["env"]["numStates"] = {env["numStates"]}, but criticStates makes the state rows {ns} '
                                 "wide (487 + the heights of a height scan + 31 privileged columns)")
            env["numStates"] = ns
        # VT:50-97 (Env.__init__)
        dev = sim_device.split(":")
        if dev[0].lower() not in ("cuda", "gpu"):
            raise ValueError("sim_device must be a CUDA device: this implementation has no CPU pipeline")
        self.device_type, self.device_id = "cuda", int(dev[1]) if len(dev) > 1 else 0
        self.device = f"cuda:{self.device_id}"
        self.rl_device = cfg.get("rl_device", self.device)
        self.headless, self.graphics_device_id = headless, graphics_device_id
        self.num_environments = env["numEnvs"]
        self.num_agents = env.get("numAgents", 1)
        self.num_observations, self.num_states, self.num_actions = env["numObservations"], env.get("numStates", 0), env["numActions"]
        self.control_freq_inv = env.get("controlFrequencyInv", 1)
        self.obs_space = Box(np.ones(self.num_obs) * -np.inf, np.ones(self.num_obs) * np.inf)
        self.state_space = Box(np.ones(self.num_states) * -np.inf, np.ones(self.num_states) * np.inf)
        self.act_space = Box(np.ones(self.num_actions) * -1., np.ones(self.num_actions) * 1.)
        self.clip_obs = env.get("clipObservations", np.inf)
        self.clip_actions = env.get("clipActions", np.inf)
        if self.clip_actions != 1.0:
            raise ValueError("clipActions is fixed to 1.0 in the prologue kernel (DyrosDynamicWalk.yaml:13)")
        self.randomize = cfg.get("task", {}).get("randomize", False)
        self.randomization_params = cfg.get("task", {}).get("randomization_params", {})
        self.max_episode_length_s = env["episodeLength"]
        self.death_cost, self.initial_height = env["deathCost"], env["initialHieght"]
        self.perturb = env["perturbation"]
        self.gen = torch.Generator(device=self.device)
        self.gen.manual_seed(seed + rank)
        self.core_cfg = core_config_from_cfg(cfg, self.gen)  # (draws the initial terrain levels, if any, from self.gen)
        self.dt, self.skipframe = self.core_cfg.dt, self.control_freq_inv
        self.dt_policy = self.dt * self.skipframe
        self.max_episode_length = self.max_episode_length_s / (self.dt * self.skipframe)  # T:35
        self.core = DyrosCore(self.num_environments, self.device, self.core_cfg, seed=seed, rank=rank)
        assert self.core.obs_width == self.num_observations
        assert self.core.states_width == (self.num_states if self.critic_states else 0)
        self.num_height_points = self.core.num_height_points
        self._bind_buffers()
        self._initial_randoms()
        self.extras: Dict[str, Any] = {}
        self.obs_dict: Dict[str, torch.Tensor] = {}
        self._actions_static = torch.zeros(self.num_envs, self.num_actions, device=self.device)
        self._graph: Optional[torch.cuda.CUDAGraph] = None
        self._use_graph = use_cuda_graph
        self._pipe: Optional["_HostPipe"] = None
        self._inplace_graphs: Dict[int, torch.cuda.CUDAGraph] = {}
        self._seen_action_ptrs: set = set()
        self.first_randomization = True

    # ------------------------------------------------------------------ VT:129-152
    @property
    def observation_space(self):
        return self.obs_space

    @property
    def action_space(self):
        return self.act_space

    @property
    def num_envs(self) -> int:
        return self.num_environments

    @property
    def num_acts(self) -> int:
        return self.num_actions

    @property
    def num_obs(self) -> int:
        return self.num_observations

    # ------------------------------------------------------------------ buffers (VT:233-256, T:87-195)
    def _bind_buffers(self):
        t, s, N = self.core.task_t, self.core.sim_t, self.num_envs
        self.obs_buf, self.rew_buf, self.reset_buf = t["obs_buf"], t["rew_buf"], t["reset_buf"]
        self.timeout_buf, self.progress_buf, self.randomize_buf = t["timeout_buf"], t["progress_buf"], t["randomize_buf"]
        # critic states (criticStates): the kernels' privileged rows (DESIGN.md section 4); else VecTask's zero buffer
        self.states_buf = t["states_buf"] if self.critic_states else torch.zeros(N, self.num_states, device=self.device)
        self.root_states = s["root_states"]
        self.dof_state = s["dof_state"]
        self.dof_pos = s["dof_state"].view(N, 33, 2)[..., 0]
        self.dof_vel = s["dof_state"].view(N, 33, 2)[..., 1]
        self.contact_forces = s["net_contact_force"].view(N, 38, 3)
        self.stacked_rewards = t["stacked_rewards"]
        # terrain (cfg["env"]["terrain"]): level (row) and type (column) of each env's sub-terrain, the sub-terrain
        # origins; with the curriculum the reset stage updates terrain_levels and terrain_level_mean
        self.terrain_levels, self.terrain_types = t.get("terrain_levels"), t.get("terrain_types")
        self.terrain_origins, self.terrain_level_mean = t.get("terrain_origins"), t.get("terrain_level_mean")
        # height scan (terrain measure_heights): (N, P) terrain heights in m under the points of height_points, of the
        # root the observation describes (obs_buf columns 487.. hold them scaled); None without the scan
        self.measured_heights, self.height_points = t.get("measured_heights"), t.get("height_points")
        for k in ("actions", "actions_pre", "time", "target_vel", "motor_constant_scale", "qpos_noise", "qvel_noise",
                  "qpos_bias", "quat_bias", "epi_len", "epi_len_log", "contact_reward_mean", "total_mass"):
            setattr(self, k, t[k])

    def _initial_randoms(self):
        """Per-env draws the reference makes in __init__ (T:129-153, T:175) and the creation pose of episode 0:
        env origin + U(-1,1) m in x, y (T:350-353, SURVEY A7)."""
        t, s, N, g, dev = self.core.task_t, self.core.sim_t, self.num_envs, self.gen, self.device
        r = lambda *shape: torch.rand(*shape, device=dev, generator=g)
        t["target_vel"][:, 0] = r(N) * 0.8
        t["motor_constant_scale"].copy_(r(N, 12) * 0.4 + 0.8)
        t["qpos_bias"].copy_(r(N, 12) * 6.28 / 100 - 3.14 / 100)
        t["quat_bias"].copy_(r(N, 3) * 6.28 / 150 - 3.14 / 150)
        t["pert_duration"].copy_(torch.randint(1, 100, (N,), device=dev, generator=g, dtype=torch.int32))
        s["root_states"][:, 0:2] = t["env_origins"][:, 0:2] + (r(N, 2) * 2 - 1)
        if self.randomize:  # first_randomization: every env (VT:536-538); mass is setup_only (CFG:81-88)
            c = self.core_cfg
            lo, hi = c.dr_mass_range
            s["body_mass_scale"].copy_(lo + r(N, 38) * (hi - lo))
            lo, hi = c.dr_damping_range
            s["dof_damping"].copy_(c.dof_damping + lo + r(N, 33) * (hi - lo))
            lo, hi = c.dr_armature_range
            s["dof_armature"].mul_(lo + r(N, 33) * (hi - lo))
            if "contact_friction" in s:
                lo, hi = c.dr_friction_range
                s["contact_friction"].copy_(c.friction * (lo + r(N) * (hi - lo)))
            if "pd_gain_scale" in t:
                lo, hi = c.dr_pd_gain_range
                t["pd_gain_scale"].copy_(lo + r(N, 2) * (hi - lo))
            masses = torch.tensor(self.core.tables.body_inertia[:, 0], dtype=torch.float32, device=dev)
            t["total_mass"].copy_((s["body_mass_scale"] * masses).sum(1))  # T:221-225

    # ------------------------------------------------------------------ step / reset (VT:293-374)
    def step(self, actions: torch.Tensor):
        """VT:293-344: returns (obs_dict, rew_buf, reset_buf, extras); tensors are the env's own buffers."""
        if actions.device.type == "cpu" and actions.is_pinned() and actions.dtype == torch.float32 and actions.is_contiguous():
            # host-side policy: the first kernel reads the actions straight from the pinned buffer (no staging copy, no
            # graph: the pointer differs per call); the caller keeps the tensor alive and unchanged until the step has
            # run, as with every tensor handed to the reference's gym setters (DOCT:348-369)
            self.core.step(actions)
        elif self._use_graph:
            g = self._graph_reading(actions)
            if g is not None:
                g.replay()  # the step's first kernel reads the caller's tensor in place
            else:
                self._actions_static.copy_(actions, non_blocking=True)
                if self._graph is None:
                    self._capture()
                self._graph.replay()
        else:
            self._actions_static.copy_(actions, non_blocking=True)
            self.core.step(self._actions_static)
        self.extras["time_outs"] = self.timeout_buf.to(self.rl_device)
        self.extras["stacked_rewards"] = self.stacked_rewards
        self.extras["reward_names"] = REWARD_NAMES
        if self.terrain_level_mean is not None:  # legged_gym's episode log; written by the step's kernels
            self.extras.setdefault("episode", {})["terrain_level"] = self.terrain_level_mean
        self.obs_dict["obs"] = self._obs_out()
        if self.critic_states:  # VT:340-341 (num_states > 0)
            self.obs_dict["states"] = self.get_state()
        return self.obs_dict, self.rew_buf.to(self.rl_device), self.reset_buf.to(self.rl_device), self.extras

    def _obs_out(self) -> torch.Tensor:
        """VT:338 `torch.clamp(obs_buf, -clip_obs, clip_obs).to(rl_device)`. With a finite clipObservations that is a
        fresh clamped tensor, as in the reference. With the yaml's default (no clipObservations: inf, VT:97-98) the clamp
        is the identity and the env's own buffer is returned WITHOUT the copy the reference makes (8 MB per step at 4096
        envs): the next `step` overwrites it, so a caller that keeps observations across steps must clone them (rl_games
        copies them into its rollout buffer, a2c_common_dyros.py:641)."""
        if np.isfinite(self.clip_obs):
            return torch.clamp(self.obs_buf, -self.clip_obs, self.clip_obs).to(self.rl_device)
        return self.obs_buf.to(self.rl_device)

    # ------------------------------------------------------------------ host-facing pipelined step
    def step_async(self, actions: torch.Tensor) -> int:
        """`step` for a caller whose buffers live in HOST memory, split as in gym's VecEnv.step_async / step_wait.

        Enqueues VT:293-344 for `actions` (pinned host or device tensor), gathers what `step` returns
        (obs_dict["obs"], rew_buf, reset_buf, extras["time_outs"]: VT:336-344) into one device block (dyros_task_pack_results) and hands that
        block to the copy engine on a second stream as ONE device->host transfer into pinned memory. Returns a ticket
        for `step_wait`. Up to cfg["async_depth"] (default 3) tickets may be in flight: the transfer of step k overlaps the kernels of step k+1, so a
        rollout whose actions do not wait for the newest observation runs at max(kernels, PCIe) instead of their sum.
        `self.obs_buf` is not updated by these steps (the observation kernel writes the ticket's block directly); rew_buf,
        reset_buf and the state tensors are. The only host wait is for the slot of step k-async_depth to be free again."""
        if self.critic_states:
            raise RuntimeError("step_async: the host pipeline carries obs / rew / reset / time_outs only, no critic states; "
                               "use step() on an env with criticStates")
        if self._pipe is None:
            self._pipe = _HostPipe(self)
        return self._pipe.submit(actions)

    def step_wait(self, ticket: int):
        """Blocks until the results of `ticket` are in host memory; returns (obs_dict, rew, reset, extras) as pinned
        host tensors, valid until async_depth further `step_async` calls have been made."""
        if self._pipe is None:
            raise RuntimeError("step_wait without step_async")
        return self._pipe.wait(ticket)

    _MAX_INPLACE_GRAPHS = 32

    def _graph_reading(self, actions: torch.Tensor) -> Optional[torch.cuda.CUDAGraph]:
        """A rollout loop hands `step` the same few action tensors over and over (the policy's output buffer): for a
        contiguous float32 (N,13) tensor on the env's device, one CUDA graph per storage address whose first kernel
        reads that address directly, so the step needs no staging copy (a launch and ~5 us). The graph is captured the
        second time an address is seen; any other tensor, or more than _MAX_INPLACE_GRAPHS distinct addresses, goes
        through the staging buffer."""
        if (not actions.is_cuda or actions.dtype != torch.float32 or not actions.is_contiguous()
                or tuple(actions.shape) != (self.num_envs, self.num_actions) or actions.device != self.core.device):
            return None
        key = actions.data_ptr()
        g = self._inplace_graphs.get(key)
        if g is None and key not in self._seen_action_ptrs:
            if len(self._seen_action_ptrs) < 4 * self._MAX_INPLACE_GRAPHS:
                self._seen_action_ptrs.add(key)
            return None
        if g is None and len(self._inplace_graphs) < self._MAX_INPLACE_GRAPHS:
            torch.cuda.synchronize()
            side = self._capture_stream()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                self.core.step(actions)
            self._inplace_graphs[key] = g
        return g

    def _capture(self):
        torch.cuda.synchronize()
        side = self._capture_stream()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            self.core.step(self._actions_static)
        self._graph = g

    def _capture_stream(self) -> "torch.cuda.Stream":
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        if self.core.l2_persist:  # kernel nodes inherit the stream's access-policy window at capture
            self.core.set_l2_persistence(True, side)
        return side

    def set_l2_persistence(self, on: bool = True) -> int:
        """Keep the env state in the persisting part of the 126 MB L2 (dyros_sim_set_l2_persistence): the step then runs
        at its back-to-back speed even when other kernels (the policy network) stream through L2 between two steps.
        Drops the CUDA graphs captured so far (their kernel nodes carry the previous setting). Returns the bytes set aside."""
        n = self.core.set_l2_persistence(on)
        self._graph, self._inplace_graphs, self._pipe = None, {}, None
        return n

    def zero_actions(self) -> torch.Tensor:
        return torch.zeros(self.num_envs, self.num_actions, dtype=torch.float32, device=self.rl_device)

    def reset(self) -> Dict[str, torch.Tensor]:
        """VT:362-374: returns the observation buffer as is (zeros before the first step); resets nothing."""
        self.obs_dict["obs"] = self._obs_out()
        if self.critic_states:
            self.obs_dict["states"] = self.get_state()
        return self.obs_dict

    def reset_done(self):
        """VT:376-391."""
        done = self.reset_buf.nonzero(as_tuple=False).squeeze(-1)
        if len(done) > 0:
            self.reset_idx(done)
        self.obs_dict["obs"] = self._obs_out()
        if self.critic_states:
            self.obs_dict["states"] = self.get_state()
        return self.obs_dict, done

    def reset_idx(self, env_ids: torch.Tensor):
        """T:598-669 for an explicit id list (the per-step path resets inside the fused kernel)."""
        self.core.reset_idx(env_ids.to(device=self.device, dtype=torch.int64).contiguous())

    def get_state(self):
        return self.states_buf.to(self.rl_device)

    # staged methods with the reference's names (T:449, T:543, T:581, T:387, T:430)
    def pre_physics_step(self, actions: torch.Tensor):
        c = self.core
        c.prologue(actions.contiguous())
        for k in range(self.skipframe):
            c.substep_torque()
            native_push = k == 0
            self._simulate_with_push(native_push)
            c.sensor_noise(k)

    def _simulate_with_push(self, first: bool):
        import ctypes as C
        from .. import native
        c = self.core
        if first and "rb_force" in c.sim_t:
            c.sim_t["rb_force"].zero_()
            c.sim_t["rb_torque"].zero_()
            c.sim_t["rb_force"].view(self.num_envs, 38, 3)[:, 0, :] = c.task_t["push_force"]
            c.simulate(apply_wrench=True)
        elif first:
            raise native.DyrosError("staged pre_physics_step needs CoreConfig.with_rb_force_tensors (apply_rigid_body_force_tensors path)")
        else:
            c.simulate()

    def post_physics_step(self):
        c = self.core
        c.epilogue()
        c.check_termination()
        c.compute_reward()
        c.compact_resets()
        c.reset_idx(None)
        c.compute_observations()
        c.late_update()
        c.end_step()

    def check_termination(self):
        self.core.check_termination()

    def compute_reward(self):
        self.core.compute_reward()

    def compute_observations(self):
        self.core.compute_observations()

    def close(self):
        self._graph = None
        self._pipe = None
        self._inplace_graphs = {}
        self.core.close()


class _HostPipe:
    """Behind step_async / step_wait: per slot a pinned host action buffer, a device result block, a pinned host result
    block and ONE CUDA graph (dyros_task_step reading the slot's action buffer + dyros_task_pack_results into the slot's
    block); a copy stream carries the device->host transfers. Launching the step's kernels one by one from Python costs
    more host time (~180 us) than the kernels run (~105 us), hence the graphs."""
    DEPTH = 3

    def __init__(self, env: DyrosDynamicWalk):
        self.env, N = env, env.num_envs
        self.DEPTH = int(env.cfg.get("async_depth", self.DEPTH))
        if self.DEPTH < 1:
            raise ValueError("async_depth must be at least 1")
        nbytes = env.core.result_bytes()
        self.copy_stream = torch.cuda.Stream(device=env.device)
        self.h_actions = [torch.zeros(N, env.num_actions).pin_memory() for _ in range(self.DEPTH)]
        self.dev = [torch.empty(nbytes, dtype=torch.uint8, device=env.device) for _ in range(self.DEPTH)]
        self.host = [torch.empty(nbytes, dtype=torch.uint8).pin_memory() for _ in range(self.DEPTH)]
        self.packed = [torch.cuda.Event() for _ in range(self.DEPTH)]
        self.landed = [torch.cuda.Event() for _ in range(self.DEPTH)]
        o, r, t, end = env.core.result_offsets()
        W = env.core.obs_width
        self.views = [({"obs": h[:o].view(torch.float32).view(N, W)}, h[o:o + N * 4].view(torch.float32),
                       h[r:t].view(torch.int64), h[t:end].view(torch.int64)) for h in self.host]
        self.graphs: Dict[Any, torch.cuda.CUDAGraph] = {}
        self.count = 0

    def _run(self, slot: int, src: torch.Tensor, kind: str):
        env = self.env

        def launches():
            # the observation kernel writes the slot's block itself (no copy of the 8 MB by another kernel, which would
            # cost the next step's first kernel its L2-resident state); env.obs_buf is not updated by these steps
            env.core.set_obs_buf(self.dev[slot])
            try:
                env.core.step(src)
                env.core.pack_results(self.dev[slot])
            finally:
                env.core.set_obs_buf(env.obs_buf)

        if not env._use_graph:
            launches()
            return
        g = self.graphs.get((slot, kind))
        if g is None:
            torch.cuda.synchronize(env.device)
            side = env._capture_stream()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                launches()
            self.graphs[(slot, kind)] = g
        g.replay()

    def submit(self, actions: torch.Tensor) -> int:
        env, k = self.env, self.count
        slot = k % self.DEPTH
        cur = torch.cuda.current_stream(env.device)
        if k >= self.DEPTH:
            # step k-DEPTH used this slot: its kernels have read h_actions[slot] and its block has left the device
            self.landed[slot].synchronize()
        if actions.device.type == "cpu":
            self.h_actions[slot].copy_(actions)  # host memcpy (213 KB at N = 4096); the step's first kernel reads it over PCIe
            self._run(slot, self.h_actions[slot], "host")
        else:
            env._actions_static.copy_(actions, non_blocking=True)
            self._run(slot, env._actions_static, "dev")
        self.packed[slot].record(cur)
        self.copy_stream.wait_event(self.packed[slot])
        with torch.cuda.stream(self.copy_stream):
            self.host[slot].copy_(self.dev[slot], non_blocking=True)
            self.landed[slot].record(self.copy_stream)
        self.count = k + 1
        return k

    def wait(self, ticket: int):
        if not (self.count - self.DEPTH <= ticket < self.count) or ticket < 0:
            raise RuntimeError(f"ticket {ticket} is not in flight (tickets {max(0, self.count - self.DEPTH)}..{self.count - 1} are)")
        slot = ticket % self.DEPTH
        self.landed[slot].synchronize()
        obs, rew, rst, tmo = self.views[slot]
        return obs, rew, rst, {"time_outs": tmo, "reward_names": REWARD_NAMES}
