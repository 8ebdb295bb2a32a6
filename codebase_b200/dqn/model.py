"""IDQN / VDN learners on the B200 path -- drop-in for marlbase/dqn/model.py (QNetwork 14-196, VDNetwork 199-269).

Same constructor signature and Hydra `_target_` role (configs/algorithm/idqn.yaml:6-14, vdn.yaml:11-13), same
`state_dict()` key names (`critic.independent.{i}.network.{0,2,4}.{weight,bias}`, `target.…`; shared:
`critic.networks.{k}.…`) so checkpoints interchange with the reference's eval.py.  All arithmetic runs in
libmarlb200.so (marl_dqn_*); torch is used for parameter initialisation (nn.init on the host, once) and as the
owner of device buffers.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import random
import math
from collections import OrderedDict

import numpy as np
import torch

from .. import _native as nat
from ..lbf import TrajStore

HIDDEN = 128
MAX_IN_DIM = 128   # widest network input the learner kernels take (per-agent observation, or a centralised critic's joint observation)


def check_in_dim(width, what):
    if width > MAX_IN_DIM:
        raise NotImplementedError(f"{what} is {width} wide; the learner kernels take at most {MAX_IN_DIM} input features")


def _dim(space) -> int:
    """gymnasium.spaces.flatdim for the two space kinds the reference uses (dqn/model.py:32-33)."""
    if getattr(space, "n", None) is not None:
        return int(space.n)
    return int(np.prod(space.shape))


def sharing_to_nets(parameter_sharing, n_agents):
    """utils/models.py:189-196: True -> one network, False -> one per agent, list -> seps indices (renumbered densely)."""
    if parameter_sharing is True:
        return [0] * n_agents
    if parameter_sharing is False or parameter_sharing is None:
        return list(range(n_agents))
    order = []
    for i in parameter_sharing:
        if i not in order:
            order.append(i)
    return [order.index(i) for i in parameter_sharing]


def init_flat_params(n_nets, in_dim, out_dim, use_orthogonal_init=True):
    """utils/models.py:8-11,35-44 (host side, once): nn.Linear default init, optionally orthogonal(gain sqrt 2) + zero bias."""
    parts = []
    for _ in range(n_nets):
        for o, i in ((HIDDEN, in_dim), (HIDDEN, HIDDEN), (out_dim, HIDDEN)):
            lin = torch.nn.Linear(i, o)
            if use_orthogonal_init:
                torch.nn.init.orthogonal_(lin.weight.data, gain=math.sqrt(2))
                torch.nn.init.constant_(lin.bias.data, 0)
            parts += [lin.weight.data.reshape(-1), lin.bias.data.reshape(-1)]
    return torch.cat(parts).float()


def flat_to_state_dict(flat, prefix, n_nets, in_dim, out_dim):
    sd, o = OrderedDict(), 0
    for k in range(n_nets):
        for layer, shape in ((0, (HIDDEN, in_dim)), (2, (HIDDEN, HIDDEN)), (4, (out_dim, HIDDEN))):
            n = shape[0] * shape[1]
            sd[f"{prefix}.{k}.network.{layer}.weight"] = flat[o:o + n].view(*shape).clone()
            o += n
            sd[f"{prefix}.{k}.network.{layer}.bias"] = flat[o:o + shape[0]].clone()
            o += shape[0]
    return sd


def state_dict_to_flat(sd, prefix, n_nets):
    parts = []
    for k in range(n_nets):
        for layer in (0, 2, 4):
            parts += [sd[f"{prefix}.{k}.network.{layer}.weight"].reshape(-1), sd[f"{prefix}.{k}.network.{layer}.bias"].reshape(-1)]
    return torch.cat([p.float() for p in parts])


class QNetwork:
    mixer = 0

    def __init__(self, obs_space, action_space, cfg, layers, parameter_sharing, use_rnn, use_orthogonal_init, device, max_batch=None, max_episode_length=None):
        if use_rnn:
            raise NotImplementedError("use_rnn=True (GRU) is out of scope of the B200 hot path (every shipped config has use_rnn: False)")
        if list(layers) != [HIDDEN, HIDDEN]:
            raise NotImplementedError(f"layers={list(layers)}: the fused kernels implement the shipped [128, 128] MLP only")
        opt = getattr(cfg, "optimizer", "Adam")
        if (opt if isinstance(opt, str) else opt.__name__) != "Adam":
            raise NotImplementedError("only optimizer=Adam is implemented")
        if not torch.cuda.is_available() or not str(device).startswith("cuda"):
            raise nat.NativeError("the B200 learners need algorithm.model.device=cuda (no CPU fallback)")
        self.device = torch.device(device if ":" in str(device) else f"cuda:{torch.cuda.current_device()}")
        self.n_agents = len(obs_space)
        obs_dims, act_dims = [_dim(o) for o in obs_space], [_dim(a) for a in action_space]
        if len(set(obs_dims)) != 1 or len(set(act_dims)) != 1:
            raise NotImplementedError("agents with different observation / action sizes are not implemented")
        self.in_dim, self.n_actions = obs_dims[0], act_dims[0]
        check_in_dim(self.in_dim, "the observation")
        self.action_space = action_space
        self.agent_net = sharing_to_nets(parameter_sharing, self.n_agents)
        self.n_nets = max(self.agent_net) + 1
        self._kind = "independent" if not parameter_sharing else "networks"
        self.gamma, self.grad_clip, self.double_q = float(cfg.gamma), cfg.grad_clip, bool(cfg.double_q)
        self.target_update_interval_or_tau = float(cfg.target_update_interval_or_tau)
        self.max_batch = int(max_batch or getattr(cfg, "batch_size", 1024))
        self.max_T = int(max_episode_length or getattr(cfg, "max_episode_length", 0) or 500)
        self._lib = nat.lib()
        mcfg = nat.MlpCfg(self.n_agents, self.n_nets, (C.c_int32 * 32)(*self.agent_net), self.in_dim, HIDDEN, self.n_actions)
        hp = nat.DqnHP(float(cfg.lr), self.gamma, float(self.grad_clip or 0.0), int(self.double_q), self.target_update_interval_or_tau,
                       0.9, 0.999, 1e-8, self.mixer)
        self._h = C.c_void_p()
        with torch.cuda.device(self.device):
            nat.check(self._lib.marl_dqn_create(C.byref(mcfg), C.byref(hp), C.c_int32(self.max_batch), C.c_int32(self.max_T), C.c_int32(self.device.index),
                                                C.byref(self._h)), "marl_dqn_create")
        ptrs = [C.c_void_p() for _ in range(5)]
        n = C.c_int64()
        nat.check(self._lib.marl_dqn_param_ptrs(self._h, *[C.byref(p) for p in ptrs], C.byref(n)), "marl_dqn_param_ptrs")
        self.n_params = int(n.value)
        self.theta, self.theta_tgt, self.adam_m, self.adam_v = [nat.device_view(p.value, self.n_params, self.device) for p in ptrs[:4]]
        self.grad = nat.device_view(ptrs[4].value, self.n_params + 4, self.device)  # + (loss numerator, filled count, 2 spare)
        self.theta.copy_(init_flat_params(self.n_nets, self.in_dim, self.n_actions, use_orthogonal_init))
        self.params_changed()
        self.hard_update()
        self._metrics = torch.zeros(6, dtype=torch.float32, device=self.device)
        self._idx = torch.zeros(self.max_batch, dtype=torch.int32, device=self.device)
        self.standardise_returns = bool(getattr(cfg, "standardise_returns", False))   # dqn/model.py:82-84 (VDN: 221-222)
        if self.standardise_returns:
            nat.check(self._lib.marl_dqn_standardise_returns(self._h, C.c_int32(1)), "marl_dqn_standardise_returns")

    def ret_ms(self):
        """(mean, var, count) of the RunningMeanStd over the TD targets (standardise_returns): one entry per agent; VDN: per batch entry."""
        pm, pc, n = C.c_void_p(), C.c_void_p(), C.c_int32()
        nat.check(self._lib.marl_dqn_ret_ms_ptrs(self._h, C.byref(pm), C.byref(pc), C.byref(n)), "marl_dqn_ret_ms_ptrs")
        ms = nat.device_view(pm.value, 2 * n.value, self.device).cpu()
        return ms[: n.value], ms[n.value:], float(nat.device_view(pc.value, 1, self.device, "<f8").cpu()[0])

    # ---- reference API ------------------------------------------------------------------------------------------
    def init_hiddens(self, batch_size):
        return [None] * self.n_agents

    def q_values(self, obs: torch.Tensor, target: bool = False, out: torch.Tensor | None = None) -> torch.Tensor:
        """Network pass of model.act (dqn/model.py:96-99) for E envs: obs f32[E,N,D] -> q f32[E,N,A]."""
        E = obs.shape[0]
        if out is None:
            out = torch.empty(E, self.n_agents, self.n_actions, dtype=torch.float32, device=self.device)
        nat.check(self._lib.marl_dqn_forward(self._h, nat.ptr(obs), C.c_int32(E), C.c_int32(int(target)), nat.ptr(out), nat.stream_ptr()), "marl_dqn_forward")
        return out

    def act(self, inputs, hiddens, epsilon, action_masks=None):
        """dqn/model.py:94-116 for API parity (single env or a stack of envs).  The training / evaluation loops use the fused
        marl_lbf_rollout_step instead, which draws exploration from the Philox stream inside the env kernel."""
        if action_masks is not None:
            raise NotImplementedError("action masks only exist for smaclite in the reference (out of scope)")
        obs = torch.as_tensor(np.stack([np.asarray(i, np.float32) for i in inputs], 0), device=self.device)
        obs = obs.view(self.n_agents, -1, self.in_dim).transpose(0, 1).contiguous()
        q = self.q_values(obs)
        # the reference's stream: ONE `random.random()` per call decides the joint exploration (dqn/model.py:105), the random joint
        # action comes from Python's `random` as well (seed it with random.seed, as the reference's users do)
        if epsilon > random.random():
            actions = torch.tensor([[random.randrange(self.n_actions) for _ in range(self.n_agents)] for _ in range(obs.shape[0])])
        else:
            actions = q.argmax(-1).cpu()
        return (actions[0].tolist() if actions.shape[0] == 1 else actions.T.tolist()), hiddens

    def update_from_store(self, traj: TrajStore, idx: torch.Tensor):
        """QNetwork.update on episodes `idx` (int32 device tensor) of a device trajectory store."""
        nat.check(self._lib.marl_dqn_update(self._h, traj.ref(), nat.ptr(idx), C.c_int32(idx.numel()), nat.ptr(self._metrics), nat.stream_ptr()), "marl_dqn_update")
        return self._metrics

    def update_grads(self, traj: TrajStore, idx: torch.Tensor):
        nat.check(self._lib.marl_dqn_update_grads(self._h, traj.ref(), nat.ptr(idx), C.c_int32(idx.numel()), nat.stream_ptr()), "marl_dqn_update_grads")

    def update_apply(self):
        nat.check(self._lib.marl_dqn_update_apply(self._h, nat.ptr(self._metrics), nat.stream_ptr()), "marl_dqn_update_apply")
        return self._metrics

    def update_n(self, traj: TrajStore, batch_size: int, n_valid: int, seed: int, first_update_idx: int, n_updates: int):
        """`rb.sample(batch); model.update(batch)` n times on device (dqn/train.py:308-311)."""
        nat.check(self._lib.marl_dqn_update_n(self._h, traj.ref(), C.c_int32(batch_size), C.c_int32(n_valid), C.c_uint64(seed & (2**64 - 1)),
                                              C.c_uint64(first_update_idx), C.c_int32(n_updates), nat.ptr(self._metrics), nat.stream_ptr()), "marl_dqn_update_n")
        return self._metrics

    def update(self, batch):
        """Reference signature (dqn/model.py:165-174): `batch` is the reference's Batch namedtuple (obss (N,T+1,B,obs), actions
        (N,T,B), rewards (N,T,B), dones (T+1,B), filled (T,B)); converted to the device layout, then the native update."""
        obss = batch.obss
        N, T1, B, D = obss.shape
        store = TrajStore(B, N, T1 - 1, D, self.device)
        store.obs.copy_(obss.permute(2, 0, 1, 3))
        store.act.copy_(batch.actions.permute(2, 0, 1))
        store.rew.copy_(batch.rewards.permute(2, 0, 1))
        store.done.copy_(batch.dones.permute(1, 0))
        store.filled.copy_(batch.filled.permute(1, 0))
        idx = torch.arange(B, dtype=torch.int32, device=self.device)
        m = self.update_from_store(store, idx)
        return {"loss": float(m[0].item())}

    def timing(self, enable: bool):
        """CUDA-event timing of the training kernel: timing(True) starts, timing(False) -> (total_ms, launches)."""
        ms, n = C.c_float(), C.c_int32()
        nat.check(self._lib.marl_dqn_timing(self._h, C.c_int32(int(enable)), C.byref(ms), C.byref(n)), "marl_dqn_timing")
        return float(ms.value), int(n.value)

    peers_attached = False

    def attach_peers(self, group=None):
        """Several ranks, one process per GPU: exchange CUDA IPC handles through torch.distributed and let `update` / `update_n` sum
        the gradients of all ranks over NVLink peer memory inside the fused reduce + Adam kernel (no all-reduce call per update)."""
        import torch.distributed as dist

        world, rank = dist.get_world_size(group), dist.get_rank(group)
        mine = (C.c_ubyte * 64)()
        nat.check(self._lib.marl_dqn_peer_handle(self._h, mine), "marl_dqn_peer_handle")
        handles = [None] * world
        dist.all_gather_object(handles, bytes(mine), group=group)
        blob = b"".join(handles)
        nat.check(self._lib.marl_dqn_peer_attach(self._h, C.c_int32(rank), C.c_int32(world), blob), "marl_dqn_peer_attach")
        self.peers_attached = True
        dist.barrier(group)

    def peer_timed_out(self) -> bool:
        """True when an in-kernel gradient exchange gave up waiting for a peer (bounded spin): every result since is invalid."""
        v = C.c_int32()
        nat.check(self._lib.marl_dqn_peer_status(self._h, C.byref(v)), "marl_dqn_peer_status")
        return bool(v.value)

    def timing_kernels(self):
        """After timing(False): (ms of online forward + TD head, ms of dH1, ms of weight gradients), launches -- tensor-core pass only."""
        ms3, n = (C.c_float * 3)(), C.c_int32()
        nat.check(self._lib.marl_dqn_timing_kernels(self._h, ms3, C.byref(n)), "marl_dqn_timing_kernels")
        return [float(x) for x in ms3], int(n.value)

    @property
    def updates(self) -> int:
        u = C.c_int64()
        nat.check(self._lib.marl_dqn_counters(self._h, C.byref(u), None), "marl_dqn_counters")
        return int(u.value)

    def hard_update(self):
        nat.check(self._lib.marl_dqn_sync_target(self._h, nat.stream_ptr()), "marl_dqn_sync_target")

    def params_changed(self):
        """Call after writing `theta` / `theta_tgt` directly (checkpoint load, tests): cached derived data is rebuilt."""
        nat.check(self._lib.marl_dqn_params_changed(self._h), "marl_dqn_params_changed")

    def state_dict(self):
        sd = flat_to_state_dict(self.theta.detach().cpu(), f"critic.{self._kind}", self.n_nets, self.in_dim, self.n_actions)
        sd.update(flat_to_state_dict(self.theta_tgt.detach().cpu(), f"target.{self._kind}", self.n_nets, self.in_dim, self.n_actions))
        return sd

    def load_state_dict(self, sd):
        self.theta.copy_(state_dict_to_flat(sd, f"critic.{self._kind}", self.n_nets))
        self.theta_tgt.copy_(state_dict_to_flat(sd, f"target.{self._kind}", self.n_nets))
        self.params_changed()

    def parameters(self):
        return [self.theta]

    def close(self):
        if getattr(self, "_h", None):
            self._lib.marl_dqn_destroy(self._h)
            self._h = None
            # the views below aliased library-owned device memory that no longer exists
            self.theta = self.theta_tgt = self.adam_m = self.adam_v = self.grad = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class VDNetwork(QNetwork):
    """marlbase/dqn/model.py:199-269: Q_tot = sum_i Q_i, reward of agent 0 (CooperativeReward makes them equal)."""

    mixer = 1


MIXER_KEYS = ("hyper_w_1.0", "hyper_w_1.2", "hyper_w_final.0", "hyper_w_final.2", "hyper_b_1", "V.0", "V.2")


def mixer_shapes(n_agents, state_dim, embed_dim, hypernet_embed):
    """(out, in) of the mixing network's seven Linear layers in the reference's state_dict order (dqn/model.py:283-311, hypernet_layers == 2)."""
    N, S, E, He = n_agents, state_dim, embed_dim, hypernet_embed
    return ((He, S), (N * E, He), (He, S), (E, He), (E, S), (E, S), (1, E))


class QMixNetwork(QNetwork):
    """marlbase/dqn/model.py:343-443: the agents' Q-values of the chosen (target: double-Q) actions go through a monotonic mixing network conditioned
    on the state (all observations concatenated); one Adam over critic + mixer, the gradient clip covers the critic only, target updates include
    the mixer.  The mixer runs in qmix.cuh's kernels next to the tensor-core training pass of the agents' networks (csrc/dqn.cu, mixer == 2)."""

    mixer = 2

    def __init__(self, obs_space, action_space, cfg, layers, parameter_sharing, use_rnn, use_orthogonal_init, mixing, device, max_batch=None, max_episode_length=None):
        if bool(getattr(cfg, "standardise_returns", False)):
            raise NotImplementedError("standardise_returns with QMIX is not implemented (qmix.yaml inherits standardise_returns: False)")
        if int(dict(mixing)["hypernet_layers"]) != 2:
            raise NotImplementedError(f"mixing.hypernet_layers={dict(mixing)['hypernet_layers']}: only the shipped two-layer hypernetworks (qmix.yaml) are implemented")
        super().__init__(obs_space, action_space, cfg, layers, parameter_sharing, use_rnn, use_orthogonal_init, device, max_batch, max_episode_length)
        mixing = dict(mixing)
        self.embed_dim, self.hypernet_embed = int(mixing["embed_dim"]), int(mixing["hypernet_embed"])
        self.state_dim = self.n_agents * self.in_dim
        with torch.cuda.device(self.device):
            nat.check(self._lib.marl_dqn_qmix_init(self._h, C.c_int32(self.embed_dim), C.c_int32(int(mixing["hypernet_layers"])), C.c_int32(self.hypernet_embed)), "marl_dqn_qmix_init")
        ptrs = [C.c_void_p() for _ in range(5)]
        n = C.c_int64()
        nat.check(self._lib.marl_dqn_qmix_ptrs(self._h, *[C.byref(p) for p in ptrs], C.byref(n)), "marl_dqn_qmix_ptrs")
        self.n_mix = int(n.value)
        self.mix, self.mix_tgt, self.mix_m, self.mix_v = [nat.device_view(p.value, self.n_mix, self.device) for p in ptrs[:4]]
        self.mix_grad = nat.device_view(ptrs[4].value, self.n_mix + 4, self.device)
        # QMixer's layers are plain nn.Linear (PyTorch's default initialisation), created in this order (dqn/model.py:283-311)
        parts = []
        for (o, i) in mixer_shapes(self.n_agents, self.state_dim, self.embed_dim, self.hypernet_embed):
            lin = torch.nn.Linear(i, o)
            parts += [lin.weight.data.reshape(-1), lin.bias.data.reshape(-1)]
        self.mix.copy_(torch.cat(parts).float())
        self.hard_update()

    def _mixer_sd(self, flat, prefix):
        sd, o = {}, 0
        for k, (no, ni) in zip(MIXER_KEYS, mixer_shapes(self.n_agents, self.state_dim, self.embed_dim, self.hypernet_embed)):
            sd[f"{prefix}.{k}.weight"] = flat[o:o + no * ni].view(no, ni).clone(); o += no * ni
            sd[f"{prefix}.{k}.bias"] = flat[o:o + no].clone(); o += no
        return sd

    def state_dict(self):
        sd = super().state_dict()
        sd.update(self._mixer_sd(self.mix.detach().cpu(), "mixer"))
        sd.update(self._mixer_sd(self.mix_tgt.detach().cpu(), "target_mixer"))
        return sd

    def load_state_dict(self, sd):
        super().load_state_dict(sd)
        for dst, prefix in ((self.mix, "mixer"), (self.mix_tgt, "target_mixer")):
            dst.copy_(torch.cat([sd[f"{prefix}.{k}.{p}"].reshape(-1).float() for k in MIXER_KEYS for p in ("weight", "bias")]))

    def parameters(self):
        return [self.theta, self.mix]

    def attach_peers(self, group=None):
        raise NotImplementedError("QMIX runs on one GPU: the mixer's gradient is not part of the peer-memory exchange")

    def close(self):
        super().close()
        self.mix = self.mix_tgt = self.mix_m = self.mix_v = self.mix_grad = None
