"""Independent actor-critic learner on the B200 path -- drop-in for marlbase/ac/model.py A2CNetwork (22-246).

Same constructor signature / Hydra `_target_` role (configs/algorithm/ia2c.yaml:8-26) and the reference's
`state_dict()` key names (`actor.independent.{i}.network.…`, `critic.…`, `target_critic.…`; shared: `.networks.{k}.`).
All arithmetic runs in libmarlb200.so (marl_a2c_*): actor forward, target-critic pass, n-step returns
(utils/utils.py:38-63), fused forward / loss / backward of critic and actor, Adam, target sync.  No CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import torch

from .. import _native as nat
from ..dqn.model import HIDDEN, _dim, check_in_dim, flat_to_state_dict, init_flat_params, sharing_to_nets, state_dict_to_flat
from ..lbf import TrajStore


class A2CNetwork:
    def __init__(self, obs_space, action_space, cfg, actor, critic, device, max_envs=None, max_episode_length=None):
        for part, name in ((actor, "actor"), (critic, "critic")):
            if part.use_rnn:
                raise NotImplementedError(f"{name}.use_rnn=True (GRU) is out of scope of the B200 hot path")
            if list(part.layers) != [HIDDEN, HIDDEN]:
                raise NotImplementedError(f"{name}.layers={list(part.layers)}: the fused kernels implement the shipped [128, 128] MLP only")
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
        # critic.centralised (MAA2C / MAPPO, ac/model.py:62-65): every agent's critic reads the concatenation of all agents' observations
        self.centralised = bool(critic.centralised) and self.n_agents > 1
        self.critic_in = self.n_agents * self.in_dim if self.centralised else self.in_dim
        check_in_dim(self.in_dim, "the observation")
        check_in_dim(self.critic_in, "critic.centralised: the joint observation")
        self.gamma, self.entropy_coef, self.n_steps = float(cfg.gamma), float(cfg.entropy_coef), int(cfg.n_steps)
        self.grad_clip, self.value_loss_coef = cfg.grad_clip, float(cfg.value_loss_coef)
        self.target_update_interval_or_tau = float(cfg.target_update_interval_or_tau)
        self.actor_net = sharing_to_nets(actor.parameter_sharing, self.n_agents)
        self.critic_net = sharing_to_nets(critic.parameter_sharing, self.n_agents)
        self.n_actor_nets, self.n_critic_nets = max(self.actor_net) + 1, max(self.critic_net) + 1
        self._akind = "independent" if not actor.parameter_sharing else "networks"
        self._ckind = "independent" if not critic.parameter_sharing else "networks"
        self.max_envs = int(max_envs or 1024)
        self.max_T = int(max_episode_length or 500)
        self._lib = nat.lib()
        acfg = nat.MlpCfg(self.n_agents, self.n_actor_nets, (C.c_int32 * 32)(*self.actor_net), self.in_dim, HIDDEN, self.n_actions)
        ccfg = nat.MlpCfg(self.n_agents, self.n_critic_nets, (C.c_int32 * 32)(*self.critic_net), self.critic_in, HIDDEN, 1)
        hp = nat.A2cHP(float(cfg.lr), self.gamma, float(self.grad_clip or 0.0), self.n_steps, self.entropy_coef, self.value_loss_coef,
                       self.target_update_interval_or_tau, 0.9, 0.999, 1e-8)
        self._h = C.c_void_p()
        with torch.cuda.device(self.device):
            nat.check(self._lib.marl_a2c_create(C.byref(acfg), C.byref(ccfg), C.byref(hp), C.c_int32(self.max_envs), C.c_int32(self.max_T),
                                                C.c_int32(self.device.index), C.byref(self._h)), "marl_a2c_create")
        ptrs = [C.c_void_p() for _ in range(5)]
        na, nc = C.c_int64(), C.c_int64()
        nat.check(self._lib.marl_a2c_param_ptrs(self._h, *[C.byref(p) for p in ptrs], C.byref(na), C.byref(nc)), "marl_a2c_param_ptrs")
        self.n_actor, self.n_critic = int(na.value), int(nc.value)
        n = self.n_actor + self.n_critic
        self.theta = nat.device_view(ptrs[0].value, n, self.device)
        self.theta_tgt = nat.device_view(ptrs[1].value, self.n_critic, self.device)
        self.adam_m, self.adam_v = nat.device_view(ptrs[2].value, n, self.device), nat.device_view(ptrs[3].value, n, self.device)
        self.grad = nat.device_view(ptrs[4].value, n + 4, self.device)
        self.theta[: self.n_actor].copy_(init_flat_params(self.n_actor_nets, self.in_dim, self.n_actions, actor.use_orthogonal_init))
        self.theta[self.n_actor:].copy_(init_flat_params(self.n_critic_nets, self.critic_in, 1, critic.use_orthogonal_init))
        self.soft_update(1.0)
        self._metrics = torch.zeros(6, dtype=torch.float32, device=self.device)
        self.standardise_returns = bool(getattr(cfg, "standardise_returns", False))   # ac/model.py:112-114
        if self.standardise_returns:
            nat.check(self._lib.marl_a2c_standardise_returns(self._h, C.c_int32(1)), "marl_a2c_standardise_returns")

    def ret_ms(self):
        """(mean[N], var[N], count) of the RunningMeanStd over the returns (standardise_returns), as CPU values."""
        pm, pc = C.c_void_p(), C.c_void_p()
        nat.check(self._lib.marl_a2c_ret_ms_ptrs(self._h, C.byref(pm), C.byref(pc)), "marl_a2c_ret_ms_ptrs")
        ms = nat.device_view(pm.value, 2 * self.n_agents, self.device).cpu()
        cnt = nat.device_view(pc.value, 1, self.device, "<f8").cpu()
        return ms[: self.n_agents], ms[self.n_agents:], float(cnt[0])

    # ---- views into the flat parameter vector ------------------------------------------------------------------
    @property
    def actor_params(self):
        return self.theta[: self.n_actor]

    @property
    def critic_params(self):
        return self.theta[self.n_actor:]

    def scratch(self, n_envs, T):
        """(target values [N,P,T+1], n-step returns [N,P,T], advantages [N,P,T]) of the last update -- device views for tests."""
        ptrs = [C.c_void_p() for _ in range(3)]
        nat.check(self._lib.marl_a2c_scratch_ptrs(self._h, *[C.byref(p) for p in ptrs]), "marl_a2c_scratch_ptrs")
        N = self.n_agents
        return (nat.device_view(ptrs[0].value, N * n_envs * (T + 1), self.device).view(N, n_envs, T + 1),
                nat.device_view(ptrs[1].value, N * n_envs * T, self.device).view(N, n_envs, T),
                nat.device_view(ptrs[2].value, N * n_envs * T, self.device).view(N, n_envs, T))

    # ---- reference API ------------------------------------------------------------------------------------------------
    def init_actor_hiddens(self, batch_size):
        return [None] * self.n_agents

    def init_critic_hiddens(self, batch_size, target=False):
        return [None] * self.n_agents

    def logits(self, obs: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        """Actor pass of act (ac/model.py:148-150): obs f32[E,N,D] -> logits f32[E,N,A]."""
        E = obs.shape[0]
        if out is None:
            out = torch.empty(E, self.n_agents, self.n_actions, dtype=torch.float32, device=self.device)
        nat.check(self._lib.marl_a2c_forward_actor(self._h, nat.ptr(obs), C.c_int32(E), nat.ptr(out), nat.stream_ptr()), "marl_a2c_forward_actor")
        return out

    def values(self, obs: torch.Tensor, target: bool = False) -> torch.Tensor:
        """get_value (ac/model.py:155-163): obs f32[E,N,D] -> f32[E,N] (centralised critic: each agent's network reads all N x D values of its env)."""
        E = obs.shape[0]
        out = torch.empty(E, self.n_agents, 1, dtype=torch.float32, device=self.device)
        nat.check(self._lib.marl_a2c_forward_critic(self._h, nat.ptr(obs), C.c_int32(E), C.c_int32(int(target)), nat.ptr(out), nat.stream_ptr()), "marl_a2c_forward_critic")
        return out.squeeze(-1)

    def act(self, inputs, actor_hiddens, action_mask=None):
        """ac/model.py:147-153 for API parity: list of N tensors [P, obs] -> i64[N, P, 1].  The training loop uses the fused
        marl_lbf_rollout_step(policy=2) which samples from the Philox stream inside the env kernel."""
        if action_mask is not None:
            raise NotImplementedError("action masks only exist for smaclite in the reference (out of scope)")
        obs = torch.stack([torch.as_tensor(i, dtype=torch.float32, device=self.device) for i in inputs], 1).contiguous()
        dist = torch.distributions.Categorical(logits=self.logits(obs))
        return dist.sample().T.unsqueeze(-1).contiguous(), actor_hiddens

    def update_from_store(self, batch: TrajStore, n_envs: int, step: int):
        """One `model.update(batch, step)` on the device batch (ac/train.py:176)."""
        nat.check(self._lib.marl_a2c_update(self._h, batch.ref(), C.c_int32(n_envs), C.c_int64(int(step)), nat.ptr(self._metrics), nat.stream_ptr()), "marl_a2c_update")
        return self._metrics

    def update_grads(self, batch: TrajStore, n_envs: int):
        nat.check(self._lib.marl_a2c_update_grads(self._h, batch.ref(), C.c_int32(n_envs), nat.stream_ptr()), "marl_a2c_update_grads")

    def update_apply(self, step: int):
        nat.check(self._lib.marl_a2c_update_apply(self._h, C.c_int64(int(step)), nat.ptr(self._metrics), nat.stream_ptr()), "marl_a2c_update_apply")
        return self._metrics

    def metrics_dict(self, m=None):
        """ac/model.py:241-246 from the device statistics (policy-gradient term, grad norm, entropy, value loss, ...)."""
        m = (self._metrics if m is None else m).tolist()
        actor_loss = m[0] - self.entropy_coef * m[2]
        return {"loss": actor_loss + self.value_loss_coef * m[3], "actor_loss": actor_loss, "value_loss": m[3], "entropy": m[2]}

    def update(self, batch, step):
        """Reference signature (ac/model.py:189): Batch(obss (T+1,P,N*obs), actions (T,P,N), rewards (T,P,N), dones (T+1,P), filled (T,P))."""
        T1, P, ND = batch.obss.shape
        N, D = self.n_agents, self.in_dim
        store = TrajStore(P, N, T1 - 1, D, self.device)
        store.obs.copy_(batch.obss.view(T1, P, N, D).permute(1, 2, 0, 3))
        store.act.copy_(batch.actions.permute(1, 2, 0))
        store.rew.copy_(batch.rewards.permute(1, 2, 0))
        store.done.copy_(batch.dones.permute(1, 0))
        store.filled.copy_(batch.filled.permute(1, 0))
        return self.metrics_dict(self.update_from_store(store, P, step))

    def soft_update(self, t):
        if t != 1.0:
            self.theta_tgt.copy_((1 - t) * self.theta_tgt + t * self.critic_params)
        else:
            nat.check(self._lib.marl_a2c_sync_target(self._h, nat.stream_ptr()), "marl_a2c_sync_target")

    def state_dict(self):
        th, tg = self.theta.detach().cpu(), self.theta_tgt.detach().cpu()
        sd = flat_to_state_dict(th[: self.n_actor], f"actor.{self._akind}", self.n_actor_nets, self.in_dim, self.n_actions)
        sd.update(flat_to_state_dict(th[self.n_actor:], f"critic.{self._ckind}", self.n_critic_nets, self.critic_in, 1))
        sd.update(flat_to_state_dict(tg, f"target_critic.{self._ckind}", self.n_critic_nets, self.critic_in, 1))
        return sd

    def load_state_dict(self, sd):
        self.theta[: self.n_actor].copy_(state_dict_to_flat(sd, f"actor.{self._akind}", self.n_actor_nets))
        self.theta[self.n_actor:].copy_(state_dict_to_flat(sd, f"critic.{self._ckind}", self.n_critic_nets))
        self.theta_tgt.copy_(state_dict_to_flat(sd, f"target_critic.{self._ckind}", self.n_critic_nets))

    def parameters(self):
        return [self.theta]

    def close(self):
        if getattr(self, "_h", None):
            self._lib.marl_a2c_destroy(self._h)
            self._h = None
            self.theta = self.theta_tgt = self.adam_m = self.adam_v = self.grad = None  # views of freed library memory

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PPONetwork(A2CNetwork):
    """Independent PPO -- drop-in for marlbase/ac/model.py PPONetwork (249-352; `_target_: ac.model.PPONetwork`, configs/algorithm/ippo.yaml).
    Same networks, rollout and n-step returns as A2CNetwork; `update` re-uses one batch for `num_epochs` optimisation steps with the clipped
    surrogate (marl_ppo_update: collecting-policy log-probabilities once, then per epoch critic pass -> actor pass -> clip + Adam on the device,
    target critic after the last epoch).  Metrics are the epochs' means, as the reference returns them."""

    def __init__(self, obs_space, action_space, cfg, actor, critic, device, max_envs=None, max_episode_length=None):
        super().__init__(obs_space, action_space, cfg, actor, critic, device, max_envs=max_envs, max_episode_length=max_episode_length)
        self.num_epochs, self.ppo_clip = int(cfg.num_epochs), float(cfg.ppo_clip)

    def update_from_store(self, batch: TrajStore, n_envs: int, step: int):
        nat.check(self._lib.marl_ppo_update(self._h, batch.ref(), C.c_int32(n_envs), C.c_int64(int(step)), C.c_int32(self.num_epochs), C.c_float(self.ppo_clip),
                                            nat.ptr(self._metrics), nat.stream_ptr()), "marl_ppo_update")
        return self._metrics

    def update_grads(self, batch, n_envs):
        raise NotImplementedError("PPO's epochs each need their own optimiser step: the grads / apply split of the data-parallel A2C path does not apply")
