"""CPU restatement (PyTorch float32, autograd) of the reference learner arithmetic.  TEST INFRASTRUCTURE ONLY.

Written functionally over FLAT parameter vectors in the device layout ([n_nets][P], reference state_dict order), so
that it also pins the layout conversion.  Pinned against committed golden vectors generated from the live reference
classes (tests/golden/: make_golden.py and the make_reference_cases functions of the tests).

Restated from (path:line under /root/reference/marlbase):
  utils/models.py:14-48      FCNetwork = Linear-ReLU-Linear-ReLU-Linear
  utils/models.py:133-300    independent / shared per-agent network containers
  dqn/model.py:118-163       QNetwork._compute_loss (double-Q TD target, MSE summed over agents, masked mean)
  dqn/model.py:224-269       VDNetwork._compute_loss (agent-summed Q, rewards[0])
  dqn/model.py:165-196       update: clip_grad_norm_, Adam, hard / soft target update
  dqn/train.py:19-124        episode ReplayBuffer; :127-174 epsilon schedule
  utils/utils.py:38-63       compute_nstep_returns
  ac/model.py:189-246        A2CNetwork.update
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np
import torch
import torch.nn.functional as F

H = 128


# ---- parameter layout ------------------------------------------------------------------------------------------
def net_size(in_dim, out_dim):
    return H * in_dim + H + H * H + H + out_dim * H + out_dim


def split_net(flat, in_dim, out_dim):
    """views (w1, b1, w2, b2, w3, b3) into one network's flat parameter vector"""
    o = 0
    out = []
    for shape in ((H, in_dim), (H,), (H, H), (H,), (out_dim, H), (out_dim,)):
        n = int(np.prod(shape))
        out.append(flat[o:o + n].view(*shape))
        o += n
    return out


def flat_from_state_dict(sd, prefix, n_nets):
    """prefix e.g. 'critic.independent' or 'critic.networks' -> flat [n_nets*P]"""
    parts = []
    for k in range(n_nets):
        for layer in (0, 2, 4):
            parts.append(sd[f"{prefix}.{k}.network.{layer}.weight"].reshape(-1))
            parts.append(sd[f"{prefix}.{k}.network.{layer}.bias"].reshape(-1))
    return torch.cat(parts).clone().float()


def state_dict_from_flat(flat, prefix, n_nets, in_dim, out_dim):
    P = net_size(in_dim, out_dim)
    sd = {}
    for k in range(n_nets):
        w1, b1, w2, b2, w3, b3 = split_net(flat[k * P:(k + 1) * P], in_dim, out_dim)
        for layer, (w, b) in zip((0, 2, 4), ((w1, b1), (w2, b2), (w3, b3))):
            sd[f"{prefix}.{k}.network.{layer}.weight"] = w.clone()
            sd[f"{prefix}.{k}.network.{layer}.bias"] = b.clone()
    return sd


def init_flat(n_nets, in_dim, out_dim, orthogonal=True, generator=None):
    """utils/models.py:8-11,35-44: orthogonal(gain sqrt 2) weights + zero bias on every Linear (or nn.Linear default)."""
    parts = []
    for _ in range(n_nets):
        for (o, i) in ((H, in_dim), (H, H), (out_dim, H)):
            lin = torch.nn.Linear(i, o)
            if orthogonal:
                torch.nn.init.orthogonal_(lin.weight.data, gain=math.sqrt(2), generator=generator) if generator is not None else torch.nn.init.orthogonal_(lin.weight.data, gain=math.sqrt(2))
                torch.nn.init.constant_(lin.bias.data, 0)
            parts += [lin.weight.data.reshape(-1), lin.bias.data.reshape(-1)]
    return torch.cat(parts).float()


_TAPS = None   # kink_risk(): hidden pre-/post-activations of the differentiated (online) passes


def mlp(flat_net, x, in_dim, out_dim):
    w1, b1, w2, b2, w3, b3 = split_net(flat_net, in_dim, out_dim)
    if _TAPS is not None and flat_net.requires_grad:
        z1 = F.linear(x, w1, b1); h1 = F.relu(z1); h1.retain_grad()
        z2 = F.linear(h1, w2, b2); h2 = F.relu(z2); h2.retain_grad()
        _TAPS.append((z1, h1, x)); _TAPS.append((z2, h2, h1))
        return F.linear(h2, w3, b3)
    return F.linear(F.relu(F.linear(F.relu(F.linear(x, w1, b1)), w2, b2)), w3, b3)


def agents_forward(flat, agent_net, xs, in_dim, out_dim):
    """xs: list (per agent) of (..., in_dim) tensors -> list of (..., out_dim).  Agents sharing a network share the flat slice."""
    P = net_size(in_dim, out_dim)
    return [mlp(flat[k * P:(k + 1) * P], x, in_dim, out_dim) for k, x in zip(agent_net, xs)]


# ---- Adam / clipping exactly as torch.optim.Adam (single tensor path) + clip_grad_norm_ -----------------------------
def clip_coef(grad, max_norm):
    total = torch.linalg.vector_norm(grad)
    return torch.clamp(max_norm / (total + 1e-6), max=1.0), total


def adam_step(theta, m, v, grad, step, lr, beta1=0.9, beta2=0.999, eps=1e-8):
    m.lerp_(grad, 1 - beta1)
    v.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
    bc1 = 1 - beta1 ** step
    bc2 = 1 - beta2 ** step
    denom = (v.sqrt() / (bc2 ** 0.5)).add_(eps)
    theta.addcdiv_(m, denom, value=-(lr / bc1))


# ---- DQN family ----------------------------------------------------------------------------------------------------
@dataclass
class DqnHP:
    lr: float = 3e-4
    gamma: float = 0.99
    grad_clip: float = 1.0
    double_q: bool = True
    target_update_interval_or_tau: float = 200
    mixer: int = 0  # 0 independent, 1 VDN


@dataclass
class DqnState:
    theta: torch.Tensor
    theta_tgt: torch.Tensor
    agent_net: list
    in_dim: int
    out_dim: int
    m: torch.Tensor = None
    v: torch.Tensor = None
    updates: int = 0
    last_target_update: int = 0
    ret_ms: object = None   # RunningMeanStdRef when cfg.standardise_returns (dqn/model.py:82-84: shape (n_agents,); VDN 221-222: shape (1,))

    def __post_init__(self):
        if self.m is None:
            self.m = torch.zeros_like(self.theta)
        if self.v is None:
            self.v = torch.zeros_like(self.theta)


def dqn_loss(theta, theta_tgt, agent_net, in_dim, out_dim, batch, hp: DqnHP, ret_ms=None):
    """batch = dict(obss (N,T+1,B,D) f32, actions (N,T,B) i64, rewards (N,T,B), dones (T+1,B) f32, filled (T,B) f32)"""
    obss, actions, rewards, dones, filled = (batch[k] for k in ("obss", "actions", "rewards", "dones", "filled"))
    N = obss.shape[0]
    q = torch.stack(agents_forward(theta, agent_net, list(obss), in_dim, out_dim))          # (N,T+1,B,A)
    chosen = q[:, :-1].gather(-1, actions.unsqueeze(-1)).squeeze(-1)                         # (N,T,B)
    with torch.no_grad():
        tq = torch.stack(agents_forward(theta_tgt, agent_net, list(obss), in_dim, out_dim))[:, 1:]
        if hp.double_q:
            a_prime = q.detach()[:, 1:].argmax(-1, keepdim=True)
            target = tq.gather(-1, a_prime).squeeze(-1)
        else:
            target = tq.max(-1)[0]
    if hp.mixer == 1:
        chosen = chosen.sum(0)
        target = target.sum(0)
        if ret_ms is not None:                                           # dqn/model.py:256-257
            target = target * torch.sqrt(ret_ms.var) + ret_ms.mean
        returns = rewards[0] + hp.gamma * target * (1 - dones[1:])
        if ret_ms is not None:                                           # dqn/model.py:262-264: update() reshapes the (E, B) returns with reshape(-1, B)
            ret_ms.update(returns)
            returns = (returns - ret_ms.mean) / torch.sqrt(ret_ms.var)
        loss = (chosen - returns.detach()) ** 2
    else:
        if ret_ms is not None:                                           # dqn/model.py:147-150 ("A E B -> E B A", per-agent statistics)
            target = (target.permute(1, 2, 0) * torch.sqrt(ret_ms.var) + ret_ms.mean).permute(2, 0, 1)
        returns = rewards + hp.gamma * target * (1 - dones[1:].unsqueeze(0).repeat(N, 1, 1))
        if ret_ms is not None:                                           # dqn/model.py:154-158
            r = returns.permute(1, 2, 0)
            ret_ms.update(r)
            returns = ((r - ret_ms.mean) / torch.sqrt(ret_ms.var)).permute(2, 0, 1)
        loss = ((chosen - returns.detach()) ** 2).sum(0)
    return (loss * filled).sum() / filled.sum()


def double_q_margin(st: DqnState, batch, hp: DqnHP):
    """Smallest gap between the best and the second-best ONLINE Q-value over every (agent, filled step t, episode) whose row t + 1 feeds the
    double-Q argmax (VDN: the same, per agent).  The argmax is discontinuous: when this margin is below the forward passes' ~1e-6 agreement, two
    correct implementations may pick different target actions and their gradients then differ by ~1 / filled-steps -- not a defect."""
    if not hp.double_q:
        return float("inf")
    with torch.no_grad():
        q = torch.stack(agents_forward(st.theta, st.agent_net, list(batch["obss"]), st.in_dim, st.out_dim))[:, 1:]     # (N, T, B, A)
        top2 = q.topk(2, dim=-1).values
        gap = (top2[..., 0] - top2[..., 1]) / top2[..., 0].abs().clamp_min(1.0)
        mask = batch["filled"].unsqueeze(0).expand_as(gap) > 0
        return float(gap[mask].min()) if bool(mask.any()) else float("inf")


def kink_risk(loss_fn, theta, near=2e-6):
    """ReLU is the learners' other discontinuity (next to the double-Q argmax): a hidden pre-activation z within the implementations' ~1e-6
    agreement of zero may be "on" in one and "off" in the other, which moves the gradient by dL/dh[r][j] x (the unit's input row) -- not a defect.
    Returns the largest such potential move over all hidden units with |z| < near (0 when there is none): loss_fn(theta) -> scalar loss."""
    global _TAPS
    _TAPS = []
    try:
        th = theta.clone().requires_grad_(True)
        loss_fn(th).backward()
        risk = 0.0
        for z, h, inp in _TAPS:
            if h.grad is None:
                continue
            m = (z.detach().abs() < near) & (z.detach() != 0)
            if bool(m.any()):
                scale_in = inp.detach().abs().amax(dim=-1, keepdim=True).clamp_min(1.0).expand_as(z)
                risk = max(risk, float((h.grad.abs() * scale_in)[m].max()))
        return risk
    finally:
        _TAPS = None


def dqn_kink_risk(st: DqnState, batch, hp: DqnHP):
    return kink_risk(lambda th: dqn_loss(th, st.theta_tgt, st.agent_net, st.in_dim, st.out_dim, batch, hp), st.theta)


def dqn_update(st: DqnState, batch, hp: DqnHP):
    """QNetwork.update: returns dict(loss, grad (before clipping), grad_norm)."""
    theta = st.theta.clone().requires_grad_(True)
    loss = dqn_loss(theta, st.theta_tgt, st.agent_net, st.in_dim, st.out_dim, batch, hp, st.ret_ms)
    (grad,) = torch.autograd.grad(loss, theta)
    raw = grad.clone()
    norm = torch.linalg.vector_norm(grad)
    if hp.grad_clip:
        coef, norm = clip_coef(grad, hp.grad_clip)
        grad = grad * coef
    st.updates += 1
    adam_step(st.theta, st.m, st.v, grad, st.updates, hp.lr)
    tu = hp.target_update_interval_or_tau
    if tu > 1.0 and (st.updates - st.last_target_update) >= tu:
        st.theta_tgt.copy_(st.theta)
        st.last_target_update = st.updates
    elif tu < 1.0:
        st.theta_tgt.copy_((1 - tu) * st.theta_tgt + tu * st.theta)
    return dict(loss=float(loss.detach()), grad=raw, grad_norm=float(norm), grad_clipped=grad.detach().clone())


def epsilon_schedule(decay_style, decay_over, eps_start, eps_end, exp_decay_rate, total_steps):
    """dqn/train.py:127-174"""
    if decay_style in ("linear", "lin"):
        return lambda step: max(eps_end + (eps_start - eps_end) * (1 - step / (total_steps * decay_over)), eps_end)
    if decay_style in ("exponential", "exp"):
        k = (eps_start - eps_end) / (total_steps * decay_over) * exp_decay_rate
        return lambda step: max(eps_end + (eps_start - eps_end) * math.exp(-k * step), eps_end)
    raise ValueError("decay_style must be one of 'linear' or 'exponential'")


# ---- trajectory store (episode-major, the device layout) <-> the reference's Batch ----------------------------------
def batch_from_store(store, idx, device="cpu"):
    """store: dict of numpy/torch arrays obs [cap,N,T+1,D], act [cap,N,T], rew [cap,N,T], done [cap,T+1], filled [cap,T];
    idx: episode slots [B].  Returns the reference Batch layout of ReplayBuffer.sample (dqn/train.py:96-124)."""
    t = {k: torch.as_tensor(np.asarray(v)) for k, v in store.items()}
    idx = torch.as_tensor(np.asarray(idx)).long()
    return dict(
        obss=t["obs"][idx].permute(1, 2, 0, 3).float().contiguous(),
        actions=t["act"][idx].permute(1, 2, 0).long().contiguous(),
        rewards=t["rew"][idx].permute(1, 2, 0).float().contiguous(),
        dones=t["done"][idx].permute(1, 0).float().contiguous(),
        filled=t["filled"][idx].permute(1, 0).float().contiguous(),
    )


class ReplayRef:
    """Episode ring with the reference's add/init_episode/sample semantics (dqn/train.py:19-124), stored episode-major."""

    def __init__(self, capacity, n_agents, T, obs_dim):
        self.capacity, self.N, self.T = capacity, n_agents, T
        self.store = dict(obs=np.zeros((capacity, n_agents, T + 1, obs_dim), np.float32), act=np.zeros((capacity, n_agents, T), np.int32),
                          rew=np.zeros((capacity, n_agents, T), np.float32), done=np.zeros((capacity, T + 1), np.uint8),
                          filled=np.zeros((capacity, T), np.uint8))
        self.pos = self.cur = self.t = 0

    def __len__(self):
        return min(self.pos, self.capacity)

    def init_episode(self, obss):
        self.t = 0
        self.store["obs"][self.cur, :, 0] = np.stack(obss)

    def add(self, obss, acts, rews, done):
        assert self.t < self.T
        s = self.store
        s["obs"][self.cur, :, self.t + 1] = np.stack(obss)
        s["act"][self.cur, :, self.t] = acts
        s["rew"][self.cur, :, self.t] = rews
        s["done"][self.cur, self.t + 1] = done
        s["filled"][self.cur, self.t] = 1
        self.t += 1
        if done:
            self.pos += 1
            self.cur = self.pos % self.capacity
            self.t = 0


# ---- actor-critic ----------------------------------------------------------------------------------------------------
def nstep_returns(rewards, done, next_values, nsteps, gamma):
    """utils/utils.py:38-63.  rewards (T,B,N); done, next_values (>=T,B,N)."""
    T = rewards.size(0)
    out = torch.zeros_like(rewards)
    for t0 in range(T):
        acc = torch.zeros_like(rewards[0])
        for step in range(nsteps + 1):
            t = t0 + step
            if t >= T:
                break
            src = next_values[t] if step == nsteps else rewards[t]
            acc = acc + gamma ** step * src * (1 - done[t])
        out[t0] = acc
    return out


class RunningMeanStdRef:
    """utils/standardise_stream.py:6-43 restated (float32 tensors, Python-float count)"""

    def __init__(self, shape, epsilon=1e-4):
        self.mean, self.var, self.count = torch.zeros(shape, dtype=torch.float32), torch.ones(shape, dtype=torch.float32), epsilon

    def update(self, arr):
        arr = arr.reshape(-1, arr.size(-1))
        batch_mean, batch_var, batch_count = torch.mean(arr, dim=0), torch.var(arr, dim=0), arr.shape[0]
        delta = batch_mean - self.mean
        tot_count = self.count + batch_count
        new_mean = self.mean + delta * batch_count / tot_count
        m_2 = self.var * self.count + batch_var * batch_count + torch.square(delta) * self.count * batch_count / (self.count + batch_count)
        self.mean, self.var, self.count = new_mean, m_2 / (self.count + batch_count), batch_count + self.count


@dataclass
class A2CHP:
    lr: float = 3e-4
    gamma: float = 0.99
    grad_clip: float = 0.0
    n_steps: int = 5
    entropy_coef: float = 0.001
    value_loss_coef: float = 0.5
    target_update_interval_or_tau: float = 200


@dataclass
class A2CState:
    actor: torch.Tensor        # flat [n_actor_nets * P_actor]
    critic: torch.Tensor       # flat [n_critic_nets * P_critic]
    target: torch.Tensor
    actor_net: list
    critic_net: list
    in_dim: int
    n_actions: int
    m: dict = field(default_factory=dict)
    v: dict = field(default_factory=dict)
    steps: int = 0             # optimiser steps taken
    ret_ms: object = None      # RunningMeanStdRef(shape=(n_agents,)) when cfg.standardise_returns (ac/model.py:112-114), else None
    centralised: bool = False  # critic.centralised (ac/model.py:62-65,156-157): every agent's critic reads the concatenated observations

    def critic_inputs(self, obs):
        """get_value's inputs: the per-agent list, or n_agents x the concatenation (and the matching input width)"""
        if not self.centralised:
            return obs, self.in_dim
        return len(obs) * [torch.cat(obs, dim=-1)], len(obs) * self.in_dim

    def __post_init__(self):
        for k in ("actor", "critic"):
            self.m.setdefault(k, torch.zeros_like(getattr(self, k)))
            self.v.setdefault(k, torch.zeros_like(getattr(self, k)))


def a2c_losses(actor, critic, target, st: A2CState, batch, hp: A2CHP):
    """batch = dict(obss (T+1,P,N*D), actions (T,P,N) i64, rewards (T,P,N), dones (T+1,P) f32/bool, filled (T,P))"""
    N, D = len(st.actor_net), st.in_dim
    obs = list(torch.split(batch["obss"], D, dim=-1))
    cobs, CD = st.critic_inputs(obs)
    with torch.no_grad():
        next_value = torch.cat(agents_forward(target, st.critic_net, cobs, CD, 1), dim=-1)                # (T+1,P,N)
    if st.ret_ms is not None:                                                                             # ac/model.py:195-196
        next_value = next_value * torch.sqrt(st.ret_ms.var) + st.ret_ms.mean
    done = batch["dones"].float().unsqueeze(-1).repeat(1, 1, N)
    returns = nstep_returns(batch["rewards"], done, next_value, hp.n_steps, hp.gamma)
    if st.ret_ms is not None:                                                                             # ac/model.py:202-204
        st.ret_ms.update(returns)
        returns = (returns - st.ret_ms.mean) / torch.sqrt(st.ret_ms.var)
    obs_t = [o[:-1] for o in obs]
    values = torch.cat(agents_forward(critic, st.critic_net, [o[:-1] for o in cobs], CD, 1), dim=-1)     # (T,P,N)
    logits = agents_forward(actor, st.actor_net, obs_t, D, st.n_actions)
    logp_all = [F.log_softmax(l, dim=-1) for l in logits]
    acts = batch["actions"]
    logp = torch.cat([lp.gather(-1, acts[..., i:i + 1]) for i, lp in enumerate(logp_all)], dim=-1)     # (T,P,N)
    entropy = torch.stack([-(lp.exp() * lp).sum(-1) for lp in logp_all], dim=-1).sum(-1)                 # (T,P)
    adv = returns - values
    filled = batch["filled"]
    actor_loss = ((-(logp * adv.detach()).sum(-1) - hp.entropy_coef * entropy) * filled).sum() / filled.sum()
    value_loss = ((returns - values).pow(2).sum(-1) * filled).sum() / filled.sum()
    ent = (entropy * filled).sum() / filled.sum()
    return actor_loss, value_loss, ent, returns


def ppo_update(st: A2CState, batch, hp: A2CHP, step: int, num_epochs: int = 4, ppo_clip: float = 0.2):
    """PPONetwork.update (ac/model.py:265-352): returns and the collecting policy's log-probabilities once, then num_epochs steps on the clipped
    surrogate; target critic after the last epoch; the metrics are the epochs' means.  Returns also the first epoch's raw gradients."""
    N, D = len(st.actor_net), st.in_dim
    obs = list(torch.split(batch["obss"], D, dim=-1))
    obs_t = [o[:-1] for o in obs]
    acts, filled = batch["actions"], batch["filled"]
    cobs, CD = st.critic_inputs(obs)
    cobs_t = [o[:-1] for o in cobs]
    with torch.no_grad():
        next_value = torch.cat(agents_forward(st.target, st.critic_net, cobs, CD, 1), dim=-1)
        if st.ret_ms is not None:                                                                         # ac/model.py:272-273
            next_value = next_value * torch.sqrt(st.ret_ms.var) + st.ret_ms.mean
        done = batch["dones"].float().unsqueeze(-1).repeat(1, 1, N)
        returns = nstep_returns(batch["rewards"], done, next_value, hp.n_steps, hp.gamma)
        if st.ret_ms is not None:                                                                         # ac/model.py:279-281
            st.ret_ms.update(returns)
            returns = (returns - st.ret_ms.mean) / torch.sqrt(st.ret_ms.var)
        old = [F.log_softmax(l, dim=-1) for l in agents_forward(st.actor, st.actor_net, obs_t, D, st.n_actions)]
        old_logp = torch.cat([lp.gather(-1, acts[..., i:i + 1]) for i, lp in enumerate(old)], dim=-1)
    out = dict(loss=[], actor_loss=[], value_loss=[], entropy=[])
    first = None
    for _ in range(num_epochs):
        actor = st.actor.clone().requires_grad_(True)
        critic = st.critic.clone().requires_grad_(True)
        values = torch.cat(agents_forward(critic, st.critic_net, cobs_t, CD, 1), dim=-1)
        logp_all = [F.log_softmax(l, dim=-1) for l in agents_forward(actor, st.actor_net, obs_t, D, st.n_actions)]
        logp = torch.cat([lp.gather(-1, acts[..., i:i + 1]) for i, lp in enumerate(logp_all)], dim=-1)
        entropy = torch.stack([-(lp.exp() * lp).sum(-1) for lp in logp_all], dim=-1).sum(-1)
        adv = returns - values
        value_loss = adv.pow(2).sum(-1)
        ratio = torch.exp(logp - old_logp)
        surr1, surr2 = ratio * adv.detach(), torch.clamp(ratio, 1.0 - ppo_clip, 1.0 + ppo_clip) * adv.detach()
        actor_loss = -torch.min(surr1, surr2).sum(-1) - hp.entropy_coef * entropy
        actor_loss = (actor_loss * filled).sum() / filled.sum()
        value_loss = (value_loss * filled).sum() / filled.sum()
        loss = actor_loss + hp.value_loss_coef * value_loss
        g_actor, g_critic = torch.autograd.grad(loss, (actor, critic))
        if first is None:
            first = dict(actor=g_actor.clone(), critic=g_critic.clone())
        if hp.grad_clip:
            total = torch.linalg.vector_norm(torch.cat([g_actor, g_critic]))
            coef = torch.clamp(hp.grad_clip / (total + 1e-6), max=1.0)
            g_actor, g_critic = g_actor * coef, g_critic * coef
        st.steps += 1
        adam_step(st.actor, st.m["actor"], st.v["actor"], g_actor, st.steps, hp.lr)
        adam_step(st.critic, st.m["critic"], st.v["critic"], g_critic, st.steps, hp.lr)
        for k, v in (("loss", loss), ("actor_loss", actor_loss), ("value_loss", value_loss), ("entropy", (entropy * filled).sum() / filled.sum())):
            out[k].append(float(v.detach()))
    tu = hp.target_update_interval_or_tau
    if tu > 1.0 and step % tu == 0:
        st.target.copy_(st.critic)
    elif tu < 1.0:
        st.target.copy_((1 - tu) * st.target + tu * st.critic)
    res = {k: sum(v) / len(v) for k, v in out.items()}
    res.update(grad=first, returns=returns, per_epoch=out)
    return res


def a2c_update(st: A2CState, batch, hp: A2CHP, step: int):
    actor = st.actor.clone().requires_grad_(True)
    critic = st.critic.clone().requires_grad_(True)
    actor_loss, value_loss, ent, returns = a2c_losses(actor, critic, st.target, st, batch, hp)
    loss = actor_loss + hp.value_loss_coef * value_loss
    g_actor, g_critic = torch.autograd.grad(loss, (actor, critic))
    raw = dict(actor=g_actor.clone(), critic=g_critic.clone())
    if hp.grad_clip:
        total = torch.linalg.vector_norm(torch.cat([g_actor, g_critic]))
        coef = torch.clamp(hp.grad_clip / (total + 1e-6), max=1.0)
        g_actor, g_critic = g_actor * coef, g_critic * coef
    st.steps += 1
    adam_step(st.actor, st.m["actor"], st.v["actor"], g_actor, st.steps, hp.lr)
    adam_step(st.critic, st.m["critic"], st.v["critic"], g_critic, st.steps, hp.lr)
    tu = hp.target_update_interval_or_tau
    if tu > 1.0 and step % tu == 0:
        st.target.copy_(st.critic)
    elif tu < 1.0:
        st.target.copy_((1 - tu) * st.target + tu * st.critic)
    return dict(loss=float(loss.detach()), actor_loss=float(actor_loss.detach()), value_loss=float(value_loss.detach()), entropy=float(ent.detach()), grad=raw, returns=returns.detach(),
                grad_clipped=dict(actor=g_actor.detach().clone(), critic=g_critic.detach().clone()))
