"""CPU restatement (PyTorch float32, autograd) of the reference's QMIX learner.  TEST INFRASTRUCTURE ONLY.

Restated from (path:line under /root/reference/marlbase):
  dqn/model.py:272-340   QMixer: hypernetworks |W1(s)|, b1(s), |w_final(s)|, V(s); Q_tot = elu(q W1 + b1) w_final + V
  dqn/model.py:343-384   QMixNetwork.__init__: state = the agents' observations concatenated, one Adam over critic + mixer
  dqn/model.py:386-443   _compute_loss (double-Q target per agent, target mixer on the next state, rewards[0]) and soft / hard updates of the mixer
  dqn/model.py:165-174   update: clip_grad_norm_ over the CRITIC's parameters only, then the shared Adam step

The mixer's parameters are one flat vector in the reference's state_dict order (hypernet_layers == 2):
  hyper_w_1.0.{weight [He,S], bias [He]}, hyper_w_1.2.{weight [N*E,He], bias [N*E]}, hyper_w_final.0.{weight [He,S], bias [He]},
  hyper_w_final.2.{weight [E,He], bias [E]}, hyper_b_1.{weight [E,S], bias [E]}, V.0.{weight [E,S], bias [E]}, V.2.{weight [1,E], bias [1]}
Pinned by tests/test_qmix.py against outputs of the live reference classes recorded under tests/golden/ (ref_qmix.npz, qmix_indep.npz).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch
import torch.nn.functional as F

from . import learner_ref as lr

MIXER_KEYS = ("hyper_w_1.0", "hyper_w_1.2", "hyper_w_final.0", "hyper_w_final.2", "hyper_b_1", "V.0", "V.2")


def mixer_shapes(n_agents, state_dim, embed_dim, hypernet_embed):
    N, S, E, He = n_agents, state_dim, embed_dim, hypernet_embed
    return ((He, S), (N * E, He), (He, S), (E, He), (E, S), (E, S), (1, E))


def mixer_size(n_agents, state_dim, embed_dim, hypernet_embed):
    return sum(o * i + o for o, i in mixer_shapes(n_agents, state_dim, embed_dim, hypernet_embed))


def split_mixer(flat, n_agents, state_dim, embed_dim, hypernet_embed):
    out, o = [], 0
    for (no, ni) in mixer_shapes(n_agents, state_dim, embed_dim, hypernet_embed):
        out.append(flat[o:o + no * ni].view(no, ni)); o += no * ni
        out.append(flat[o:o + no]); o += no
    return out


def mixer_flat_from_state_dict(sd, prefix="mixer"):
    return torch.cat([sd[f"{prefix}.{k}.{p}"].reshape(-1) for k in MIXER_KEYS for p in ("weight", "bias")]).clone().float()


def mixer_state_dict_from_flat(flat, prefix, n_agents, state_dim, embed_dim, hypernet_embed):
    parts = split_mixer(flat, n_agents, state_dim, embed_dim, hypernet_embed)
    sd = {}
    for j, k in enumerate(MIXER_KEYS):
        sd[f"{prefix}.{k}.weight"] = parts[2 * j].clone(); sd[f"{prefix}.{k}.bias"] = parts[2 * j + 1].clone()
    return sd


def init_mixer_flat(n_agents, state_dim, embed_dim, hypernet_embed):
    """QMixer builds plain nn.Linear layers (PyTorch's default initialisation, no orthogonal init), in this order."""
    parts = []
    for (no, ni) in mixer_shapes(n_agents, state_dim, embed_dim, hypernet_embed):
        lin = torch.nn.Linear(ni, no)
        parts += [lin.weight.data.reshape(-1), lin.bias.data.reshape(-1)]
    return torch.cat(parts).float()


def mixer_forward(flat, agent_qs, states, n_agents, embed_dim, hypernet_embed):
    """agent_qs (N, T, B), states (T, B, S) -> Q_tot (T, B)   (dqn/model.py:314-340)"""
    N, T, B = agent_qs.shape
    S = states.shape[-1]
    w1a, b1a, w1b, b1b, wfa, bfa, wfb, bfb, wb, bb, wva, bva, wvb, bvb = split_mixer(flat, n_agents, S, embed_dim, hypernet_embed)
    qs = agent_qs.permute(1, 2, 0).reshape(T * B, 1, N)
    x = states.reshape(-1, S)
    w1 = torch.abs(F.linear(F.relu(F.linear(x, w1a, b1a)), w1b, b1b)).view(-1, N, embed_dim)
    b1 = F.linear(x, wb, bb).view(-1, 1, embed_dim)
    hidden = F.elu(torch.bmm(qs, w1) + b1)
    wf = torch.abs(F.linear(F.relu(F.linear(x, wfa, bfa)), wfb, bfb)).view(-1, embed_dim, 1)
    v = F.linear(F.relu(F.linear(x, wva, bva)), wvb, bvb).view(-1, 1, 1)
    return (torch.bmm(hidden, wf) + v).view(T, B)


@dataclass
class QmixState:
    theta: torch.Tensor        # agents' networks, device layout of learner_ref
    theta_tgt: torch.Tensor
    mix: torch.Tensor
    mix_tgt: torch.Tensor
    agent_net: list
    in_dim: int
    out_dim: int
    embed_dim: int = 64
    hypernet_embed: int = 32
    m: torch.Tensor = None
    v: torch.Tensor = None
    mix_m: torch.Tensor = None
    mix_v: torch.Tensor = None
    updates: int = 0
    last_target_update: int = 0

    def __post_init__(self):
        for name, ref in (("m", self.theta), ("v", self.theta), ("mix_m", self.mix), ("mix_v", self.mix)):
            if getattr(self, name) is None:
                setattr(self, name, torch.zeros_like(ref))


def qmix_loss(theta, mix, st: QmixState, batch, hp: lr.DqnHP):
    obss, actions, rewards, dones, filled = (batch[k] for k in ("obss", "actions", "rewards", "dones", "filled"))
    N = obss.shape[0]
    q = torch.stack(lr.agents_forward(theta, st.agent_net, list(obss), st.in_dim, st.out_dim))            # (N, T+1, B, A)
    chosen = q[:, :-1].gather(-1, actions.unsqueeze(-1)).squeeze(-1)
    chosen = mixer_forward(mix, chosen, torch.concat(list(obss[:, :-1]), dim=-1), N, st.embed_dim, st.hypernet_embed)
    with torch.no_grad():
        tq = torch.stack(lr.agents_forward(st.theta_tgt, st.agent_net, list(obss), st.in_dim, st.out_dim))[:, 1:]
        if hp.double_q:
            target = tq.gather(-1, q.detach()[:, 1:].argmax(-1, keepdim=True)).squeeze(-1)
        else:
            target = tq.max(-1)[0]
        target = mixer_forward(st.mix_tgt, target, torch.concat(list(obss[:, 1:]), dim=-1), N, st.embed_dim, st.hypernet_embed)
    returns = rewards[0] + hp.gamma * target * (1 - dones[1:])
    loss = (chosen - returns.detach()) ** 2
    return (loss * filled).sum() / filled.sum()


def qmix_update(st: QmixState, batch, hp: lr.DqnHP):
    """QMixNetwork.update: returns dict(loss, grad / mix_grad (before clipping), grad_norm of the critic part)."""
    theta = st.theta.clone().requires_grad_(True)
    mix = st.mix.clone().requires_grad_(True)
    loss = qmix_loss(theta, mix, st, batch, hp)
    grad, mgrad = torch.autograd.grad(loss, (theta, mix))
    raw, mraw = grad.clone(), mgrad.clone()
    norm = torch.linalg.vector_norm(grad)
    if hp.grad_clip:                                  # the critic's parameters only (dqn/model.py:169-170)
        coef, norm = lr.clip_coef(grad, hp.grad_clip)
        grad = grad * coef
    st.updates += 1
    lr.adam_step(st.theta, st.m, st.v, grad, st.updates, hp.lr)
    lr.adam_step(st.mix, st.mix_m, st.mix_v, mgrad, st.updates, hp.lr)
    tu = hp.target_update_interval_or_tau
    if tu > 1.0 and (st.updates - st.last_target_update) >= tu:
        st.theta_tgt.copy_(st.theta); st.mix_tgt.copy_(st.mix)
        st.last_target_update = st.updates
    elif tu < 1.0:
        st.theta_tgt.copy_((1 - tu) * st.theta_tgt + tu * st.theta)
        st.mix_tgt.copy_((1 - tu) * st.mix_tgt + tu * st.mix)
    return dict(loss=float(loss.detach()), grad=raw, mix_grad=mraw, grad_norm=float(norm))


def qmix_kink_risk(st: QmixState, batch, hp: lr.DqnHP):
    """Largest gradient move a ReLU unit of the AGENT networks at its kink could cause (learner_ref.kink_risk), through the mixer."""
    return lr.kink_risk(lambda th: qmix_loss(th, st.mix, st, batch, hp), st.theta)


def random_batch(N, T, B, D, A, seed=0, ragged=True):
    g = torch.Generator().manual_seed(seed)
    obss = torch.randn(N, T + 1, B, D, generator=g)
    actions = torch.randint(0, A, (N, T, B), generator=g)
    rew = torch.randn(1, T, B, generator=g).repeat(N, 1, 1)
    dones = torch.zeros(T + 1, B); filled = torch.ones(T, B)
    if ragged:
        for b in range(B):
            L = int(torch.randint(1, T + 1, (1,), generator=g))
            dones[L:, b] = 1.0; filled[L:, b] = 0.0
    return dict(obss=obss, actions=actions, rewards=rew, dones=dones, filled=filled)
