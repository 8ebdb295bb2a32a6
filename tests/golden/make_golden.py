"""Generates the learner fixtures under tests/golden/ from the LIVE reference learner classes of a marlbase checkout.
Run:  MARLBASE_SRC=<directory holding marlbase/> python tests/golden/make_golden.py
Every fixture stores the inputs in the device ("trajectory store") layout plus the reference's outputs, so that both
the CPU oracle (oracle/learner_ref.py) and the CUDA path are checked against numbers the reference itself produced."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import learner_ref as lr  # noqa: E402
from oracle import ref_shim  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
N, D, A, T = 2, 15, 6, 25
# fixed integers: Python's hash() of a str is salted per process, which made the fixtures irreproducible
SEEDS = {"idqn_indep": 101, "idqn_single_q_polyak_noclip": 202, "idqn_shared": 303, "vdn_indep": 404, "ia2c_indep": 505, "ia2c_shared": 606}


def optimizer_state_flat(model, module_name, prefix, n_nets, key):
    """Adam's exp_avg / exp_avg_sq of one sub-module as a flat vector in the device layout (zeros where a parameter never got a gradient)."""
    mod = getattr(model, module_name)
    sd = {}
    for k, p in mod.named_parameters():
        st = model.optimizer.state.get(p, {})
        sd[f"{module_name}.{k}"] = st[key].detach().clone() if key in st else torch.zeros_like(p)
    return lr.flat_from_state_dict(sd, prefix, n_nets).numpy()


def grads_flat(model, module_name, prefix, n_nets):
    mod = getattr(model, module_name)
    sd = {f"{module_name}.{k}": (p.grad.detach().clone() if p.grad is not None else torch.zeros_like(p)) for k, p in mod.named_parameters()}
    return lr.flat_from_state_dict(sd, prefix, n_nets).numpy()


def random_store(rng, cap, n_agents=N):
    """Synthetic episodes with LBF-like value ranges, ragged lengths and terminal flags."""
    obs = rng.integers(-1, 8, size=(cap, n_agents, T + 1, D)).astype(np.float32)
    act = rng.integers(0, A, size=(cap, n_agents, T)).astype(np.int32)
    rew = (rng.random((cap, n_agents, T)) < 0.1).astype(np.float32) * rng.random((cap, n_agents, T)).astype(np.float32)
    length = rng.integers(3, T + 1, size=cap)
    done = np.zeros((cap, T + 1), np.uint8)
    filled = np.zeros((cap, T), np.uint8)
    for e in range(cap):
        filled[e, : length[e]] = 1
        done[e, length[e]] = 1
    return dict(obs=obs, act=act, rew=rew, done=done, filled=filled)


def to_ref_batch(mod, store, idx):
    b = lr.batch_from_store(store, idx)
    return mod.Batch(b["obss"], b["actions"], b["rewards"], b["dones"], b["filled"], None)


def dqn_case(name, cls_name, sharing, n_updates=3, B=8, **cfgkw):
    ref = ref_shim.load()
    torch.manual_seed(SEEDS[name])
    rng = np.random.default_rng(SEEDS[name])
    spaces_o = [ref_shim.Space(shape=(D,)) for _ in range(N)]
    spaces_a = [ref_shim.Space(n=A) for _ in range(N)]
    model = getattr(ref.dqn_model, cls_name)(spaces_o, spaces_a, ref_shim.dqn_cfg(**cfgkw), [128, 128], sharing, False, True, "cpu")
    n_nets = 1 if sharing else N
    prefix = "critic.networks" if sharing else "critic.independent"
    theta0 = lr.flat_from_state_dict(model.state_dict(), prefix, n_nets)
    out = dict(theta0=theta0.numpy(), n_nets=n_nets, agent_net=np.array([0] * N if sharing else list(range(N))),
               mixer=int(cls_name == "VDNetwork"), hp=np.array([cfgkw.get("lr", 3e-4), cfgkw.get("gamma", 0.99), float(cfgkw.get("grad_clip", 1.0) or 0.0),
                                                            float(cfgkw.get("double_q", True)), cfgkw.get("target_update_interval_or_tau", 200)], np.float64))
    losses = []
    for u in range(n_updates):
        store = random_store(rng, 16)
        idx = rng.integers(0, 16, size=B).astype(np.int32)
        for k, v in store.items():
            out[f"u{u}_{k}"] = v
        out[f"u{u}_idx"] = idx
        if cls_name == "VDNetwork":  # cooperative reward: all agents carry the same reward
            store["rew"][:] = store["rew"][:, :1]
            out[f"u{u}_rew"] = store["rew"]
        batch = to_ref_batch(ref.dqn_train, store, idx)
        model.optimizer.zero_grad()
        loss = model._compute_loss(batch)
        loss.backward()
        if u == 0:
            sd_grad = {k: p.grad for k, p in model.critic.named_parameters()}
            sd_grad = {f"critic.{k}": v for k, v in sd_grad.items()}
            out["grad0"] = lr.flat_from_state_dict(sd_grad, prefix, n_nets).numpy()
        losses.append(model.update(batch)["loss"])
        if u == 0:  # update() clips in place before optimizer.step(): p.grad now holds what Adam consumed
            out["grad0_clipped"] = grads_flat(model, "critic", prefix, n_nets)
    out["adam_m_final"] = optimizer_state_flat(model, "critic", prefix, n_nets, "exp_avg")
    out["adam_v_final"] = optimizer_state_flat(model, "critic", prefix, n_nets, "exp_avg_sq")
    out["losses"] = np.array(losses, np.float64)
    sd = model.state_dict()
    out["theta_final"] = lr.flat_from_state_dict(sd, prefix, n_nets).numpy()
    out["target_final"] = lr.flat_from_state_dict(sd, prefix.replace("critic", "target"), n_nets).numpy()
    np.savez_compressed(os.path.join(OUT, f"{name}.npz"), **out)
    print(name, losses)


def a2c_case(name, sharing, n_updates=2, P=6, **cfgkw):
    ref = ref_shim.load()
    torch.manual_seed(SEEDS[name])
    rng = np.random.default_rng(SEEDS[name])
    spaces_o = [ref_shim.Space(shape=(D,)) for _ in range(N)]
    spaces_a = [ref_shim.Space(n=A) for _ in range(N)]
    cfg = ref_shim.a2c_cfg(**cfgkw)
    model = ref.ac_model.A2CNetwork(spaces_o, spaces_a, cfg, ref_shim.net_cfg(sharing), ref_shim.net_cfg(sharing), "cpu")
    n_nets = 1 if sharing else N
    kind = "networks" if sharing else "independent"
    sd = model.state_dict()
    out = dict(actor0=lr.flat_from_state_dict(sd, f"actor.{kind}", n_nets).numpy(), critic0=lr.flat_from_state_dict(sd, f"critic.{kind}", n_nets).numpy(),
               target0=lr.flat_from_state_dict(sd, f"target_critic.{kind}", n_nets).numpy(), n_nets=n_nets,
               agent_net=np.array([0] * N if sharing else list(range(N))),
               hp=np.array([cfg.lr, cfg.gamma, float(cfg.grad_clip or 0.0), cfg.n_steps, cfg.entropy_coef, cfg.value_loss_coef, cfg.target_update_interval_or_tau], np.float64))
    metrics = []
    steps = [0, 150]  # step % 200 == 0 on the first update -> exercises the target sync branch
    for u in range(n_updates):
        store = random_store(rng, P)
        for k, v in store.items():
            out[f"u{u}_{k}"] = v
        batch = ref.ac_model  # noqa
        t = {k: torch.as_tensor(v) for k, v in store.items()}
        obss = t["obs"].permute(2, 0, 1, 3).reshape(T + 1, P, N * D).float()
        b = ref.dqn_train.Batch  # placeholder to keep flake quiet
        from collections import namedtuple
        AB = namedtuple("Batch", ["obss", "actions", "rewards", "dones", "filled", "action_masks"])
        acb = AB(obss, t["act"].permute(2, 0, 1).long(), t["rew"].permute(2, 0, 1).float(), t["done"].permute(1, 0).bool(), t["filled"].permute(1, 0).float(), None)
        if u == 0:
            with torch.no_grad():
                nv, _ = model.get_value(model.split_obs(acb.obss), None, target=True)
            done = acb.dones.float().unsqueeze(-1).repeat(1, 1, N)
            out["returns0"] = ref.utils.compute_nstep_returns(acb.rewards, done, nv, cfg.n_steps, cfg.gamma).numpy()
        m = model.update(acb, steps[u])
        if u == 0:
            out["actor_grad0_clipped"] = grads_flat(model, "actor", f"actor.{kind}", n_nets)
            out["critic_grad0_clipped"] = grads_flat(model, "critic", f"critic.{kind}", n_nets)
        metrics.append([m["loss"], m["actor_loss"], m["value_loss"], m["entropy"]])
    for mod in ("actor", "critic"):
        out[f"{mod}_adam_m_final"] = optimizer_state_flat(model, mod, f"{mod}.{kind}", n_nets, "exp_avg")
        out[f"{mod}_adam_v_final"] = optimizer_state_flat(model, mod, f"{mod}.{kind}", n_nets, "exp_avg_sq")
    out["metrics"] = np.array(metrics, np.float64)
    out["steps"] = np.array(steps[:n_updates])
    sd = model.state_dict()
    out["actor_final"] = lr.flat_from_state_dict(sd, f"actor.{kind}", n_nets).numpy()
    out["critic_final"] = lr.flat_from_state_dict(sd, f"critic.{kind}", n_nets).numpy()
    out["target_final"] = lr.flat_from_state_dict(sd, f"target_critic.{kind}", n_nets).numpy()
    np.savez_compressed(os.path.join(OUT, f"{name}.npz"), **out)
    print(name, metrics)


def misc_case():
    ref = ref_shim.load()
    steps = np.array([0, 1, 999, 25000, 49999, 50000, 80000, 100000])
    lin = ref.dqn_train._epsilon_schedule("linear", 0.5, 1.0, 0.05, 6.5, 100000)
    exp = ref.dqn_train._epsilon_schedule("exponential", 0.5, 1.0, 0.05, 6.5, 100000)
    rng = np.random.default_rng(0)
    rew = torch.tensor(rng.random((25, 4, 2)), dtype=torch.float32)
    done = torch.tensor(rng.random((26, 4, 2)) < 0.1, dtype=torch.float32)
    nv = torch.tensor(rng.standard_normal((26, 4, 2)), dtype=torch.float32)
    out = dict(steps=steps, eps_linear=np.array([lin(int(s)) for s in steps]), eps_exp=np.array([exp(int(s)) for s in steps]),
               ns_rew=rew.numpy(), ns_done=done.numpy(), ns_nv=nv.numpy())
    for n in (1, 5, 30):
        out[f"ns_ret_{n}"] = ref.utils.compute_nstep_returns(rew, done, nv, n, 0.99).numpy()
    np.savez_compressed(os.path.join(OUT, "misc.npz"), **out)


if __name__ == "__main__":
    dqn_case("idqn_indep", "QNetwork", False, target_update_interval_or_tau=2)
    dqn_case("idqn_single_q_polyak_noclip", "QNetwork", False, double_q=False, grad_clip=False, target_update_interval_or_tau=0.05)
    dqn_case("idqn_shared", "QNetwork", True, target_update_interval_or_tau=2)
    dqn_case("vdn_indep", "VDNetwork", False, target_update_interval_or_tau=2)
    a2c_case("ia2c_indep", False)
    a2c_case("ia2c_shared", True, grad_clip=0.5)
    misc_case()
