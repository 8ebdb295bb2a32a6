#!/usr/bin/env python
"""bench.py -- env-steps/sec of the marlbase hot path on B200 (BASELINE.json metric) next to the CPU reference loop.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config idqn|vdn15|ia2c] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Default workload (`--config idqn`) = BASELINE.json configs[1], the configuration the metric is quoted on: IDQN on
Foraging-8x8-2p-3f-v3, 4096 envs per GPU, batch_size 1024.  A "step" is one training iteration of the hot path on every GPU: E envs
collect one episode each (<= 25 env steps; fused forward + epsilon-greedy + transition + replay write per env step) followed by
`updates_per_iteration` updates (replay sample + target forward + forward/TD/backward + reduce + clip/Adam/target), default E updates =
the reference's one update per collected episode (marlbase/dqn/train.py:299-311).  `value` counts real env transitions (sum of episode
lengths) per second with the whole loop device resident; `e2e` runs the same iteration with every env step's observations / rewards /
flags crossing pinned HOST buffers (the gym-style plugin boundary), copies inside the timed region.
`--config vdn15` = configs[3] (VDN, Foraging-15x15-4p-5f-v3, 4096 envs/GPU, CooperativeReward); `--config ia2c` = configs[2] (IA2C, full
parameter sharing, 8192 envs, n_steps 5: one update per vector rollout, marlbase/ac/train.py:170-204).  Same JSON contract for all three.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

TIME_LIMIT = 25
HIDDEN = 128
WORKLOADS = {
    "idqn": dict(algo="idqn", baseline_config=1, env="lbforaging:Foraging-8x8-2p-3f-v3", lbf=dict(rows=8, cols=8, n_agents=2, max_num_food=3, sight=8),
                 envs=4096, batch=1024, buffer=65536, wrappers=None),
    "vdn15": dict(algo="vdn", baseline_config=3, env="lbforaging:Foraging-15x15-4p-5f-v3", lbf=dict(rows=15, cols=15, n_agents=4, max_num_food=5, sight=15, cooperative_reward=1),
                  envs=4096, batch=1024, buffer=32768, wrappers=["CooperativeReward"]),
    "ia2c": dict(algo="ia2c", baseline_config=2, env="lbforaging:Foraging-8x8-2p-3f-v3", lbf=dict(rows=8, cols=8, n_agents=2, max_num_food=3, sight=8),
                 envs=8192, batch=0, buffer=0, wrappers=None),
}
# dram__bytes_read.sum + dram__bytes_write.sum of one launch of the idqn workload: ncu --set full, one kernel at a time with ncu's cache flush in
# front (cold L2; profiles/r1_tc_pipeline.md).  The warm, pipelined figure of the whole update is in profiles/r2_dram_traffic.md.
TRAFFIC_NCU = {"tc_dqn_fwd_kernel": 9303552, "tc_dh1_kernel": 3705344, "tc_dw_kernel": 92672512,
               # on-chip pass (round 2): dram__bytes of one launch inside the running pipeline (ncu --cache-control none, profiles/r2_dram_traffic.md)
               "tc_dqn_fwd3_kernel": 4300000, "tc_dh1w1_kernel": 10300000, "tc_dw2_kernel": 10300000}
DUMP_EPISODES = 1024   # --dump-outputs: episodes of the last step kept (a fixed, seeded sample), so that the files stay small at any --envs


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="idqn", choices=sorted(WORKLOADS), help="idqn = BASELINE configs[1] (default, what the driver runs), vdn15 = configs[3], ia2c = configs[2]")
    ap.add_argument("--envs", type=int, default=0, help="env instances per GPU (0 = the workload's value)")
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--buffer", type=int, default=0, help="replay ring capacity in episodes (per GPU)")
    ap.add_argument("--updates-per-iter", type=int, default=0, help="0 = one update per collected episode (= --envs)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--collective", default="peer", choices=["peer", "nccl"],
                    help="N > 1: gradient exchange inside the fused reduce + Adam kernel over NVLink peer memory (default), or one NCCL all-reduce per update")
    ap.add_argument("--tc-backward", type=int, default=1, help="1 = tcgen05 training pipeline (default), 0 = fused FP32 FFMA training kernel")
    ap.add_argument("--tc-onchip", type=int, default=1, help="1 = training pass with H1 / H2 / dH1 kept on chip (tc_train3.cu, default), 0 = streamed through global memory (tc_train.cu)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32): parameters, target parameters, update "
                         f"metrics, every env's episode length and return, and a fixed sample of at most {DUMP_EPISODES} of the episodes it collected")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")
    wl = WORKLOADS[a.config]
    a.envs = a.envs or wl["envs"]
    a.batch = a.batch or wl["batch"]
    a.buffer = a.buffer or wl["buffer"]
    return a


def dims(wl):
    n, f = wl["lbf"]["n_agents"], wl["lbf"]["max_num_food"]
    return n, 3 * f + 3 * n, 6   # agents, observation width, actions


def fwd_flop_per_row(obs_dim, out):
    return 2 * (obs_dim * HIDDEN + HIDDEN * HIDDEN + HIDDEN * out)   # 38 144 at 8x8-2p-3f with 6 outputs (SURVEY section 8d)


# ---- clocks ------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(gpu_index)],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush(); self.f.seek(0)
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2])); power.append(float(parts[3]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


# ---- reference arm: the CPU loop on all host cores this process may use -------------------------------------------------------
def host_cores():
    try:
        return len(os.sched_getaffinity(0))   # the cores this process may run on (cgroup / taskset aware), not the machine's count
    except AttributeError:
        return os.cpu_count() or 1


def plan_a(args, seconds=120.0):
    """BASELINE.md section 3, Plan A: the reference AS SHIPPED (run.py + lbforaging + gymnasium + hydra).  Returns (dict | None, why-not)."""
    try:
        import gymnasium  # noqa: F401
        import hydra  # noqa: F401
        import lbforaging  # noqa: F401
        import omegaconf  # noqa: F401
    except Exception as e:  # noqa: BLE001
        return None, f"{type(e).__name__}: {e}"
    marlbase = os.path.join(ROOT, "baseline", "_ref", "marlbase")   # a driver-provided install; /root/reference does not exist on the GPU box
    if not os.path.exists(os.path.join(marlbase, "run.py")):
        return None, "third-party packages import, but no marlbase/run.py under baseline/_ref"
    wl = WORKLOADS[args.config]
    if wl["algo"] not in ("idqn", "vdn"):
        return None, "Plan A is wired for the DQN-family configs only"
    out = tempfile.mkdtemp(prefix="plan_a_")
    cmd = [sys.executable, "run.py", f"+algorithm={wl['algo']}", f"env.name={wl['env']}", f"env.time_limit={TIME_LIMIT}", f"algorithm.batch_size={args.batch}",
           "seed=0", "algorithm.total_steps=100000000", "algorithm.eval_interval=2000", "algorithm.log_interval=2000", f"hydra.run.dir={out}"]
    t0 = time.perf_counter()
    p = subprocess.Popen(cmd, cwd=marlbase, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    try:
        p.wait(timeout=seconds)
    except subprocess.TimeoutExpired:
        p.terminate(); p.wait()
    wall = time.perf_counter() - t0
    try:
        import pandas as pd

        df = pd.read_csv(os.path.join(out, "results.csv"))
        steps = float(df["environment_steps"].iloc[-1])
    except Exception as e:  # noqa: BLE001
        return None, f"run.py produced no results.csv ({type(e).__name__})"
    return {"value": steps / wall, "unit": "env-steps/s", "cores": 1, "kind": "reference",
            "sample": f"marlbase/run.py as shipped for {wall:.0f} s (1 torch thread, run.py:29); last logged environment_steps / wall clock"}, ""


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import cpu_loop

    wl = WORKLOADS[args.config]
    cores = host_cores()
    got, why_not = plan_a(args)
    # Plan B: `cores` independent single-thread copies of the restated reference loop; each "step" = every copy runs `eps` iterations, the
    # step ends when the slowest copy is done, and the step's wall clock (the parent's, around the whole pool) is what is reported
    eps = 3 if wl["algo"] != "ia2c" else 1
    pool = cpu_loop.WorkerPool(cores, dict(algo=wl["algo"], lbf=wl["lbf"], time_limit=TIME_LIMIT, batch=args.batch or 128, prefill=args.batch or 0))
    t_run0 = time.perf_counter()
    rounds = [pool.run_round(eps) for _ in range(args.warmup + args.steps)]
    pool.close()
    timed = rounds[args.warmup:]
    steps = sum(r[0] for r in timed)
    secs = sum(r[1] for r in timed)
    value = steps / secs
    what = ("one 25-step episode with one env + one update at batch_size=%d" % args.batch) if wl["algo"] != "ia2c" else "one 10-env vector rollout + one A2C update (ia2c.yaml: parallel_envs 10)"
    line = {
        "impl": "reference", "metric": "env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * secs / max(args.steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, 1),
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port",
                         "sample": f"{cores} independent single-thread copies (torch.set_num_threads(1), marlbase/run.py:29) of the restated reference loop on the cores of "
                                   f"os.sched_getaffinity; per step every copy runs {eps} x ({what}) and the step ends with the slowest copy; pure-Python LBF restatement + "
                                   f"PyTorch-CPU learner; pool wall clock {time.perf_counter() - t_run0:.1f} s",
                         "per_copy_env_steps_per_s": value / cores, "plan_a": got if got is not None else f"unavailable: {why_not}"},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def workload_config(args, world):
    wl = WORKLOADS[args.config]
    n_agents, obs_dim, _ = dims(wl)
    if wl["algo"] == "ia2c":
        return {"workload": f"IA2C (full parameter sharing, n_steps=5) {wl['env']} time_limit={TIME_LIMIT}, {args.envs} vectorised envs/GPU, one update per vector rollout "
                            f"(BASELINE.json configs[{wl['baseline_config']}])",
                "envs_per_gpu": args.envs, "parallelism": f"dp{world}" if world > 1 else "single",
                "collective": "one NCCL all-reduce of the gradient buffer per update" if world > 1 else None,
                "l2": "inputs larger than L2: every iteration rewrites and re-reads a %.0f MB on-policy batch" % (args.envs * n_agents * (TIME_LIMIT + 1) * obs_dim * 4 / 1e6)}
    upi = args.updates_per_iter or args.envs
    ep_bytes = n_agents * ((TIME_LIMIT + 1) * obs_dim * 4 + TIME_LIMIT * 8) + 2 * TIME_LIMIT + 1
    return {"workload": f"{wl['algo'].upper()} {wl['env']} time_limit={TIME_LIMIT}, {args.envs} vectorised envs/GPU, batch_size={args.batch}, "
                        f"{upi} updates per iteration of {args.envs} episodes (BASELINE.json configs[{wl['baseline_config']}])",
            "envs_per_gpu": args.envs, "batch_size": args.batch, "updates_per_iteration": upi, "buffer_episodes": args.buffer,
            "parallelism": f"dp{world}" if world > 1 else "single", "global_batch": args.batch * world,
            "collective": (("gradient sum over NVLink peer memory inside the fused reduce + Adam kernel" if args.collective == "peer"
                            else "one NCCL all-reduce of the gradient buffer per update") if world > 1 else None),
            "l2": "inputs larger than L2: each update gathers %d random episodes from a %.0f MB replay ring" % (args.batch, args.buffer * ep_bytes / 1e6)}


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        return {}


# ---- B200 arm: shared scaffolding ------------------------------------------------------------------------------------------------
class Harness:
    """Process-group set-up, the timed-region protocol (barrier + synchronize on both sides, CUDA events, max over ranks), clocks."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        self.torch, self.dist, self.args = torch, dist, args
        self.rank, self.world, self.local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device -- the B200 path has no CPU fallback")
        torch.cuda.set_device(self.local)
        torch.manual_seed(args.seed)   # the networks' initialisation: with the same arguments every run computes the same (--dump-outputs)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.steps_dev = torch.zeros((), dtype=torch.int64, device=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, k, fn):
        torch = self.torch
        self.steps_dev.zero_()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=self.dev)
        n = self.steps_dev.clone()
        if self.world > 1:
            self.dist.all_reduce(ms, op=self.dist.ReduceOp.MAX)
            self.dist.all_reduce(n, op=self.dist.ReduceOp.SUM)
        self.barrier()
        return float(ms.item()), int(n.item())

    def finish(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def dump_outputs(torch, out_dir, model, nat_env, store, slot0):
    """--dump-outputs: what the last timed step computed -- the parameters and target parameters after its updates, the metrics of its last update,
    each env's episode length and return, and a fixed, seeded sample of the episodes it wrote to `store` from slot `slot0` on -- as float32 .npy files."""
    import numpy as np

    E = nat_env.E
    pick = np.sort(np.random.default_rng(0).choice(E, min(E, DUMP_EPISODES), replace=False))
    slots = torch.as_tensor((slot0 + pick) % store.capacity, device=store.obs.device)
    arrays = {"theta": model.theta, "theta_target": model.theta_tgt, "metrics": model._metrics, "episode_length": nat_env.final_len,
              "episode_return": nat_env.final_ret, "episode_index": pick}
    arrays.update({f"episodes_{k}": getattr(store, k)[slots] for k in ("obs", "act", "rew", "done", "filled")})
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else t
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float32))


def theta_fingerprint(torch, theta):
    """Two order-sensitive 64-bit integers over the raw bits of the parameters (equal on two ranks <=> bit-identical parameters, up to a 2^-64 collision)."""
    bits = theta.detach().view(torch.int32).to(torch.int64)
    w = torch.arange(1, bits.numel() + 1, dtype=torch.int64, device=bits.device) % 65521 + 1
    return torch.stack([bits.sum(), (bits * w).sum()])


# ---- IDQN / VDN ------------------------------------------------------------------------------------------------------------------
def run_dqn_family(args, wl):
    import ctypes as C

    H = Harness(args)
    torch, dist, dev, rank, world = H.torch, H.dist, H.dev, H.rank, H.world
    from codebase_b200 import _native as nat
    from codebase_b200.config import Config
    from codebase_b200.dqn.model import QNetwork, VDNetwork
    from codebase_b200.dqn.train import Collector
    from codebase_b200.lbf import TrajStore
    from codebase_b200.utils.envs import make_env

    E, B, T = args.envs, args.batch, TIME_LIMIT
    U = args.updates_per_iter or E
    n_agents, obs_dim, n_act = dims(wl)
    env = make_env(args.seed, name=wl["env"], time_limit=T, parallel_envs=E, env_gid0=rank * E, wrappers=wl["wrappers"])
    cfg = Config(dict(optimizer="Adam", lr=3e-4, gamma=0.99, grad_clip=1.0, double_q=True, target_update_interval_or_tau=200, standardise_returns=False))
    cls = VDNetwork if wl["algo"] == "vdn" else QNetwork
    model = cls(env.single_observation_space, env.single_action_space, cfg, [128, 128], False, False, True, "cuda", max_batch=B, max_episode_length=T)
    if world > 1 and args.collective == "peer":
        try:
            model.attach_peers()
        except Exception as e:  # e.g. no peer access between the GPUs of this box: fall back to the NCCL exchange, and say so
            print(f"[bench] peer-memory exchange unavailable ({e}); using one NCCL all-reduce per update", file=sys.stderr)
            args.collective = "nccl"
        flag = torch.tensor([1 if args.collective == "peer" else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)   # all ranks or none
        if int(flag.item()) == 0:
            args.collective = "nccl"
    if world > 1:
        dist.broadcast(model.theta, 0)
        model.params_changed()
        model.hard_update()
    rb = TrajStore(args.buffer, env.n_agents, T, env.cfg.obs_dim, dev)
    coll = Collector(env, model, T)
    lib = nat.lib()
    nat.check(lib.marl_set_option(b"tensor_core_backward", C.c_int32(int(args.tc_backward))), "marl_set_option")
    nat.check(lib.marl_set_option(b"tensor_core_onchip", C.c_int32(int(args.tc_onchip))), "marl_set_option")
    state = dict(pos=0, updates=0)
    steps_dev = H.steps_dev
    # pinned host mirrors for the e2e leg
    nat_env = env.native
    h_obs = torch.empty_like(nat_env.obs, device="cpu").pin_memory()
    h_rew = torch.empty_like(nat_env.rew, device="cpu").pin_memory()
    h_done = torch.empty_like(nat_env.done, device="cpu").pin_memory()
    h_trunc = torch.empty_like(nat_env.trunc, device="cpu").pin_memory()
    h_loss = torch.empty(6, dtype=torch.float32).pin_memory()
    d_obs_in = torch.empty_like(nat_env.obs)
    sample_seed = args.seed + 7919 * rank

    def nccl_update(update_idx, n_valid):
        nat.check(lib.marl_replay_sample(C.c_uint64(sample_seed), C.c_uint64(update_idx), C.c_int32(B), C.c_int32(n_valid), nat.ptr(model._idx), nat.stream_ptr()), "marl_replay_sample")
        model.update_grads(rb, model._idx[:B])
        dist.all_reduce(model.grad)  # [sum-gradients | loss numerator | filled count], one exchange per update (SURVEY section 8e)
        model.update_apply()

    def do_updates():
        n_valid = min(state["pos"], args.buffer)
        if world == 1 or args.collective == "peer":   # peer: the gradient sum of all ranks happens inside the fused reduce + Adam kernel
            model.update_n(rb, B, n_valid, sample_seed, state["updates"], U)
        else:
            for u in range(U):
                nccl_update(state["updates"] + u, n_valid)
        state["updates"] += U

    def iteration(host_boundary: bool):
        slot0 = state["pos"] % args.buffer
        eps = 0.5
        if not host_boundary:
            final_len, _ = coll.collect(rb, slot0, eps)
        else:  # every env step's observations enter through pinned host memory and its results return to it
            nat_env.reset(traj=rb, slot0=slot0)
            h_obs.copy_(nat_env.obs, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            for _ in range(T):
                d_obs_in.copy_(h_obs, non_blocking=True)                                  # H2D: this step's inputs
                model.q_values(d_obs_in, out=coll.q)
                nat_env.rollout_step(coll.q, policy=1, epsilon=eps, traj=rb, slot0=slot0)
                h_obs.copy_(nat_env.obs, non_blocking=True); h_rew.copy_(nat_env.rew, non_blocking=True)      # D2H: this step's results
                h_done.copy_(nat_env.done, non_blocking=True); h_trunc.copy_(nat_env.trunc, non_blocking=True)
                torch.cuda.current_stream().synchronize()                                 # the host "sees" the step before the next one
            final_len = nat_env.final_len
        steps_dev.add_(final_len.sum())
        state["pos"] += E
        do_updates()
        if host_boundary:
            h_loss.copy_(model._metrics, non_blocking=True)

    for _ in range(max(args.warmup, 3)):
        iteration(False)
    sampler = ClockSampler(H.local) if rank == 0 else None
    ms, n_steps = H.timed(args.steps, lambda: iteration(False))
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, args.dump_outputs, model, nat_env, rb, (state["pos"] - E) % args.buffer)

    # ---- multi-GPU correctness, driver visible: replicated parameters must be BIT-identical on every rank after the timed region, and the in-kernel
    # peer-memory exchange must agree with the plain NCCL all-reduce path on one update from the same state (tests/test_peer_exchange_gpu.py asserts
    # the same; the driver's GPU test box has one GPU, so the evidence is emitted here) ------------------------------------------------------------
    multi = None
    if world > 1:
        fp = theta_fingerprint(torch, model.theta)
        fps = [torch.zeros_like(fp) for _ in range(world)]
        dist.all_gather(fps, fp)
        identical = all(bool(torch.equal(f, fps[0])) for f in fps)
        multi = {"ranks_bit_identical": identical, "theta_fingerprint": [int(x) for x in fps[0].tolist()]}
        if args.collective == "peer":
            upd, last = C.c_int64(), C.c_int64()
            nat.check(lib.marl_dqn_counters(model._h, C.byref(upd), C.byref(last)), "marl_dqn_counters")
            saved = [t.clone() for t in (model.theta, model.theta_tgt, model.adam_m, model.adam_v)]
            n_valid = min(state["pos"], args.buffer)

            def restore():
                for dst, src in zip((model.theta, model.theta_tgt, model.adam_m, model.adam_v), saved):
                    dst.copy_(src)
                model.params_changed()
                nat.check(lib.marl_dqn_set_counters(model._h, upd, last), "marl_dqn_set_counters")

            model.update_n(rb, B, n_valid, sample_seed, state["updates"], 1)          # in-kernel exchange over peer memory
            theta_peer = model.theta.clone()
            restore()
            nccl_update(state["updates"], n_valid)                                     # same batch, same state, NCCL all-reduce between grads and apply
            delta = (model.theta - theta_peer).abs().max()
            dist.all_reduce(delta, op=dist.ReduceOp.MAX)
            restore()
            multi["peer_vs_nccl_max_abs_dtheta"] = float(delta.item())
            multi["peer_vs_nccl_ok"] = float(delta.item()) <= 1e-6

    # roofline leg: one more iteration with the library's CUDA events around (and inside) the training pass of its first 1024
    # updates -- outside the headline region, because in-stream events serialise launches that otherwise overlap (PDL)
    model.timing(True)
    iteration(False)
    torch.cuda.synchronize()
    train_ms, train_n = model.timing(False)
    kernel_ms, kernel_n = model.timing_kernels()
    e2e = None
    if not args.no_e2e:
        iteration(True)
        ms_e, n_e = H.timed(args.steps, lambda: iteration(True))
        e2e = {"value": n_e / (ms_e / 1e3), "unit": "env-steps/s",
               "h2d_bytes_per_step": T * h_obs.numel() * 4,
               "d2h_bytes_per_step": T * (h_obs.numel() * 4 + h_rew.numel() * 4 + h_done.numel() + h_trunc.numel()) + 8}
    if rank != 0:
        H.finish()
        return
    value = n_steps / (ms / 1e3)
    rows = n_agents * (T + 1) * B
    FWD = fwd_flop_per_row(obs_dim, n_act)
    train_flop = 3 * rows * FWD             # online forward (1x) + backward (2x) of one update
    train_avg_s = (train_ms / max(train_n, 1)) / 1e3
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    fp32_peak = n_sm * 128 * 2 * sm_mhz * 1e6 / 1e12    # FFMA lanes x 2 flop x clock actually seen during the run
    peaks = load_peaks()
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    tensor_peak = peaks.get("bf16_tflops_sustained", 1443.2)   # sustained figure: the kernel is timed inside a long step
    per_update_us = 1e3 * (ms / args.steps) / U   # upper bound: includes the rollout's share of the iteration
    if kernel_n:
        # tensor-core training pass (DESIGN.md section 4.3): three kernels; the roofline object describes the slowest one
        P_net = model.n_params // model.n_nets
        if args.tc_onchip:
            names = ["tc_dqn_fwd3_kernel", "tc_dh1w1_kernel", "tc_dw2_kernel"]
            flops = [rows * FWD + rows * 2 * (n_act * HIDDEN + n_act),                  # online forward, dW3 | db3
                     rows * 2 * HIDDEN * HIDDEN + rows * 2 * HIDDEN * (obs_dim + 1),     # dH1 = dH2 x W2, dW1 | db1
                     rows * 2 * HIDDEN * (HIDDEN + 1)]                                   # dW2 | db2 (the recomputed layer 1, rows * 2 * obs * 128, is overhead and not counted)
            # algorithmic HBM bytes: what crosses the kernels is the gathered observation row (stored 32 floats wide) and the 64-byte row record
            inter = [rows * (obs_dim * 4 + n_act * 4) + rows * (128 + 64) + n_sm * 4 * (n_act * HIDDEN + n_act),
                     rows * (128 + 64) + n_sm * 4 * HIDDEN * (obs_dim + 1), rows * (128 + 64) + n_sm * 4 * HIDDEN * (HIDDEN + 1)]
        else:
            names = ["tc_dqn_fwd_kernel", "tc_dh1_kernel", "tc_dw_kernel"]
            flops = [rows * FWD,                                                       # online forward
                     rows * 2 * HIDDEN * HIDDEN,                                       # dH1 = dH2 x W2
                     rows * 2 * (HIDDEN * HIDDEN + HIDDEN * obs_dim + n_act * HIDDEN + HIDDEN + HIDDEN + n_act)]   # dW2, dW1, dW3 and the bias sums
            # algorithmic HBM bytes per update: H1, H2 written + read, dH1 written + read (FP32), 64-byte row records written + read twice,
            # gathered observations, target outputs, per-CTA gradient partials
            inter = [rows * (2 * 512 + 64) + rows * obs_dim * 4 + rows * n_act * 4, rows * (512 + 64), rows * (3 * 512 + 64 + obs_dim * 4) + n_sm * 4 * P_net]
        us = [1e3 * m / kernel_n for m in kernel_ms]
        k = max(range(3), key=lambda i: us[i])
        achieved = flops[k] / (us[k] * 1e-6) / 1e12
        roofline = {"bound": "tensor", "kernel": names[k], "achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s", "frac": achieved / tensor_peak,
                    "traffic": TRAFFIC_NCU.get(names[k]) if args.config == "idqn" else None,   # dram bytes of one launch (ncu)
                    "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (dense bf16; TF32 runs at half of it and 3xTF32 needs three MMAs per "
                                   "FP32-accurate product: the FP32-equivalent ceiling of this arithmetic is peak / 6)",
                    "fp32_equivalent_peak": tensor_peak / 6, "frac_of_fp32_equivalent_peak": achieved / (tensor_peak / 6),
                    "launch_us": us[k], "launches_timed": kernel_n, "flop_per_launch": flops[k],
                    "kernels": {names[i]: {"launch_us": us[i], "flop": flops[i], "tflops": flops[i] / (us[i] * 1e-6) / 1e12,
                                           "algorithmic_bytes": inter[i], "gbs": inter[i] / (us[i] * 1e-6) / 1e9, "hbm_frac": inter[i] / (us[i] * 1e-6) / 1e9 / hbm_peak}
                                for i in range(3)},
                    "training_pass": {"launch_us": 1e6 * train_avg_s, "flop": train_flop, "tflops": train_flop / train_avg_s / 1e12,
                                      "frac_of_fp32_cuda_core_peak": train_flop / train_avg_s / 1e12 / fp32_peak, "fp32_cuda_core_peak": fp32_peak,
                                      "note": "events between the three kernels serialise them; the headline run overlaps their heads and tails (PDL)"},
                    "whole_update": {"us_upper_bound": per_update_us, "flop": 4 * rows * FWD, "tflops": 4 * rows * FWD / (per_update_us * 1e-6) / 1e12,
                                     "frac_of_fp32_equivalent_peak": 4 * rows * FWD / (per_update_us * 1e-6) / 1e12 / (tensor_peak / 6),
                                     "note": "headline ms_per_step / updates_per_iteration (rollout included): target forward + training pass + reduce/Adam, pipelined"},
                    "hbm_peak_gbs": hbm_peak, "hbm_peak_source": "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"}
    else:
        train_bytes = B * 3421 + 7 * 4 * model.n_params       # gathered episodes + parameter / Adam traffic (SURVEY section 8d)
        achieved = train_flop / train_avg_s / 1e12 if train_n else None
        roofline = {"bound": "fp32-fma", "kernel": "train_kernel<16, kHeadDqn>", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s",
                    "frac": (achieved / fp32_peak) if achieved else None,
                    "traffic": 5524224,  # dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full (profiles/r1_train_kernel_final.md)
                    "peak_source": f"{n_sm} SMs x 128 FP32 lanes x 2 x {sm_mhz:.0f} MHz median SM clock sampled during the run (MEASURED_PEAKS.json holds no FP32 figure)",
                    "launch_us": 1e6 * train_avg_s, "launches_timed": train_n, "flop_per_launch": train_flop,
                    "hbm": {"achieved_gbs": (train_bytes / train_avg_s / 1e9) if train_n else None, "peak_gbs": hbm_peak,
                            "peak_source": "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)",
                            "frac": (train_bytes / train_avg_s / 1e9 / hbm_peak) if train_n else None, "bytes_per_launch": train_bytes,
                            "note": "the fused learner is compute-bound (~1 750 FLOP/B, SURVEY F7): the HBM fraction is small by construction"},
                    "bf16_tensor_peak_tflops": peaks.get("bf16_tflops_sustained")}
    # reset; per env step: forward, env; per update: target forward, training pass (3 kernels | 1 fused FP32 kernel), reduce + Adam (which also draws the
    # next update's replay indices); VDN adds an online forward and the TD kernel per update; one sample kernel per iteration
    per_update = (5 if kernel_n else 3) + (2 if wl["algo"] == "vdn" else 0)
    launches_per_step = 1 + 2 * T + U * per_update + 1
    line = {"metric": "env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, world), "clocks": clocks, "e2e": e2e, "gpu_launches": launches_per_step * args.steps,
            "roofline": roofline, "updates_per_sec": U * args.steps * world / (ms / 1e3), "env_steps_timed": n_steps}
    if multi is not None:
        line["multi_gpu"] = multi
        line["ranks_bit_identical"] = multi["ranks_bit_identical"]
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(args)
    emit(line)
    H.finish()


# ---- IA2C ------------------------------------------------------------------------------------------------------------------------
def run_ia2c(args, wl):
    import types

    H = Harness(args)
    torch, dist, dev, rank, world = H.torch, H.dist, H.dev, H.rank, H.world
    from codebase_b200.ac.model import A2CNetwork
    from codebase_b200.ac.train import Collector
    from codebase_b200.utils.envs import make_env

    P, T = args.envs, TIME_LIMIT
    n_agents, obs_dim, n_act = dims(wl)
    env = make_env(args.seed, name=wl["env"], time_limit=T, parallel_envs=P, env_gid0=rank * P)
    cfg = types.SimpleNamespace(optimizer="Adam", lr=3e-4, gamma=0.99, grad_clip=False, n_steps=5, entropy_coef=0.001, value_loss_coef=0.5,
                                target_update_interval_or_tau=200, standardise_returns=False)
    net = types.SimpleNamespace(layers=[128, 128], parameter_sharing=True, use_rnn=False, use_orthogonal_init=True, centralised=False)
    model = A2CNetwork(env.single_observation_space, env.single_action_space, cfg, net, net, "cuda", max_envs=P, max_episode_length=T)
    if world > 1:
        dist.broadcast(model.theta, 0)
        model.soft_update(1.0)
    coll = Collector(env, model, T)
    nat_env, b = env.native, coll.batch
    state = dict(step=0)
    h_obs = torch.empty_like(nat_env.obs, device="cpu").pin_memory()
    h_rew = torch.empty_like(nat_env.rew, device="cpu").pin_memory()
    h_done = torch.empty_like(nat_env.done, device="cpu").pin_memory()
    h_trunc = torch.empty_like(nat_env.trunc, device="cpu").pin_memory()
    h_met = torch.empty(6, dtype=torch.float32).pin_memory()
    d_obs_in = torch.empty_like(nat_env.obs)

    def update():
        if world == 1:
            model.update_from_store(b, P, state["step"])
        else:   # data-parallel: un-normalised gradient sums + filled count, one all-reduce, identical Adam step on every rank
            model.update_grads(b, P)
            dist.all_reduce(model.grad)
            model.update_apply(state["step"])

    def iteration(host_boundary: bool):
        if not host_boundary:
            final_len, _ = coll.collect()
        else:
            b.obs.zero_(); b.act.zero_(); b.rew.zero_(); b.filled.zero_(); b.done.zero_()
            nat_env.reset(traj=b, slot0=0)
            h_obs.copy_(nat_env.obs, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            for _ in range(T):
                d_obs_in.copy_(h_obs, non_blocking=True)
                model.logits(d_obs_in, out=coll.logits)
                nat_env.rollout_step(coll.logits, policy=2, traj=b, slot0=0)
                h_obs.copy_(nat_env.obs, non_blocking=True); h_rew.copy_(nat_env.rew, non_blocking=True)
                h_done.copy_(nat_env.done, non_blocking=True); h_trunc.copy_(nat_env.trunc, non_blocking=True)
                torch.cuda.current_stream().synchronize()
            final_len = nat_env.final_len
        H.steps_dev.add_(final_len.sum())
        update()
        state["step"] += T * P
        if host_boundary:
            h_met.copy_(model._metrics, non_blocking=True)

    for _ in range(max(args.warmup, 3)):
        iteration(False)
    sampler = ClockSampler(H.local) if rank == 0 else None
    ms, n_steps = H.timed(args.steps, lambda: iteration(False))
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, args.dump_outputs, model, nat_env, b, 0)
    multi = None
    if world > 1:
        fp = theta_fingerprint(torch, model.theta)
        fps = [torch.zeros_like(fp) for _ in range(world)]
        dist.all_gather(fps, fp)
        multi = {"ranks_bit_identical": all(bool(torch.equal(f, fps[0])) for f in fps)}
    # roofline leg: the update alone (CUDA events on torch's current stream = the stream every library call is enqueued on)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    torch.cuda.synchronize(); e0.record()
    for _ in range(reps):
        model.update_from_store(b, P, 1)
    e1.record(); torch.cuda.synchronize()
    upd_s = e0.elapsed_time(e1) / reps / 1e3
    e2e = None
    if not args.no_e2e:
        iteration(True)
        ms_e, n_e = H.timed(args.steps, lambda: iteration(True))
        e2e = {"value": n_e / (ms_e / 1e3), "unit": "env-steps/s", "h2d_bytes_per_step": T * h_obs.numel() * 4,
               "d2h_bytes_per_step": T * (h_obs.numel() * 4 + h_rew.numel() * 4 + h_done.numel() + h_trunc.numel()) + 24}
    if rank != 0:
        H.finish()
        return
    rows_t1, rows_t = n_agents * (T + 1) * P, n_agents * T * P
    f_actor, f_critic = fwd_flop_per_row(obs_dim, n_act), fwd_flop_per_row(obs_dim, 1)
    flop = rows_t1 * f_critic + 3 * rows_t * (f_actor + f_critic)     # target critic forward + forward/backward of critic and actor
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    fp32_peak = n_sm * 128 * 2 * sm_mhz * 1e6 / 1e12
    peaks = load_peaks()
    achieved = flop / upd_s / 1e12
    roofline = {"bound": "fp32-fma", "kernel": "marl_a2c_update (target critic forward, n-step returns, critic pass, actor pass, reduce, Adam)", "achieved": achieved, "peak": fp32_peak,
                "unit": "TFLOP/s", "frac": achieved / fp32_peak, "traffic": None, "launch_us": 1e6 * upd_s, "launches_timed": reps, "flop_per_launch": flop,
                "peak_source": f"{n_sm} SMs x 128 FP32 lanes x 2 x {sm_mhz:.0f} MHz median SM clock sampled during the run",
                "update_share_of_iteration": upd_s / (ms / args.steps / 1e3), "bf16_tensor_peak_tflops": peaks.get("bf16_tflops_sustained")}
    line = {"metric": "env-steps/sec", "value": n_steps / (ms / 1e3), "unit": "env-steps/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, world), "clocks": clocks, "e2e": e2e, "gpu_launches": (1 + 5 + 2 * T + 8) * args.steps,
            "roofline": roofline, "updates_per_sec": args.steps * world / (ms / 1e3), "env_steps_timed": n_steps}
    if multi is not None:
        line["multi_gpu"] = multi
        line["ranks_bit_identical"] = multi["ranks_bit_identical"]
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(args)
    emit(line)
    H.finish()


def cpu_baseline(args):
    """The reference loop (oracle port) on ONE core -- the reference pins torch to one thread (run.py:29) -- bounded sample."""
    from oracle import cpu_loop

    wl = WORKLOADS[args.config]
    kw = dict(algo=wl["algo"], lbf=wl["lbf"], time_limit=TIME_LIMIT, seed=args.seed)
    if wl["algo"] == "ia2c":
        loop = cpu_loop.make_loop(batch=0, **kw)
        loop.run(1)
        n = 6
        steps, secs = loop.run(n)
        return {"value": steps / secs, "unit": "env-steps/s", "cores": 1, "kind": "port",
                "sample": f"{n} iterations of the reference IA2C loop (one 10-env vector rollout, ia2c.yaml parallel_envs=10, + one update), 1 thread, pure-Python LBF "
                          f"restatement + PyTorch-CPU learner, {secs:.1f} s"}
    loop = cpu_loop.make_loop(batch=args.batch, **kw)
    loop.prefill(args.batch)
    loop.run(1)
    n = 30 if args.config == "idqn" else 8
    steps, secs = loop.run(n)
    out = {"value": steps / secs, "unit": "env-steps/s", "cores": 1, "kind": "port",
           "sample": f"{n} iterations of the reference loop (one 25-step episode with one env + one update at batch_size={args.batch}), 1 thread, "
                     f"pure-Python LBF restatement + PyTorch-CPU learner, {secs:.1f} s"}
    # the reference AS SHIPPED trains at batch_size=128 (BASELINE.json configs[0]; marlbase/configs/algorithm/idqn.yaml): timed next to it
    small = cpu_loop.make_loop(batch=128, **kw)
    small.prefill(128)
    small.run(1)
    s2, t2 = small.run(60)
    out["as_shipped_batch_128"] = {"value": s2 / t2, "unit": "env-steps/s", "cores": 1,
                                   "sample": f"60 iterations at the reference's own batch_size=128 (configs[0]), {t2:.1f} s"}
    return out


def emit(line: dict):
    """The ONE JSON line goes to the real stdout; everything else (NCCL banners, library prints) was redirected to stderr."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1

if __name__ == "__main__":
    a = parse()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # stray prints of other libraries must not pollute the JSON contract
    if a.impl == "reference":
        run_reference(a)
    elif WORKLOADS[a.config]["algo"] == "ia2c":
        run_ia2c(a, WORKLOADS[a.config])
    else:
        run_dqn_family(a, WORKLOADS[a.config])
