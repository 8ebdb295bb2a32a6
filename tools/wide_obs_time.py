"""Time of the FP32 FFMA training pass and of a whole IDQN update at observation widths 27..128 (batch 1024 episodes x 25 steps, 2 agents with
independent networks, 6 actions): python tools/wide_obs_time.py [out.json]

Widths above 32 take the K-chunked first layer (mlp.cuh, mlp_forward_tile_wide); 27 runs with tensor_core_backward=0, i.e. the KP = 32 FFMA pass
the wide one is compared with.  Achieved FLOP/s count 3 x the forward's 2 (D*128 + 128*128 + 128*A) FLOPs per gathered row (N x B x (T + 1) rows).
The card's name and power limit are recorded with the numbers."""
import ctypes as C
import json
import os
import subprocess
import sys
import types

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from codebase_b200 import _native as nat  # noqa: E402
from codebase_b200.dqn import model as M  # noqa: E402
from codebase_b200.lbf import TrajStore  # noqa: E402

N, A, T, B, CAP = 2, 6, 25, 1024, 4096
WARMUP, STEPS = 20, 200


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def one(D, tc_backward):
    nat.check(nat.lib().marl_set_option(b"tensor_core_backward", C.c_int32(tc_backward)), "marl_set_option")
    cfg = types.SimpleNamespace(optimizer="Adam", lr=3e-4, gamma=0.99, grad_clip=1.0, double_q=True, target_update_interval_or_tau=200, standardise_returns=False)
    sp = lambda **kw: types.SimpleNamespace(shape=kw.get("shape"), n=kw.get("n"))
    m = M.QNetwork([sp(shape=(D,))] * N, [sp(n=A)] * N, cfg, [128, 128], False, False, True, "cuda", max_batch=B, max_episode_length=T)
    ts = TrajStore(CAP, N, T, D, m.device)
    ts.obs.copy_(torch.randn_like(ts.obs)); ts.act.copy_(torch.randint(0, A, ts.act.shape)); ts.rew.copy_(torch.rand_like(ts.rew))
    ts.filled.fill_(1)
    m.update_n(ts, B, CAP, 1, 0, WARMUP)
    torch.cuda.synchronize()
    # the training pass alone: CUDA events around it on every update
    m.timing(True)
    m.update_n(ts, B, CAP, 1, WARMUP, STEPS)
    torch.cuda.synchronize()
    train_ms, launches = m.timing(False)
    # the whole update (target forward, training pass, fused reduce + Adam, next replay indices)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); m.update_n(ts, B, CAP, 1, WARMUP + STEPS, STEPS); e1.record(); torch.cuda.synchronize()
    update_us = e0.elapsed_time(e1) / STEPS * 1e3
    m.close()
    rows = N * B * (T + 1)
    flops = 3 * 2 * (D * 128 + 128 * 128 + 128 * A) * rows
    train_us = train_ms / max(launches, 1) * 1e3
    return dict(D=D, tensor_core_backward=tc_backward, path="FFMA KP=32" if D <= 32 else f"FFMA K-chunked ({(D + 31) // 32} chunks)", rows=rows,
                train_pass_us=round(train_us, 1), train_tflops=round(flops / train_us * 1e-6, 2), update_us=round(update_us, 1), timed_updates=launches)


def main():
    torch.cuda.set_device(0)
    res = dict(card=card(), batch=B, T=T, n_agents=N, n_actions=A, warmup=WARMUP, updates=STEPS, results=[])
    print(res["card"], flush=True)
    for D, tcb in ((27, 0), (45, 1), (64, 1), (108, 1), (128, 1)):
        r = one(D, tcb)
        res["results"].append(r)
        print(json.dumps(r), flush=True)
    nat.check(nat.lib().marl_set_option(b"tensor_core_backward", C.c_int32(1)), "marl_set_option")
    if len(sys.argv) > 1:
        os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
        with open(sys.argv[1], "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
