"""Cost of a push (mb200_apply_impulse): one JSON line on stdout.

* k_apply_impulse_<kind> per call at 16 384 envs for every env kind: CUDA events around each call, >= 200 timed calls
  after a warm-up, a 256 MB buffer overwritten between calls so the state rows come from HBM, not from L2.  Every env
  is pushed (on a foot, at the base COM; the sign alternates so the velocities stay bounded).
* Walker3DCustomEnv-v0 env-steps/s with a push on 10 % of the envs after every step vs no pushes, in alternating
  blocks in the same process.
* the GPU's name and power limit, read in the same run.

Usage: python tools/impulse_bench.py [--envs 16384] [--calls 200] [--steps 200] [--rounds 5]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mocca_envs_b200 import vec_env as V  # noqa: E402

KINDS = {  # name -> VecEnv class, kwargs, pushed link (URDF name)
    "walker3d_custom": ("Walker3DCustomVecEnv", {}, "right_foot"),
    "walker3d_stepper": ("Walker3DStepperVecEnv", {}, "right_foot"),
    "walker3d_stepper_pillar": ("Walker3DStepperVecEnv", {"plank_class": "Pillar"}, "right_foot"),
    "monkey3d_custom": ("Monkey3DCustomVecEnv", {}, "right_foot"),
    "cassie": ("CassieVecEnv", {}, "right_toe"),
    "child3d_custom": ("Child3DCustomVecEnv", {}, "right_foot"),
    "mike_stepper": ("MikeStepperVecEnv", {}, "right_foot"),
    "walker2d_custom": ("Walker2DCustomVecEnv", {}, "foot"),
    "crab2d_custom": ("Crab2DCustomVecEnv", {}, "foot"),
}


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        return float(out.strip().splitlines()[0])
    except Exception:
        return None


def kernel_time(cls, kw, link_name, n, calls, warmup, flush):
    env = getattr(V, cls)(n, seed=0, **kw)
    try:
        env.reset()
        # (every input prepared outside the timed window: the window holds the kernel launch only)
        link = torch.full((n,), env.link_index(link_name), dtype=torch.int32, device="cuda")
        point = env.get_state()[:, 0:3].contiguous()
        g = torch.Generator(device="cuda").manual_seed(0)
        imp = torch.randn(n, 3, device="cuda", generator=g)
        imp = 5.0 * imp / imp.norm(dim=1, keepdim=True)
        imps = (imp, (-imp).contiguous())
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(calls)]
        for i in range(warmup + calls):
            flush.zero_()
            if i >= warmup:
                ev[i - warmup][0].record()
            env.apply_impulse(imps[i % 2], link=link, point=point)
            if i >= warmup:
                ev[i - warmup][1].record()
        torch.cuda.synchronize()
        ms = np.array([a.elapsed_time(b) for a, b in ev])
        assert np.isfinite(env.get_state().cpu().numpy()).all()
    finally:
        env.close()
    return {"median_us": float(np.median(ms) * 1e3), "min_us": float(ms.min() * 1e3), "calls": calls}


def step_rate(n, steps, rounds, warmup):
    env = V.Walker3DCustomVecEnv(n, seed=0)
    try:
        env.reset()
        g = torch.Generator(device="cuda").manual_seed(1)
        act = torch.rand(n, env.act_dim, device="cuda", generator=g) * 2 - 1
        pushed = torch.rand(n, device="cuda", generator=g) < 0.1
        link = torch.full((n,), -2, dtype=torch.int32, device="cuda")
        link[pushed] = -1  # the base, at its COM; -2 leaves the other envs untouched
        rates = {"no_push": [], "push_10pct": []}

        def block(push, k):
            for _ in range(k):
                env.step(act)
                if push:
                    env.apply_impulse(torch.randn(n, 3, device="cuda", generator=g) * 5.0, link=link,
                                      point=env.get_state()[:, 0:3])

        block(False, warmup)
        block(True, warmup)
        for _ in range(rounds):
            for name, push in (("no_push", False), ("push_10pct", True)):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                block(push, steps)
                b.record()
                b.synchronize()
                rates[name].append(n * steps / (a.elapsed_time(b) * 1e-3))
        stats = env.stats()
    finally:
        env.close()
    out = {k: float(np.median(v)) for k, v in rates.items()}
    out["ratio"] = out["push_10pct"] / out["no_push"]
    out["nonfinite"] = stats["nonfinite"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=16384)
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "impulse_bench measures on a CUDA device; there is no CPU measurement"
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device="cuda")  # 256 MB > the 126 MB L2
    res = {"gpu": torch.cuda.get_device_name(), "power_limit_w": power_limit_w(), "envs": a.envs, "kernel": {}}
    for name, (cls, kw, link) in KINDS.items():
        res["kernel"][name] = kernel_time(cls, kw, link, a.envs, a.calls, a.warmup, flush)
    res["walker3d_step_rate"] = step_rate(a.envs, a.steps, a.rounds, a.warmup)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
