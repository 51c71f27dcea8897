"""Cost of camera images (mb200_render): one JSON line on stdout.

* every env kind at 16 384 envs x 64 x 64 (one tracking camera per env) and at 16 envs x 640 x 480: CUDA events
  around each VecEnv.render call (camera matrices prepared outside the window), median over the timed calls after a
  warm-up; frames/s and rays/s from it.
* the split between the scene pass (k_render_scene_<kind>) and the ray pass (k_render_rays): device time per call of
  each kernel from torch.profiler (CUDA activities) over a separate run of calls.
* Walker3DCustomEnv-v0 env-steps/s stepping alone vs stepping with a 64 x 64 render of every env after every step, in
  alternating blocks in the same process.
* the GPU's name and power limit, read in the same run.

Usage: python tools/render_bench.py [--envs 16384] [--calls 50] [--steps 100] [--rounds 5]
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

KINDS = {  # name -> VecEnv class, kwargs
    "walker3d_custom": ("Walker3DCustomVecEnv", {}),
    "walker3d_stepper": ("Walker3DStepperVecEnv", {}),
    "walker3d_stepper_pillar": ("Walker3DStepperVecEnv", {"plank_class": "Pillar"}),
    "monkey3d_custom": ("Monkey3DCustomVecEnv", {}),
    "cassie": ("CassieVecEnv", {}),
    "child3d_custom": ("Child3DCustomVecEnv", {}),
    "mike_stepper": ("MikeStepperVecEnv", {}),
    "walker2d_custom": ("Walker2DCustomVecEnv", {}),
    "crab2d_custom": ("Crab2DCustomVecEnv", {}),
}
SHAPES = ((16384, 64, 64), (16, 640, 480))  # envs, width, height


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        return float(out.strip().splitlines()[0])
    except Exception:
        return None


def render_time(env, w, h, calls, warmup):
    st = env.get_state()[:, 0:3]
    view, proj = V.camera_matrices(st, aspect=w / h, **V.TRACKING_CAMERA)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(calls)]
    for i in range(warmup + calls):
        if i >= warmup:
            ev[i - warmup][0].record()
        out = env.render(width=w, height=h, view=view, proj=proj)
        if i >= warmup:
            ev[i - warmup][1].record()
    torch.cuda.synchronize()
    ms = np.array([a.elapsed_time(b) for a, b in ev])
    robot = float((out["seg"] >= 99).float().mean())
    # kernel split, in a run of its own
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(10):
            env.render(width=w, height=h, view=view, proj=proj)
        torch.cuda.synchronize()
    scene = rays = 0.0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if e.key.startswith("k_render_rays"):
            rays += t / 10
        elif "k_render_scene_" in e.key:
            scene += t / 10
    med = float(np.median(ms))
    n = env.num_envs
    return {"median_ms": med, "min_ms": float(ms.min()), "frames_per_s": n / (med * 1e-3),
            "rays_per_s": n * w * h / (med * 1e-3), "scene_pass_us": scene, "ray_pass_us": rays,
            "robot_pixel_fraction": robot, "calls": calls}


def step_rate(n, steps, rounds, warmup):
    env = V.Walker3DCustomVecEnv(n, seed=0)
    try:
        env.reset()
        g = torch.Generator(device="cuda").manual_seed(1)
        act = torch.rand(n, env.act_dim, device="cuda", generator=g) * 2 - 1
        rates = {"step": [], "step_render_64": []}

        def block(render, k):
            for _ in range(k):
                env.step(act)
                if render:
                    env.render(width=64, height=64)

        block(False, warmup)
        block(True, warmup)
        for _ in range(rounds):
            for name, render in (("step", False), ("step_render_64", True)):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                block(render, steps)
                b.record()
                b.synchronize()
                rates[name].append(n * steps / (a.elapsed_time(b) * 1e-3))
    finally:
        env.close()
    out = {k: float(np.median(v)) for k, v in rates.items()}
    out["ratio"] = out["step_render_64"] / out["step"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=16384)
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "render_bench measures on a CUDA device; there is no CPU measurement"
    res = {"gpu": torch.cuda.get_device_name(), "power_limit_w": power_limit_w(), "render": {}}
    for name, (cls, kw) in KINDS.items():
        res["render"][name] = {}
        for n, w, h in SHAPES:
            n = a.envs if n == 16384 else n
            env = getattr(V, cls)(n, seed=0, **kw)
            try:
                env.reset()
                g = torch.Generator(device="cuda").manual_seed(0)
                for _ in range(3):
                    env.step(torch.rand(n, env.act_dim, device="cuda", generator=g) * 2 - 1)
                res["render"][name]["%dx%dx%d" % (n, w, h)] = render_time(env, w, h, a.calls, a.warmup)
            finally:
                env.close()
    res["walker3d_step_rate"] = step_rate(a.envs, a.steps, a.rounds, a.warmup)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
