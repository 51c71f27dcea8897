#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched Walker3DCustomEnv-v0 hot path (BASELINE.json configs[1]).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--envs E] [--actions random|pd] [--impl reference]
                  [--dump-outputs DIR]

One "step" = one fused kernel launch stepping E envs per GPU through one control step (4 Bullet substeps +
obs/reward/done/auto-reset).  Prints ONE JSON line (rank 0).  See DESIGN.md section "Measurement".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (it may be read-only)

WORKLOAD = "Walker3DCustomEnv-v0 batched 16384 envs/GPU, flat ground"
METRIC = "env-steps/sec (Walker3DCustomEnv-v0, 16384 envs/GPU, random actions)"


# DRAM bytes per launch of k_step_walker3d_custom at 16384 envs from the last committed ncu --set full capture
NCU_TRAFFIC = {"bytes": 8.06e6, "source": "ncu --set full capture profiles/r3z_step_kernel_raw.csv (8.06 MB read, < 0.01 MB "
                                          "written per launch), not measured by this run"}

ENV_NAMES = {"custom": "Walker3DCustomEnv", "stepper": "Walker3DStepperEnv", "monkey": "Monkey3DCustomEnv",
             "cassie": "CassieEnv", "child": "Child3DCustomEnv", "mike": "MikeStepperEnv",
             "walker2d": "Walker2DCustomEnv", "crab2d": "Crab2DCustomEnv"}


def flops_per_env_step(rows_per_substep, S=4, n=27, L=17, G=22, I=5, P=0):
    """SURVEY.md section 8(d): F = S*[60L + 430n + 30G + 60P + R*150n + I*R*(4n+10) + 20n] + 1000
    (P = self-collision candidate pairs tested per substep)."""
    R = rows_per_substep
    return S * (60 * L + 430 * n + 30 * G + 60 * P + R * 150 * n + I * R * (4 * n + 10) + 20 * n) + 1000


def bytes_per_env_step(S_state=55, A=21, O=52, S_env=12):
    """SURVEY.md section 8(d): B = 4*(2*S_state + A + O + 2*S_env) + 6."""
    return 4 * (2 * S_state + A + O + 2 * S_env) + 6


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe): an in-process NVML
    poll every 10 ms (so that even a sub-second timed region is covered), nvidia-smi -lms as the fallback."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
            0x80: "hw_power_brake_slowdown"}

    def __init__(self, gpu_index, uuid=None):
        self.rows = []
        self.sm, self.mx, self.reasons = [], [], set()
        self.proc = None
        self.gpu = gpu_index
        self.uuid = uuid
        self.nvml = None
        self.handle = None
        self.stop_flag = False
        self.source = None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            h = None
            if self.uuid:
                try:
                    h = pynvml.nvmlDeviceGetHandleByUUID(self.uuid if isinstance(self.uuid, bytes) else self.uuid.encode())
                except Exception:
                    h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self.nvml, self.handle = pynvml, h
            self.mx.append(float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)))
            self.source = "nvml poll 10 ms"
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi -lms 20"
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def sample(self):
        if self.nvml is None:
            return
        n, h = self.nvml, self.handle
        try:
            self.sm.append(float(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)))
            try:
                r = n.nvmlDeviceGetCurrentClocksEventReasons(h)
            except Exception:
                r = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            for bit, nm in self.BITS.items():
                if r & bit:
                    self.reasons.add(nm)
        except Exception:
            pass

    def _poll(self):
        while not self.stop_flag:
            self.sample()
            time.sleep(0.01)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.t.join(timeout=2)
            sm = sorted(self.sm)
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                    "reasons": sorted(self.reasons), "samples": len(sm), "source": self.source}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower() == "active":
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": self.source}


def cpu_reference_run(n_envs, steps, warmup, threads, time_budget=None, kind="custom"):
    """The reference-side CPU implementation of the path: the float64 oracle port (oracle/mocca_oracle.c; the
    reference's own arithmetic is the un-installable third-party pybullet), OpenMP over envs."""
    import ctypes as C

    import numpy as np

    from mocca_envs_b200.model_compiler import load_table
    from oracle import oracle as O

    model, struct, pre, A, OB = {"child": ("child3d", O.W3DEnv, "orc_w3d", 21, 52),
                                 "walker2d": ("walker2d", O.W3DEnv, "orc_w3d", 7, 24),
                                 "crab2d": ("crab2d", O.W3DEnv, "orc_w3d", 6, 22),
                                 "mike": ("mike", O.StepperEnv, "orc_stepper", 21, 65),
                                 "cassie": ("cassie", O.CassieEnvS, "orc_cassie", 10, 36),
                                 "custom": ("walker3d", O.W3DEnv, "orc_w3d", 21, 52),
                                 "stepper": ("walker3d", O.StepperEnv, "orc_stepper", 21, 65),
                                 "monkey": ("monkey3d", O.MonkeyEnv, "orc_monkey", 23, 69)}[kind]
    t = load_table(os.path.join(ROOT, "mocca_envs_b200", "models", model + ".json"))
    m = O.model_from_table(t)
    p = O.cassie_params() if kind == "cassie" else O.default_params()
    L = O.lib()
    envs = (struct * n_envs)()
    obs = np.zeros((n_envs, OB))
    seed_fn = getattr(L, pre + "_seed", None)  # CassieEnv draws no random numbers
    reset_fn, batch_fn = getattr(L, pre + "_reset"), getattr(L, pre + "_step_batch")
    for i in range(n_envs):
        words = O.gym_seed_words(1000 + i)
        key = (C.c_uint32 * len(words))(*words)
        if kind in ("stepper", "mike"):
            envs[i].curriculum = (0, 5, 9)[i % 3]
        if seed_fn is not None:
            seed_fn(C.byref(envs[i]), key, len(words), 1)
        reset_fn(C.byref(m), C.byref(p), C.byref(envs[i]), obs[i].ctypes.data_as(C.c_void_p))
    rew = np.zeros(n_envs)
    done = np.zeros(n_envs, dtype=np.int32)
    rng = np.random.RandomState(1)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)

    def one():
        a = rng.uniform(-1, 1, (n_envs, A)) * (0.1 if kind == "cassie" else 1.0)
        batch_fn(C.byref(m), C.byref(p), envs, n_envs, vp(a), vp(obs), vp(rew), vp(done), threads)

    for _ in range(warmup):
        one()
    t0 = time.perf_counter()
    done_steps = 0
    for _ in range(steps):
        one()
        done_steps += 1
        if time_budget and time.perf_counter() - t0 > time_budget:
            break
    dt = time.perf_counter() - t0
    return n_envs * done_steps / dt, dt, done_steps


_REAL_STDOUT = None


def _quiet_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints "NCCL version ..." at
    communicator creation): keep a private handle on the real stdout and point fd 1 at stderr for the rest of the run."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def _emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000, help="timed steps of every measured loop")
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--envs", type=int, default=16384, help="envs per GPU")
    ap.add_argument("--actions", default="random", choices=["random", "pd"])
    ap.add_argument("--env", default="custom", choices=["custom", "stepper", "monkey", "cassie", "child", "mike", "walker2d", "crab2d"],
                    help="custom = BASELINE configs[1] (headline); stepper = configs[2] (curriculum 0/5/9 per env); "
                         "monkey = configs[4] (Monkey3DCustomEnv-v0); cassie = configs[3] (CassieEnv-v0, 50 substeps per step); "
                         "child / mike = SURVEY 8 f3 (Child3DCustomEnv-v0, MikeStepperEnv-v0)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", dest="also", action="store_false",
                    help="skip the short runs of BASELINE configs 2-5 (scripted PD, Stepper, Monkey3D, Cassie at 8192 envs) "
                         "that the default headline run appends under \"also\"")
    ap.add_argument("--self-collision", type=int, default=1, choices=[0, 1],
                    help="1 = the reference's URDF_USE_SELF_COLLISION flags (robots.py:259-264); 0 = ablation")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the run, write what the last timed step of the headline workload returned (rank 0's "
                         "envs) as DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the CUDA path (--impl b200)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cores = os.cpu_count() or 1

    if args.impl == "reference":
        if rank != 0:
            return
        # size the per-step sample so that K steps take about a minute on this box's cores
        v0, _, _ = cpu_reference_run(256, 8, 1, cores, kind=args.env)
        sample_envs = int(min(4096, max(64, v0 * 60.0 / max(args.steps, 1))))
        v, dt, ks = cpu_reference_run(sample_envs, args.steps, min(max(args.warmup, 1), 10), cores, kind=args.env)
        line = {
            "impl": "reference",
            "metric": METRIC.replace("Walker3DCustomEnv", ENV_NAMES[args.env]),
            "value": v, "unit": "env-steps/s", "n_gpus": args.gpus,
            "steps": ks, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(ks, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "envs_per_gpu": args.envs, "actions": "random-uniform U(-1,1)^21",
                       "envs_stepped_per_sample": sample_envs,
                       "note": "a CPU loop over independent envs: throughput does not depend on the batch size, so each "
                               "timed step advances a bounded sample of %d envs of the %d-env workload" % (sample_envs, args.envs)},
            "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": cores, "kind": "port",
                             "sample": "%d envs x %d control steps per step-sample, OpenMP over envs; float64 oracle "
                                       "port (PyBullet itself is not installable: no wheel, no network)" % (sample_envs, ks)},
            "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        _emit(line)
        return

    import numpy as np
    import torch

    from mocca_envs_b200 import _lib
    from mocca_envs_b200.distributed import shard_seed
    from mocca_envs_b200.vec_env import (CassieVecEnv, Child3DCustomVecEnv, MikeStepperVecEnv, Monkey3DCustomVecEnv,
                                         Walker3DCustomVecEnv, Walker3DStepperVecEnv)

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    dist = None
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    N, K, W = args.envs, args.steps, max(args.warmup, 3)
    ctx = dict(np=np, torch=torch, _lib=_lib, dist=dist, dev=dev, rank=rank, world=world, local_rank=local_rank)
    outputs = {} if args.dump_outputs else None
    line = measure(ctx, args.env, N, K, W, args.actions, args.self_collision, outputs)
    if args.also and args.env == "custom" and args.actions == "random" and args.self_collision:
        # BASELINE configs 2-5 next to the headline, every default run (so the 1/2/4/8-GPU scaling runs carry them):
        # device + e2e measurements with their own roofline fractions
        also = {}
        Wa = 20
        for name, kind, n_envs, acts in (("walker3d_custom_pd", "custom", N, "pd"),
                                         ("walker3d_stepper", "stepper", N, "random"),
                                         ("monkey3d", "monkey", N, "random"),
                                         ("cassie_8192", "cassie", min(N, 8192), "random")):
            r = measure(ctx, kind, n_envs, K, Wa, acts, 1)
            if r is not None:
                also[name] = {k: r[k] for k in ("metric", "value", "unit", "ms_per_step", "steps", "warmup", "roofline",
                                                "e2e", "gpu_launches", "episodes")}
                also[name]["config"] = {k: r["config"][k] for k in ("workload", "envs_per_gpu", "actions", "frame_skip")}
        if line is not None:
            line["also"] = also
    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if not args.no_cpu_baseline:
        ce = 256 if args.env == "cassie" else 2048
        v, dt, ks = cpu_reference_run(ce, 2000, 2, cores, time_budget=15.0, kind=args.env)
        line["cpu_baseline"] = {"value": v, "unit": "env-steps/s", "cores": cores, "kind": "port",
                                "sample": str(ce) + " envs x %d control steps (%.1f s), same action distribution; float64 "
                                          "oracle port with OpenMP over envs (PyBullet not installable here)" % (ks, dt)}
    _emit(line)
    if dist:
        dist.destroy_process_group()


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, outputs):
    """Write `outputs` (arrays with one row per env) as <out_dir>/<name>.npy in float32, and env_index.npy (float64):
    the envs whose rows were written.  That is every env unless the files would exceed DUMP_BYTES; then it is a fixed,
    seeded sample of them, the same from run to run."""
    import numpy as np

    n = len(outputs["obs"])
    row_bytes = 8 + sum(4 * (a.size // n) for a in outputs.values())
    keep = min(n, (DUMP_BYTES - 4096) // row_bytes)  # 4 KiB for the .npy headers
    idx = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "env_index.npy"), idx.astype(np.float64))
    for name, a in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a[idx], dtype=np.float32))


def measure(ctx, env_kind, N, K, W, actions, self_collision, outputs=None):
    """One workload: W warm-up steps, K device-timed steps (CUDA events, L2 flushed in between, max over ranks) and the
    host-buffer e2e leg over K steps.  Returns the JSON line (rank 0) or None.  `outputs`, when given, receives as
    NumPy arrays what the last timed step returned: obs, reward, done and truncated."""
    np, torch, _lib, dist, dev = ctx["np"], ctx["torch"], ctx["_lib"], ctx["dist"], ctx["dev"]
    rank, world, local_rank = ctx["rank"], ctx["world"], ctx["local_rank"]
    from mocca_envs_b200.distributed import shard_seed
    from mocca_envs_b200.vec_env import (CassieVecEnv, Child3DCustomVecEnv, MikeStepperVecEnv, Monkey3DCustomVecEnv,
                                         Walker3DCustomVecEnv, Walker3DStepperVecEnv)

    # env i of rank r is global env r*N + i: seeds are independent of the GPU count (SURVEY 8e)
    phys = {"self_collision": self_collision}
    if env_kind in ("stepper", "mike"):
        cls = Walker3DStepperVecEnv if env_kind == "stepper" else MikeStepperVecEnv
        env = cls(N, device=dev, seed=shard_seed(1234, rank, N), physics=phys)
        env.set_env_params({"curriculum": np.array([0, 5, 9] * (N // 3 + 1))[:N]})
    elif env_kind == "child":
        env = Child3DCustomVecEnv(N, device=dev, seed=shard_seed(1234, rank, N), physics=phys)
    elif env_kind in ("walker2d", "crab2d"):
        from mocca_envs_b200.vec_env import Crab2DCustomVecEnv, Walker2DCustomVecEnv
        cls = Walker2DCustomVecEnv if env_kind == "walker2d" else Crab2DCustomVecEnv
        env = cls(N, device=dev, seed=shard_seed(1234, rank, N), physics=phys)
    elif env_kind == "monkey":
        env = Monkey3DCustomVecEnv(N, device=dev, seed=shard_seed(1234, rank, N), physics=phys)
    elif env_kind == "cassie":
        env = CassieVecEnv(N, device=dev, seed=shard_seed(1234, rank, N), physics=phys)
    else:
        env = Walker3DCustomVecEnv(N, device=dev, seed=shard_seed(1234, rank, N), physics=phys)
    env.reset()
    A = env.act_dim
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    pool = 64
    act_pool = torch.rand(pool, N, A, device=dev, generator=gen) * 2 - 1
    if env_kind == "cassie":
        act_pool *= 0.1  # SURVEY 8d config 4: a ~ U(-0.1, 0.1)^10 residual on the PD targets
    if actions == "pd":
        q_ref = torch.tensor(env.table["base_joint_angles"], device=dev, dtype=torch.float32)
        lo = torch.tensor(env.table["lower"], device=dev, dtype=torch.float32)
        hi = torch.tensor(env.table["upper"], device=dev, dtype=torch.float32)
        ref_norm = 2 * (q_ref - lo) / (hi - lo) - 1

    def action(i, obs):
        if actions == "random":
            return act_pool[i % pool]
        # scripted PD toward the running_start pose in normalised units (SURVEY 8d config 2: kp=1, kd=0.1)
        return torch.clamp(1.0 * (ref_norm - obs[:, 6:6 + A]) - 0.1 * (obs[:, 6 + A:6 + 2 * A] * 10.0), -1, 1)

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    obs = env.obs
    for i in range(W):
        obs, _, _, _ = env.step(action(i, obs))
    torch.cuda.synchronize(dev)
    rec0 = env.get_record()
    rows0 = float(rec0[:, 15].double().sum())
    cont0 = float(rec0[:, 16].double().sum())
    env.stats(reset=True)
    try:
        uuid = "GPU-" + str(torch.cuda.get_device_properties(dev).uuid)
    except Exception:
        uuid = None
    try:
        gpu_index = int(os.environ["CUDA_VISIBLE_DEVICES"].split(",")[local_rank])
    except Exception:
        gpu_index = local_rank
    sampler = ClockSampler(gpu_index, uuid)
    launches0 = env.launch_count()
    if dist:
        dist.barrier()
    torch.cuda.synchronize(dev)
    if rank == 0:
        sampler.start()  # polls from here to the closing synchronize: the timed region only
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    wall0 = time.perf_counter()
    for i in range(K):
        flush.zero_()  # evict L2 between timed steps (not inside the event pair)
        a = action(W + i, obs)
        evs[i][0].record()
        obs, rew, done, info = env.step(a)
        evs[i][1].record()
    if rank == 0:
        sampler.sample()  # the GPU is still draining the queued steps here
    if dist:
        dist.barrier()
    torch.cuda.synchronize(dev)
    wall = time.perf_counter() - wall0
    if outputs is not None:  # copied now: the e2e leg below steps the same env again
        outputs.update((k, v.float().cpu().numpy()) for k, v in (
            ("obs", obs), ("reward", rew), ("done", done), ("truncated", info["TimeLimit.truncated"])))
    launches = env.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    step_ms = [a.elapsed_time(b) for a, b in evs]
    total_ms = float(sum(step_ms))
    tmax = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if dist:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    total_ms_max = float(tmax.item())
    rec1 = env.get_record()
    rows = float(rec1[:, 15].double().sum()) - rows0
    conts = float(rec1[:, 16].double().sum()) - cont0
    st = env.stats()
    # the path's only collective: all-reduce of episode statistics over NCCL (SURVEY 8e)
    stat_vec = torch.tensor([st["episodes"], st["return_sum"], st["length_sum"], st["nonfinite"], st["overflow"],
                             rows, conts], device=dev, dtype=torch.float64)
    if dist:
        dist.all_reduce(stat_vec, op=dist.ReduceOp.SUM)
    episodes, ret_sum, len_sum, nonfinite, overflow, rows_all, conts_all = [float(x) for x in stat_vec.tolist()]

    # ---- e2e: same step through the host-buffer C-ABI entry point (pinned host memory, H2D + D2H in the timed region)
    # the same action stream as the device-timed loop, held in pinned host memory (a constant action per env would
    # be a different workload: joints pinned at their limits, more constraint rows)
    h_pool = act_pool.cpu().pin_memory()
    h_obs = torch.empty(N, env.obs_dim, dtype=torch.float32).pin_memory()
    h_rew = torch.empty(N, dtype=torch.float32).pin_memory()
    h_done = torch.empty(N, dtype=torch.uint8).pin_memory()
    h_trunc = torch.empty(N, dtype=torch.uint8).pin_memory()
    outs = (h_obs.numpy(), h_rew.numpy(), h_done.numpy(), h_trunc.numpy())
    h_pool_np = [h_pool[k].numpy() for k in range(pool)]
    for k in range(3):
        env.step_host(h_pool_np[k % pool], outs)
    if dist:
        dist.barrier()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for i in range(K):
        env.step_host(h_pool_np[(W + i) % pool], outs)  # returns once the D2H copies have completed
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if dist:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = N * world * K / float(te.item())
    h2d = N * A * 4
    d2h = N * (env.obs_dim * 4 + 4 + 1 + 1)

    env.close()
    del flush, act_pool, h_pool
    if rank != 0:
        return None

    ms_per_step = total_ms_max / K
    value = N * world * K / (total_ms_max * 1e-3)
    S_sub = 50 * env.physics.substeps if env_kind == "cassie" else env.physics.substeps  # substeps per env step
    R_mean = rows_all / (K * N * world * S_sub)
    n_self = len(env.table.get("self_pairs", [])) if self_collision else 0
    if env_kind == "cassie":  # Cassie: 50 x 1 substeps, n = 24 generalised coordinates, 17 massive links, 158 points
        F = flops_per_env_step(R_mean, S=S_sub, n=24, L=17, G=158)
        B_step = bytes_per_env_step(S_state=49, A=10, O=36, S_env=20)
    elif env_kind == "monkey":  # Monkey3D: n = 29 generalised coordinates, 20 massive links, 29 geoms, obs 69
        F = flops_per_env_step(R_mean, n=29, L=20, G=29, P=n_self)
        B_step = bytes_per_env_step(S_state=59, A=23, O=69, S_env=40)
    elif env_kind in ("stepper", "mike"):
        F = flops_per_env_step(R_mean, L=len([x for x in env.table["mass"] if x > 0]) + 1, G=len(env.table["geoms"]),
                               P=n_self)
        B_step = bytes_per_env_step(O=65, S_env=40)
    elif env_kind in ("walker2d", "crab2d"):  # planar walkers: n = 6 + A, every link massive
        F = flops_per_env_step(R_mean, n=6 + A, L=len(env.table["mass"]) + 1, G=len(env.table["geoms"]), P=n_self)
        B_step = bytes_per_env_step(S_state=13 + 2 * A, A=A, O=env.obs_dim)
    else:
        F = flops_per_env_step(R_mean, P=n_self)
        B_step = bytes_per_env_step()
    kernel_s = (total_ms / K) * 1e-3  # this rank's average launch duration (one kernel per step)
    achieved_tf = F * N / kernel_s / 1e12
    if "fp32_peak" not in ctx:
        ctx["fp32_peak"] = C_peak(_lib, local_rank)
    peak = ctx["fp32_peak"]
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_ach = B_step * N / kernel_s / 1e9
    line = {
        "metric": METRIC.replace("Walker3DCustomEnv", ENV_NAMES[env_kind]
                                 ).replace("16384", str(N)),
        "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": {"custom": WORKLOAD,
                                "stepper": "Walker3DStepperEnv-v0 batched 16384 envs/GPU, seeded stepping stones, "
                                           "curriculum 0/5/9",
                                "monkey": "Monkey3DCustomEnv-v0 batched, seeded monkey bars",
                                "cassie": "CassieEnv-v0 batched, residual PD control, 50 substeps per env step",
                                "child": "Child3DCustomEnv-v0 batched, flat ground, crawl start pose",
                                "walker2d": "Walker2DCustomEnv-v0 batched, flat ground, planar base (SURVEY 8 f3)",
                                "crab2d": "Crab2DCustomEnv-v0 batched, flat ground, planar base (SURVEY 8 f3)",
                                "mike": "MikeStepperEnv-v0 batched, seeded stepping stones, curriculum 0/5/9"}[env_kind],
                   "envs_per_gpu": N, "actions": "random-uniform U(-1,1)^%d (device pool)" % A
                   if actions == "random" else "scripted PD toward running_start (kp=1, kd=0.1, normalised)",
                   "frame_skip": S_sub, "solver_iterations": 5,
                   "self_collision": "on, %d candidate geom pairs per substep" % n_self if n_self else "off", "rng": "mt19937 (NumPy-compatible)",
                   "l2": "flushed between timed steps (256 MiB memset outside the per-step CUDA-event pairs)",
                   "timing": "sum of per-step CUDA-event durations on the launch stream, max over ranks",
                   "parallelism": "env-sharded x%d, no data-path collective" % world},
        "roofline": {"bound": "fp32", "achieved": achieved_tf, "peak": peak, "unit": "TFLOP/s",
                     "frac": achieved_tf / peak if peak else None,
                     # dram__bytes_read.sum + dram__bytes_write.sum per launch of this kernel at 16384 envs: NOT measured
                     # by this run (ncu cannot run inside a timed bench) -- the figure of the committed ncu --set full
                     # capture named in traffic_source; null for other workloads
                     "traffic": NCU_TRAFFIC["bytes"] if (env_kind == "custom" and N == 16384 and self_collision and actions == "random") else None,
                     "traffic_source": NCU_TRAFFIC["source"] if (env_kind == "custom" and N == 16384 and self_collision and actions == "random") else None,
                     "peak_source": "FP32 FMA probe kernel measured in this run (mb200_measure_fp32_peak)",
                     "flops_per_env_step": F, "rows_per_substep": R_mean,
                     "contacts_per_substep": conts_all / (K * N * world * S_sub),
                     "hbm": {"achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                             "bytes_per_env_step": B_step,
                             "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"}},
        "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": K, "api": "mb200_step_host (pinned host buffers, returns when the D2H copies have landed)",
                "actions": "the device loop's random pool, read from pinned host memory"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "episodes": {"finished": episodes, "mean_return": ret_sum / episodes if episodes else None,
                     "mean_length": len_sum / episodes if episodes else None, "nonfinite": nonfinite,
                     "cap_overflows": overflow, "reduced_with": "nccl all_reduce" if dist else "single rank"},
        "wall_s": wall,
    }
    return line


def C_peak(_lib, device):
    import ctypes as C

    out = C.c_double(0.0)
    _lib.check(_lib.lib().mb200_measure_fp32_peak(device, C.byref(out)))
    return out.value


if __name__ == "__main__":
    main()
