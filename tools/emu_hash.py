#!/usr/bin/env python
"""Bit-level fingerprint of the kernel source (g++ lane-loop emulation, tests/emu): seeded rollouts of every env kind,
CRC of every observation / reward / state / record and of the accumulated episode statistics.  A refactoring that only moves addressing around (no change of the
floating-point operations or their order) must leave every line unchanged:

    python tools/emu_hash.py > /tmp/before.txt;  <edit>;  python tools/emu_hash.py | diff /tmp/before.txt -
"""
import os
import sys
import zlib

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from tests.emu import emu  # noqa: E402


def mt_state(seed):
    return np.random.RandomState(seed).get_state()[1].astype(np.uint32).tolist() + [624]


def rollout(env, act_dim, steps, seed, scale=1.0):
    rng = np.random.RandomState(seed)
    crc = zlib.crc32(env.reset().tobytes())
    ndone = 0
    for _ in range(steps):
        obs, rew, done, trunc, fin = env.step(scale * rng.uniform(-1, 1, act_dim))
        crc = zlib.crc32(obs.tobytes() + np.float32(rew).tobytes() + env.state.tobytes() + env.rec.tobytes() +
                         env.stats.tobytes(), crc)
        ndone += done
    return "%08x episodes %d" % (crc, ndone)


def main():
    steps = int(sys.argv[1]) if len(sys.argv) > 1 else 60
    for seed in (1, 2):
        m = np.zeros(625, dtype=np.uint32)
        m[:] = mt_state(seed)
        print("w3d", seed, rollout(emu.EmuW3D(m), 21, steps, seed))
        print("child", seed, rollout(emu.EmuChild(m), 21, steps, seed))
        print("walker2d", seed, rollout(emu.EmuWalker2D(m), 7, steps, seed))
        print("crab2d", seed, rollout(emu.EmuCrab2D(m), 6, steps, seed))
        for cur in (0, 9):
            print("stepper c%d" % cur, seed, rollout(emu.EmuStepper(m, cur), 21, steps, seed, 0.4))
        print("pillar", seed, rollout(emu.EmuPillar(m, 5), 21, steps, seed, 0.4))
        print("mike", seed, rollout(emu.EmuMike(m, 5), 21, steps, seed, 0.4))
        print("monkey", seed, rollout(emu.EmuMonkey(m), 23, steps, seed))
        print("cassie", seed, rollout(emu.EmuCassie(), 10, max(steps // 6, 4), seed))


if __name__ == "__main__":
    main()
