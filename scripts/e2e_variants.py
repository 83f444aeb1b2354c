"""A/B of the host step path variants (run on a GPU box): prints us per BlueSkyVectorEnv.step()."""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from bluesky_gym_sasha_b200.vector_env import BlueSkyVectorEnv

E = int(os.environ.get("E", 4096))
v = BlueSkyVectorEnv("HorizontalCREnv-v0", E, seed=0, cd_enabled=True, n_intruders=20, autoreset_mode=os.environ.get("MODE", "same_step"))
v.reset()
a = np.random.default_rng(0).uniform(-1, 1, (E, 1)).astype(np.float32)
for _ in range(30):
    v.step(a)
torch.cuda.synchronize()
t0 = time.perf_counter()
for _ in range(500):
    v.step(a)
torch.cuda.synchronize()
print("threads=%s mode=%s copy=True : %.1f us" % (os.environ.get("BSG_HOST_THREADS", "4"), v.autoreset_mode,
                                                 (time.perf_counter() - t0) / 500 * 1e6))
v.copy = False
t0 = time.perf_counter()
for _ in range(500):
    v.step(a)
torch.cuda.synchronize()
print("   copy=False: %.1f us" % ((time.perf_counter() - t0) / 500 * 1e6))
