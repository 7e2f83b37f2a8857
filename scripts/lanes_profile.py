"""Cycle budget of each warp of the lanes physics kernel: kernel entry to the first substep (prologue: staging the
records and inputs, TakeActions), the substep loop, and observe + write-back.  Needs a -DWB_PHASE_PROFILE build:
scripts/build_variant.sh prof -DWB_PHASE_PROFILE; WB_LIB_PATH=.../libwalker_b200_prof.so python scripts/lanes_profile.py N K WARM L.
Each of the K timed env-steps is read back on its own; the statistics run over all (warp, env-step) samples.  Profiled
builds are for the cycle split only, never for timing."""
import ctypes as C
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import __graft_entry__ as ge

n, K, warm, lanes = (int(v) for v in sys.argv[1:5])
wb = ge.load_package()
wb.init(0)
L = wb.lib()
env = wb.EnvBatch(n, floor_materials="Wood")
env.set_variant(lanes)
ctas = (n * lanes + 31) // 32
rng = np.random.default_rng(0)
acts = [torch.from_numpy(rng.uniform(-1, 1, (n, 4)).astype(np.float32)).cuda() for _ in range(8)]
obs = torch.empty(n, 12, device="cuda")
rew = torch.empty(n, device="cuda")
done = torch.empty(n, dtype=torch.uint8, device="cuda")
env.set_stream(torch.cuda.current_stream().cuda_stream)
for i in range(warm):
    env.step_dev(acts[i % 8], obs, rew, done)
buf = (C.c_uint64 * (3 * ctas))()
samples = []
for i in range(K):
    env.step_dev(acts[i % 8], obs, rew, done)
    assert L.wb_lanes_prof_read(buf, ctas) == 0
    samples.append(np.frombuffer(buf, np.uint64).reshape(ctas, 3).astype(np.float64))
s = np.concatenate(samples)
tot = s.sum(axis=1)
print(f"n={n} lanes={lanes} warps={ctas} samples={len(s)} (cycles per warp-launch)")
for name, v in (("prologue", s[:, 0]), ("substeps", s[:, 1]), ("observe+writeback", s[:, 2]), ("total", tot)):
    print(f"  {name:18s} mean {v.mean():9.0f}  p99 {np.percentile(v, 99):9.0f}  max {v.max():9.0f}  "
          f"share of the mean total {100 * v.mean() / tot.mean():5.1f}%")
slow = np.argmax(tot)
print(f"  slowest warp: total {tot[slow]:.0f}, prologue {s[slow, 0]:.0f}, substeps {s[slow, 1]:.0f}, observe+writeback {s[slow, 2]:.0f}")
