#!/usr/bin/env python
"""Per-phase SM-cycle breakdown of spf_batch_kernel on the C2 workload (debug aid).

usage: phase_profile.py [delta] [general|general_kahn]   (the kernel path, default general)"""
import ctypes as C
import sys

import numpy as np

sys.path.insert(0, ".")
from holo_b200 import capi, synth  # noqa: E402

delta = int(sys.argv[1]) if len(sys.argv) > 1 else 0
path = sys.argv[2] if len(sys.argv) > 2 else "general"
t = synth.random_topology(10000, 40000, synth.SEED_BASE + 2)
csr = synth.topology_csr(t, delta=delta)
ctx = capi.Context(0)
g = ctx.upload(csr)
lib = ctx.lib
lib.hspf_debug_phase_profile.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_uint64)]
roots = np.arange(1000, dtype=np.uint32)
with ctx.path(path):
    ctx.run(g, roots)
    lib.hspf_debug_phase_profile(ctx.handle, 1, None)
    ctx.run(g, roots)
out = (C.c_uint64 * 16)()
lib.hspf_debug_phase_profile(ctx.handle, 0, out)
jump = path != "general_kahn"
names = ["init", "sssp", "parents", "dist_wb", "jump_nh" if jump else "kahn", "jump_hops" if jump else "hops_wb"]
tot = sum(out[k] for k in range(6))
print("delta", delta, "total Mcycles", tot / 1e6, "per job kcycles", tot / 1000 / 1e3)
print("  kahn rounds/job", out[6] / 1000, " sssp rounds/job", out[7] / 1000)
print("  sssp per job: frontier entries", out[12] / 1000, " kcycles: expand(t0)", out[8] / 1e6, " barrier1", out[9] / 1e6,
      " compact", out[10] / 1e6, " barrier2", out[11] / 1e6)
if jump:
    print("  jump per job: hop rounds", out[13] / 1000, " nh rounds", out[14] / 1000, " closure sweeps", out[15] / 1000)
else:
    print("  kahn per job kcycles: expand(t0)", out[13] / 1e6, " barrier1", out[14] / 1e6, " compact+barrier2", out[15] / 1e6)
for k, n in enumerate(names):
    print(f"  {n:8s} {100 * out[k] / tot:5.1f}%  {out[k] / 1000 / 1e3:8.1f} kcycles/job")
