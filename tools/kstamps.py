"""Kernel-level timeline of one step in steady state (debug build with -DGCA_PHASE_TIMING).
Usage on the GPU box: python tools/kstamps.py   (builds lib/libgca_timing.so first)"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "gym-guidance-collision-avoidance-single_b200")
sys.path[:0] = [ROOT, PKG]
lib_path = os.path.join(PKG, "lib", "libgca_timing.so")
if not os.path.exists(lib_path) or os.environ.get("GCA_REBUILD"):
    csrc = os.path.join(PKG, "csrc")
    cu = sorted(os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cu"))
    subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-fmad=false", "-std=c++17",
                           "-DGCA_PHASE_TIMING", "-Xcompiler", "-fPIC", "-shared", "-I" + os.path.join(ROOT, "include"), "-I" + csrc]
                          + cu + ["-o", lib_path])
os.environ["GCA_LIB"] = lib_path
import torch  # noqa: E402
from gca_b200 import abi  # noqa: E402
from gca_b200.batched import BatchedAircraftEnv  # noqa: E402
from gym_guidance_collision_avoidance_single.envs.config import Config  # noqa: E402

B, N = 65536, int(os.environ.get("GCA_N", "80"))
PRE = int(os.environ.get("GCA_PRESTEPS", "300"))
env = BatchedAircraftEnv("SingleAircraft2Env", B, Config, n_intruders=N, mode="fast", seed=1)
env.reset()
acts = [torch.rand((B, 2), device="cuda") * 2 - 1 for _ in range(8)]
lib = abi.load()
lib.gca_debug_kstamps.argtypes = [C.c_void_p, C.c_int]
buf = np.zeros(8, np.uint64)
g1 = torch.cuda.CUDAGraph()
side = torch.cuda.Stream()
with torch.cuda.stream(side):
    for i in range(PRE):
        env.step(acts[i % 8])
torch.cuda.synchronize()
with torch.cuda.graph(g1):
    env.step(acts[0])
g8 = torch.cuda.CUDAGraph()
with torch.cuda.graph(g8):
    for i in range(8):
        env.step(acts[i])


def show(st, label):
    t0 = int(min(st[0], st[2], st[4]))
    rel = lambda v: (int(v) - t0) / 1e3
    print(label)
    print("  ownship kernel    first in %7.2f   last out %7.2f" % (rel(st[0]), rel(st[1])))
    print("  finish kernel     first in %7.2f   last out %7.2f" % (rel(st[4]), rel(st[5])))
    print("  streaming kernel  first in %7.2f   last out %7.2f   first record seen %7.2f" % (rel(st[2]), rel(st[3]), rel(st[7])))


for rep in range(3):
    g8.replay()
    lib.gca_debug_kstamps(buf.ctypes.data, 1)          # (syncs through the symbol copy)
    g8.replay()
    torch.cuda.synchronize()
    lib.gca_debug_kstamps(buf.ctypes.data, 1)
    st = buf.astype(np.int64)
    print("8-step graph: first in .. last out = %.2f us per step" % ((max(st[1], st[3], st[5]) - min(st[0], st[2], st[4])) / 8e3))
    g1.replay()
    torch.cuda.synchronize()
    lib.gca_debug_kstamps(buf.ctypes.data, 1)
    show(buf.astype(np.int64), "single-step graph (us, relative to the first block of the step):")
env.check()
# per-block timeline of the streaming kernel of the last single-step graph
cb = np.zeros(8192 * 2, np.uint64)
lib.gca_debug_cta.argtypes = [C.c_void_p]
lib.gca_debug_cta(cb.ctypes.data)
c = cb.astype(np.int64).reshape(8192, 2)
c = c[(c[:, 0] > 0) & (c[:, 1] > 0)]
t0 = c[:, 0].min()
start, end = (c[:, 0] - t0) / 1e3, (c[:, 1] - t0) / 1e3
print("streaming blocks: %d, lifetime us mean %.2f p50 %.2f p90 %.2f max %.2f" % (len(c), (end - start).mean(), np.median(end - start), np.percentile(end - start, 90), (end - start).max()))
edges = np.arange(0, end.max() + 4, 4.0)
for lo in edges:
    m = (end >= lo) & (end < lo + 4)
    if m.any():
        print("  t=%5.1f..%5.1f  blocks finished %5d  mean lifetime %.2f  resident at t %d" % (lo, lo + 4, m.sum(), (end - start)[m].mean(), ((start <= lo) & (end > lo)).sum()))
# per-tile phases of the finish kernel: start, loads, replay, reward + stores, reset + counters, spawn (i)
fb = np.zeros(2048 * 8, np.uint64)
lib.gca_debug_fin.argtypes = [C.c_void_p]
lib.gca_debug_fin(fb.ctypes.data)
f = fb.astype(np.int64).reshape(2048, 8)
f = f[f[:, 0] > 0]
dur = (f[:, 1] - f[:, 0]) / 1e3
print("finish_tile per tile (us): mean %.2f p50 %.2f p90 %.2f p99 %.2f max %.2f" % (dur.mean(), np.median(dur), np.percentile(dur, 90), np.percentile(dur, 99), dur.max()))
print("finish phases (us, mean): loads %.2f  replay %.2f  reward+stores %.2f  reset+counters %.2f  spawn phase (i) %.2f" % (
    ((f[:, 4] - f[:, 0]) / 1e3).mean(), ((f[:, 5] - f[:, 4]) / 1e3).mean(), ((f[:, 6] - f[:, 5]) / 1e3).mean(),
    ((f[:, 1] - f[:, 6]) / 1e3).mean(), ((f[:, 7] - f[:, 1]) / 1e3).mean()))
print("per tile (mean): respawn records %.2f, resets %.2f" % (f[:, 2].mean(), f[:, 3].mean()))
t0 = f[:, 0].min()
print("relative to the first finish warp: finish_tile starts p50 %.2f max %.2f; ends max %.2f; spawn (i) ends max %.2f" % (
    (np.median(f[:, 0]) - t0) / 1e3, (f[:, 0].max() - t0) / 1e3, (f[:, 1].max() - t0) / 1e3, (f[:, 7].max() - t0) / 1e3))
# position-load latency of the streaming pass (clock64 cycles from issue to data), by eighth of the walk order:
# what the previous step wrote last is read first - L2 hits there show as a low-latency mode
lb = np.zeros(8 * 64, np.uint32)
lib.gca_debug_lat.argtypes = [C.c_void_p, C.c_int]
lib.gca_debug_lat(lb.ctypes.data, 1)
for rep in range(2):
    g8.replay()
    torch.cuda.synchronize()
    lib.gca_debug_lat(lb.ctypes.data, 1)
    h = lb.astype(np.int64).reshape(8, 64)
    print("position-load latency histogram (work items per 256-cycle bin: 0-255, 256-511, ...; last bin = 3840+), 8 steps:")
    for o in range(8):
        row = h[o].reshape(16, 4).sum(1)
        cdf = np.cumsum(h[o]) / max(1, h[o].sum())
        med = int(np.searchsorted(cdf, 0.5)) * 64
        print("  eighth %d of the walk: median %5d cycles  " % (o, med) + " ".join("%5d" % v for v in row))
