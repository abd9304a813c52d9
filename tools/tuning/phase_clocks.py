"""Phase timeline of fot_sweep_items (tuning aid): runs the bench workload against a library built
with -DFOT_PHASE_CLOCKS and prints the share of warp-cycles spent between the kernel's barriers.

  nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false -Xcompiler -fPIC -shared \\
       -DFOT_PHASE_CLOCKS -I include -o tools/tuning/libfot_clk.so integrated_path_planning_b200/csrc/fot_api.cu
"""
import ctypes as C, os, sys
os.environ["FOT_SWEEP"] = "items"     # the only kernel with phase marks; the default fot_sweep_pairs has none
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))  # repo root
sys.path.insert(0, ROOT)
from integrated_path_planning_b200 import _lib
_lib.LIB_PATH = os.path.join(ROOT, "tools/tuning/libfot_clk.so")
import torch
import bench
from tests import scenarios
from integrated_path_planning_b200 import BatchFrenetPlanner, DeviceBatch
nq = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
spline, frenet, dyn = bench.make_queries(0, nq)
planner = BatchFrenetPlanner(spline, device=0, **scenarios.S1_KNOBS)
batch = DeviceBatch(planner, frenet, bench.TARGET_SPEED, dyn, _lib.FOT_DYN_SINGLE)
lib = _lib.load()
buf = (C.c_ulonglong * 16)()
for _ in range(3):
    batch.launch(None)
lib.fot_debug_phase_clocks(buf)
batch.launch(None)
lib.fot_debug_phase_clocks(buf)
v = list(buf)
names = ["A work", "A barrier", "B work (items, jerk)", "B barrier", "C work (lists, validity loop)", "C barrier",
         "D cull", "D cull barrier", "D process+slow", "D process barrier", "E work", "E barrier"]
tot = sum(v[:12])
for n, x in zip(names, v[:12]):
    print(f"{n:32s} {x / tot * 100:6.2f} %   {x / (nq * 12 * 10):9.0f} cycles per warp per block")
print("total cycles per warp per block", tot / (nq * 12 * 10))

print(f"validity screen: valid items {v[12]:.3e}, dirty items {v[13]:.3e} ({v[13] / max(v[12], 1) * 100:.1f} %), warps with valid items "
      f"{v[14] & 0xffffffff:.3e}, of them skipped {v[15]:.3e} ({v[15] / max(v[14] & 0xffffffff, 1) * 100:.1f} %), full-chain warps "
      f"{v[14] >> 32:.3e} ({(v[14] >> 32) / max(v[14] & 0xffffffff, 1) * 100:.1f} %)")
