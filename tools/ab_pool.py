"""Kernel 2 timing on one workload, cold (GPU idle before) and hot (right after 20 full calls, i.e. under the power cap,
which is the state it runs in inside a denoising loop)."""
import json, os, subprocess, sys
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO); sys.path.insert(0, os.path.join(REPO, "rectified-spaattn_b200"))
name = sys.argv[1] if len(sys.argv) > 1 else "c3b"
sys.argv = [sys.argv[0]]
import torch
import bench
from rsa_b200 import ops
dev = torch.device("cuda:0")
wp = bench.workload_params(name)
q, k, v = bench.synth_heads_device(wp["heads"], 0, wp["s"], "walk", dev)
nbr = ops.gilbert_block_neighbors(*wp["grid"])
plan = ops.Plan(q, k, v, bench.product_geometry(wp), wp["top_k"], bench.P_REMAIN, nbr)
x = torch.empty(1 << 28, dtype=torch.bfloat16, device=dev); y = torch.empty_like(x)

def smi():
    o = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,clocks.mem,power.draw", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return o

def t(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n

b = 3 * q.numel() * 2
res = {"workload": name}
for _ in range(5):
    plan.pool_stats()
torch.cuda.synchronize()
ms = t(plan.pool_stats, 50); res["cold_ms"] = ms; res["cold_frac"] = b / ms / 1e6 / 6469.9
ms = t(lambda: y.copy_(x), 20); res["cold_copy_GBps"] = 2 * x.numel() * 2 / ms / 1e6
for _ in range(20):
    plan.run()
ms = t(plan.pool_stats, 20); res["hot_ms"] = ms; res["hot_frac"] = b / ms / 1e6 / 6469.9; res["smi_after_hot"] = smi()
for _ in range(20):
    plan.run()
ms = t(lambda: y.copy_(x), 20); res["hot_copy_GBps"] = 2 * x.numel() * 2 / ms / 1e6
for _ in range(20):
    plan.run()
ms = t(plan.pool_stats, 200); res["hot_then_200_ms"] = ms
print(json.dumps(res))
