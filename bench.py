#!/usr/bin/env python
"""bench.py -- rectified block-sparse attention call on B200: ms per attention call and dense-equivalent TFLOP/s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3a] [--regime walk] [--impl ours|reference]
                  [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one call of the reference's inner surface (rectified_block_sparse_attention) on one batch of synthetic
bf16 Q/K/V: block pooling -> scores/GAPR -> selection -> C -> block-sparse attention with the fused rectification
epilogue.  Heads are independent, so at N > 1 the heads of ONE call are sharded across ranks with no collective
("scaling": "strong"); value = dense-equivalent FLOP of the whole call / max-over-ranks time.
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(REPO, "rectified-spaattn_b200")
for _p in (REPO, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

# name: family, grid (t,h,w), text tokens, valid text tokens, heads, sa_drop_rate, first-frame rule
WORKLOADS = {
    "c1": dict(desc="synthetic 4x16x16 (1024 tokens), wan path", fam="wan", grid=(4, 16, 16), text=0, text_valid=0,
               heads=12, drop=0.75, ffb=True),
    "c2": dict(desc="Wan2.1-T2V-1.3B 480p 81f, 21x30x52 (32760 tokens)", fam="wan", grid=(21, 30, 52), text=0,
               text_valid=0, heads=12, drop=0.75, ffb=True),
    "c3a": dict(desc="HunyuanVideo 720p 128f (reference default), 32x45x80 + 256 text = 115456 tokens", fam="hunyuan",
                grid=(32, 45, 80), text=256, text_valid=200, heads=24, drop=0.8, ffb=False),
    "c3b": dict(desc="HunyuanVideo 720p 129f (BASELINE.json configs[2]), 33x45x80 + 256 text = 119056 tokens; the "
                     "ragged visual segment (928 blocks + 16 tokens) is zero-padded to 929 blocks inside the kernels",
                fam="hunyuan", grid=(33, 45, 80), text=256, text_valid=200, heads=24, drop=0.8, ffb=False),
    "c4": dict(desc="Wan2.1-T2V-14B 720p 81f, 21x45x80 (75600 tokens)", fam="wan", grid=(21, 45, 80), text=0,
               text_valid=0, heads=40, drop=0.75, ffb=True),
    "c5": dict(desc="Flux.1-dev 4096x4096, 1x256x256 + 512 text = 66048 tokens", fam="flux", grid=(1, 256, 256),
               text=512, text_valid=512, heads=24, drop=0.9, ffb=False),
}
P_REMAIN = 0.3
FLOP_PER_PAIR = 4 * 128 * 128 * 128  # QK^T + PV of one kept (q-block, kv-block) pair at D = 128


def workload_params(name):
    w = WORKLOADS[name]
    t, h, ww = w["grid"]
    nv = t * h * ww
    s = nv + w["text"]
    img_blocks = (nv + 127) // 128 if w["fam"] == "wan" else nv // 128
    top_k = int((1 - w["drop"]) * img_blocks)          # reference scripts/main_hunyuan.py:253 (float truncation)
    ffb = (img_blocks // t) if w["ffb"] else 0         # scripts/main_wan21t2v.py:259
    return dict(w, nv=nv, s=s, top_k=top_k, ffb_blocks=ffb, num_true=nv + w["text_valid"],
                dense_flop_per_head=4.0 * s * s * 128)


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        self.stop_flag = True
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        busy = [x for x in sm if x > 0]
        return {"sm_mhz": busy[len(busy) // 2] if busy else None,
                "sm_max_mhz": int(float(self.rows[0][1])) if self.rows else None,
                "samples": len(self.rows), "reasons": sorted(reasons)}


def parse_cpulist(text):
    """sysfs cpulist ("0-7,16-23", "5") -> set of CPU numbers."""
    cpus = set()
    for part in text.strip().split(","):
        if part:
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def bind_to_gpu_numa_node(local_rank):
    """Multi-rank runs: pin this process to the CPUs of its GPU's NUMA node before any host buffer is allocated, so that
    the pinned tensors of the end-to-end leg live in the memory next to the GPU's PCIe root (what `numactl
    --cpunodebind` does for a one-process-per-GPU launch).  At 8 ranks the H2D copies otherwise fall from 55 to 23 GB/s
    per GPU (`profiles/r01_bench_c3b_8gpu.json`): the buffers of all ranks sit in one socket's memory.  Returns the node
    or None (no NUMA information, or anything unexpected: the run simply goes on unbound)."""
    try:
        import torch
        p = torch.cuda.get_device_properties(local_rank)
        bus = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = parse_cpulist(f.read())
        allowed = os.sched_getaffinity(0) & cpus
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return node
    except Exception:  # noqa: BLE001
        return None


def ncu_traffic(workload):
    """DRAM bytes per launch of kernel 4 from the committed ncu --set full capture of this workload (or None)."""
    # the capture of the shipped kernel (2-CTA clusters, round 2) where there is one, else the round-1 capture of the
    # workload (same kernel without the multicast prefix: 3 % more DRAM bytes at C3b)
    cands = [os.path.join(REPO, "profiles", f"r02_ncu_summary_{workload}_kernel4_cluster.json"),
             os.path.join(REPO, "profiles", f"r02_ncu_summary_{workload}.json"),
             os.path.join(REPO, "profiles", f"r01_ncu_summary_{workload}.json")]
    p = next((c for c in cands if os.path.exists(c)), None)
    if p is None:
        return None
    k = json.load(open(p))["kernels"].get("attn_tc5_kernel", {})
    rd = next((v * (1e9 if "Gbyte" in m else 1e6) for m, v in k.items() if m.startswith("dram__bytes_read.sum")), None)
    wr = next((v * (1e9 if "Gbyte" in m else 1e6) for m, v in k.items() if m.startswith("dram__bytes_write.sum")), None)
    return None if rd is None or wr is None else rd + wr


def kernel0_leg(wp, geo, nbr, heads, dev, timed, peaks, steps):
    """Kernel 0 (rsa_qkv_prep: head split + QK norm + rotary embedding + re-layout + block pooling in one pass over the
    projection outputs; what a processor calls per layer instead of kernel 2) on this workload's shape and family form,
    against the copy bandwidth: algorithmic bytes = Q, K, V read once and written once."""
    import torch

    from rsa_b200 import ops
    s, nv = wp["s"], wp["nv"]
    wan = wp["fam"] == "wan"
    g = torch.Generator(device=dev).manual_seed(0)
    src = [torch.randn(1, s, heads * 128, generator=g, device=dev).to(torch.bfloat16) for _ in range(3)]
    nw = heads * 128 if wan else 128      # Wan: RMSNorm across heads; the joint families: per head
    wq = (1 + 0.1 * torch.randn(nw, generator=g, device=dev)).to(torch.bfloat16)
    wk = (1 + 0.1 * torch.randn(nw, generator=g, device=dev)).to(torch.bfloat16)
    ang = torch.outer(torch.arange(nv, dtype=torch.float32, device=dev),
                      1.0 / (256.0 ** (torch.arange(0, 128, 2, device=dev) / 128)))
    cos, sin = ang.cos().repeat_interleave(2, 1).contiguous(), ang.sin().repeat_interleave(2, 1).contiguous()
    q0, k0, v0 = (torch.empty(1, heads, s, 128, dtype=torch.bfloat16, device=dev) for _ in range(3))
    plan0 = ops.Plan(q0, k0, v0, geo, wp["top_k"], P_REMAIN, nbr, private_workspace=True)

    def fused():
        if wp["text"] and geo.gap:          # ragged visual segment: two sources (dual-stream form)
            plan0.qkv_prep(*(x[:, :nv] for x in src), dst_row=0, q_weight=wq, k_weight=wk, rope=(cos, sin))
            plan0.qkv_prep(*(x[:, nv:] for x in src), dst_row=nv, q_weight=wq, k_weight=wk)
        else:
            plan0.qkv_prep(*src, dst_row=0, q_weight=wq, k_weight=wk, rope=(cos, sin), rope_rows=nv)

    for _ in range(3):      # the first call checks the rotary tables' form once (a host sync) and configures the kernel
        fused()
    ms = timed(fused, steps)
    b_alg = 6 * s * heads * 128 * 2
    del plan0, q0, k0, v0, src
    torch.cuda.empty_cache()
    return {"kernel": "qkv_prep (kernel 0; per layer, replaces kernel 2)", "algorithmic_bytes": b_alg, "ms": ms,
            "achieved_gbs": b_alg / (ms * 1e-3) / 1e9, "peak_gbs": peaks["hbm"],
            "frac": b_alg / (ms * 1e-3) / 1e9 / peaks["hbm"],
            "form": "norm across heads + rotary embedding (Wan)" if wan else "per-head RMSNorm + rotary embedding (joint families)",
            "note": "issue-bound (about 190 instructions per row and thread around diffusers' rounding points), not in the headline call"}


def measured_peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained"), hbm=d["hbm_gbs"],
                    source="measured")
    return dict(bf16=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback")


def synth_heads_device(heads, head0, s, regime, dev, seed=0, d=128):
    """Q, K, V [1, heads, s, d] bf16 on the device (SURVEY 8d regimes), one generator stream per global head."""
    import torch
    nb = (s + 127) // 128
    outs = [torch.empty(1, heads, s, d, dtype=torch.bfloat16, device=dev) for _ in range(3)]
    for hi in range(heads):
        g = torch.Generator(device=dev).manual_seed(seed * 1000 + head0 + hi)
        for ti in range(3):
            x = torch.randn(nb * 128, d, generator=g, device=dev)
            if ti < 2 and regime != "iid":
                mu = torch.randn(nb, d, generator=g, device=dev) * (0.35 if regime == "walk" else 1.0)
                if regime == "walk":
                    mu = torch.cumsum(mu, dim=0)
                x = x + mu.repeat_interleave(128, dim=0)
            outs[ti][0, hi] = x[:s].to(torch.bfloat16)
    return outs


DUMP_BYTES = 32 << 20     # --dump-outputs: float32 bytes written at most (larger outputs are sampled by token row)


def dump_outputs(out_dir, out):
    """--dump-outputs: the attention output [B, S, heads, D] of the timed call as out_dir/output.npy, float32
    [rows, heads, D] of batch 0.  An output above DUMP_BYTES is sampled: a fixed, seeded set of token rows (ascending, all
    heads and columns), the same for every run of a workload, so two builds can be compared element for element."""
    import numpy as np
    import torch
    o = out[0]
    row_bytes = o[0].numel() * 4
    if o.shape[0] * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(o.shape[0], DUMP_BYTES // row_bytes, replace=False))
        o = o[torch.from_numpy(rows).to(o.device)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "output.npy"), o.float().cpu().numpy())


def product_geometry(wp):
    from rsa_b200 import geometry as G
    if wp["fam"] == "wan":
        return G.wan(wp["s"], wp["ffb_blocks"])
    if wp["fam"] == "hunyuan":
        return G.hunyuan(wp["s"], wp["num_true"])
    if wp["fam"] == "flux":
        return G.flux(wp["s"], wp["text"])
    return G.cogvideo(wp["s"], wp["text"])


def entry_point(wp):
    """The reference-facing public call for this family (what a user of the reference calls)."""
    if wp["fam"] == "wan":
        from rectified_spaattn.rectified_wan21_attn import rectified_block_sparse_attention as f
        return lambda q, k, v, nbr: f(q, k, v, None, wp["top_k"], block_neighbor_list=nbr, p_remain_rates=P_REMAIN,
                                      first_frame_blocks=wp["ffb_blocks"])
    if wp["fam"] == "hunyuan":
        from rectified_spaattn.rectified_hunyuan_attn import rectified_block_sparse_attention as f
        cu = [0, wp["num_true"], wp["s"]]
        return lambda q, k, v, nbr: f(q, k, v, None, wp["top_k"], cu_seqlens_q=cu, cu_seqlens_kv=cu,
                                      max_seqlen_q=wp["s"], max_seqlen_kv=wp["s"], block_neighbor_list=nbr,
                                      p_remain_rates=P_REMAIN)
    from rectified_spaattn.rectified_flux_attn import rectified_block_sparse_attention as f
    cu = [0, wp["s"], wp["s"]]
    return lambda q, k, v, nbr: f(q, k, v, None, wp["top_k"], cu_seqlens_q=cu, cu_seqlens_kv=cu, max_seqlen_q=wp["s"],
                                  max_seqlen_kv=wp["s"], block_neighbor_list=nbr, p_remain_rates=P_REMAIN,
                                  text_length=wp["text"])


# --------------------------------------------------------------------------------------------- CPU baseline
class CpuArm:
    """The reference's CPU path on the host cores.  Unit of work = ONE HEAD through the whole call (heads are independent
    and cost the same; a CPU runs them one after the other), every stage and every query block of it -- no proration.

    kind "reference": the reference's own PyTorch code from baseline/_ref (mask builder, GAPR, IPAR, sort / cumsum /
    scatter, R, C, epilogue, cat / permute) on fp32 CPU tensors, with its two CUDA-only pieces -- the Triton launch and
    the flash-attn call -- restated (oracle/ref_cpu.py).  kind "port": the oracle's restatement of all of it, when the
    reference files are not on the box.  Nothing of the product (rsa_b200, librsa_b200.so) is imported here."""

    def __init__(self, wp, regime, threads=None, heads=1):
        import torch

        from oracle import gilbert_oracle as GO
        from oracle import ref_cpu
        from oracle import rsa_oracle as O

        # all the host threads this process may use (torchrun exports OMP_NUM_THREADS=1, which would silently make
        # this a single-thread baseline)
        torch.set_num_threads(threads or len(os.sched_getaffinity(0)))
        self.cores = torch.get_num_threads()
        self.wp, self.O, self.torch = wp, O, torch
        s = wp["s"]
        self.heads = heads
        q, k, v = O.synth_qkv(heads, s, 128, regime, 0)
        t, h, w = wp["grid"]
        self.nbr = GO.gilbert_block_neighbors(t, h, w)
        self.kind = "reference" if ref_cpu.available() else "port"
        if self.kind == "reference":
            self.runner = ref_cpu.ReferenceOnCpu(wp["fam"])
            self.q, self.k, self.v = (torch.from_numpy(x) for x in (q, k, v))
            self.nbr_t = torch.from_numpy(self.nbr)
        else:
            self.q, self.k, self.v = q, k, v
            if wp["fam"] == "wan":
                self.geo = O.geometry_wan(s, wp["top_k"], P_REMAIN, wp["ffb_blocks"])
            elif wp["fam"] == "hunyuan":
                self.geo = O.geometry_hunyuan(s, wp["num_true"], wp["top_k"], P_REMAIN)
            else:
                self.geo = O.geometry_flux(s, wp["text"], wp["top_k"], P_REMAIN)

    def head(self):
        """`heads` heads (default ONE) through the whole call; returns seconds."""
        wp = self.wp
        t0 = time.perf_counter()
        if self.kind == "reference":
            self.runner.call(self.q, self.k, self.v, self.nbr_t, wp["top_k"], P_REMAIN, num_true=wp["num_true"],
                             text_len=wp["text"], first_frame_blocks=wp["ffb_blocks"] or None)
        else:
            self.O.forward(self.q, self.k, self.v, self.geo, self.nbr)
        return time.perf_counter() - t0

    def describe(self, t_head, n_heads_timed):
        wp = self.wp
        what = ("the reference's own PyTorch mask builder / GAPR / R / C / epilogue from baseline/_ref on fp32 CPU tensors, "
                "its Triton launch and flash-attn call restated (oracle/ref_cpu.py)" if self.kind == "reference"
                else "oracle port (reference files not on this box)")
        return dict(value=wp["dense_flop_per_head"] / t_head / 1e12, unit="TFLOP/s (dense-equivalent)", cores=self.cores,
                    kind=self.kind,
                    sample=f"{wp['name']}: ONE head of {wp['heads']} through the whole call (all stages, all "
                           f"{(wp['s'] + 127) // 128} query blocks), {t_head:.2f} s per head, median of {n_heads_timed}; "
                           f"heads are independent and run one after the other on a CPU; {what}",
                    s_per_head=t_head,
                    ms_per_call_all_heads_extrapolated=t_head * wp["heads"] * 1e3)


def cpu_c1_full(regime):
    """BASELINE.json configs[0] (C1: 4x16x16 = 1024 tokens, 12 heads) through the CPU arm IN FULL: all 12 heads,
    median of 5 calls -- no extrapolation."""
    wp = workload_params("c1")
    wp["name"] = "c1"
    arm = CpuArm(wp, regime, heads=wp["heads"])
    arm.head()
    ts = sorted(arm.head() for _ in range(5))
    return {"workload": "c1: " + wp["desc"], "heads": wp["heads"], "ms_per_call": ts[2] * 1e3, "cores": arm.cores,
            "kind": arm.kind, "dense_equiv_tflops": wp["dense_flop_per_head"] * wp["heads"] / ts[2] / 1e12,
            "note": "the whole call, all 12 heads in one invocation, median of 5, no extrapolation"}


# ------------------------------------------------------------------------------------- the reference on the GPU
def load_reference_from_baseline(names):
    """The UNMODIFIED reference's hot-path modules from baseline/_ref (staged by __graft_entry__.build(); git-ignored,
    travels with gpurun).  diffusers / matplotlib are not installed: empty stand-ins for the names the reference imports
    at module scope.  The reference keeps the package name `rectified_spaattn`, which this repo mirrors, so it is aliased."""
    import importlib
    import types
    root = os.path.join(REPO, "baseline", "_ref")
    if not os.path.isdir(os.path.join(root, "rectified_spaattn")):
        return None

    def stub(name, **attrs):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.__dict__.update(attrs)
            sys.modules[name] = m
    try:
        import diffusers  # noqa: F401
    except Exception:  # noqa: BLE001
        for n in ("diffusers", "diffusers.models", "diffusers.models.transformers"):
            stub(n)
        stub("diffusers.models.attention_processor", Attention=object, AttentionProcessor=object)
        stub("diffusers.models.transformers.transformer_wan", _get_qkv_projections=None, _get_added_kv_projections=None)
    # its own alias: the CPU arm (oracle/ref_cpu.py) patches the two CUDA-only functions of ITS copy of these modules
    if "refgpu_rectified_spaattn" not in sys.modules:
        pkg = types.ModuleType("refgpu_rectified_spaattn")
        pkg.__path__ = [os.path.join(root, "rectified_spaattn")]
        sys.modules["refgpu_rectified_spaattn"] = pkg
    return {n: importlib.import_module("refgpu_rectified_spaattn." + n) for n in names}


def reference_on_gpu(name, regime, dev, ours_ms_fn):
    """SURVEY 8d "Reference beside it -- GPU": the unmodified reference (PyTorch eager mask builder in bf16, its Triton
    JIT kernel, flash-attn for the text rows) through its own public entry point on the SAME inputs on this B200, and
    this repository's call on them.  C3a (128 frames) is the largest HunyuanVideo shape the reference runs: on the
    129-frame shape of the headline it raises (rectified_hunyuan_attn.py:356)."""
    import torch
    from rsa_b200 import ops
    wp = workload_params(name)
    wp["name"] = name
    modname = {"wan": "rectified_wan21_attn", "hunyuan": "rectified_hunyuan_attn", "flux": "rectified_flux_attn"}[wp["fam"]]
    try:
        mods = load_reference_from_baseline([modname])
    except Exception as e:  # noqa: BLE001
        return {"unavailable": f"reference import failed: {e!r}"[:300]}
    if mods is None:
        return {"unavailable": "baseline/_ref is not on this box (run __graft_entry__.build() where /root/reference exists)"}
    ref = mods[modname]
    t, h, w = wp["grid"]
    nbr = ops.gilbert_block_neighbors(t, h, w)
    q, k, v = synth_heads_device(wp["heads"], 0, wp["s"], regime, dev)
    s = wp["s"]

    def call_ref():
        if wp["fam"] == "wan":
            return ref.rectified_block_sparse_attention(q, k, v, None, wp["top_k"], block_neighbor_list=nbr,
                                                        p_remain_rates=P_REMAIN, first_frame_blocks=wp["ffb_blocks"])
        if wp["fam"] == "hunyuan":
            am = (torch.arange(s, device=dev) < wp["num_true"]).view(1, 1, 1, s)
            cu = torch.tensor([0, wp["num_true"], s], dtype=torch.int32, device=dev)
            return ref.rectified_block_sparse_attention(q, k.clone(), v.clone(), am, wp["top_k"], cu_seqlens_q=cu,
                                                        cu_seqlens_kv=cu, max_seqlen_q=s, max_seqlen_kv=s,
                                                        block_neighbor_list=nbr, p_remain_rates=P_REMAIN)
        cu = torch.tensor([0, s, s], dtype=torch.int32, device=dev)
        return ref.rectified_block_sparse_attention(q, k, v, None, wp["top_k"], cu_seqlens_q=cu, cu_seqlens_kv=cu,
                                                    max_seqlen_q=s, max_seqlen_kv=s, block_neighbor_list=nbr,
                                                    p_remain_rates=P_REMAIN, text_length=wp["text"])

    stage = {}
    orig_build = ref._build_block_index_with_importance_optimized
    orig_kernel = ref._triton_block_sparse_attention_onehot

    def wrap(key, fn):
        def inner(*a, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a, **kw)
            e1.record()
            torch.cuda.synchronize()
            stage.setdefault(key, []).append(e0.elapsed_time(e1))
            if key == "kernel":
                stage["kept_pairs"] = int(a[4].sum().item())
            return r
        return inner

    def one():
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        o = call_ref()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), o

    try:
        for _ in range(3):      # Triton JIT + warm-up
            one()
        tot = sorted(one()[0] for _ in range(5))
        ref._build_block_index_with_importance_optimized = wrap("mask_build", orig_build)
        ref._triton_block_sparse_attention_onehot = wrap("kernel", orig_kernel)
        for _ in range(3):
            _, o_ref = one()
    except Exception as e:  # noqa: BLE001
        return {"unavailable": f"reference call failed: {e!r}"[:300]}
    finally:
        ref._build_block_index_with_importance_optimized = orig_build
        ref._triton_block_sparse_attention_onehot = orig_kernel
    geo = product_geometry(wp)
    plan = ops.Plan(q, k, v, geo, wp["top_k"], P_REMAIN, nbr)
    ours_ms = ours_ms_fn(plan.run)
    o_ours = plan.run()
    torch.cuda.synchronize()
    rows = min(wp["num_true"], s)
    a, b = o_ours.reshape(1, s, -1)[0, :rows].float(), o_ref.reshape(1, s, -1)[0, :rows].float()
    cos = float(torch.nn.functional.cosine_similarity(a.flatten(), b.flatten(), dim=0))
    ms_ref = tot[len(tot) // 2]
    dense = wp["dense_flop_per_head"] * wp["heads"]
    return {"workload": f"{name}: {wp['desc']}", "regime": regime, "impl": "unmodified reference from baseline/_ref: "
            "rectified_block_sparse_attention -> PyTorch eager mask builder (bf16) + Triton JIT kernel + flash-attn text rows",
            "ms_per_call": ms_ref, "ms_all": tot, "mask_build_ms": sorted(stage["mask_build"])[1],
            "kernel_ms": sorted(stage["kernel"])[1], "kept_pairs": stage.get("kept_pairs"),
            "dense_equiv_tflops": dense / (ms_ref * 1e-3) / 1e12,
            "ours_ms_per_call": ours_ms, "ours_dense_equiv_tflops": dense / (ours_ms * 1e-3) / 1e12,
            "speedup": ms_ref / ours_ms, "output_cosine_ours_vs_reference": cos,
            "note": "same synthetic bf16 inputs, same B200, same process; CUDA events around the whole public call; the "
                    "reference's bf16 mask differs from the fp32 one on near-tie entries (SURVEY 0.5), so outputs agree "
                    "in cosine, not element-wise"}


# ------------------------------------------------------------------- sequence-parallel host models (world > 1)
def ulysses_leg(wp, dev, rank, world, steps=10):
    """SURVEY 8e / 8f rank 3, measured beside the headline (not part of it): the same attention layer for a host model
    that keeps the SEQUENCE sharded over the ranks (Ulysses).  Every rank holds tokens [r S/P, (r+1) S/P) of the Q/K/V
    projection outputs and must end up with the same tokens of the result.
      fused: rsa_b200.parallel.FusedUlysses -- kernel 0 gathers each token's rows from the owning rank's peer-mapped
             buffer over NVLink while it normalises / rotates / pools, kernel 4's epilogue scatters every output row into
             the owning rank's buffer; two one-element all-reduces as barriers, no data collective;
      nccl:  all_to_all_single x3 in, kernel 0 + kernels 3a-4 locally, all_to_all_single out (+ staging copies).
    Both must produce the same bits on every rank."""
    import torch
    import torch.distributed as dist
    from rsa_b200 import ops, parallel
    heads, s, nv = wp["heads"], wp["s"], wp["nv"]
    if heads % world or s % world:
        return {"unavailable": f"{heads} heads / {s} tokens do not divide by {world} ranks"}
    geo = product_geometry(wp)
    t, h, w = wp["grid"]
    nbr = ops.gilbert_block_neighbors(t, h, w)
    rows, hl = s // world, heads // world
    g = torch.Generator(device=dev).manual_seed(1234)            # the same stream on every rank: the full tensors
    full = [torch.randn(1, s, heads * 128, generator=g, device=dev).to(torch.bfloat16) for _ in range(3)]
    mu = torch.cumsum(torch.randn(1, (s + 127) // 128, heads * 128, generator=g, device=dev) * 0.35, dim=1)
    for x in full[:2]:                                           # block structure, as in the headline's inputs
        x.add_(mu.repeat_interleave(128, dim=1)[:, :s].to(torch.bfloat16))
    del mu
    wq = (1 + 0.1 * torch.randn(128, generator=g, device=dev)).to(torch.bfloat16)
    wk = (1 + 0.1 * torch.randn(128, generator=g, device=dev)).to(torch.bfloat16)
    ang = torch.outer(torch.arange(nv, dtype=torch.float32, device=dev),
                      1.0 / (256.0 ** (torch.arange(0, 128, 2, device=dev) / 128)))
    rope = (ang.cos().repeat_interleave(2, 1).contiguous(), ang.sin().repeat_interleave(2, 1).contiguous())
    del ang
    mine = slice(rank * rows, (rank + 1) * rows)
    norm = {} if wp["fam"] == "wan" else dict(q_weight=wq, k_weight=wk, eps=1e-6)   # the fused gather has the per-head norm
    fu = parallel.FusedUlysses(1, heads, geo, wp["top_k"], P_REMAIN, nbr)
    for dst, src in zip((fu.q_src, fu.k_src, fu.v_src), full):
        dst.copy_(src[:, mine])
    run_fused = lambda: fu.run(norm.get("q_weight"), norm.get("k_weight"), 1e-6, rope, nv)
    out = run_fused().clone()
    q, k, v = (torch.empty(1, hl, s, 128, dtype=torch.bfloat16, device=dev) for _ in range(3))
    plan = ops.Plan(q, k, v, geo, wp["top_k"], P_REMAIN, nbr)

    def run_nccl():
        srcs = []
        for x in full:
            loc = x[:, mine].reshape(1, rows, world, hl * 128).permute(2, 0, 1, 3).contiguous()   # [P(dst), 1, rows, hl*128]
            rcv = torch.empty_like(loc)
            dist.all_to_all_single(rcv, loc)
            srcs.append(rcv.permute(1, 0, 2, 3).reshape(1, s, hl * 128))                         # all tokens, my heads
        if geo.gap:
            plan.qkv_prep(*(x[:, :nv] for x in srcs), dst_row=0, rope=rope, **norm)
            plan.qkv_prep(*(x[:, nv:] for x in srcs), dst_row=nv, **norm)
        else:
            plan.qkv_prep(*srcs, dst_row=0, rope=rope, rope_rows=nv, **norm)
        o = plan.run_pooled()                                                                     # [1, S, hl, 128]
        return parallel.head_to_seq_shard(o).reshape(1, rows, heads * 128)

    ref = run_nccl().clone()
    torch.cuda.synchronize()
    same = bool(torch.equal(out.view(torch.int16), ref.view(torch.int16)))

    def timed_max(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        tt = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    ms_fused, ms_nccl = timed_max(run_fused), timed_max(run_nccl)
    oks = [None] * world
    dist.all_gather_object(oks, same)
    fu.close()
    return {"fused_ms": ms_fused, "nccl_all_to_all_form_ms": ms_nccl, "fused_over_nccl": ms_fused / ms_nccl,
            "bitwise_equal": all(oks), "tokens_per_rank": rows, "heads_per_rank": hl,
            "note": "one attention layer of a sequence-parallel (Ulysses) host model: kernel 0 (head split, QK norm, rotary "
                    "embedding, pooling) + kernels 3a-4; fused = gather inside kernel 0 and scatter inside kernel 4's "
                    "epilogue over peer memory; nccl = all_to_all_single x4 + staging copies around the same kernels; "
                    "max over ranks, CUDA events"}


# ------------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3b", choices=list(WORKLOADS))
    ap.add_argument("--regime", default="walk", choices=["walk", "iid", "cluster"])
    ap.add_argument("--attn-flags", type=int, default=0,
                    help="kernel 4 A/B switches (rsa_debug_set_attention_flags): 4 = head_dim 64 through the 128-column "
                         "form, 16 = kernel 4 grid in the former order")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-reference-gpu", action="store_true",
                    help="skip the reference_gpu key (the unmodified reference from baseline/_ref on this GPU)")
    ap.add_argument("--no-permute", action="store_true")
    ap.add_argument("--no-ulysses", action="store_true", help="world > 1: skip the sequence-parallel (Ulysses) leg")
    ap.add_argument("--host-chunk", type=int, default=0,
                    help="heads per chunk of the pipelined host-buffer call (0 = library default: 2, or 1 below 8 heads)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the output of the last timed call to DIR/output.npy (float32; rank 0's heads; token "
                         "rows sampled with a fixed seed when it exceeds 32 MiB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3)

    # stdout carries exactly ONE JSON line.  Native libraries write to file descriptor 1 behind Python's back (NCCL
    # prints "NCCL version ..." there when NCCL_DEBUG is set), so fd 1 is pointed at stderr for the whole run and the
    # result line is written to a private duplicate of the original stdout.
    sys.stdout.flush()
    result_fd = os.dup(1)
    os.dup2(2, 1)
    emit = lambda obj: os.write(result_fd, (json.dumps(obj) + "\n").encode())
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wp = workload_params(args.workload)
    wp["name"] = args.workload
    config = {"workload": f"{args.workload}: {wp['desc']}", "heads": wp["heads"], "tokens": wp["s"], "head_dim": 128,
              "top_k": wp["top_k"], "p_remain_rates": P_REMAIN, "regime": args.regime,
              "parallelism": f"head-parallel x{world}" if world > 1 else "single GPU",
              "l2": "inputs (Q,K,V >= 0.4 GB) exceed the 126 MB L2; no explicit flush"}

    if args.impl == "reference":
        # The reference's own CPU implementation of the path, on the box's host cores, rank 0 only: ONE step = ONE head
        # of this arm's workload through the whole call (CpuArm).  W warm-up steps, then exactly K timed steps.
        if rank != 0:
            return
        arm = CpuArm(wp, args.regime)
        for _ in range(args.warmup):
            arm.head()
        ts = [arm.head() for _ in range(args.steps)]
        t_head = sum(ts) / len(ts)
        base = arm.describe(sorted(ts)[len(ts) // 2], len(ts))
        v = wp["dense_flop_per_head"] / t_head / 1e12
        line = {"impl": "reference", "metric": "dense-equiv TFLOP/s per rectified sparse-attention call", "value": v,
                "unit": "TFLOP/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": t_head * 1e3, "step": "one head of the call (1/%d of its work) on the CPU" % wp["heads"],
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config, "cpu_baseline": dict(base, value=v),
                "e2e": {"value": v, "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "c1_full": cpu_c1_full(args.regime)}
        emit(line)
        return

    import torch
    import torch.distributed as dist

    from rsa_b200 import native, ops

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback on the product path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_node = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert native.lib().rsa_device_ok() == 1
    ops.set_attention_flags(args.attn_flags)

    heads = wp["heads"]
    if heads % world:
        raise SystemExit(f"{heads} heads do not split over {world} ranks")
    h_loc = heads // world
    head0 = rank * h_loc
    t, h, w = wp["grid"]
    nbr = ops.gilbert_block_neighbors(t, h, w)
    q, k, v = synth_heads_device(h_loc, head0, wp["s"], args.regime, dev)
    geo = product_geometry(wp)
    plan = ops.Plan(q, k, v, geo, wp["top_k"], P_REMAIN, nbr)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        """CUDA events on the launching stream; returns max-over-ranks milliseconds per step."""
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        if world > 1:
            tt = torch.tensor([ms], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = float(tt.item())
        sync_all()
        return ms

    def timed_median(fn, steps):
        """Median over `steps` individually event-timed launches (local, no collective): for the short HBM-bound kernels,
        whose mean over a few launches one stray hiccup on the box can double."""
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        ev[0].record()
        for i in range(steps):
            fn()
            ev[i + 1].record()
        torch.cuda.synchronize()
        ts = sorted(ev[i].elapsed_time(ev[i + 1]) for i in range(steps))
        return ts[len(ts) // 2]

    for _ in range(args.warmup):
        plan.run()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_step = timed(plan.run, args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, plan.out)     # before the legs below run the plan again

    # per-stage device times (same launches, timed alone) and the roofline of the dominant kernel
    stages = {}
    for name, fn in (("pool_stats", plan.pool_stats), ("block_scores", plan.block_scores),
                     ("block_select", plan.block_select), ("rect_c", plan.rect_c),
                     ("sparse_attention", plan.sparse_attention)):
        stages[name] = timed(fn, max(3, args.steps))
    # mask re-use (SURVEY 8f rank 4, off in the headline): the same call with the selection of the previous call kept
    reuse = {"keep_lists_ms": timed(lambda: plan.run(native.MASK_KEEP_LISTS), max(3, args.steps // 2)),
             "keep_all_ms": timed(lambda: plan.run(native.MASK_KEEP_ALL), max(3, args.steps // 2)),
             "note": "rsa_rectified_attention_reuse on unchanged inputs: RSA_MASK_KEEP_LISTS skips 3b's sort/threshold/"
                     "scatter and the pair schedule, RSA_MASK_KEEP_ALL runs kernel 4 only; ms_per_step rebuilds every call"}
    # kernel 1 (per transformer forward, not per attention call): Gilbert permute of the hidden states [1, Nv, 3072]
    hbm_kernels = None
    if rank == 0 and not args.no_permute:
        peaks_ = measured_peaks()
        l2h, h2l = ops.gilbert_mapping(t, h, w)
        chans = 3072 if wp["fam"] != "wan" else (1536 if wp["heads"] == 12 else 5120)
        x = torch.randn(1, wp["nv"], chans, device=dev).to(torch.bfloat16)
        xo = torch.empty_like(x)
        idx = h2l.to(dev)
        ms_perm = timed(lambda: ops.permute_rows(x, idx, out=xo), max(5, args.steps)) if world == 1 else None
        if world > 1:   # timed() holds collectives; outside rank 0 nobody joins them, so time locally
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for _ in range(3):
                ops.permute_rows(x, idx, out=xo)
            e0.record()
            for _ in range(10):
                ops.permute_rows(x, idx, out=xo)
            e1.record()
            torch.cuda.synchronize()
            ms_perm = e0.elapsed_time(e1) / 10
        b_perm = 2 * x.numel() * 2
        b_pool = 3 * q.numel() * 2
        ms_perm_med = timed_median(lambda: ops.permute_rows(x, idx, out=xo), max(9, args.steps))
        ms_pool_med = timed_median(plan.pool_stats, max(9, args.steps))
        hbm_kernels = [
            {"kernel": "permute_rows (kernel 1)", "algorithmic_bytes": b_perm, "ms": ms_perm,
             "achieved_gbs": b_perm / (ms_perm * 1e-3) / 1e9, "peak_gbs": peaks_["hbm"],
             "frac": b_perm / (ms_perm * 1e-3) / 1e9 / peaks_["hbm"], "shape": [1, wp["nv"], chans],
             "ms_median": ms_perm_med, "frac_median": b_perm / (ms_perm_med * 1e-3) / 1e9 / peaks_["hbm"]},
            {"kernel": "pool_stats (kernel 2)", "algorithmic_bytes": b_pool, "ms": stages["pool_stats"],
             "achieved_gbs": b_pool / (stages["pool_stats"] * 1e-3) / 1e9, "peak_gbs": peaks_["hbm"],
             "frac": b_pool / (stages["pool_stats"] * 1e-3) / 1e9 / peaks_["hbm"],
             "ms_median": ms_pool_med, "frac_median": b_pool / (ms_pool_med * 1e-3) / 1e9 / peaks_["hbm"],
             "note": "ms / frac: mean over back-to-back launches; *_median: median of individually timed launches (a mean over "
                     "a few sub-millisecond launches is at the mercy of one stray stall on the box)"}]
        del x, xo
        if world == 1:
            hbm_kernels.append(kernel0_leg(wp, geo, nbr, heads, dev, timed, peaks_, max(5, args.steps)))
    clocks = sampler.summary() if rank == 0 else None
    vw = plan.view()
    pairs = int(vw["kept_cnt"].sum().item())
    if world > 1:
        tp = torch.tensor([pairs], device=dev, dtype=torch.int64)
        dist.all_reduce(tp)
        pairs_all = int(tp.item())
    else:
        pairs_all = pairs
    nqt = geo.n_blocks
    density = pairs_all / (heads * nqt * nqt)

    # end to end through the public entry point with HOST buffers (pinned): the per-family call receives host tensors
    # and returns a host tensor; inside, rsa_rectified_attention_host pipelines H2D | kernels | D2H over chunks of
    # heads.  For comparison the same call with three blocking-order copies around a device call ("serial").
    e2e = None
    if not args.no_e2e:
        call = entry_point(wp)
        ops.HOST_HEADS_PER_CHUNK = args.host_chunk or None
        host_chunk = args.host_chunk or (2 if h_loc >= 8 else 1)
        hq, hk, hv = (x.cpu().pin_memory() for x in (q, k, v))
        ho = torch.empty((1, wp["s"], h_loc * 128), dtype=torch.bfloat16).pin_memory()
        dq_, dk_, dv_ = (torch.empty_like(x) for x in (q, k, v))
        res = {}

        def e2e_step():
            res["o"] = call(hq, hk, hv, nbr)

        def serial_step():
            dq_.copy_(hq, non_blocking=True)
            dk_.copy_(hk, non_blocking=True)
            dv_.copy_(hv, non_blocking=True)
            o = call(dq_, dk_, dv_, nbr)
            ho.copy_(o, non_blocking=True)

        for _ in range(2):
            e2e_step()
            serial_step()
        n_e2e = max(3, args.steps // 2)
        ms_e2e = timed(e2e_step, n_e2e)
        ms_serial = timed(serial_step, max(3, args.steps // 4))

        def h2d_only():
            dq_.copy_(hq, non_blocking=True)
            dk_.copy_(hk, non_blocking=True)
            dv_.copy_(hv, non_blocking=True)

        ms_h2d = timed(h2d_only, 3)
        # the copy ceiling of this step on this box: the step's bytes in BOTH directions at once (H2D of Q, K, V on one
        # stream, D2H of the result on another), all ranks together, no kernels -- PCIe is not full duplex at full rate
        # here (one GPU: 55 GB/s in alone, 71 GB/s in + out together), and 8 GPUs share the host's root ports
        do_ = torch.empty((1, wp["s"], h_loc * 128), dtype=torch.bfloat16, device=dev)
        side = torch.cuda.Stream()

        def copies_only():
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                ho.copy_(do_, non_blocking=True)
            h2d_only()
            torch.cuda.current_stream().wait_stream(side)

        ms_copies = timed(copies_only, 3)
        assert torch.equal(res["o"].view(torch.int16), ho.view(torch.int16)), "pipelined and serial results differ"
        bi = 3 * q.numel() * 2 * world
        bo = ho.numel() * 2 * world
        e2e = {"value": wp["dense_flop_per_head"] * heads / (ms_e2e * 1e-3) / 1e12, "unit": "TFLOP/s",
               "ms_per_step": ms_e2e, "h2d_bytes_per_step": bi, "d2h_bytes_per_step": bo,
               "path": f"public per-family entry point on pinned host tensors -> rsa_rectified_attention_host, "
                       f"{host_chunk} head(s) per chunk (the last {host_chunk} heads one per chunk), H2D | kernels | D2H on three streams",
               "ms_per_step_unpipelined": ms_serial,
               "h2d_only_ms": ms_h2d, "copies_only_ms": ms_copies, "frac_of_copy_ceiling": ms_copies / ms_e2e,
               "copy_ceiling_note": "copies_only_ms = this step's H2D and D2H bytes moved concurrently by all ranks with no "
                                    "kernel in between: the floor of any end-to-end schedule on this box",
               "host_numa_node_rank0": numa_node}

    ulysses = None
    if world > 1 and not args.no_ulysses:
        try:
            del plan
            torch.cuda.empty_cache()
            ulysses = ulysses_leg(wp, dev, rank, world)
        except Exception as e:  # noqa: BLE001
            ulysses = {"unavailable": repr(e)[:300]}
        plan = None
    if rank == 0:
        peaks = measured_peaks()
        t_attn = stages["sparse_attention"]
        achieved = FLOP_PER_PAIR * (pairs_all / world) / (t_attn * 1e-3) / 1e12   # per GPU
        line = {
            "metric": "dense-equiv TFLOP/s per rectified sparse-attention call", "value":
                wp["dense_flop_per_head"] * heads / (ms_step * 1e-3) / 1e12,
            "unit": "TFLOP/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": config, "ms_per_attn_call": ms_step, "kept_pair_density": density, "stages_ms": stages,
            "mask_reuse": reuse,
            "attention_impl": "tcgen05 (the library's only attention kernel)",
            "attention_flags": args.attn_flags,
            "gpu_launches": 7 * args.steps,
            "roofline": {"bound": "tensor", "kernel": "rect_attn (kernel 4)", "achieved": achieved,
                         "peak": peaks["bf16"], "unit": "TFLOP/s", "frac": achieved / peaks["bf16"],
                         "peak_source": f"{peaks['source']} cuBLAS bf16 burst (kernel timed alone, back to back); "
                                        f"sustained peak {peaks['bf16_sustained']}",
                         "frac_of_sustained_peak": achieved / peaks["bf16_sustained"] if peaks["bf16_sustained"] else None,
                         "flop_per_kept_pair": FLOP_PER_PAIR, "kept_pairs_per_launch": pairs_all // world,
                         "ms_per_launch": t_attn, "traffic": ncu_traffic(args.workload) if world == 1 else None,
                         "traffic_note": "DRAM read+write bytes of one launch, ncu --set full, profiles/r02_ncu_summary_<workload>_kernel4_cluster.json (else the r01 capture)"},
            "clocks": clocks,
        }
        if hbm_kernels:
            line["hbm_kernels"] = hbm_kernels
        if e2e:
            line["e2e"] = e2e
        if ulysses:
            line["ulysses"] = ulysses
        if world == 1 and not args.no_cpu_baseline:
            arm = CpuArm(wp, args.regime)
            line["cpu_baseline"] = arm.describe(arm.head(), 1)
            line["cpu_baseline"]["c1_full"] = cpu_c1_full(args.regime)
        if world == 1 and not args.no_reference_gpu:
            # the bar to beat: the unmodified reference on this GPU, on the largest HunyuanVideo shape it can run
            del plan, q, k, v
            torch.cuda.empty_cache()
            line["reference_gpu"] = reference_on_gpu("c3a" if args.workload == "c3b" else args.workload, args.regime, dev,
                                                     lambda fn: timed(fn, max(5, args.steps // 2)))
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
