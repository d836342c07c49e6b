"""Kernel 0 in fp16 against bf16 (run on the GPU box), in one process, the two dtypes alternating:
  * kernel 0 with pooling (rsa_qkv_prep, what the sparse fused path runs) at C3b (HunyuanVideo 720p 129f: two launches,
    visual and text tokens), C4 (Wan2.1-14B 720p: RMSNorm across heads), C5 (Flux 4096^2: RMSNorm per head),
    CogVideoX1.5 (42 466 tokens x 48 heads x 64, LayerNorm(64), rotary embedding) and CogVideoX-2B (480x720 x 49
    frames: 13x30x45 + 226 = 17 776 tokens x 30 heads x 64, LayerNorm(64), no rotary embedding; pooled as one segment,
    because the CogVideoX block geometry (rsa_b200.geometry.cogvideo, the reference's rule) has no layout for 17 550
    visual tokens, which do not fill whole blocks, in front of 226 text tokens);
  * at CogVideoX-2B's head configuration, one whole fp16 attention layer through
    RectifiedCogVideoXVideoSpaAttnProcessor2_0 on a stand-in module (tests/fake_attention.py, dim 1920): fused
    (fuse_prep_fp16) against op by op (fuse_prep = False), at a sparse step and at a dense call (fuse_prep_dense).  The
    video tokens are rounded up to whole blocks (138 x 128 = 17 664, + 226 text = 17 890 tokens) for the reason above;
  * the card's name and power limit (read-only nvidia-smi query), in the same run.
Each timing is the median of 7 rounds of 10 launches (CUDA events); bf16 and fp16 alternate round by round.  The inputs
(2.2 GB of projection outputs per dtype at C3b) are larger than L2 except at the CogVideoX shapes.
One JSON line per shape; with an argument, the lines are also written to that file."""
import json
import os
import statistics
import subprocess
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [REPO, os.path.join(REPO, "rectified-spaattn_b200"), os.path.join(REPO, "tests")]
sys.argv, argv = [sys.argv[0]], sys.argv[1:]
import bench  # noqa: E402
from fake_attention import FakeAttention  # noqa: E402
from rectified_spaattn import rectified_cogvideo_attn as cog  # noqa: E402
from rsa_b200 import geometry as G  # noqa: E402
from rsa_b200 import ops  # noqa: E402

dev = torch.device("cuda:0")
DTYPES = (torch.bfloat16, torch.float16)
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True, timeout=30).stdout.strip()
lines = []


def emit(d):
    d["card"] = card
    print(json.dumps(d), flush=True)
    lines.append(d)


def alternating(fns, rounds=7, n=10):
    """Median ms per call of each function; the functions take turns round by round."""
    for fn in fns:
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    times = [[] for _ in fns]
    for _ in range(rounds):
        for i, fn in enumerate(fns):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            torch.cuda.synchronize()
            times[i].append(e0.elapsed_time(e1) / n)
    return [statistics.median(t) for t in times], [max(t) - min(t) for t in times]


def shape(name):
    """(desc, heads, head_dim, s, nv, geo, top_k, nbr, norm kind, rope rows) of a benchmark shape."""
    if name in ("c3b", "c4", "c5"):
        wp = bench.workload_params(name)
        t, h, w = wp["grid"]
        kind = {"wan": "wan", "hunyuan": "rms", "flux": "rms"}[wp["fam"]]
        return (wp["desc"], wp["heads"], 128, wp["s"], wp["nv"], bench.product_geometry(wp), wp["top_k"],
                ops.gilbert_block_neighbors(t, h, w), kind, wp["s"] if kind == "wan" else wp["nv"])
    (t, h, w), heads = ((11, 48, 80), 48) if name == "cogvideox1.5" else ((13, 30, 45), 30)
    nv, text = t * h * w, 226
    geo = G.cogvideo(nv + text, text) if name == "cogvideox1.5" else G.wan(nv + text)   # 2B: one segment (see above)
    return (f"{name} {t}x{h}x{w} + {text} text = {nv + text} tokens x {heads} heads x 64", heads, 64, nv + text, nv,
            geo, int((1 - 0.75) * (nv // 128)), ops.gilbert_block_neighbors(t, h, w) if name == "cogvideox1.5" else None,
            "layer",
            nv if name == "cogvideox1.5" else 0)


def kernel0(name):
    desc, heads, hd, s, nv, geo, top_k, nbr, kind, n_rope = shape(name)
    g = torch.Generator(device=dev).manual_seed(0)
    src32 = [torch.randn(1, s, heads * hd, generator=g, device=dev) for _ in range(3)]
    nw = heads * 128 if kind == "wan" else hd
    w32 = [1 + 0.1 * torch.randn(nw, generator=g, device=dev) for _ in range(2)]
    b32 = [0.05 * torch.randn(hd, generator=g, device=dev) for _ in range(2)]
    ang = torch.outer(torch.arange(max(n_rope, 1), dtype=torch.float32, device=dev),
                      1.0 / (256.0 ** (torch.arange(0, hd, 2, device=dev) / hd)))
    rope = (ang.cos().repeat_interleave(2, 1).contiguous(), ang.sin().repeat_interleave(2, 1).contiguous())
    calls, plans = [], []
    for dt in DTYPES:
        src = [x.to(dt) for x in src32]
        prm = dict(q_weight=w32[0].to(dt), k_weight=w32[1].to(dt), eps=1e-6, allow_fp16=True)
        if kind == "layer":
            prm.update(q_bias=b32[0].to(dt), k_bias=b32[1].to(dt))
        q, k, v = (torch.empty(1, heads, s, hd, dtype=dt, device=dev) for _ in range(3))
        plan = ops.Plan(q, k, v, geo, top_k, bench.P_REMAIN, nbr, private_workspace=True)
        plans.append(plan)

        def call(plan=plan, src=src, prm=prm):
            if geo.gap:         # ragged visual segment (C3b): the visual and the text tokens, two launches
                plan.qkv_prep(*(x[:, :nv] for x in src), dst_row=0, rope=rope, **prm)
                plan.qkv_prep(*(x[:, nv:] for x in src), dst_row=nv, **prm)
            elif n_rope:
                plan.qkv_prep(*src, dst_row=0, rope=rope, rope_rows=n_rope, **prm)
            else:
                plan.qkv_prep(*src, dst_row=0, **prm)
        calls.append(call)
    (ms_bf16, ms_f16), (sp_bf16, sp_f16) = alternating(calls)
    emit({"shape": name, "desc": desc, "what": "kernel 0 with pooling (rsa_qkv_prep)",
          "bf16_ms": ms_bf16, "fp16_ms": ms_f16, "fp16_over_bf16": ms_f16 / ms_bf16,
          "bf16_round_spread_ms": sp_bf16, "fp16_round_spread_ms": sp_f16,
          "algorithmic_bytes": 6 * s * heads * hd * 2, "fp16_q_finite": bool(torch.isfinite(plans[1].q).all())})


def cog2b_layer():
    t, h, w, text, heads, dim = 13, 30, 45, 226, 30, 1920
    nv = -(-t * h * w // 128) * 128                     # 17 664: whole blocks (see the top of this file)
    torch.manual_seed(0)
    attn = FakeAttention(dim, heads, head_dim=64, norm="layer").to(dev).to(torch.float16)
    g = torch.Generator(device=dev).manual_seed(1)
    mu = torch.cumsum(torch.randn(-(-nv // 128), dim, generator=g, device=dev) * 0.35, 0).repeat_interleave(128, 0)[:nv]
    x = (torch.randn(nv, dim, generator=g, device=dev) + mu)[None].to(torch.float16)
    txt = torch.randn(1, text, dim, generator=g, device=dev).to(torch.float16)
    for dense in (False, True):
        prs = []
        for fused in (True, False):
            pr = cog.RectifiedCogVideoXVideoSpaAttnProcessor2_0("sparse", int((1 - 0.75) * (nv // 128)), None,
                                                                bench.P_REMAIN)
            pr.fuse_prep, pr.fuse_prep_dense, pr.fuse_prep_fp16 = fused, dense and fused, fused
            prs.append(pr)

        def call(pr):
            pr.current_step = 0 if dense else 5         # call 0: dense (fullattn "flash"); from call 5 on: sparse
            with torch.no_grad():
                return pr(attn, x, txt, None, None)
        (ms_fused, ms_eager), (sp_f, sp_e) = alternating([lambda: call(prs[0]), lambda: call(prs[1])], rounds=5, n=5)
        a, b = (torch.cat(call(pr), dim=1).float() for pr in prs)
        cos = float((a * b).sum() / (a.norm() * b.norm()))
        emit({"shape": f"cogvideox-2b heads, {nv} + {text} tokens", "what": f"one fp16 attention layer, {'dense call 0' if dense else 'sparse step'}",
              "fused_ms": ms_fused, "op_by_op_ms": ms_eager, "fused_round_spread_ms": sp_f,
              "op_by_op_round_spread_ms": sp_e, "output_cosine_fused_vs_op_by_op": cos,
              "output_max_abs_diff": float((a - b).abs().max()), "module": f"stand-in, dim {dim}, LayerNorm(64) + bias"})


for name in ("c3b", "c4", "c5", "cogvideox1.5", "cogvideox-2b"):
    kernel0(name)
    torch.cuda.empty_cache()
cog2b_layer()
if argv:
    os.makedirs(os.path.dirname(os.path.abspath(argv[0])), exist_ok=True)
    with open(argv[0], "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")
