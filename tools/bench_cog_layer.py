"""CogVideoX1.5 at its real shape (run on the GPU box): 11x48x80 = 42 240 video + 226 text = 42 466 tokens, 48 heads x 64,
top_k 82 (the defaults of tools/bench_hd64.py).  Measures
  * kernel 0 at 64 columns (rsa_qkv_prep: head split + LayerNorm(64) + rotary embedding on the video tokens + re-layout
    + pooling) against the PyTorch sequence it replaces (oracle/make_golden.torch_prep_cog on q and k, then kernel 2
    pooling the result), with its algorithmic bytes 6*S*H*64*2 over the measured copy bandwidth and the fraction of
    output elements identical to the PyTorch sequence;
  * one whole CogVideoX attention layer through RectifiedCogVideoXVideoSpaAttnProcessor2_0 at a sparse step
    (current_step 5) on a stand-in module (tests/fake_attention.py, dim 3072, LayerNorm(64) with bias), fused (kernel 0)
    against fuse_prep = False (the op-by-op PyTorch pre-attention + kernels 2-4), and how closely the two outputs agree;
  * the card's name and power limit (read-only nvidia-smi query).
One JSON line."""
import json
import os
import subprocess
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [REPO, os.path.join(REPO, "rectified-spaattn_b200"), os.path.join(REPO, "tests")]
sys.argv, argv = [sys.argv[0]], sys.argv[1:]
import bench  # noqa: E402
from fake_attention import FakeAttention  # noqa: E402
from oracle import make_golden as MG  # noqa: E402
from rectified_spaattn import rectified_cogvideo_attn as cog  # noqa: E402
from rsa_b200 import geometry as G  # noqa: E402
from rsa_b200 import ops  # noqa: E402

dev = torch.device("cuda:0")
t, h, w, text, heads, dim = 11, 48, 80, 226, 48, 3072
nv = t * h * w
s = nv + text
top_k = int((1 - 0.75) * (nv // 128))
geo = G.cogvideo(s, text)
nbr = ops.gilbert_block_neighbors(t, h, w)


def timed(fn, n=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True, timeout=30).stdout.strip()
res = {"shape": f"CogVideoX1.5 {t}x{h}x{w} + {text} text = {s} tokens x {heads} heads x 64, top_k {top_k}", "card": card}

# ------------------------------------------------------------------------------------------- kernel 0 at 64
g = torch.Generator(device=dev).manual_seed(0)
src = [torch.randn(1, s, heads * 64, generator=g, device=dev).to(torch.bfloat16) for _ in range(3)]
lw = [(1 + 0.1 * torch.randn(64, generator=g, device=dev)).to(torch.bfloat16) for _ in range(2)]
lb = [(0.05 * torch.randn(64, generator=g, device=dev)).to(torch.bfloat16) for _ in range(2)]
ang = torch.outer(torch.arange(nv, dtype=torch.float32, device=dev), 1.0 / (256.0 ** (torch.arange(0, 64, 2, device=dev) / 64)))
cos, sin = ang.cos().repeat_interleave(2, 1).contiguous(), ang.sin().repeat_interleave(2, 1).contiguous()
q, k, v = (torch.empty(1, heads, s, 64, dtype=torch.bfloat16, device=dev) for _ in range(3))
plan = ops.Plan(q, k, v, geo, top_k, bench.P_REMAIN, nbr, private_workspace=True)


def kernel0():
    plan.qkv_prep(*src, q_weight=lw[0], k_weight=lw[1], q_bias=lb[0], k_bias=lb[1], eps=1e-6, rope=(cos, sin),
                  rope_rows=nv)


def torch_sequence():
    tq = MG.torch_prep_cog(src[0], heads, lw[0], lb[0], 1e-6, cos, sin, nv)
    tk = MG.torch_prep_cog(src[1], heads, lw[1], lb[1], 1e-6, cos, sin, nv)
    return tq, tk, src[2].unflatten(2, (heads, -1)).transpose(1, 2)


tq, tk, tv = torch_sequence()
tplan = ops.Plan(tq, tk, tv, geo, top_k, bench.P_REMAIN, nbr, private_workspace=True)
res["kernel0_ms"] = timed(kernel0)
res["torch_sequence_ms"] = timed(torch_sequence)
res["kernel2_on_torch_sequence_ms"] = timed(tplan.pool_stats)
res["torch_sequence_plus_kernel2_ms"] = res["torch_sequence_ms"] + res["kernel2_on_torch_sequence_ms"]
b_alg = 6.0 * s * heads * 64 * 2
peaks = bench.measured_peaks()
res["kernel0_algorithmic_bytes"] = b_alg
res["kernel0_achieved_gbs"] = b_alg / (res["kernel0_ms"] * 1e-3) / 1e9
res["copy_bandwidth_gbs"], res["copy_bandwidth_source"] = peaks["hbm"], peaks["source"]
res["kernel0_frac_of_copy_bandwidth"] = res["kernel0_achieved_gbs"] / peaks["hbm"]
kernel0()
torch.cuda.synchronize()
same = [float((a.view(torch.int16) == b.view(torch.int16)).float().mean()) for a, b in ((q, tq), (k, tk))]
res["kernel0_fraction_identical_q_k"] = same
res["kernel0_v_bit_exact"] = bool(torch.equal(v.view(torch.int16), tv.contiguous().view(torch.int16)))
del src, q, k, v, tq, tk, tv, plan, tplan
torch.cuda.empty_cache()

# --------------------------------------------------------------------------------------- one attention layer
torch.manual_seed(0)
attn = FakeAttention(dim, heads, head_dim=64, norm="layer").to(dev).to(torch.bfloat16)
# hidden states with the block structure of video (neighbouring blocks similar, the "walk" regime of tools/bench_layer.py)
mu = torch.cumsum(torch.randn(nv // 128, dim, device=dev) * 0.35, dim=0).repeat_interleave(128, dim=0)
x = (torch.randn(nv, dim, device=dev) + mu)[None].to(torch.bfloat16)
del mu
txt = torch.randn(1, text, dim, device=dev).to(torch.bfloat16)
outs = {}
with torch.no_grad():
    for key, fuse in (("layer_fused_ms", True), ("layer_op_by_op_ms", False)):
        pr = cog.RectifiedCogVideoXVideoSpaAttnProcessor2_0("sparse", top_k, nbr, bench.P_REMAIN)
        pr.fuse_prep = fuse

        def call():
            pr.current_step = 5                              # a sparse step (the processor is dense before call 5)
            outs[key] = pr(attn, x, txt, None, (cos, sin))
        res[key] = timed(call, 5)
    hs = torch.cat([x, txt], dim=1)                          # inner width heads * 64 == dim: to_out[0] takes hs too
    res["projections_alone_ms"] = timed(lambda: [f(hs) for f in (attn.to_q, attn.to_k, attn.to_v, attn.to_out[0])], 5)
a = torch.cat(outs["layer_fused_ms"], dim=1).float()
b = torch.cat(outs["layer_op_by_op_ms"], dim=1).float()
res["layer_fused_vs_op_by_op_cosine"] = float(torch.nn.functional.cosine_similarity(a.flatten(), b.flatten(), dim=0))
res["layer_fused_vs_op_by_op_max_abs_diff"] = float((a - b).abs().max())
res["layer_fused_vs_op_by_op_fraction_identical"] = float((a == b).float().mean())
res["layer_saving_ms"] = res["layer_op_by_op_ms"] - res["layer_fused_ms"]
print(json.dumps(res))
