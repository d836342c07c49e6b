"""Dense attention calls at real shapes (run on the GPU box): one whole attention layer through the processor protocol,
op by op (fuse_prep_dense = False: projections, PyTorch head split / QK norm / RoPE, fullattn(mode="flash"), output
projections) against fused (fuse_prep_dense = True: projections, kernel 0 without pooling, kernel 4's list-free dense
form, output projections).  Workloads:
  flux   Flux.1-dev 4096x4096 single-stream block 40 (dense range 37-56): 65 536 + 512 text = 66 048 tokens x 24 heads
  wan    Wan2.1-T2V-14B 720p 81f warm-up call (step 0 of layer 3): 21x45x80 = 75 600 tokens x 40 heads
  cog    CogVideoX1.5 call 0 of a layer: 11x48x80 + 226 text = 42 466 tokens x 48 heads x 64
  c3a    HunyuanVideo C3a under mode="flash": 32x45x80 + 256 text (200 valid) = 115 456 tokens x 24 heads, dual-stream
For each: the layer time both ways; in a separate instrumented pass (CUDA events at the section boundaries) the time from
the layer's start to the attention call (projections + pre-attention), the attention call and the rest; kernel 0 alone
(pool = 0); and, on random tensors of the same shape, kernel 4's list-free walk against the masked entry with an all-ones
mask (bit-identical outputs checked).  Modules are tests/fake_attention.py stand-ins with the models' widths.  Reads the
card's name and power limit (read-only nvidia-smi query).  One JSON line per workload."""
import json
import os
import subprocess
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [REPO, os.path.join(REPO, "rectified-spaattn_b200"), os.path.join(REPO, "tests")]
from fake_attention import FakeAttention  # noqa: E402
from rectified_spaattn import attn as A  # noqa: E402
from rectified_spaattn import rectified_cogvideo_attn as cog  # noqa: E402
from rectified_spaattn import rectified_flux_attn as flux  # noqa: E402
from rectified_spaattn import rectified_hunyuan_attn as hun  # noqa: E402
from rectified_spaattn import rectified_wan21_attn as wan21  # noqa: E402
from rsa_b200 import ops  # noqa: E402

dev = torch.device("cuda:0")
names = [a for a in sys.argv[1:] if not a.startswith("--")] or ["flux", "wan", "cog", "c3a"]
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True, timeout=30).stdout.strip()


def timed(fn, n=5):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def rope_real_tables(n, d, theta=256.0):
    ang = torch.outer(torch.arange(n, dtype=torch.float32, device=dev),
                      1.0 / (theta ** (torch.arange(0, d, 2, device=dev) / d)))
    return ang, (ang.cos().repeat_interleave(2, 1).contiguous(), ang.sin().repeat_interleave(2, 1).contiguous())


def video(n, dim, g):
    """Hidden states with neighbouring blocks alike (the "walk" regime of tools/bench_layer.py)."""
    mu = torch.cumsum(torch.randn((n + 127) // 128, dim, device=dev, generator=g) * 0.35, 0).repeat_interleave(128, 0)
    return (torch.randn(n, dim, device=dev, generator=g) + mu[:n])[None].to(torch.bfloat16)


def workload(name):
    """(description, attn module, make_processor(), call(processor), heads, S, head_dim, q_valid)."""
    g = torch.Generator(device=dev).manual_seed(0)
    torch.manual_seed(0)
    if name == "flux":
        nv, text, heads, dim = 256 * 256, 512, 24, 3072
        attn = FakeAttention(dim, heads).to(dev).to(torch.bfloat16)
        hs = torch.cat([video(nv, dim, g), torch.randn(1, text, dim, device=dev, generator=g).to(torch.bfloat16)], 1)
        _, rope = rope_real_tables(nv + text, 128, 10000.0)
        make = lambda: flux.RectifiedFluxSpaAttnProcessor2_0("sparse", 1, None, 0.3, processor_id=40, text_length=text)
        return ("Flux.1-dev 4096x4096 single-stream block 40", attn, make, lambda pr: pr(attn, hs, None, None, rope),
                heads, nv + text, 128, nv + text)
    if name == "wan":
        s, heads, dim = 21 * 45 * 80, 40, 5120
        attn = FakeAttention(dim, heads, norm="inner").to(dev).to(torch.bfloat16)
        x = video(s, dim, g)
        ang, _ = rope_real_tables(s, 128, 10000.0)
        emb = torch.polar(torch.ones_like(ang, dtype=torch.float64), ang.double())[None, None]

        def make():
            return wan21.RectifiedWanT2VSpaAttnProcessor2_0("sparse", 1, None, 0.3, processor_id=3)

        def call(pr):
            pr.current_step = 0                      # warm-up call: dense
            return pr(attn, x, None, None, emb)
        return "Wan2.1-T2V-14B 720p warm-up call", attn, make, call, heads, s, 128, s
    if name == "cog":
        nv, text, heads, dim = 11 * 48 * 80, 226, 48, 3072
        attn = FakeAttention(dim, heads, head_dim=64, norm="layer").to(dev).to(torch.bfloat16)
        x, txt = video(nv, dim, g), torch.randn(1, text, dim, device=dev, generator=g).to(torch.bfloat16)
        _, rope = rope_real_tables(nv, 64)

        def make():
            return cog.RectifiedCogVideoXVideoSpaAttnProcessor2_0("sparse", 1, None, 0.3)

        def call(pr):
            pr.current_step = 0                      # call 0: dense
            return pr(attn, x, txt, None, rope)
        return "CogVideoX1.5 call 0", attn, make, call, heads, nv + text, 64, nv + text
    if name == "c3a":
        nv, text, valid, heads, dim = 32 * 45 * 80, 256, 200, 24, 3072
        attn = FakeAttention(dim, heads, added=True).to(dev).to(torch.bfloat16)
        x, txt = video(nv, dim, g), torch.randn(1, text, dim, device=dev, generator=g).to(torch.bfloat16)
        _, rope = rope_real_tables(nv, 128)

        def make():
            pr = hun.RectifiedHunyuanVideoSpaAttnProcessor2_0("flash", 1, None, 0.3)
            pr.num_true = nv + valid
            return pr
        return ("HunyuanVideo C3a mode=flash (dual-stream)", attn, make, lambda pr: pr(attn, x, txt, None, rope), heads,
                nv + text, 128, nv + valid)
    raise SystemExit(f"unknown workload {name}")


class Sections:
    """CUDA events at the layer's section boundaries, recorded through wrappers of the attention entry points."""

    def __init__(self):
        self.ev = {}
        self.orig = (A._flash_like, ops.Plan.qkv_prep, ops.Plan.run_dense)

    def mark(self, key, first=False):
        if first and key in self.ev:
            return
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.ev[key] = e

    def __enter__(self):
        flash, prep, dense = self.orig
        sec = self

        def flash_w(*a, **kw):
            sec.mark("attn_start")
            out = flash(*a, **kw)
            sec.mark("attn_end")
            return out

        def prep_w(self_, *a, **kw):
            sec.mark("k0_start", first=True)
            prep(self_, *a, **kw)
            sec.mark("k0_end")

        def dense_w(self_, *a, **kw):
            sec.mark("attn_start")
            out = dense(self_, *a, **kw)
            sec.mark("attn_end")
            return out
        A._flash_like, ops.Plan.qkv_prep, ops.Plan.run_dense = flash_w, prep_w, dense_w
        return self

    def __exit__(self, *exc):
        A._flash_like, ops.Plan.qkv_prep, ops.Plan.run_dense = self.orig

    def run(self, call, n=3):
        acc = {}
        for _ in range(n):
            self.ev = {}
            self.mark("start")
            call()
            self.mark("end")
            torch.cuda.synchronize()
            t = lambda a, b: self.ev[a].elapsed_time(self.ev[b])
            parts = {"to_attention_ms": t("start", "attn_start"), "attention_ms": t("attn_start", "attn_end"),
                     "after_attention_ms": t("attn_end", "end")}
            if "k0_start" in self.ev:
                parts["kernel0_pool0_ms"] = t("k0_start", "k0_end")
            for k, v in parts.items():
                acc[k] = acc.get(k, 0.0) + v / n
        return acc


for name in names:
    desc, attn, make, call, heads, s, hd, q_valid = workload(name)
    res = {"workload": name, "shape": f"{desc}: {s} tokens x {heads} heads x {hd}", "card": card}
    outs = {}
    with torch.no_grad():
        for key, fuse in (("fused", True), ("op_by_op", False)):
            pr = make()
            pr.fuse_prep_dense = fuse

            def one():
                outs[key] = call(pr)
            res[f"layer_{key}_ms"] = timed(one)
            with Sections() as sec:
                res[f"sections_{key}"] = sec.run(one)
        a, b = (torch.cat(o, 1) if isinstance(o, tuple) else o for o in (outs["fused"], outs["op_by_op"]))
        a, b = a.float(), b.float()
        res["fused_vs_op_by_op_cosine"] = float(torch.nn.functional.cosine_similarity(a.flatten(), b.flatten(), dim=0))
        res["fused_vs_op_by_op_max_abs_diff"] = float((a - b).abs().max())
        res["layer_saving_ms"] = res["layer_op_by_op_ms"] - res["layer_fused_ms"]
        del outs, a, b
        torch.cuda.empty_cache()
        # kernel 4: the list-free walk against the masked entry on an all-ones mask, same random tensors
        g = torch.Generator(device=dev).manual_seed(1)
        q, k, v = (torch.randn(1, heads, s, hd, device=dev, generator=g).to(torch.bfloat16) for _ in range(3))
        mask = torch.ones(1, heads, (s + 127) // 128, (s + 127) // 128, dtype=torch.bool, device=dev)
        od = ops.dense_attention(q, k, v, q_valid, q_valid)     # the layer's call: kv_len = q_valid
        om = ops.masked_attention(q, k, v, mask, q_valid, fp32_scale=True)
        om[:, :, q_valid:] = 0
        torch.cuda.synchronize()
        res["kernel4_dense_bit_identical_to_masked_all_ones"] = bool(torch.equal(od.view(torch.int16), om.view(torch.int16)))
        res["kernel4_dense_ms"] = timed(lambda: ops.dense_attention(q, k, v, q_valid, q_valid, out=od), 10)
        res["kernel4_masked_all_ones_ms"] = timed(lambda: ops.masked_attention(q, k, v, mask, q_valid, out=om, fp32_scale=True), 10)
        flop = 4.0 * heads * q_valid * q_valid * hd        # QK^T + PV over the valid query rows and keys
        res["kernel4_dense_tflops"] = flop / (res["kernel4_dense_ms"] * 1e-3) / 1e12
        res["note"] = ("masked_all_ones_ms: the mask is built once outside the timed loop; each call still allocates its "
                       "workspace and runs mask_to_lists + pair_schedule before kernel 4. sections: one instrumented pass "
                       "(events at the attention entry points), to_attention = projections + pre-attention")
        del q, k, v, od, om, mask
    del attn
    torch.cuda.empty_cache()
    print(json.dumps(res), flush=True)
