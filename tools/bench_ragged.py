"""Sparse calls at ragged visual segments (run on the GPU box), in one process: the padded layout of geometry.flux /
geometry.cogvideo at the models' own token counts.
  * CogVideoX-2B (13x30x45 + 226 = 17 776 tokens x 30 heads x 64, fp16), CogVideoX-5B (the same tokens x 48 heads x 64,
    bf16), Flux.1-dev at 1360x768 (4 080 + 512 tokens) and 1920x1088 (8 160 + 512) x 24 heads x 128 (bf16):
      - the whole sparse call (Plan.run: kernels 2, 3a-3c, 4), ms per call;
      - the same call on the explicitly padded tensors (gap zero rows inserted at the visual token count) with the
        aligned geometry the reference rule gives for them -- the A/B that shows what the padded layout costs beyond
        its extra rows (the two select the same blocks: tests/test_ragged_joint.py);
      - kernel 4 alone (rsa_sparse_attention after the stages): ms, kept (query tile, key block) pairs, and TFLOP/s on
        the kept pairs (4 * 128 * 128 * head_dim FLOP per pair, a partial block counted whole);
      - kernel 4's list-free dense form (Plan.run_dense over all S tokens): ms and TFLOP/s (4 * S^2 * head_dim per head);
    the four alternate round by round; each timing is the median of 7 rounds of 10 launches (CUDA events);
    top_k = int((1 - 0.75) * visual blocks), inputs bench.py's "walk" regime;
  * one fp16 CogVideoX-2B attention layer at its own 17 550 + 226 tokens through RectifiedCogVideoXVideoSpaAttnProcessor2_0
    on a stand-in module (tests/fake_attention.py, dim 1920): fused (fuse_prep_fp16) against op by op, at a sparse step
    and at a dense call (fuse_prep_dense);
  * the card's name and power limit (read-only nvidia-smi query), in the same run.
One JSON line per measurement; with an argument, the lines are also written to that file."""
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

if not torch.cuda.is_available():
    raise SystemExit("bench_ragged.py measures on the GPU: no CUDA device")
dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True, timeout=30).stdout.strip()
lines = []
DROP = 0.75
SHAPES = {
    # name: (family, grid, text tokens, heads, head_dim, dtype)
    "cogvideox-2b": ("cogvideo", (13, 30, 45), 226, 30, 64, torch.float16),
    "cogvideox-5b": ("cogvideo", (13, 30, 45), 226, 48, 64, torch.bfloat16),
    "flux-1360x768": ("flux", (1, 48, 85), 512, 24, 128, torch.bfloat16),
    "flux-1920x1088": ("flux", (1, 68, 120), 512, 24, 128, torch.bfloat16),
}


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


def pad_rows(x, nv, gap):
    z = torch.zeros(*x.shape[:2], gap, x.shape[3], dtype=x.dtype, device=x.device)
    return torch.cat([x[:, :, :nv], z, x[:, :, nv:]], dim=2).contiguous()


def sparse_call(name):
    fam, (t, h, w), text, heads, hd, dt = SHAPES[name]
    nv = t * h * w
    s = nv + text
    make = G.flux if fam == "flux" else G.cogvideo
    geo = make(s, text)
    geo_pad = make(s + geo.gap, text)
    assert geo.gap > 0 and geo_pad.gap == 0
    top_k = int((1 - DROP) * (nv // 128))
    nbr = ops.gilbert_block_neighbors(t, h, w)
    q, k, v = (x.to(dt) for x in bench.synth_heads_device(heads, 0, s, "walk", dev, d=hd))
    qp, kp, vp = (pad_rows(x, nv, geo.gap) for x in (q, k, v))
    ragged = ops.Plan(q, k, v, geo, top_k, bench.P_REMAIN, nbr, private_workspace=True)
    padded = ops.Plan(qp, kp, vp, geo_pad, top_k, bench.P_REMAIN, nbr, private_workspace=True)
    ragged.run()
    padded.run()
    torch.cuda.synchronize()
    kept = int(ragged.view()["kept_cnt"].sum())
    kept_pad = int(padded.view()["kept_cnt"].sum())
    (ms_r, ms_p, ms_k4, ms_dense), spread = alternating(
        [ragged.run, padded.run, ragged.sparse_attention, lambda: ragged.run_dense(s, s)])
    out_r = ragged.run().clone()
    out_p = padded.run()
    out_p = torch.cat([out_p[:, :nv], out_p[:, nv + geo.gap:]], dim=1)
    torch.cuda.synchronize()
    emit({"shape": name, "tokens": f"{nv} + {text} = {s}", "heads": heads, "head_dim": hd, "dtype": str(dt)[6:],
          "geometry": dict(n_blocks=geo.n_blocks, nq_blocks=geo.nq_blocks, vis_len=geo.vis_len, gap=geo.gap,
                           kv_len=geo.kv_len),
          "top_k": top_k, "drop": DROP,
          "ms_per_call": ms_r, "ms_per_call_padded_aligned": ms_p, "padded_over_ragged": ms_p / ms_r,
          "kernel4_ms": ms_k4, "kept_pairs": kept, "kept_pairs_padded_aligned": kept_pad,
          "kernel4_tflops_on_kept_pairs": kept * 4.0 * 128 * 128 * hd / (ms_k4 * 1e-3) / 1e12,
          "dense_kernel4_ms": ms_dense, "dense_kernel4_tflops": heads * 4.0 * s * s * hd / (ms_dense * 1e-3) / 1e12,
          "round_spread_ms": dict(zip(("ragged", "padded", "kernel4", "dense"), spread)),
          "output_rows_equal_to_padded_call": float((out_r.view(torch.int16) == out_p.view(torch.int16)).float().mean()),
          "note": "median of 7 alternating rounds of 10 launches, CUDA events; q, k, v of "
                  f"{3 * heads * s * hd * 2 / 1e6:.0f} MB ({'more' if 3 * heads * s * hd * 2 > 126e6 else 'less'} "
                  "than the 126 MB of L2)"})
    del ragged, padded, q, k, v, qp, kp, vp
    torch.cuda.empty_cache()


def cog2b_layer():
    t, h, w, text, heads, dim = 13, 30, 45, 226, 30, 1920
    nv = t * h * w                                      # 17 550: the padded layout of geometry.cogvideo
    torch.manual_seed(0)
    attn = FakeAttention(dim, heads, head_dim=64, norm="layer").to(dev).to(torch.float16)
    g = torch.Generator(device=dev).manual_seed(1)
    mu = torch.cumsum(torch.randn(-(-nv // 128), dim, generator=g, device=dev) * 0.35, 0).repeat_interleave(128, 0)[:nv]
    x = (torch.randn(nv, dim, generator=g, device=dev) + mu)[None].to(torch.float16)
    txt = torch.randn(1, text, dim, generator=g, device=dev).to(torch.float16)
    for dense in (False, True):
        prs = []
        for fused in (True, False):
            pr = cog.RectifiedCogVideoXVideoSpaAttnProcessor2_0("sparse", int((1 - DROP) * (nv // 128)), None,
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
        emit({"shape": f"cogvideox-2b, {nv} + {text} tokens", "what": f"one fp16 attention layer, {'dense call 0' if dense else 'sparse step'}",
              "fused_ms": ms_fused, "op_by_op_ms": ms_eager, "fused_round_spread_ms": sp_f,
              "op_by_op_round_spread_ms": sp_e, "output_cosine_fused_vs_op_by_op": cos,
              "output_max_abs_diff": float((a - b).abs().max()), "module": f"stand-in, dim {dim}, LayerNorm(64) + bias"})


for name in SHAPES:
    sparse_call(name)
cog2b_layer()
if argv:
    os.makedirs(os.path.dirname(os.path.abspath(argv[0])), exist_ok=True)
    with open(argv[0], "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")
