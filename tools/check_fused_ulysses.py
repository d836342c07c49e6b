"""Multi-GPU check + measurement of the fused Ulysses exchange (run under torchrun on 2, 4 or 8 GPUs of one box;
workload name as the argument: a bench.py workload, or "odd" / "cog" / "cog_ragged" / "flux_ragged" below; --dense: the dense form, FusedUlysses.run(
dense=True) against kernel 0 without pooling + Plan.run_dense; --dtype float16: fp16 projection rows, norm parameters and
results, FusedUlysses(dtype=torch.float16)):
  * rank r holds tokens [r*S/P, (r+1)*S/P) of the projection outputs; FusedUlysses.run() must return exactly the rows a
    single-GPU call over all heads produces (heads are independent, same kernels => bit-identical),
  * the NCCL form (two all-to-alls around kernel 0 + the pooled call, rsa_b200.parallel.ulysses_attention-style) gives
    the same bits and is timed beside it.
Prints one JSON line from rank 0."""
import json
import os
import sys

import torch
import torch.distributed as dist

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [REPO, os.path.join(REPO, "rectified-spaattn_b200")]
sys.argv, argv = [sys.argv[0]], sys.argv[1:]
import bench  # noqa: E402
from rsa_b200 import ops, parallel  # noqa: E402

name = next((a for i, a in enumerate(argv) if not a.startswith("--") and (i == 0 or argv[i - 1] != "--dtype")), "c3a")
check = "--no-check" not in argv
dense = "--dense" in argv
dt = {"bfloat16": torch.bfloat16, "float16": torch.float16}[argv[argv.index("--dtype") + 1] if "--dtype" in argv else "bfloat16"]
f16 = dict(allow_fp16=True) if dt == torch.float16 else {}     # Plan.qkv_prep takes fp16 plans on request
rank, world, lrank = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lrank)
dev = torch.device("cuda", lrank)
dist.init_process_group("nccl", device_id=dev)
if name == "odd":
    # tokens AND heads that do not divide by the ranks (Wan form, 5 x 9 x 23 = 1035 tokens, 3 heads): the last rank owns
    # fewer rows, the first rank(s) compute one head more
    bench.WORKLOADS["odd"] = dict(desc="uneven token and head shards", fam="wan", grid=(5, 9, 23), text=0, text_valid=0,
                                  heads=3, drop=0.6, ffb=True)
if name == "cog":
    # CogVideoX form: 64-column heads, LayerNorm(64) with bias, rotary embedding on the video tokens; 2 x 8 x 24 = 384
    # video + 227 text = 611 tokens and 3 heads, so neither divides by 2 ranks
    bench.WORKLOADS["cog"] = dict(desc="CogVideoX form, uneven token and head shards", fam="cog", grid=(2, 8, 24),
                                  text=227, text_valid=227, heads=3, drop=0.5, ffb=False)
if name == "cog_ragged":
    # CogVideoX form with a ragged visual segment: 3 x 10 x 35 = 1050 video tokens (8 blocks + 26) + 226 text -> the
    # padded layout of geometry.cogvideo (gap 102), two gathers per tensor
    bench.WORKLOADS["cog_ragged"] = dict(desc="CogVideoX form, ragged visual segment", fam="cog", grid=(3, 10, 35),
                                         text=226, text_valid=226, heads=3, drop=0.5, ffb=False)
if name == "flux_ragged":
    # Flux form with a ragged visual segment: 1 x 25 x 41 = 1025 image tokens + 512 text (gap 127); the rotary
    # embedding covers the text tokens too, so the text gather rotates with table rows [nv, S)
    bench.WORKLOADS["flux_ragged"] = dict(desc="Flux form, ragged visual segment", fam="flux", grid=(1, 25, 41),
                                          text=512, text_valid=512, heads=3, drop=0.5, ffb=False)
wp = bench.workload_params(name)
heads, s, nv = wp["heads"], wp["s"], wp["nv"]
cog = wp["fam"] == "cog"
hd = 64 if cog else 128                             # head_dim
geo = bench.product_geometry(wp)
t, h, w = wp["grid"]
nbr = ops.gilbert_block_neighbors(t, h, w)
rows, hl = -(-s // world), heads // world          # rows per rank (the last rank may own fewer)
even = rows * world == s and hl * world == heads      # the NCCL form below is written for even shards only
g = torch.Generator(device=dev).manual_seed(1234)                       # same stream on every rank: the full tensors
full = [torch.randn(1, s, heads * hd, generator=g, device=dev).to(dt) for _ in range(3)]
if wp["fam"] != "wan":                                                   # give the pooled scores some structure
    mu = torch.cumsum(torch.randn(1, (s + 127) // 128, heads * hd, generator=g, device=dev) * 0.35, dim=1)
    for x in full[:2]:
        x.add_(mu.repeat_interleave(128, dim=1)[:, :s].to(dt))
wan = wp["fam"] == "wan"     # Wan: RMSNorm over all heads*128 channels of a token, rotary embedding on every token
nw = heads * 128 if wan else hd
wq = (1 + 0.1 * torch.randn(nw, generator=g, device=dev)).to(dt)
wk = (1 + 0.1 * torch.randn(nw, generator=g, device=dev)).to(dt)
# CogVideoX: LayerNorm(head_dim) with bias on q and k
norm_kw = dict(q_bias=(0.05 * torch.randn(hd, generator=g, device=dev)).to(dt),
               k_bias=(0.05 * torch.randn(hd, generator=g, device=dev)).to(dt)) if cog else {}
n_rope = s if wp["fam"] == "flux" else nv            # Flux rotates every token, the others the visual tokens only
ang = torch.outer(torch.arange(n_rope, dtype=torch.float32, device=dev), 1.0 / (256.0 ** (torch.arange(0, hd, 2, device=dev) / hd)))
rope = (ang.cos().repeat_interleave(2, 1).contiguous(), ang.sin().repeat_interleave(2, 1).contiguous())
rope_vis = (rope[0][:nv], rope[1][:nv])
rope_txt = (rope[0][nv:], rope[1][nv:]) if n_rope > nv else None
mine = slice(rank * rows, min((rank + 1) * rows, s))

fu = parallel.FusedUlysses(1, heads, geo, wp["top_k"], bench.P_REMAIN, nbr, head_dim=hd, dtype=dt)
for dst, src in zip((fu.q_src, fu.k_src, fu.v_src), full):
    dst.copy_(src[:, mine])
out = fu.run(wq, wk, 1e-6, rope, n_rope, dense=dense, **norm_kw).clone()
torch.cuda.synchronize()

# NCCL form: all-to-all the projection rows to head shards, kernel 0 + pooled call locally, all-to-all the result back
q, k, v = (torch.empty(1, max(hl, 1), s, hd, dtype=dt, device=dev) for _ in range(3))
plan = ops.Plan(q, k, v, geo, wp["top_k"], bench.P_REMAIN, nbr)


def finish(pl):
    """The attention after kernel 0: the pooled sparse call, or dense attention over the valid memory rows."""
    n_valid = geo.kv_len - geo.gap
    return pl.run_dense(n_valid, n_valid) if dense else pl.run_pooled()


def wan_norm(x, w):
    """diffusers RMSNorm over the whole row (what the Wan processor does before the head split), in PyTorch."""
    var = x.float().pow(2).mean(-1, keepdim=True)
    return (x * torch.rsqrt(var + 1e-6)).to(dt) * w


def nccl_form():
    srcs = []
    for i, x in enumerate(full):
        loc = x[:, mine]
        if wan and i < 2:      # the norm needs whole rows: before the exchange, on the tokens this rank owns
            loc = wan_norm(loc, wq if i == 0 else wk)
        loc = loc.reshape(1, rows, world, hl * hd).permute(2, 0, 1, 3).contiguous()    # [P(dst), 1, rows, hl*hd]
        rcv = torch.empty_like(loc)
        dist.all_to_all_single(rcv, loc)
        srcs.append(rcv.permute(1, 0, 2, 3).reshape(1, s, hl * hd))                          # all tokens, my heads
    if wan:
        plan.qkv_prep(*srcs, dst_row=0, rope=rope, rope_rows=nv, pool=not dense, **f16)
    elif geo.gap:
        plan.qkv_prep(*(x[:, :nv] for x in srcs), dst_row=0, q_weight=wq, k_weight=wk, eps=1e-6, rope=rope_vis,
                      pool=not dense, **norm_kw, **f16)
        plan.qkv_prep(*(x[:, nv:] for x in srcs), dst_row=nv, q_weight=wq, k_weight=wk, eps=1e-6, rope=rope_txt,
                      pool=not dense, **norm_kw, **f16)
    else:
        plan.qkv_prep(*srcs, dst_row=0, q_weight=wq, k_weight=wk, eps=1e-6, rope=rope, rope_rows=n_rope,
                      pool=not dense, **norm_kw, **f16)
    o = finish(plan)                                                                     # [1, S, hl, hd]
    return parallel.head_to_seq_shard(o).reshape(1, rows, heads * hd)


# (the NCCL form below is written for even shards; with uneven ones the single-GPU call is the only reference)
ref = nccl_form().clone() if even else out
torch.cuda.synchronize()
# Wan: the NCCL form's norm is PyTorch's (other reduction order: a bf16 rounding may flip, and with it a block selection),
# so it is a timing reference there, not a bit reference -- the bit reference is the single-GPU call below
same_as_nccl = bool(torch.equal(out.view(torch.int16), ref.view(torch.int16)))
frac_equal_nccl = float((out.view(torch.int16) == ref.view(torch.int16)).float().mean())
same_as_single = None
if check and (rank == 0 or not even):       # uneven shards: every rank checks its own rows (the shapes are small)
    # one GPU, all heads, no exchange at all
    qa, ka, va = (torch.empty(1, heads, s, hd, dtype=dt, device=dev) for _ in range(3))
    pa = ops.Plan(qa, ka, va, geo, wp["top_k"], bench.P_REMAIN, nbr)
    if geo.gap:
        pa.qkv_prep(*(x[:, :nv] for x in full), dst_row=0, q_weight=wq, k_weight=wk, eps=1e-6, rope=rope_vis,
                    pool=not dense, **norm_kw, **f16)
        pa.qkv_prep(*(x[:, nv:] for x in full), dst_row=nv, q_weight=wq, k_weight=wk, eps=1e-6, rope=rope_txt,
                    pool=not dense, **norm_kw, **f16)
    else:
        pa.qkv_prep(*full, dst_row=0, q_weight=wq, k_weight=wk, eps=1e-6, rope=rope, rope_rows=n_rope,
                    pool=not dense, **norm_kw, **f16)
    single = finish(pa).reshape(1, s, heads * hd)[:, mine]
    torch.cuda.synchronize()
    same_as_single = bool(torch.equal(out.view(torch.int16), single.view(torch.int16)))
    del qa, ka, va, pa


def timed(fn, n=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    tt = torch.tensor([e0.elapsed_time(e1) / n], device=dev)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    return float(tt.item())


ms_fused = timed(lambda: fu.run(wq, wk, 1e-6, rope, n_rope, dense=dense, **norm_kw))
ms_nccl = timed(nccl_form) if even else None
oks = [None] * world
dist.all_gather_object(oks, same_as_nccl)
singles = [None] * world
dist.all_gather_object(singles, same_as_single)
if rank == 0:
    print(json.dumps({"workload": name, "dense": dense, "dtype": str(dt).replace("torch.", ""), "n_gpus": world, "tokens": s, "heads": heads, "head_dim": hd,
                      "fused_ms_per_layer_attention": ms_fused, "nccl_all_to_all_form_ms": ms_nccl,
                      "norm": "across heads (Wan)" if wan else ("LayerNorm per head (CogVideoX)" if cog else "per head"),
                      "fused_equals_nccl_form_bitwise_all_ranks": all(oks),
                      "fraction_of_elements_equal_to_nccl_form_rank0": frac_equal_nccl,
                      "fused_equals_single_gpu_bitwise_rank0": same_as_single,
                      "fused_equals_single_gpu_bitwise_checked_ranks": [x for x in singles if x is not None],
                      "rows_per_rank": rows, "rows_last_rank": s - (world - 1) * rows, "heads_rank0": fu.heads,
                      "note": "both forms run kernel 0 + kernels 3a-4 (--dense: kernel 0 without pooling + dense kernel 4); fused = gather inside kernel 0 and scatter inside "
                              "kernel 4's epilogue over peer memory, barriers only; nccl = all_to_all_single x4 + staging copies"}))
fu.close()
dist.destroy_process_group()
