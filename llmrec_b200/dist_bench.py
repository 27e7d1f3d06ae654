"""bench.py leg for N > 1 GPUs (and the `scaling_base` leg of the N = 1 line): the ID-propagation training step on the large
synthetic bipartite graph (10 M users x 1 M items x 200 M edges, d = 128, L = 2 by default; scaled by --syn-scale),
users sharded over ranks, item-sized tensors replicated, NCCL exchanges of [ni x d] partial sums (dist.py).
STRONG scaling: the graph and the global batch (1024 sampled + aug-sized extra = 1126 triplets) are fixed as N grows.
No side features in this configuration (SURVEY.md 8d item 4) -- stated in config.workload.

Everything here is device-agnostic host code (timing helper, generators, collectives): tests/test_dist_bench_cpu.py runs it
end to end at world size 2 under gloo with torch stand-ins for the kernels, so the dictionary the driver parses is built in CI."""
from __future__ import annotations

import os
import time

import torch
import torch.distributed as dist


def _sync(dev):
    if dev.type == "cuda":
        torch.cuda.synchronize(dev)


def _time_ms(dev, fn, world):
    """Device time of fn() in ms: CUDA events on the current stream (perf_counter on the CPU stand-in), barrier + synchronize
    on both sides, MAX over ranks."""
    _sync(dev)
    if world > 1:
        dist.barrier()
    _sync(dev)
    if dev.type == "cuda":
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1)
    else:
        t0 = time.perf_counter()
        fn()
        ms = (time.perf_counter() - t0) * 1e3
    if world > 1:
        dist.barrier()
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    return ms


def _median(xs):
    s = sorted(xs)
    return s[len(s) // 2]


def _init_tables(nu_local, ni, nu_total, d, rank, dev):
    bound_u = (6.0 / (nu_total + d)) ** 0.5                                       # xavier_uniform on the full [nu x d] table
    E_u = (torch.rand(nu_local, d, device=dev, generator=torch.Generator(device=dev).manual_seed(77 + rank)) * 2 - 1) * bound_u
    E_i = (torch.rand(ni, d, device=dev, generator=torch.Generator(device=dev).manual_seed(1234)) * 2 - 1) * (6.0 / (ni + d)) ** 0.5
    return E_u, E_i                                                               # E_i: same seed on every rank = replicated


def syn_sizes(scale):
    return int(10_000_000 * scale), int(1_000_000 * scale), int(200_000_000 * scale), 128, 2


def run_single(a, dev, batches, K, W, tag="rank 0 alone"):
    """The same synthetic workload on ONE device (the strong-scaling base): -> dict(value, ms_per_step, ...)."""
    from .dist import ShardedGraph, ShardedHotPath, synthetic_shard
    from .engine import HotPathConfig
    nu, ni, ne, d, L = syn_sizes(a.syn_scale)
    B = int(batches[0][0].numel())
    ul, it, _, _ = synthetic_shard(nu, ni, ne, 0, 1, dev, seed=0)
    g1 = ShardedGraph(ul, it, nu, ni, solo=True)
    del ul, it
    Eu1, Ei1 = _init_tables(nu, ni, nu, d, 0, dev)
    hp1 = ShardedHotPath(g1, Eu1, Ei1, HotPathConfig(embed_size=d, n_layers=L, batch_size=1024), 0, solo=True,
                         demand=bool(getattr(a, "demand", 1)))
    k1 = max(3, min(K, 8))
    for i in range(min(W, 3)):
        hp1.train_step(*batches[i % len(batches)])
    blocks = []
    for _ in range(3):
        blocks.append(_time_ms(dev, lambda: [hp1.train_step(*batches[(W + i) % len(batches)]) for i in range(k1)], 1) / k1)
    ms1 = _median(blocks)
    out = {"n_gpus": 1, "value": round(B / (ms1 / 1e3), 1), "unit": "interactions/s", "ms_per_step": round(ms1, 4), "steps": k1, "blocks": 3,
           "nnz": int(g1.nnz), "note": "same synthetic workload, same code path, " + tag + "; edges of the 1-GPU graph are drawn with the 1-rank generator"}
    return out, hp1, g1


def eval_leg(a, hp, g, dev, world, rank, nu_total, nu_local, shots=5):
    """Full-catalog eval (BASELINE.json configs[4]): every rank ranks its own users against the replicated item table (users are
    independent: no exchange); tcgen05 scoring + fused top-K, train rows of the local shard as the mask.  Median of `shots`."""
    from . import ops
    n_eval = min(int(a.eval_users), nu_total)
    per = max(1, n_eval // world)
    per = min(per, nu_local)
    hp.forward()
    eu = torch.randperm(nu_local, device=dev, generator=torch.Generator(device=dev).manual_seed(5 + rank))[:per].to(torch.int32)
    K_eval = 50
    ops.score_topk(hp.U, hp.I, eu, g.rowptr_u, g.col_u, K_eval, mode=0)      # warm-up at the timed size: scratch and tensor maps exist afterwards
    box = {}

    def shot():
        box["top"] = ops.score_topk(hp.U, hp.I, eu, g.rowptr_u, g.col_u, K_eval, mode=0)
    times = [_time_ms(dev, shot, world) for _ in range(shots)]
    ms_ev = _median(times)
    ni, d = hp.ni, hp.d
    return {"metric": "eval_users_per_sec", "value": round(per * world / (ms_ev / 1e3), 1), "unit": "users/s", "n_users": per * world, "n_items": ni,
            "K": K_eval, "ms": round(ms_ev, 3), "ms_min": round(min(times), 3), "ms_max": round(max(times), 3), "shots": shots,
            "all_ranked": bool((box["top"] >= 0).all()),
            "tensor_tflops_useful": round(2.0 * ni * d * per * world / (ms_ev * 1e-3) / 1e12, 1),
            "includes": "tcgen05 3xTF32 scoring + fused top-K + exact rescoring, users sharded over ranks, item table replicated (device-resident)"}


def workload_string(nu, ni, nnz, d, L, B):
    return (f"synthetic {nu}x{ni}, {int(nnz)} unique edges (Zipf 0.8 item popularity), d={d}, L={L}, global batch {B} triplets, "
            "ID propagation + BPR/prune + dense AdamW, no side features; users sharded over ranks, items replicated")


def run_sharded(a, dev=None):
    from . import ops
    from .dist import ShardedGraph, ShardedHotPath, synthetic_shard
    from .engine import HotPathConfig
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if dev is None:
        if not torch.cuda.is_available():
            raise RuntimeError("bench: the sharded leg needs CUDA devices (no CPU fallback)")
        torch.cuda.set_device(local)
        dev = torch.device("cuda", local)
        if world > 1 and not dist.is_initialized():
            dist.init_process_group("nccl")
    nu, ni, ne, d, L = syn_sizes(a.syn_scale)
    t0 = time.perf_counter()
    ul, it, lo, hi = synthetic_shard(nu, ni, ne, rank, world, dev, seed=0)
    g = ShardedGraph(ul, it, hi - lo, ni, pieces=(a.pieces if world > 1 else 1))
    del ul, it
    if dev.type == "cuda":
        torch.cuda.empty_cache()
    E_u, E_i = _init_tables(hi - lo, ni, nu, d, rank, dev)
    cfg = HotPathConfig(embed_size=d, n_layers=L, batch_size=1024)
    hp = ShardedHotPath(g, E_u, E_i, cfg, lo, item_sharded=bool(getattr(a, "item_sharded", 0)), demand=bool(getattr(a, "demand", 1)))
    nnz = torch.tensor([g.nnz], device=dev, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(nnz)
    build_s = time.perf_counter() - t0
    K, W, B = a.steps, max(a.warmup, 3), 1126
    bg = torch.Generator(device=dev).manual_seed(99)                                  # identical batches on every rank
    batches = [(torch.randint(0, nu, (B,), device=dev, generator=bg, dtype=torch.int32),
                torch.randint(0, ni, (B,), device=dev, generator=bg, dtype=torch.int32),
                torch.randint(0, ni, (B,), device=dev, generator=bg, dtype=torch.int32)) for _ in range(W + K)]
    for i in range(W):
        hp.train_step(*batches[i])
    # ---- device-resident leg: blocks of EXACTLY K steps (barrier + synchronize on both sides, max over ranks), repeated until
    #      >= min_seconds of device time; the reported step time is the median block
    l0 = ops.STATS["launches"]; hp.comm_bytes = 0
    blocks, spent = [], 0.0
    while True:
        ms = _time_ms(dev, lambda: [hp.train_step(*batches[W + i]) for i in range(K)], world)
        blocks.append(ms); spent += ms
        if spent >= 1e3 * a.min_seconds or len(blocks) >= a.max_blocks:
            break
    launches = (ops.STATS["launches"] - l0) // len(blocks)
    comm_per_step = hp.comm_bytes // (K * len(blocks))
    ms = _median(blocks)
    # ---- end-to-end: batch indices start in pinned host memory every step, loss read back every step
    pin = (lambda t: t.pin_memory()) if dev.type == "cuda" else (lambda t: t)
    hb = [pin(torch.stack([b.cpu() for b in batches[W + i]])) for i in range(K)]
    loss_host = pin(torch.empty(K, dtype=torch.float32))
    idx = torch.empty((3, B), dtype=torch.int32, device=dev)

    def e2e_block():
        for i in range(K):
            idx.copy_(hb[i], non_blocking=True)
            loss = hp.train_step(idx[0], idx[1], idx[2])
            loss_host[i:i + 1].copy_(loss.reshape(1), non_blocking=True)
    blocks2 = [_time_ms(dev, e2e_block, world) for _ in range(max(1, min(len(blocks), 5)))]
    ms2 = _median(blocks2)
    assert bool(torch.isfinite(loss_host).all()), "non-finite loss"
    # ---- roofline of the dominant kernel: the item-side gather SpMM (iu_raw), timed alone on this rank
    seg = [(hp.Ul[1], hp.part, None, False)]
    g.iu_raw.apply(seg)
    t_spmm = _time_ms(dev, lambda: [g.iu_raw.apply(seg) for _ in range(5)], world) / 5
    nu_l = hi - lo
    nnz_local = g.nnz
    alg = 4 * nnz_local + 4 * (ni + 1) + 4 * d * nu_l + 4 * d * ni
    gather = 4 * nnz_local + 4 * d * nnz_local + 4 * d * ni
    ev = eval_leg(a, hp, g, dev, world, rank, nu, nu_l)
    item_sharded = bool(hp.item_sharded)          # read before the engine is freed for the 1-GPU base below
    demand = bool(hp.demand)
    # ---- the SAME workload on ONE GPU (rank 0 alone, other ranks wait): the strong-scaling base measured in this run ----
    base = None
    if world > 1 and a.n1_base:
        del hp, g, E_u, E_i, seg
        if dev.type == "cuda":
            torch.cuda.empty_cache()
        if rank == 0:
            base, hp1, g1 = run_single(a, dev, batches, K, W)
            del hp1, g1
            if dev.type == "cuda":
                torch.cuda.empty_cache()
        dist.barrier()
    if rank != 0:
        return None
    from .roofline import peaks
    hbm, _, src = peaks()
    value = B * K / (ms / 1e3)
    out = {"metric": "train_interactions_per_sec", "value": round(value, 1), "unit": "interactions/s", "n_gpus": world, "steps": K,
           "warmup": W, "ms_per_step": round(ms / K, 4), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic", "impl": "ours",
           "config": {"workload": workload_string(nu, ni, nnz, d, L, B),
                      "l2": "inputs larger than L2", "graph_build_s": round(build_s, 1), "exchange_bytes_per_step": comm_per_step, "item_sharded": item_sharded,
                      "demand_rows": demand, "cuda_graph": False, "timing": f"median of {len(blocks)} blocks of {K} steps",
                      "ms_per_step_min": round(min(blocks) / K, 4), "ms_per_step_max": round(max(blocks) / K, 4)},
           "e2e": {"value": round(B * K / (ms2 / 1e3), 1), "unit": "interactions/s", "h2d_bytes_per_step": 3 * 4 * B, "d2h_bytes_per_step": 4,
                   "ms_per_step": round(ms2 / K, 4)},
           "gpu_launches": launches, "same_workload_1gpu": base, "scaling_base": base,
           "roofline": {"kernel": "spmm gather (item-side product R_r^T . U, one rank)", "bound": "hbm", "achieved": round(alg / (t_spmm * 1e-3) / 1e9, 4),
                        "peak": hbm, "unit": "GB/s", "frac": round(alg / (t_spmm * 1e-3) / 1e9 / hbm, 4), "traffic": None, "peak_source": src,
                        "alg_bytes": alg, "ms": round(t_spmm, 4), "gather_bound_gbs": round(gather / (t_spmm * 1e-3) / 1e9, 1),
                        "note": "achieved uses compulsory bytes (every operand once); gather_bound_gbs counts one row read per non-zero"},
           "eval": ev}
    if base:
        out["speedup_vs_1gpu"] = round(value / base["value"], 3)
    return out
