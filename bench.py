"""bench.py -- LLMRec hot path on B200: train interactions/s (+ full-catalog eval users/s).

    python bench.py --gpus 1 --steps 20 --warmup 5            # our CUDA path, netflix-shaped synthetic (BASELINE.json configs[1])
    python bench.py --impl reference --steps 20 --warmup 3    # the reference's CPU algorithm (oracle port) on the host cores
    torchrun --nproc-per-node N bench.py --gpus N             # N > 1: the 10M x 1M x 200M synthetic, users sharded (configs[3])

One JSON line on stdout (rank 0).  A "step" is one full training step of Trainer (sampled batch of 1024 interactions +
augmented edges: forward, 8 BPR/prune heads, backward, dense AdamW).
  value         whole-job interactions/s with the batch indices already resident in HBM: EXACTLY --steps consecutive steps after
                --warmup (at least 3) untimed ones, between two CUDA events (synchronize on both sides); an event after every step gives
                the per-step min / max.  Before the timed window the same steps are replayed for --min-seconds of device time so that
                clocks and caches are in steady state; the parameter and optimizer updates of those replays are undone
  e2e           the same through Trainer's public API: host sampler -> pinned H2D of the index batch -> step -> D2H of the loss, every step
                (blocks of --steps steps, repeated until >= --min-seconds / 2 of device time; the median block is reported)
  roofline      the dominant kernel family of the step: algorithmic bytes / CUDA-event time vs MEASURED_PEAKS.json
  cpu_baseline  the oracle port (oracle/llmrec_oracle.py, torch CPU) on a bounded sample of the same workload
  gpu_torch_baseline  the same oracle ops with every tensor on cuda:0 (torch.sparse.mm / F.linear / AdamW = cuSPARSE / cuBLAS / ATen):
                BASELINE.json configs[1]'s "reference torch.sparse" on the same B200
  parity        netflix-shape end-to-end check: a fresh Trainer takes the SAME batches the CPU oracle trained on, then both rank the same users
  eval          Trainer.test() over every test user (scoring + top-50 + metrics), users/s, median of 5
  configs       the other BASELINE.json configurations measured in the same call: movielens d=128 L=3 (configs[2]); the 10M x 1M synthetic on
                this one GPU (= `scaling_base`, the strong-scaling base of the N > 1 lines, configs[3]) with its 1M-item eval leg (configs[4])
Features (704 MB) exceed the 126 MB L2, so consecutive steps cannot be served from cache ("inputs larger than L2").

--dump-outputs DIR writes what the last timed step left to its caller, one float32 array per file: DIR/loss.npy and DIR/<parameter
name>.npy for every parameter after that step's AdamW update.  Dataset, initialisation and batches are seeded, so two builds run with
the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import contextlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

WORKLOADS = {
    # name: (dataset, n_users, n_items, interactions, dims, embed, weight_size)
    "netflix": ("netflix", 13187, 17366, 68933, (512, 768, 1536), 64, "[64, 64]"),
    "movielens": ("movielens", 12495, 10322, 57960, (512, 768, 1536), 128, "[128,128,128]"),
}


def workload_string(name):
    """The one description both arms print (the driver compares the strings)."""
    ds, nu, ni, ne, dims, embed, wsize = WORKLOADS[name]
    return (f"{name}-shaped synthetic {nu}x{ni}, {ne} interactions (train/val/test split), d={embed}, L={len(eval(wsize))}, "
            f"batch=1024 (+aug edges), feature dims {list(dims)}")


def ensure_dataset(name):
    from llmrec_b200.synth import make_dataset
    ds, nu, ni, ne, dims, _, _ = WORKLOADS[name]
    base = os.environ.get("LLMREC_BENCH_DIR") or os.path.join(tempfile.gettempdir(), f"llmrec_bench_{os.getuid()}")
    root = os.path.join(base, f"{name}_seed0") + "/"
    marker = os.path.join(root, ".complete")
    if not os.path.exists(marker):
        os.makedirs(root, exist_ok=True)
        make_dataset(root, dataset=ds, n_users=nu, n_items=ni, n_inter=ne, dims=dims, seed=0)
        open(marker, "w").write("ok")
    return root


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.rows, self.stop_flag, self.index, self.proc = [], threading.Event(), index, None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
                if self.stop_flag.is_set():
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag.set()
        try:
            self.proc.terminate()
        except Exception:
            pass
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        mx = max((int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()), default=None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def _median(xs):
    s = sorted(xs)
    return s[len(s) // 2]


def make_trainer(workload, a, extra=()):
    import torch
    from llmrec_b200 import main as M
    from llmrec_b200.runtime import set_args
    from llmrec_b200.utility import batch_test
    from llmrec_b200.utility.load_data import Data
    from llmrec_b200.utility.parser import parse_args, resolve_dataset_dir
    ds, nu, ni, ne, dims, embed, wsize = WORKLOADS[workload]
    root = ensure_dataset(workload)
    args = set_args(parse_args(["--data_path", root, "--dataset", ds, "--debug", "--epoch", "1", "--embed_size", str(embed),
                                "--weight_size", wsize, "--proj_mode", a.proj_mode, "--host_sampler", a.host_sampler,
                                "--cuda_graph", str(a.graph)] + list(extra)))
    torch.cuda.set_device(0)
    M.set_seed(args.seed)
    with contextlib.redirect_stdout(sys.stderr):          # stdout carries exactly one JSON line
        gen = Data(path=resolve_dataset_dir(args.data_path, args.dataset), batch_size=args.batch_size, sampler=args.host_sampler)
        batch_test.init(gen, args)
        tr = M.Trainer(data_config={}, data_generator=gen)
    return tr, gen, args


def time_steps(tr, a, K, W, min_seconds, max_blocks, dump_dir=None):
    """-> dict(ms, value, ms_min, ms_max, launches) for EXACTLY K timed steps of the device-resident leg of Trainer `tr`."""
    import torch
    from llmrec_b200 import ops
    hp = tr.hot
    batches = [tr.sample_batch() for _ in range(W + K)]
    dev_batches = []
    for u, p, n in batches:
        t = torch.tensor([u, p, n], dtype=torch.int32, device="cuda")
        dev_batches.append((t[0], t[1], t[2]))
    step = hp.train_step_graphed if a.graph else hp.train_step
    for i in range(W):
        step(*dev_batches[i])
    snap = hp._snapshot_state()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    spent, blocks = 0.0, 0
    while spent < 1e3 * min_seconds and blocks < max_blocks:
        e0.record()
        for i in range(W, W + K):
            step(*dev_batches[i])
        e1.record()
        torch.cuda.synchronize()
        spent += e0.elapsed_time(e1); blocks += 1
    hp._restore_state(snap)
    del snap
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    l0 = ops.STATS["launches"]
    ev[0].record()
    for i in range(K):
        step(*dev_batches[W + i])
        ev[i + 1].record()
    torch.cuda.synchronize()
    launches = ops.STATS["launches"] - l0
    if dump_dir is not None:
        dump_outputs(hp, dump_dir)
    per_step = [ev[i].elapsed_time(ev[i + 1]) for i in range(K)]
    if a.graph:      # kernels per replayed step = launches of one eager step
        l1 = ops.STATS["launches"]
        snap = hp._snapshot_state(); hp.train_step(*dev_batches[0]); hp._restore_state(snap)
        launches = (ops.STATS["launches"] - l1) * K
    n_inter = sum(len(b[0]) for b in batches[W:])
    ms = ev[0].elapsed_time(ev[K])
    return {"ms": ms, "value": n_inter / (ms / 1e3), "ms_min": min(per_step), "ms_max": max(per_step), "launches": launches,
            "dev_batches": dev_batches}


DUMP_LIMIT = 64 << 20


def dump_outputs(hp, out_dir):
    """DIR/loss.npy and DIR/<parameter name>.npy (float32) as the last step left them (about 9 MB at netflix shape, 14 MB at movielens shape)."""
    import numpy as np
    arrays = {"loss": hp.loss.detach().float().cpu().numpy()}
    arrays.update({k: v.detach().float().cpu().numpy() for k, v in hp.p.items()})
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def time_e2e(tr, K, min_seconds, max_blocks):
    import torch
    loss_host = torch.empty(K, dtype=torch.float32).pin_memory()
    for _ in range(3):
        tr.train_next_batch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    blocks, spent, per_step = [], 0.0, []
    dev_sampler = getattr(tr, "device_sampler", None) is not None
    while True:
        torch.cuda.synchronize()
        n_e2e = h2d = 0
        n0 = float(tr._epoch_stats[3]) if dev_sampler else 0.0
        e0.record()
        for i in range(K):
            loss, B = tr.train_next_batch()          # the body of Trainer.train()'s loop: host sampler -> pinned staging -> H2D -> step
            loss_host[i:i + 1].copy_(loss, non_blocking=True)
            if not dev_sampler:
                n_e2e += B; h2d += tr.last_h2d_bytes
        e1.record()
        torch.cuda.synchronize()
        if dev_sampler:                              # batches drawn on the device: B' is accumulated there, nothing crosses PCIe but the loss
            n_e2e = int(float(tr._epoch_stats[3]) - n0)
        ms = e0.elapsed_time(e1)
        assert bool(torch.isfinite(loss_host).all()), "non-finite loss"
        blocks.append(ms); spent += ms; per_step.append((n_e2e / (ms / 1e3), h2d // K))
        if spent >= 1e3 * min_seconds or len(blocks) >= max_blocks:
            break
    i = sorted(range(len(blocks)), key=lambda j: blocks[j])[len(blocks) // 2]
    return {"value": round(per_step[i][0], 1), "unit": "interactions/s", "h2d_bytes_per_step": per_step[i][1], "d2h_bytes_per_step": 4,
            "ms_per_step": round(blocks[i] / K, 4), "blocks": len(blocks)}


def family_times(tr, dev_batch):
    """Per-kernel-family device time: each family's launches of one step, replayed R times from its own CUDA graph between two events."""
    import torch
    hp = tr.hot
    u0, p0, n0 = dev_batch
    hp.forward(); hp.loss_and_output_grads(u0, p0, n0); hp.backward()
    torch.cuda.synchronize()
    snap = hp._snapshot_state()
    fams = hp.families(u0, p0, n0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    R, fam = 10, {}
    for name, fn in fams.items():
        fn(); torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(R):
                fn()
        g.replay(); torch.cuda.synchronize()
        ts = []
        for _ in range(5):
            e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) / R)
        fam[name] = _median(ts)
    hp._restore_state(snap)
    return fam


def eval_leg(tr, gen, ni, shots=5):
    import torch
    users = list(gen.test_set.keys())
    tr.test(users, False)                         # warm-up at the timed size (scratch buffers exist afterwards)
    ts, res = [], None
    for _ in range(shots):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = tr.test(users, False)
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    t_eval = _median(ts)
    return {"metric": "eval_users_per_sec", "value": round(len(users) / t_eval, 1), "unit": "users/s", "n_users": len(users),
            "n_items": ni, "seconds": round(t_eval, 4), "seconds_min": round(min(ts), 4), "seconds_max": round(max(ts), 4), "shots": shots,
            "recall@20": float(res["recall"][1]), "ndcg@20": float(res["ndcg"][1]), "includes": "forward + scoring + top-50 + metrics, host buffers"}


def run_workload(name, a, K, W, min_seconds, with_families=True, hoist=False, extra=(), dump_dir=None):
    """One single-GPU configuration: device-resident leg (its outputs written to `dump_dir` if given), e2e leg, family roofline, eval leg."""
    import torch
    from llmrec_b200.roofline import peaks, step_bytes
    tr, gen, args = make_trainer(name, a, extra=(["--hoist_side", "1"] if hoist else []) + list(extra))
    ds, nu, ni, ne, dims, embed, wsize = WORKLOADS[name]
    t = time_steps(tr, a, K, W, min_seconds, a.max_blocks, dump_dir)
    e2e = time_e2e(tr, K, min_seconds / 2, a.max_blocks)
    out = {"workload": workload_string(name), "ms_per_step": round(t["ms"] / K, 4), "value": round(t["value"], 1), "unit": "interactions/s",
           "ms_per_step_min": round(t["ms_min"], 4), "ms_per_step_max": round(t["ms_max"], 4),
           "e2e": e2e, "gpu_launches": t["launches"], "train_edges": int(gen.n_train)}
    if with_families and not hoist:
        fam = family_times(tr, t["dev_batches"][0])
        bytes_ = step_bytes(tr.hot, tr.graph.nnz)
        hbm, tf, src = peaks()
        top = max((k for k in fam if k in bytes_), key=lambda k: fam[k])
        ach = bytes_[top] / (fam[top] * 1e-3) / 1e9
        traffic, traffic_src = None, None
        try:                                          # per-launch DRAM bytes of this kernel family from the committed ncu capture
            tj = json.load(open(os.path.join(REPO, "profiles", "ncu_traffic.json"))).get(top)
            if tj and name == "netflix" and not hoist:
                traffic, traffic_src = int(tj["bytes"]), tj["source"]
        except Exception:
            pass
        out["roofline"] = {"kernel": top, "bound": "hbm", "achieved": round(ach, 1), "peak": hbm, "unit": "GB/s", "frac": round(ach / hbm, 4),
                           "traffic": traffic, "traffic_source": traffic_src, "peak_source": src, "alg_bytes_per_step": bytes_[top],
                           "ms_per_step": round(fam[top], 4),
                           "families_ms": {k: round(v, 4) for k, v in sorted(fam.items(), key=lambda kv: -kv[1])},
                           "families_gbs": {k: round(bytes_[k] / (fam[k] * 1e-3) / 1e9, 1) for k in fam if k in bytes_},
                           "families_frac": {k: round(bytes_[k] / (fam[k] * 1e-3) / 1e9 / hbm, 3) for k in fam if k in bytes_},
                           "families_sum_ms": round(sum(fam.values()), 4),
                           "note": "each family is timed alone from its own CUDA graph; the step overlaps independent families as parallel graph "
                                   "branches (ID-layer products beside the projections / weight gradients, gradient init, bias column sums), so "
                                   "ms_per_step < families_sum_ms"}
    out["eval"] = eval_leg(tr, gen, ni)
    return out, tr, gen


def parity_leg(a, side):
    """A fresh Trainer (same seed -> same init, asserted by the golden tests) trains on the batches the CPU oracle trained on,
    then both rank the same test users: losses, Recall@20 / NDCG@20 (north_star: within 1e-4) and the top-50 lists."""
    import torch
    from llmrec_b200.utility import batch_test
    tr, gen, args = make_trainer(a.workload, a)
    losses = [float(tr.train_batch(u, p, n)) for (u, p, n) in side["batches"]]
    users = side["users"]
    res = tr.test(users, False)
    idx, _ = batch_test.rank_block(tr.hot.U, tr.hot.I, users, False)
    top = idx.cpu().numpy()
    same = sum(1 for j, u in enumerate(users) if list(top[j]) == list(side["tops"][u]))
    same_set = sum(1 for j, u in enumerate(users) if set(top[j].tolist()) == set(side["tops"][u]))
    ol = side["losses"]
    return {"steps": len(losses), "users_ranked": len(users), "loss_max_rel_diff": float(max(abs(x - y) / max(1.0, abs(y)) for x, y in zip(losses, ol))),
            "recall@20_gpu": float(res["recall"][1]), "recall@20_oracle": float(side["res"]["recall"][1]),
            "ndcg@20_gpu": float(res["ndcg"][1]), "ndcg@20_oracle": float(side["res"]["ndcg"][1]),
            "recall@20_abs_diff": float(abs(res["recall"][1] - side["res"]["recall"][1])), "ndcg@20_abs_diff": float(abs(res["ndcg"][1] - side["res"]["ndcg"][1])),
            "top50_identical_lists": round(same / max(1, len(users)), 5), "top50_identical_sets": round(same_set / max(1, len(users)), 5),
            "tolerance": "north_star: Recall@20 / NDCG@20 within 1e-4, identical top-K sets except fp32 near-ties"}


def gpu_torch_baseline(a, steps, eval_users=256):
    """The oracle's torch ops with every tensor on cuda:0 -- torch.sparse.mm (cuSPARSE), F.linear (cuBLAS), autograd, torch.optim.AdamW,
    host argsort per BPR head and float(loss) per step as main.py:159,280 do -- i.e. the reference's own GPU path on this B200."""
    import torch
    from oracle import llmrec_oracle as O
    from llmrec_b200.synth import DATASET_DIR
    ds, nu, ni, ne, dims, embed, wsize = WORKLOADS[a.workload]
    data = O.load_dataset(os.path.join(ensure_dataset(a.workload), DATASET_DIR[ds]))
    cfg = O.OracleConfig(embed_size=embed, weight_size=tuple(eval(wsize)))
    O.set_seed(cfg.seed)
    tr = O.OracleTrainer(data, cfg, device="cuda")
    batches = [O.sample_batch(data, cfg) for _ in range(steps + 3)]
    for b in batches[:3]:
        tr.step(*b)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); n = 0
    for b in batches[3:]:
        tr.step(*b); n += len(b[0])
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    users = list(data.test_set.keys())[:eval_users]
    t1 = time.perf_counter()
    tr.test(users, faithful=True)
    de = time.perf_counter() - t1
    return {"value": round(n / (ms / 1e3), 1), "unit": "interactions/s", "ms_per_step": round(ms / steps, 3), "steps": steps, "kind": "port on cuda",
            "what": f"oracle port with tensors on cuda:0, torch {torch.__version__}: torch.sparse.mm + F.linear + autograd + torch.optim.AdamW, host argsort per head and float(loss) per step as the reference",
            "eval": {"value": round(len(users) / de, 1), "unit": "users/s", "sample": f"{len(users)} users: device matmul, D2H of the score block, per-user heapq on the host (batch_test.py:150-157)"}}


def cpu_baseline(a, steps, eval_users, warmup=1, side=None):
    """The oracle port timed on the host cores: `steps` training steps + eval of `eval_users` users."""
    import torch
    from oracle import llmrec_oracle as O
    ds, nu, ni, ne, dims, embed, wsize = WORKLOADS[a.workload]
    root = ensure_dataset(a.workload)
    from llmrec_b200.synth import DATASET_DIR
    data = O.load_dataset(os.path.join(root, DATASET_DIR[ds]))
    cores = os.cpu_count()
    cfg = O.OracleConfig(embed_size=embed, weight_size=tuple(eval(wsize)))
    # torch's intra-op pool oversubscribes badly on many-core hosts (128 threads: 5 s/step vs 0.25 s at 8): use the
    # thread count that runs one step fastest ("all the host threads it can use" without thrashing)
    O.set_seed(cfg.seed + 1)
    probe = O.OracleTrainer(data, cfg)
    best_t, best_dt = None, None
    for nt in sorted({min(cores, c) for c in (8, 16, 32, 64)}):
        torch.set_num_threads(nt)
        b = O.sample_batch(data, cfg)
        probe.step(*b)
        t0 = time.perf_counter(); probe.step(*b); dt = time.perf_counter() - t0
        if best_dt is None or dt < best_dt:
            best_t, best_dt = nt, dt
    del probe
    torch.set_num_threads(best_t)
    O.set_seed(cfg.seed)                       # the run that is timed starts from the reference's seeded state (main.py:363)
    tr = O.OracleTrainer(data, cfg)
    batches, losses = [], []
    t0 = time.perf_counter(); n = 0; t_warm = 0.0
    for i in range(warmup + steps):
        if i == warmup:
            t_warm = time.perf_counter() - t0
        u, p, ng = O.sample_batch(data, cfg)
        l, _ = tr.step(u, p, ng)
        batches.append((u, p, ng)); losses.append(l)
        if i >= warmup:
            n += len(u)
    dt = time.perf_counter() - t0 - t_warm
    users = list(data.test_set.keys())[:eval_users]
    t1 = time.perf_counter()
    res, tops = (tr.test(users, faithful=True) if users else (None, None))
    de = time.perf_counter() - t1
    if side is not None:
        side.update(batches=batches, losses=losses, users=users, res=res, tops=tops)
    return {"value": round(n / dt, 1), "unit": "interactions/s", "cores": best_t, "host_cores": cores, "kind": "port",
            "sample": f"{steps} training steps ({dt:.1f} s) of the same workload, torch {torch.__version__} CPU with {torch.get_num_threads()} threads",
            "ms_per_step": round(dt / steps * 1e3, 2),
            "eval": {"value": round(len(users) / de, 1) if users else None, "unit": "users/s", "sample": f"{len(users)} test users, per-user heapq ranking ({de:.1f} s)"}}


def run_ours(a):
    import torch
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    if world > 1 or a.workload == "synthetic":
        from llmrec_b200.dist_bench import run_sharded
        return run_sharded(a)
    K, W = a.steps, max(a.warmup, 3)
    ds, nu, ni, ne, dims, embed, wsize = WORKLOADS[a.workload]
    clocks = ClockSampler(0); clocks.start()      # samples clocks / throttle reasons across the value and e2e legs
    main, tr, gen = run_workload(a.workload, a, K, W, a.min_seconds, dump_dir=a.dump_outputs)
    clk = clocks.finish()
    out = {"metric": "train_interactions_per_sec", "value": main["value"], "unit": "interactions/s", "n_gpus": 1, "steps": K, "warmup": W,
           "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic", "impl": "ours",
           "config": {"workload": workload_string(a.workload), "train_edges": main["train_edges"],
                      "interactions_counted": "sum(len(users)) incl. augmented edges", "l2": "inputs larger than L2 (704 MB of features per step)",
                      "proj_mode": a.proj_mode, "host_sampler": a.host_sampler, "cuda_graph": bool(a.graph),
                      "timing": f"{K} consecutive steps between CUDA events after {W} untimed ones",
                      "ms_per_step_min": main["ms_per_step_min"], "ms_per_step_max": main["ms_per_step_max"]},
           "e2e": main["e2e"], "gpu_launches": main["gpu_launches"], "clocks": clk, "roofline": main["roofline"], "eval": main["eval"]}
    del tr
    torch.cuda.empty_cache()
    side = {}
    if not a.no_cpu:
        out["cpu_baseline"] = cpu_baseline(a, steps=a.cpu_steps, eval_users=a.cpu_eval_users, side=side)
        out["parity"] = parity_leg(a, side)
    if a.gpu_baseline:
        out["gpu_torch_baseline"] = gpu_torch_baseline(a, steps=K)
        torch.cuda.empty_cache()
    if a.extra:
        cfgs = {}
        try:
            h, _, _ = run_workload(a.workload, a, K, W, min(a.min_seconds, 1.0), hoist=True)
            cfgs[a.workload + "_hoisted"] = dict(h, note="--hoist_side 1: constant side-feature propagation precomputed (SURVEY.md 8f-3); same results within the golden tolerances")
            torch.cuda.empty_cache()
        except Exception as e:                                        # an extra leg must never take the headline down
            cfgs[a.workload + "_hoisted"] = {"error": repr(e)[:300]}
        if a.extra == 2:                                              # quick A/B runs: the hoisted line only
            out["configs"] = cfgs
            return out
        try:
            dsm, _, _ = run_workload(a.workload, a, K, W, min(a.min_seconds, 1.0), with_families=False, hoist=True, extra=["--device_sampler", "1"])
            cfgs[a.workload + "_hoisted_device_sampler"] = dict(dsm, note="--hoist_side 1 --device_sampler 1: batches drawn on the GPU inside the replayed graph "
                                                                "(SURVEY.md 8f-1; same distributions, not the reference's RNG streams); e2e moves no index bytes")
            torch.cuda.empty_cache()
        except Exception as e:
            cfgs[a.workload + "_hoisted_device_sampler"] = {"error": repr(e)[:300]}
        other = "movielens" if a.workload == "netflix" else "netflix"
        try:
            m, _, _ = run_workload(other, a, K, W, min(a.min_seconds, 1.0))
            cfgs[other] = m
            torch.cuda.empty_cache()
        except Exception as e:
            cfgs[other] = {"error": repr(e)[:300]}
        try:
            from llmrec_b200 import dist_bench
            dev = torch.device("cuda", 0)
            nu_s, ni_s, ne_s, d_s, L_s = dist_bench.syn_sizes(a.syn_scale)
            bg = torch.Generator(device=dev).manual_seed(99)
            B = 1126
            batches = [(torch.randint(0, nu_s, (B,), device=dev, generator=bg, dtype=torch.int32),
                        torch.randint(0, ni_s, (B,), device=dev, generator=bg, dtype=torch.int32),
                        torch.randint(0, ni_s, (B,), device=dev, generator=bg, dtype=torch.int32)) for _ in range(8)]
            base, hp1, g1 = dist_bench.run_single(a, dev, batches, 5, 3, tag="this GPU")
            base["workload"] = dist_bench.workload_string(nu_s, ni_s, base["nnz"], d_s, L_s, B)
            base["eval"] = dist_bench.eval_leg(a, hp1, g1, dev, 1, 0, nu_s, nu_s)
            del hp1, g1
            torch.cuda.empty_cache()
            cfgs["synthetic_1gpu"] = base
            out["scaling_base"] = {k: base[k] for k in ("n_gpus", "value", "unit", "ms_per_step", "workload")}
        except Exception as e:
            cfgs["synthetic_1gpu"] = {"error": repr(e)[:300]}
        out["configs"] = cfgs
    return out


def run_reference(a):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return None
    cb = cpu_baseline(a, steps=max(1, a.steps), eval_users=a.cpu_eval_users, warmup=max(1, min(a.warmup, 3)))
    cfg_note = {}
    if a.gpus > 1:
        # our arm runs the 10M x 1M synthetic workload at N > 1; one step of it on the host cores (8 SpMMs over 200 M non-zeros, 25 GB of
        # fp32 state) does not fit a few-minute arm, so the CPU line stays on the workload the reference itself can run
        cfg_note = {"n_gpus_note": "CPU arm: rank 0 only, netflix-shaped workload at every N (the reference pins one device, main.py:23; "
                                   "the 10M x 1M synthetic of the N>1 GPU arm is out of reach of its CPU path within the arm's time limit)"}
    return {"metric": "train_interactions_per_sec", "value": cb["value"], "unit": "interactions/s", "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": workload_string(a.workload),
                       "note": "reference algorithm as the CPU oracle port (the Python reference has no installable package and cannot travel to the GPU box)",
                       **cfg_note},
            "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "interactions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "eval": cb["eval"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed training steps (N=1: exactly this many; the e2e leg times blocks of this many)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="netflix", choices=list(WORKLOADS) + ["synthetic"])
    ap.add_argument("--min-seconds", dest="min_seconds", type=float, default=2.0, help="N=1: untimed replays of the K timed steps before they are timed, and the e2e leg's repeated K-step blocks; N>1: repeat the K-step block until this much device time, the median block is reported")
    ap.add_argument("--max-blocks", dest="max_blocks", type=int, default=400)
    ap.add_argument("--pieces", type=int, default=1, help="N>1: item-row pieces of the exchange SpMMs (all-reduce of piece k overlaps SpMM of piece k+1)")
    ap.add_argument("--item-sharded", dest="item_sharded", type=int, default=0, help="N>1: reduce-scatter / row-local work / all-gather form of the item-side exchanges, AdamW of the item table sharded by item")
    ap.add_argument("--demand", type=int, default=1, help="synthetic workload: training forward/backward restricted to the rows the batch can reach (identical results)")
    ap.add_argument("--n1-base", dest="n1_base", type=int, default=1, help="N>1: also time the same synthetic workload on rank 0 alone")
    ap.add_argument("--eval-users", dest="eval_users", type=int, default=102400, help="users ranked in the synthetic eval leg")
    ap.add_argument("--syn-scale", dest="syn_scale", type=float, default=1.0, help="size factor of the 10M x 1M x 200M synthetic graph")
    ap.add_argument("--proj_mode", default="3xtf32")
    ap.add_argument("--host_sampler", default="native")
    ap.add_argument("--no-cpu", dest="no_cpu", action="store_true")
    ap.add_argument("--gpu-baseline", dest="gpu_baseline", type=int, default=1)
    ap.add_argument("--extra", type=int, default=1, help="N=1: also measure the hoisted mode, the other small configuration and the synthetic 1-GPU scaling base (2: the hoisted mode only)")
    ap.add_argument("--graph", type=int, default=1)
    ap.add_argument("--cpu-steps", dest="cpu_steps", type=int, default=24)
    ap.add_argument("--cpu-eval-users", dest="cpu_eval_users", type=int, default=1500)
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="N=1: write the loss and the parameters after the last timed step to DIR/<name>.npy (float32)")
    a = ap.parse_args()
    if a.dump_outputs is not None and (a.impl != "ours" or a.gpus > 1 or a.workload == "synthetic"):
        ap.error("--dump-outputs covers the single-GPU CUDA path (--impl ours --gpus 1, workload netflix or movielens)")
    if a.workload == "synthetic" and a.impl == "reference":
        a.workload = "netflix"
    out = run_reference(a) if a.impl == "reference" else run_ours(a)
    if out is not None and int(os.environ.get("RANK", 0)) == 0:
        print(json.dumps(out), flush=True)
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    main()
