#!/usr/bin/env python
"""bench.py -- boosting rounds/sec on synthetic 10M x 100 (BASELINE.json metric, config C3).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" is one boosting round (gradient -> all tree levels -> prediction-cache update, including
the per-level histogram allreduce) over the fixed synthetic matrix; the 10M rows are row-sharded
INTERLEAVED over the N ranks (strong scaling, one process per GPU).  `value` is timed with the
quantised matrix resident in HBM; `e2e` goes through the xgb.train() replacement with HOST buffers
(upload + GPU sketch/binning + K rounds + a per-round metric read-back, all inside the timed region).
`--impl reference` times the CPU path (the oracle port of XGBoost hist; `xgboost` itself is not
installable here) on the host cores for the same config.
`--dump-outputs DIR` writes, after the timed steps, what the timed path computed in its last step (see dump_outputs);
the synthetic inputs depend on the arguments only, so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PARAMS = {"objective": "reg:squarederror", "max_depth": 8, "eta": 0.3, "lambda": 1.0, "gamma": 0.0,
          "min_child_weight": 1.0, "max_bin": 256, "base_score": 0.5, "tree_method": "hist"}


WORKLOADS = {   # SURVEY.md 8(d); C3 is the configuration the metric is quoted on, the others are opt-in (--workload)
    "C2": {"rows": 11_000_000, "cols": 28, "depth": 6, "objective": "binary:logistic"},
    "C3": {"rows": 10_000_000, "cols": 100, "depth": 8, "objective": "reg:squarederror"},
    "C4": {"rows": 100_000_000, "cols": 50, "depth": 10, "objective": "binary:logistic"},
    "C5": {"rows": 50_000_000, "cols": 200, "depth": 6, "objective": "multi:softprob", "num_class": 10},
}


def feature_types(workload, cols):
    """C5: the last quarter of the columns is categorical with cardinalities 4/16/64/256 cycling."""
    if workload != "C5":
        return None
    n_cat = cols // 4
    return ["q"] * (cols - n_cat) + ["c"] * n_cat


def synth_block(block, rows, cols, seed=1234, workload="C3"):
    """Deterministic block of a synthetic dataset (SURVEY.md 8d).
    C3: x~U[0,10), y = sum_{j<10} a_j x_j + sin(x_10) + N(0,0.1).
    C2: 3/4 of the columns N(0,1), the rest exp(N(0,1)) (HIGGS-like); label ~ Bernoulli(sigmoid(w.x[:8] + 0.5 x0 x1)).
    C4: x~U[0,10); label as C2 on centred features."""
    rng = np.random.default_rng([seed, block])
    a = np.random.default_rng(seed).normal(size=10).astype(np.float32)
    if workload == "C3":
        X = rng.random((rows, cols), dtype=np.float32) * np.float32(10.0)
        k = min(10, cols)
        y = X[:, :k] @ a[:k]
        if cols > 10:
            y = y + np.sin(X[:, 10])
        y = y + rng.normal(scale=0.1, size=rows).astype(np.float32)
        return X, y.astype(np.float32)
    if workload == "C5":
        n_cat = cols // 4
        n_num = cols - n_cat
        X = np.empty((rows, cols), np.float32)
        X[:, :n_num] = rng.random((rows, n_num), dtype=np.float32) * np.float32(10.0)
        cards = [(4, 16, 64, 256)[j % 4] for j in range(n_cat)]
        for j, c in enumerate(cards):
            X[:, n_num + j] = rng.integers(0, c, size=rows)
        wrng = np.random.default_rng(seed + 5)
        k_num, k_cat = min(20, n_num), min(8, n_cat)
        W = wrng.normal(size=(k_num, 10)).astype(np.float32)
        score = (X[:, :k_num] - np.float32(5.0)) @ W
        for j in range(k_cat):
            eff = wrng.normal(scale=4.0, size=(cards[j], 10)).astype(np.float32)
            score += eff[X[:, n_num + j].astype(np.int64)]
        score += rng.normal(scale=1.0, size=score.shape).astype(np.float32)
        return X, score.argmax(axis=1).astype(np.float32)
    if workload == "C2":
        X = rng.standard_normal((rows, cols), dtype=np.float32)
        heavy = cols - (3 * cols) // 4
        np.exp(X[:, cols - heavy:], out=X[:, cols - heavy:])
        Z = X
    else:
        X = rng.random((rows, cols), dtype=np.float32) * np.float32(10.0)
        Z = (X[:, :8] - np.float32(5.0)) * np.float32(0.4)
    k = min(8, cols)
    s = Z[:, :k] @ a[:k] + np.float32(0.5) * Z[:, 0] * Z[:, 1]
    y = (rng.random(rows, dtype=np.float32) < 1.0 / (1.0 + np.exp(-s))).astype(np.float32)
    return X, y


def synth_block_gpu(block, rows, cols, seed=1234, workload="C4", device="cuda"):
    """The large configurations (C4 100M x 50, C5 50M x 200) generate their blocks with torch's Philox generator on the
    GPU (numpy needs minutes of host time for 10^10 values); same distributions as synth_block, returned as host arrays.
    The stream depends on (seed, block) only, so every rank count sees the same global matrix."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed * 100003 + block)
    a = torch.from_numpy(np.random.default_rng(seed).normal(size=10).astype(np.float32)).to(device)
    if workload == "C5":
        n_cat = cols // 4
        n_num = cols - n_cat
        X = torch.empty((rows, cols), dtype=torch.float32, device=device)
        X[:, :n_num] = torch.rand((rows, n_num), generator=g, device=device) * 10.0
        cards = [(4, 16, 64, 256)[j % 4] for j in range(n_cat)]
        for j, c in enumerate(cards):
            X[:, n_num + j] = torch.randint(0, c, (rows,), generator=g, device=device).float()
        wrng = np.random.default_rng(seed + 5)
        k_num, k_cat = min(20, n_num), min(8, n_cat)
        W = torch.from_numpy(wrng.normal(size=(k_num, 10)).astype(np.float32)).to(device)
        score = (X[:, :k_num] - 5.0) @ W
        for j in range(k_cat):
            eff = torch.from_numpy(wrng.normal(scale=4.0, size=(cards[j], 10)).astype(np.float32)).to(device)
            score += eff[X[:, n_num + j].long()]
        score += torch.randn(score.shape, generator=g, device=device)
        return X.cpu().numpy(), score.argmax(dim=1).float().cpu().numpy()
    if workload == "C3":
        X = torch.rand((rows, cols), generator=g, device=device) * 10.0
        k = min(10, cols)
        y = X[:, :k] @ a[:k]
        if cols > 10:
            y = y + torch.sin(X[:, 10])
        y = y + torch.randn(rows, generator=g, device=device) * 0.1
        return X.cpu().numpy(), y.cpu().numpy()
    if workload == "C2":
        X = torch.randn((rows, cols), generator=g, device=device)
        heavy = cols - (3 * cols) // 4
        X[:, cols - heavy:] = torch.exp(X[:, cols - heavy:])
        Z = X
    else:
        X = torch.rand((rows, cols), generator=g, device=device) * 10.0
        Z = (X[:, :8] - 5.0) * 0.4
    k = min(8, cols)
    sc = Z[:, :k] @ a[:k] + 0.5 * Z[:, 0] * Z[:, 1]
    y = (torch.rand(rows, generator=g, device=device) < torch.sigmoid(sc)).float()
    return X.cpu().numpy(), y.cpu().numpy()


GPU_GEN = {"on": False}     # set by main() for the configurations with more than 2e9 values (or --gen gpu)


def synth_shard(n_rows, cols, rank, world, block_rows=1_000_000, workload="C3"):
    """Rows rank, rank+world, ... of the global matrix (INTERLEAVED sharding, matrix.py:1100)."""
    n_local = len(range(rank, n_rows, world))
    cache = os.environ.get("B2_BENCH_CACHE")   # optional .npy cache of the generated shard (A/B runs inside one gpurun call)
    cpath = os.path.join(cache, "%s%s_%d_%d_%d_%d.npz" % (workload, "g" if GPU_GEN["on"] else "", n_rows, cols, rank, world)) if cache else None
    if cpath and os.path.exists(cpath):
        z = np.load(cpath)
        return z["X"], z["y"]
    Xs = np.empty((n_local, cols), dtype=np.float32)
    ys = np.empty(n_local, dtype=np.float32)
    at = 0
    for b, start in enumerate(range(0, n_rows, block_rows)):
        rows = min(block_rows, n_rows - start)
        X, y = (synth_block_gpu if GPU_GEN["on"] else synth_block)(b, rows, cols, workload=workload)
        first = (rank - start) % world
        m = len(range(first, rows, world))
        Xs[at:at + m] = X[first::world]
        ys[at:at + m] = y[first::world]
        at += m
    if cpath:
        os.makedirs(cache, exist_ok=True)
        np.savez(cpath, X=Xs, y=ys)
    return Xs, ys


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons sampled through NVML every 5 ms during the timed region."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.err = index, [], threading.Event(), None

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis else self.index
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            while not self.stop_flag.is_set():
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                try:
                    rs = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    rs = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append((sm, rs))
                self.stop_flag.wait(0.005)
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable: %s" % self.err]}
        sm = sorted(s[0] for s in self.samples)
        mask = 0
        for _, rs in self.samples:
            mask |= rs
        return {"sm_mhz": float(sm[len(sm) // 2]), "sm_max_mhz": float(self.max_sm),
                "reasons": [n for n, bit in self.REASONS if mask & bit], "samples": len(sm)}


def workload_string(args):
    """Identical on both arms (the driver compares the config of the reference arm with ours)."""
    return "%s synthetic %dx%d %s depth %d 256 bins" % (args.workload, args.rows, args.cols, args.objective, args.depth)


def _sha(*arrays):
    import hashlib
    h = hashlib.sha256()
    for a in arrays:
        h.update(a if isinstance(a, (bytes, bytearray)) else np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def parity_check(E, args, rank, world, dm_kw, bst_timed, dm_timed):
    """Outside the timed region: (1) hashes of the timed model and of its cut points -- integer histograms make them
    independent of the GPU count, so the SCALE lines must carry the same values at N = 1/2/4/8; (2) a 200k-row, 3-round
    sub-problem of the same workload trained on all N ranks and compared tree for tree with the fixed-point CPU oracle
    on rank 0 (split feature / bin / default direction bit-exact, leaf values within 1e-5)."""
    dump = "\n".join(bst_timed.get_dump(dump_format="json", with_stats=True)).encode()
    ptrs, vals, mins, hm = dm_timed.get_cuts()
    out = {"model_sha256": _sha(dump), "cuts_sha256": _sha(ptrs, vals, mins, hm), "oracle_match": None}
    n_sub, rounds = min(200_000, args.rows), 3
    Xs, ys = synth_shard(n_sub, args.cols, rank, world, workload=args.workload)
    params = dict(PARAMS, max_depth=min(args.depth, 8), objective=args.objective, profile=0)
    if args.num_class:
        params["num_class"] = args.num_class
    d = E.DMatrix(Xs, label=ys, **dm_kw)
    b = E.train(params, d, num_boost_round=rounds, verbose_eval=False)
    trees = b.get_trees()
    out["sub_model_sha256"] = _sha("\n".join(b.get_dump(dump_format="json", with_stats=True)).encode())
    if rank == 0:
        from oracle import oracle as O
        O.build()
        O.use_all_cores()
        Xf, yf = synth_shard(n_sub, args.cols, 0, 1, workload=args.workload)
        is_cat = [1 if t == "c" else 0 for t in args.feature_types] if args.feature_types else None
        ob, _ = O.train(params, Xf, yf, rounds, is_cat=is_cat)
        ok = len(trees) == ob.num_trees
        worst = 0.0
        for i, t in enumerate(trees):
            if not ok:
                break
            o = ob.tree(i)
            ok = (np.array_equal(t["split_feature"], o.split_feature) and np.array_equal(t["split_bin"], o.split_bin)
                  and np.array_equal(t["default_left"], o.default_left))
            if ok:
                leaf = o.split_feature < 0
                worst = max(worst, float(np.max(np.abs(t["value"][leaf] - o.value[leaf]))))
        out["oracle_match"] = bool(ok and worst <= 1e-5)
        out["oracle_sub_problem"] = "%d rows x %d cols, %d rounds, depth %d, %d rank(s); max |leaf - oracle| %.3g" % (
            n_sub, args.cols, rounds, params["max_depth"], world, worst)
    del b, d
    return out


TREE_FIELDS = ("left", "right", "parent", "split_feature", "split_bin", "split_cond", "default_left", "value",
               "base_weight", "loss_chg", "sum_hess", "split_type", "cat_bits")
DUMP_MARGIN_VALUES = 12_000_000     # float32: 48 MB, which keeps a dump (trees included) under 64 MB


def dump_outputs(out_dir, trees, margin):
    """Write the outputs of one boosting round as .npy files (float32 / float64) under out_dir:
    tree_<field>.npy -- the node arrays of the trees the round added, concatenated in tree order (integer fields as
                        float64, which holds them exactly); tree_nodes.npy -- the node count of each of those trees;
    margin.npy       -- the training margin (prediction cache) after the round, rows x outputs; above
                        DUMP_MARGIN_VALUES values only the rows of a fixed sample (numpy default_rng(0), sorted)."""
    files = {"tree_nodes": np.array([len(t["left"]) for t in trees], np.float64)}
    for k in TREE_FIELDS:
        a = np.concatenate([np.asarray(t[k]) for t in trees])
        files["tree_" + k] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
    m = np.asarray(margin, np.float32)
    m = m.reshape(m.shape[0], -1)
    if m.size > DUMP_MARGIN_VALUES:
        rows = np.random.default_rng(0).choice(m.shape[0], DUMP_MARGIN_VALUES // m.shape[1], replace=False)
        m = m[np.sort(rows)]
    files["margin"] = m
    os.makedirs(out_dir, exist_ok=True)
    for name, a in files.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def hist_traffic_per_launch():
    """dram bytes per launch of the histogram kernel from the committed ncu --set full capture."""
    p = os.path.join(ROOT, "profiles", "hist_traffic.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return d.get("dram_bytes_per_launch"), d.get("algorithmic_bytes_per_launch_same_capture")
        except Exception:
            return None, None
    return None, None


def run_reference(args, rank, world):
    """CPU arm: the oracle port (kind "port") with all host threads, full config."""
    if rank != 0:
        return
    from oracle import oracle as O
    O.build()
    cores = O.use_all_cores()
    X, y = synth_shard(args.rows, args.cols, 0, 1, workload=args.workload)
    params = dict(PARAMS, max_depth=args.depth, hist_qbits=0, objective=args.objective)   # qbits=0: float64 histograms = XGBoost CPU hist
    if args.num_class:
        params["num_class"] = args.num_class
    is_cat = [1 if t == "c" else 0 for t in args.feature_types] if args.feature_types else None
    t0 = time.time()
    cuts = O.Cuts.from_data(X, 256, is_cat=is_cat)
    bins = cuts.bin(X)
    t_quant = time.time() - t0
    bst = O.Booster(params, cuts)
    bst.init_margin(X.shape[0])
    for _ in range(args.warmup):
        bst.boost(bins, y)
    t0 = time.time()
    for _ in range(args.steps):
        bst.boost(bins, y)
    dt = time.time() - t0
    if args.dump_outputs:
        trees = [bst.tree(i) for i in range(bst.num_trees - bst.K, bst.num_trees)]
        dump_outputs(args.dump_outputs, [{k: getattr(t, k) for k in TREE_FIELDS} for t in trees], bst.margin)
    v = args.steps / dt
    line = {"impl": "reference", "metric": "boosting rounds/sec", "value": v, "unit": "rounds/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_string(args),
                       "rows": args.rows, "cols": args.cols, "max_depth": args.depth, "max_bin": 256},
            "cpu_baseline": {"value": v, "unit": "rounds/s", "cores": cores, "kind": "port",
                             "sample": "full workload, %d timed rounds; CPU quantisation %.1fs not in the timed region" % (args.steps, t_quant)},
            "e2e": {"value": v, "unit": "rounds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C3", choices=sorted(WORKLOADS), help="SURVEY.md 8(d) configuration (default C3, the headline)")
    ap.add_argument("--rows", type=int, default=None)
    ap.add_argument("--cols", type=int, default=None)
    ap.add_argument("--depth", type=int, default=None)
    ap.add_argument("--qbits", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--gen", default="auto", choices=["auto", "cpu", "gpu"],
                    help="synthetic data generator: numpy on the host, or torch Philox on the GPU (default for > 2e9 values)")
    ap.add_argument("--no-public-e2e", action="store_true", help="skip the end-to-end run through train(RayDMatrix, RayParams)")
    ap.add_argument("--profile", type=int, default=1, help="2 = per-phase CUDA-event timers (adds event records)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the trees of the last step and the training margin as .npy files "
                         "(rank 0; with several ranks, the margin of rank 0's rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    wl = WORKLOADS[args.workload]
    args.rows = args.rows or wl["rows"]
    args.cols = args.cols or wl["cols"]
    args.depth = args.depth or wl["depth"]
    args.objective = wl["objective"]
    args.num_class = wl.get("num_class")
    args.feature_types = feature_types(args.workload, args.cols)
    GPU_GEN["on"] = args.gen == "gpu" or (args.gen == "auto" and args.rows * args.cols > 2_000_000_000)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from xgboost_ray_b200 import engine as E

    torch.cuda.set_device(local_rank)
    os.environ["B2_DEVICE"] = str(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    params = dict(PARAMS, max_depth=args.depth, profile=args.profile, objective=args.objective)
    if args.num_class:
        params["num_class"] = args.num_class
    dm_kw = {"feature_types": args.feature_types, "enable_categorical": True} if args.feature_types else {}
    if args.qbits is not None:
        params["hist_qbits"] = args.qbits

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- communicator: rank 0's NCCL id broadcast through torch.distributed (plumbing only)
    comm_args = {"b2_world": world, "b2_rank": rank, "b2_device": local_rank}
    if world > 1:
        uid = [E.get_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        comm_args["b2_uid"] = uid[0]

    X, y = synth_shard(args.rows, args.cols, rank, world, workload=args.workload)
    sampler = ClockSampler(local_rank)
    with E.CommunicatorContext(**comm_args):
        # ================= device-resident arm: matrix quantised and resident before timing
        if rank == 0:
            sampler.start()      # NVML init takes longer than a short timed region; samples are reset below
        dm = E.DMatrix(X, label=y, **dm_kw)
        if world > 1:
            E.collective.allreduce([0.0])    # NCCL connects its peers lazily on the first collective: keep that out of quantise_seconds
        t0 = time.time()
        dm._ensure_quantized(256)
        t_quant = time.time() - t0
        bst = E.Booster(params, cache=[dm])
        for r in range(args.warmup):
            bst.update(dm, r)
        bst.get_timers(reset=True)
        barrier()
        sampler.samples.clear()
        t0 = time.perf_counter()
        for r in range(args.steps):
            bst.update(dm, args.warmup + r)
        barrier()
        wall = time.perf_counter() - t0
        sampler.stop_flag.set()
        timers = bst.get_timers(reset=True)
        wall = max_over_ranks(wall)
        dev_ms = max_over_ranks(timers["round_ms"])
        hist_ms = max_over_ranks(timers["hist_ms"])
        ms_per_step = 1e3 * wall / args.steps
        value = args.steps / wall
        if args.dump_outputs and rank == 0:
            n_trees, per_round = bst.num_trees(), bst.num_class * bst.num_parallel_tree
            dump_outputs(args.dump_outputs, [bst.get_tree(i) for i in range(n_trees - per_round, n_trees)],
                         bst.predict(dm, output_margin=True, training=True))
        final_metric = bst.eval_set([(dm, "train")], 0).split("\t", 1)[-1]
        exchange_kind = "none (1 GPU)" if world == 1 else ("nccl" if os.environ.get("B2_EXCHANGE", "").lower() == "nccl" else "nvlink peer memory (nccl if peers cannot be mapped)")
        parity = None if args.no_parity else parity_check(E, args, rank, world, dm_kw, bst, dm)
        del bst

        # ================= e2e arm: host buffers -> xgb.train replacement, copies inside the timed region
        e2e = None
        if not args.no_e2e:
            barrier()
            t0 = time.perf_counter()
            d2 = E.DMatrix(X, label=y, **dm_kw)             # host -> device upload
            t_up = time.perf_counter() - t0
            d2._ensure_quantized(256)                       # GPU sketch + binning (train() would do it itself)
            t_q = time.perf_counter() - t0 - t_up
            res = {}
            b2 = E.train(params, d2, num_boost_round=args.steps, evals=[(d2, "train")], evals_result=res, verbose_eval=False)
            barrier()
            e2e_wall = max_over_ranks(time.perf_counter() - t0)
            e2e = {"value": args.steps / e2e_wall, "unit": "rounds/s",
                   "h2d_bytes_per_step": int((X.nbytes + y.nbytes) / args.steps),
                   "d2h_bytes_per_step": 8, "seconds_total": e2e_wall, "seconds_upload": t_up, "seconds_quantise": t_q,
                   "api": "xgboost_ray_b200.engine.train (the xgb.train replacement an actor calls, host numpy in)",
                   "final_train_metric": {k: v[-1] for k, v in res["train"].items()}}
            del b2, d2

        # ================= CPU baseline (rank 0, N=1): oracle port on the host cores, bounded sample
        cpu = None
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            from oracle import oracle as O
            O.build()
            O.use_all_cores()
            ptrs, vals, mins, hm = dm.get_cuts()
            is_cat = [1 if t == "c" else 0 for t in args.feature_types] if args.feature_types else None
            cuts = O.Cuts.from_arrays(ptrs, vals, mins, hm, 256, is_cat=is_cat)
            bins = dm.get_bins()
            ob = O.Booster(dict(params, hist_qbits=0), cuts)
            ob.init_margin(X.shape[0])
            ob.boost(bins, y)  # warm-up round
            n_cpu, t0 = 0, time.time()
            while n_cpu < 3 or (time.time() - t0 < 10 and n_cpu < 20):
                ob.boost(bins, y)
                n_cpu += 1
            dt = time.time() - t0
            cpu = {"value": n_cpu / dt, "unit": "rounds/s", "cores": int(O.lib().or_num_threads()), "kind": "port",
                   "sample": "%d full-size rounds (%dx%d, depth %d) of the oracle port, float64 histograms, %.1fs" % (
                       n_cpu, args.rows, args.cols, args.depth, dt)}
    # ================= e2e through the PUBLIC API (the call a user of the reference makes):
    #   train(params, RayDMatrix(X, y), num_boost_round=K, ray_params=RayParams(num_actors=N))
    # issued by rank 0 alone with the WHOLE matrix in host memory; it shards the rows, hands the shards to N actor
    # processes (one per GPU), they upload, sketch, bin, train K rounds (per-round metric read back) and return the model.
    # One untimed warm-up call on a small matrix starts the actor processes, their CUDA contexts and the communicator,
    # the counterpart of the W warm-up steps of the device-resident arm (Ray keeps warm workers the same way); a second
    # untimed call has the timed shape (warm device-memory pools).
    e2e_public = None
    if not args.no_e2e and not args.no_public_e2e:
        del dm
        torch.cuda.empty_cache()
        cpu_group = dist.new_group(backend="gloo") if world > 1 else None
        if rank == 0:
            try:
                from xgboost_ray_b200 import RayDMatrix, RayParams, main as M, train as ray_train
                Xf, yf = (X, y) if world == 1 else synth_shard(args.rows, args.cols, 0, 1, workload=args.workload)
                pub_params = {k: v for k, v in params.items() if k != "profile"}
                nw = min(200_000, args.rows)
                ray_train(pub_params, RayDMatrix(Xf[:nw], yf[:nw], **dm_kw), num_boost_round=3, verbose_eval=False,
                          ray_params=RayParams(num_actors=world))
                # ... and one untimed call of the timed shape: the actors' device-memory pools then hold blocks of the right
                # sizes, like the pool of this process does for the engine-level arm (its device-resident arm ran first).
                # Its wall time is reported as first_call_seconds (cold pools: every large block is a cudaMalloc).
                t0 = time.perf_counter()
                dwarm = RayDMatrix(Xf, yf, **dm_kw)
                ray_train(pub_params, dwarm, num_boost_round=args.steps, evals=[(dwarm, "train")], verbose_eval=False,
                          ray_params=RayParams(num_actors=world))
                first_call = time.perf_counter() - t0
                del dwarm
                time.sleep(1.0)      # the actors tear the previous call's boosters down after replying; not part of the next call
                t0 = time.perf_counter()
                dmat = RayDMatrix(Xf, yf, **dm_kw)
                res, extra = {}, {}
                bpub = ray_train(pub_params, dmat, num_boost_round=args.steps, evals=[(dmat, "train")], evals_result=res,
                                 additional_results=extra, verbose_eval=False, ray_params=RayParams(num_actors=world))
                pub_wall = time.perf_counter() - t0
                e2e_public = {"value": args.steps / pub_wall, "unit": "rounds/s",
                              "h2d_bytes_per_step": int((Xf.nbytes + yf.nbytes) / args.steps), "d2h_bytes_per_step": 8,
                              "seconds_total": pub_wall, "first_call_seconds": first_call, "seconds_in_train_call": extra.get("total_time_s"),
                              "seconds_training_attempt": extra.get("training_time_s"), "timing": extra.get("timing"),
                              "api": "xgboost_ray_b200.train(params, RayDMatrix(X, y), num_boost_round=K, evals=[(dtrain, 'train')], "
                                     "ray_params=RayParams(num_actors=%d)) -- whole host matrix in, Booster out; warm actor pool (one untimed call of the same shape before)" % world,
                              "trees": bpub.num_trees(), "final_train_metric": {k: v[-1] for k, v in res["train"].items()}}
                M.shutdown_actors()
            except Exception as exc:  # noqa: BLE001 -- the bench line must still be printed
                e2e_public = {"error": repr(exc)[:500]}
        if cpu_group is not None:
            dist.barrier(group=cpu_group)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if e2e_public is not None and "value" in e2e_public:
        # the headline end-to-end number is the public API; the engine-level number (what one actor does) stays beside it
        e2e_engine, e2e = e2e, dict(e2e_public, engine_level=e2e)
    peak, peak_kind = measured_peak()
    # ncu --set full capture of one boosting round (C3): dram bytes per launch and the algorithmic bytes of the SAME launches
    traffic, traffic_alg = hist_traffic_per_launch() if args.workload == "C3" else (None, None)
    hist_bytes_per_launch = timers["hist_bytes"] / max(1, timers["hist_launches"])
    hist_ms_per_launch = hist_ms / max(1, timers["hist_launches"])
    achieved = hist_bytes_per_launch / (hist_ms_per_launch * 1e-3) / 1e9 if hist_ms_per_launch > 0 else 0.0
    line = {
        "metric": "boosting rounds/sec", "value": value, "unit": "rounds/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "int64 fixed-point histograms (int32 shared-memory cells), f64 gain", "data": "synthetic",
        "config": {"workload": workload_string(args), "sharding": "rows INTERLEAVED over %d rank(s)" % world,
                   "rows": args.rows, "cols": args.cols, "max_depth": args.depth, "max_bin": 256, "parallelism": "dp%d" % world,
                   "hist_qbits": params.get("hist_qbits", 18), "l2": "inputs_larger_than_l2",
                   "device_ms_per_step": dev_ms / args.steps, **({"phase_ms_per_step": {k: v / args.steps for k, v in timers.get("phase_ms", {}).items()}} if args.profile >= 2 else {}),
                   "quantise_seconds": t_quant, "exchange": exchange_kind, "cuda_graph": os.environ.get("B2_GRAPH", "1") != "0", "final_train_metric": final_metric},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "peak_source": peak_kind, "kernel": "b2::hist_build_kernel",
                     "algorithmic_bytes_per_launch": hist_bytes_per_launch, "ms_per_launch": hist_ms_per_launch,
                     "launches": timers["hist_launches"], "share_of_step": hist_ms / max(dev_ms, 1e-9),
                     "traffic": traffic, "traffic_capture_algorithmic_bytes": traffic_alg},
        "cpu_baseline": cpu, "e2e": e2e, "parity": parity, "gpu_launches": int(timers["kernel_launches"]),
        "clocks": sampler.summary(),
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
