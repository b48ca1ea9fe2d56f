#!/usr/bin/env python
"""bench.py — one "step" = one pass of the CTR hot path (gather → attention → MLP → BCE → backward →
scatter-add + SGD(rows) + Adam(dense)) over one batch of synthetic MovieLens-shaped input.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload NAME] [--dump-outputs DIR]

Prints ONE JSON line (see the task contract).  `value` = whole-job train samples/s with inputs
resident in HBM; `e2e` = same metric through the C-ABI entry point ctr_train_step_idx with pinned
HOST buffers (H2D of the indices/labels and D2H of the cost inside the timed region);
`roofline` = the dominant kernel's algorithmic bytes / its CUDA-event duration vs the measured HBM
peak; `cpu_baseline` = the CPU oracle port timed on this box's host cores on a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[3] — the north-star placement: DIN over a 100M-row item table (25.6 GB + 22.4 GB of item
    # features), row-sharded row % N over the N GPUs of the box and gathered / updated over NVLink peer memory;
    # N = 1 keeps the whole table on one GPU (HBM regime).  65536 samples per GPU and step (weak scaling).
    "din_100m": dict(model="din", U=138493, I=100_000_000, D=64, S=50, uP=52, cF=53, B=65536, zipf=False,
                     note="BASELINE.json configs[3]: DIN, 100M-row table (row-sharded row%N for N>1, NVLink peer gather / red.add), batch 65536 per GPU, S=50, uniform ids"),
    # BASELINE.json configs[1]: DIN on synthetic MovieLens-20M-shaped batches (138k users, 27k items, dim 64)
    "din_ml20m": dict(model="din", U=138493, I=27278, D=64, S=50, uP=52, cF=53, B=65536, zipf=True,
                      note="BASELINE.json configs[1]; item table 7 MB is L2-resident (reported, not an HBM reading); replicated for N>1"),
    # BASELINE.json configs[2]: YouTube DNN, 10M-item table dim 64, batch 16384
    "youtube_10m": dict(model="youtube", U=138493, I=10_000_000, D=64, S=50, uP=52, cF=53, B=16384, zipf=False,
                        note="BASELINE.json configs[2]"),
    "din_100m_shard": dict(model="din", U=138493, I=12_500_000, D=64, S=50, uP=52, cF=53, B=65536, zipf=False,
                           note="one GPU's 1/8 row shard of configs[3] held locally; uniform indices"),
}

# NVLink 5 per GPU and direction: nominal, and what a random 256-byte-row gather / red.add.v4 reaches between two
# processes' VMM mappings on this pool (tests/cuda/peer_probe.cu, profiles/r02/peer_probe.md)
NVLINK_NOMINAL_GBS = 900.0
NVLINK_PROBE_GBS = {"gather": 487.0, "red_add": 677.0}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi polled every 10 ms from before the warm-up; stop() keeps the samples whose timestamp falls inside
    [t0, t1] = the timed region plus a short untimed tail of the same load (the timed region alone is often shorter
    than nvidia-smi's start-up + polling latency)."""
    Q = "timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "10"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self, t0=None, t1=None):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush(); self.f.seek(0)
        rows = []
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(c[2]), float(c[3]), c[5:9]))
            except ValueError:
                continue
        os.unlink(self.f.name)
        inside = [r for r in rows if t0 is None or (t0 - 0.005 <= r[0] <= t1 + 0.005)]
        sm, mx, reasons = [], [], set()
        for ts, a, m, flags in inside:
            sm.append(a); mx.append(m)
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), flags):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm),
                       window="timed region + untimed tail of the same steps, %.2f s" % (t1 - t0) if t0 is not None else "whole run")
        return out


def synth_batch(w, rng, B):
    from tests.util import make_batch
    return make_batch(rng, w["U"], w["I"], B, w["S"], pad_frac=0.2, zipf=w["zipf"])


def algorithmic_bytes(w, hist, ir):
    """SURVEY.md §8(d): fp32 table, int32 ids, duplicates counted, caches ignored; only rows that
    exist (hist >= 0) are counted."""
    B = hist.shape[0]
    rows = int((hist >= 0).sum()) + int((ir >= 0).sum())
    row_bytes = w["D"] * 4
    gather = rows * row_bytes + B * (w["S"] + 2) * 4 + B * (w["uP"] + w["cF"]) * 4
    scatter = 2 * rows * row_bytes
    return gather, scatter, rows


def dump_rows(batch, nrows=32768, seed=0):
    """A fixed, seeded sample of `nrows` ITEM_EMB rows among those the batch updates (the whole table is up to 25.6 GB),
    in ascending order."""
    ur, ir, hist, y = batch
    rows = np.unique(np.concatenate([hist[hist >= 0], ir[ir >= 0]]))
    return np.sort(np.random.default_rng(seed).choice(rows, min(nrows, rows.size), replace=False))


def step_outputs(eng, w, rows):
    """What a caller of the timed step receives from its last call: the batch cost and the model the step leaves behind,
    i.e. the dense weights in full and the ITEM_EMB rows `rows` (dump_rows of the step's batch).  The rows are read back
    through the gather entry point, S rows per history slot; it gathers locally, so the table must not be row-sharded."""
    S, D, uP = w["S"], w["D"], w["uP"]
    slots = np.concatenate([rows, np.full(-rows.size % S, -1)]).astype(np.int32).reshape(-1, S)
    none = np.full(slots.shape[0], -1, np.int32)
    X = eng.gather_rows(none, none, slots)
    out = {"cost": np.array([eng.last_cost()], np.float32)}
    out.update(zip(("mlp0", "mlp1", "mlp2", "att0"), eng.get_weights()))
    if w["model"] != "din":
        del out["att0"]                  # the YouTube graph has no attention weights
    out["item_emb_rows"] = X[:, uP:uP + S * D].reshape(-1, D)[:rows.size]
    return out


def config_of(args, w, wname, world):
    """identical keys for both arms (the driver compares them)"""
    return {"workload": wname, "note": w["note"], "graph": w["model"], "users": w["U"], "items": w["I"], "D": w["D"], "S": w["S"],
            "uP": w["uP"], "cF": w["cF"], "per_gpu_batch": w["B"], "global_batch": w["B"] * world,
            "ids": "zipf(1.05)" if w["zipf"] else "uniform", "history_padding": "20% of samples have a -1 padded tail",
            "l2": "GPU arm: a 256 MiB buffer is written before every timed step (outside the event pair), per-step event pairs are summed; "
                  "CPU arm: host caches as they are"}


def cpu_arm(w, seconds, Bc, threads, seed=43, min_steps=2, state=None):
    """The reference's CPU path for this workload on the host cores: oracle/cpu_fast.c (float32, blocked thread-parallel
    SGEMMs like gonum's under gorgonia, Hogwild row update) stepping Bc-sample batches for ~`seconds`.  The item table is
    capped at 2M rows (512 MB) so the arm fits any host; ids are drawn in that range."""
    from oracle import oracle as orc
    from tests.util import make_batch
    I = min(w["I"], 2_000_000)
    if state is not None and state.get("Bc") == Bc:
        tr, batches = state["tr"], state["batches"]
    else:
        rng = np.random.default_rng(seed)
        model = orc.DIN_COS if w["model"] == "din" else orc.YOUTUBE
        ocfg = orc.make_cfg(model, w["uP"], w["S"], w["D"], w["cF"], 200, 80, 0.005, 0.005)
        uf = rng.random((w["U"], w["uP"]), dtype=np.float32); itf = rng.random((I, w["cF"]), dtype=np.float32)
        emb = (rng.standard_normal((I, w["D"]), dtype=np.float32) / np.sqrt(w["D"])).astype(np.float32)
        tr = orc.IdxTrainer(ocfg, orc.default_solver(0), orc.init_weights(ocfg, 0), uf, itf, emb)
        batches = [make_batch(rng, w["U"], I, Bc, w["S"], zipf=w["zipf"]) for _ in range(2)]
        tr.step_fast(*batches[0], table_lr=0.05, nthreads=threads)           # warm
        if state is not None:
            state.update(Bc=Bc, tr=tr, batches=batches)
    n = 0; t0 = time.perf_counter()
    while True:
        tr.step_fast(*batches[n % 2], table_lr=0.05, nthreads=threads); n += 1
        dt = time.perf_counter() - t0
        if dt >= seconds and n >= min_steps:
            break
    return Bc * n / dt, n, dt, I


def host_threads():
    """threads the process may really use: the affinity mask, cut by a cgroup CPU quota if one is set"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except (OSError, ValueError):
        pass
    return n


def pick_threads(step, cores):
    """The CPU arm at its best: one timed step at each of a few thread counts (all threads, half — one per physical core
    under SMT —, a quarter, 32, 16), keep the fastest.  `step(threads)` runs one warm step and returns its seconds."""
    cand = sorted({c for c in (cores, cores // 2, cores // 4, 32, 16) if 1 <= c <= cores}, reverse=True)
    tried = {}
    for c in cand:
        step(c)
        tried[c] = step(c)
    best = min(tried, key=tried.get)
    return best, {str(k): round(v, 4) for k, v in tried.items()}


def run_reference(args, w, wname):
    """--impl reference: the reference's own CPU implementation of the path.  The reference is Go (gorgonia + gonum) and
    cannot be built here (no Go toolchain, modules not vendored), so this times the C restatement of its CPU path
    (oracle/cpu_fast.c: blocked f32 SGEMMs, all host threads) on the SAME step shape as the engine arm: every step is one
    65536-sample batch of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as orc
    from tests.util import make_batch
    avail = host_threads()
    rng = np.random.default_rng(42)
    Bc = w["B"]
    I = min(w["I"], 2_000_000)
    model = orc.DIN_COS if w["model"] == "din" else orc.YOUTUBE
    ocfg = orc.make_cfg(model, w["uP"], w["S"], w["D"], w["cF"], 200, 80, 0.005, 0.005)
    uf = rng.random((w["U"], w["uP"]), dtype=np.float32); itf = rng.random((I, w["cF"]), dtype=np.float32)
    emb = (rng.standard_normal((I, w["D"]), dtype=np.float32) / np.sqrt(w["D"])).astype(np.float32)
    tr = orc.IdxTrainer(ocfg, orc.default_solver(0), orc.init_weights(ocfg, 0), uf, itf, emb)
    batches = [make_batch(rng, w["U"], I, Bc, w["S"], zipf=w["zipf"]) for _ in range(2)]
    steps = args.steps; warm = max(1, min(args.warmup, 2))

    def one(th):
        t = time.perf_counter(); tr.step_fast(*batches[0], table_lr=0.05, nthreads=th); return time.perf_counter() - t
    cores, tried = pick_threads(one, avail)
    for i in range(warm):
        tr.step_fast(*batches[i % 2], table_lr=0.05, nthreads=cores)
    t0 = time.perf_counter()
    for i in range(steps):
        tr.step_fast(*batches[i % 2], table_lr=0.05, nthreads=cores)
    dt = time.perf_counter() - t0
    v = Bc * steps / dt
    v1, n1, dt1, _ = cpu_arm(w, 3.0, 4096, 1)
    line = {"impl": "reference", "metric": "ctr_train_samples_per_sec", "value": v, "unit": "samples/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_of(args, w, wname, args.gpus),
            "cpu_baseline": {"value": v, "unit": "samples/s", "cores": cores, "kind": "port",
                             "sample": "%d steps x %d samples (the engine arm's step), OpenMP %d threads (fastest of %s on %d usable), blocked-SGEMM C restatement of go-ctr's CPU path "
                                       "(Go reference unbuildable here); item table capped at %d rows; 1 thread: %.0f samples/s" % (steps, Bc, cores, sorted(int(k) for k in tried), avail, I, v1),
                             "one_thread_value": v1, "seconds_per_step_by_threads": tried},
            "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def cpu_baseline(w, seconds=10.0):
    avail = host_threads()
    state = {}

    def one(th):
        v, n, dt, _ = cpu_arm(w, 0.0, w["B"], th, min_steps=1, state=state); return dt / n
    cores, tried = pick_threads(one, avail)
    v, n, dt, I = cpu_arm(w, seconds, w["B"], cores, state=state)
    v1, n1, dt1, _ = cpu_arm(w, 3.0, 4096, 1)
    return {"value": v, "unit": "samples/s", "cores": cores, "kind": "port", "one_thread_value": v1, "seconds_per_step_by_threads": tried, "usable_threads": avail,
            "sample": "%d steps x %d samples of the same workload shape in %.1f s (item table capped at %d rows), OpenMP %d threads (the fastest count tried); "
                      "blocked-SGEMM f32 C restatement of the reference's CPU path (oracle/cpu_fast.c), cross-checked against the "
                      "double-accumulating checker by tests/test_oracle_fast.py; 1 thread: %.0f samples/s on 4096-sample steps" % (n, w["B"], dt, I, cores, v1)}


def run_item2vec(args):
    """BASELINE configs[4] (item2vec SkipGram-HS, window 5): a step = one pass of the trainer over the synthetic item
    stream — `--i2v-tokens` tokens PER GPU (weak scaling; 8 x 125 M = the 1 B-token stream of configs[4]).  value = stream
    tokens of all ranks / device time of the training segments (max over ranks; includes the replica averaging for N > 1);
    e2e = stream tokens / wall time of the whole call (device-side dictionary / filter / path build, host Huffman merge,
    H2D of the tokens, training, D2H of the table).  The only throughput the reference publishes is for this loop: 555 k
    words/s on an Apple M1 Max (README.md:140)."""
    import go_ctr_b200 as g
    from oracle import oracle as orc
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    V, n, D = args.i2v_vocab, args.i2v_tokens, args.i2v_dim
    rng = np.random.default_rng(42 + rank)
    # Zipf(1.0)-like item popularity over V items (log-uniform ranks); ids are popularity ranks
    toks = (np.floor(np.exp(rng.random(n) * np.log(V))).astype(np.int64) - 1).clip(0, V - 1).astype(np.int32)
    hbm_peak, peak_src = load_peaks()
    if args.impl == "reference":
        if rank != 0:
            return
        m = min(n, args.i2v_cpu_tokens)
        cfg = orc.i2v_cfg(dim=D, window=5, iters=1, seed=1, rng_mode=0)
        t0 = time.perf_counter(); emb, trained = orc.i2v_train(cfg, toks[:m], V); dt = time.perf_counter() - t0
        v = m / dt
        print(json.dumps({"impl": "reference", "metric": "item2vec_words_per_sec", "value": v, "unit": "words/s", "n_gpus": args.gpus, "steps": 1, "warmup": 0,
                          "ms_per_step": 1e3 * dt, "higher_is_better": True, "scaling": "weak", "vs_baseline": v / 555000.0, "dtype": "f64", "data": "synthetic",
                          "config": {"workload": "item2vec", "vocab": V, "dim": D, "window": 5, "tokens_per_gpu": n},
                          "cpu_baseline": {"value": v, "unit": "words/s", "cores": 1, "kind": "port", "sample": "%d tokens of the same stream, single-threaded float64 port" % m},
                          "e2e": {"value": v, "unit": "words/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    import torch
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cfg = g.i2v_default_config(dim=D, window=5, iter=1, seed=1, device=local)
    best = None
    for i in range(2 + max(0, min(args.steps, 2) - 1)):
        nid = [None]
        if world > 1:
            if rank == 0:
                nid[0] = g.Engine(g.engine.default_config(g.MODEL_YOUTUBE, batch=1, pred_batch=1, device=local)).comm_unique_id()
            dist.broadcast_object_list(nid, src=0)
            dist.barrier()
        t0 = time.perf_counter()
        if world > 1:
            emb, st = g.i2v_train_dist(toks, V, rank, world, nid[0], sync_every=args.i2v_sync, cfg=cfg, want_table=(rank == 0))   # the averaged table goes to the host once
        else:
            emb, st = g.i2v_train_ids(toks, V, cfg=cfg)
        wall = time.perf_counter() - t0
        ms = st.ms_device
        if world > 1:
            t = torch.tensor([ms, wall], dtype=torch.float64, device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms, wall = float(t[0]), float(t[1])
        if i >= 1 and (best is None or ms < best[1]):
            best = (st, ms, wall)
    st, ms, wall = best
    value = n * world / (ms * 1e-3)
    ach = st.algorithmic_bytes / (st.ms_device * 1e-3) / 1e9
    line = {"metric": "item2vec_words_per_sec", "value": value, "unit": "words/s", "n_gpus": world, "steps": 1, "warmup": 1, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": value / 555000.0, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "item2vec", "note": "BASELINE.json configs[4]: %d tokens per GPU (%d in total)" % (n, n * world), "vocab": V, "dim": D, "window": 5,
                       "tokens_per_gpu": n, "optimizer": "hierarchical softmax", "ids": "zipf(1.0)", "l2": "vector tables (%.0f MB) exceed L2; no flush" % (2.0 * V * D * 4 / 1e6),
                       "placement": "single GPU" if world == 1 else "a full replica of both tables per GPU; counts all-reduced, replicas averaged every %d positions (NCCL)" % (args.i2v_sync or (4 << 20)),
                       "vs_baseline_note": "published 555k words/s is MovieLens-10M on an Apple M1 Max (README.md:140), different data and dim"},
            "e2e": {"value": n * world / wall, "unit": "words/s", "h2d_bytes_per_step": int(n * 4), "d2h_bytes_per_step": int(V * D * 4)},
            "gpu_launches": int(st.launches),
            "roofline": {"bound": "hbm", "kernel": "k_i2v_skipgram_hs", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "traffic": None,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": st.algorithmic_bytes, "ms_per_launch": st.ms_device,
                         "pairs": int(st.pairs), "node_visits": int(st.node_visits),
                         "note": "rank 0's kernel; Zipf item popularity: most node/context rows are served by L2 and the top Huffman nodes by shared memory "
                                 "(ncu: DRAM traffic << algorithmic bytes, profiles/r01/ncu_item2vec_v2.md) - this is SURVEY 8(d)'s algorithmic-bytes figure, "
                                 "not a DRAM reading; the kernel is L2-latency / issue bound"},
            "stats": {"doc_len": int(st.doc_len), "trained_positions": int(st.trained_positions)}}
    if rank == 0:
        if not args.no_cpu_baseline:
            m = min(n, args.i2v_cpu_tokens)
            ocfg = orc.i2v_cfg(dim=D, window=5, iters=1, seed=1, rng_mode=0)
            t0 = time.perf_counter(); orc.i2v_train(ocfg, toks[:m], V); dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": m / dt, "unit": "words/s", "cores": 1, "kind": "port", "sample": "%d tokens of the same stream, single-threaded float64 port" % m}
        print(json.dumps(line))
    if world > 1:
        dist.barrier(); dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="din_100m", choices=list(WORKLOADS) + ["item2vec"])
    ap.add_argument("--i2v-vocab", type=int, default=10_000_000)
    ap.add_argument("--i2v-tokens", type=int, default=50_000_000)
    ap.add_argument("--i2v-dim", type=int, default=64)
    ap.add_argument("--i2v-cpu-tokens", type=int, default=2_000_000)
    ap.add_argument("--i2v-sync", type=int, default=0, help="item2vec, N > 1: positions between replica averagings (0 = 4 Mi)")
    ap.add_argument("--batch", type=int, default=0, help="override per-GPU batch")
    ap.add_argument("--table-opt", default="sgd", choices=["sgd", "det", "frozen", "adam"])
    ap.add_argument("--gemm", default="auto", choices=["auto", "fp32", "tcgen05"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-side-legs", action="store_true", help="only the timed workload (+ roofline, e2e)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (cost, dense weights, a seeded "
                    "sample of the updated ITEM_EMB rows) as DIR/<name>.npy, to compare two builds on identical inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload == "item2vec"):
        ap.error("--dump-outputs covers the engine's CTR training step (--impl ours, not item2vec)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    wname = args.workload
    if wname == "item2vec":
        return run_item2vec(args)
    w = dict(WORKLOADS[wname])
    if args.batch:
        w["B"] = args.batch
    sharded = args.gpus > 1 and w["I"] * w["D"] * 4 > 32 * 2**20         # the engine row-shards ITEM_* tables above 32 MiB
    if args.dump_outputs and sharded:
        ap.error("--dump-outputs reads rows back through a local gather, which a row-sharded item table "
                 "(%s on %d GPUs) does not serve" % (wname, args.gpus))
    if args.impl == "reference":
        return run_reference(args, w, wname)

    import torch
    import go_ctr_b200 as g
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d: launch with torch.distributed.run --nproc-per-node N" % (args.gpus, world))
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this engine has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    hbm_peak, peak_src = load_peaks()
    dev = torch.device("cuda", local)

    def build_engine(w, B, placement=0, world_=None, rank_=None, table_opt=None, dropout=None, hot=None):
        wd = world if world_ is None else world_; rk = rank if rank_ is None else rank_
        model = g.MODEL_DIN_COS if w["model"] == "din" else g.MODEL_YOUTUBE
        topt = {"sgd": g.TABLE_SGD, "det": g.TABLE_SGD_DETERMINISTIC, "frozen": g.TABLE_FROZEN, "adam": g.TABLE_ADAM}[table_opt or args.table_opt]
        gm = {"auto": g.GEMM_AUTO, "fp32": g.GEMM_FP32, "tcgen05": g.GEMM_TCGEN05_3XTF32}[args.gemm]
        kw = {} if dropout is None else dict(dropout0=dropout, dropout1=dropout)
        cfg = g.engine.default_config(model, uP=w["uP"], S=w["S"], D=w["D"], cF=w["cF"], batch=B, pred_batch=B,
                                      table_opt=topt, table_lr=0.05, gemm=gm, device=local, rank=rk, world=wd, seed=1, **kw)
        cfg.reserved[1] = placement          # ITEM_* under world > 1: 0 = by size (> 32 MB shards), 1 = row-sharded, 2 = replicated
        # popular-row handling (replica accumulators; on sharded tables also a replica of rows [0, 32768) on every rank with an
        # all-reduce of their gradient sums): a uniform id stream has no popular rows — switched off there, default for Zipf ids
        zipf_ids = w["zipf"] if hot is None else hot
        cfg.reserved[0] = 0 if zipf_ids else -1
        eng = g.Engine(cfg)
        if wd > 1:
            ids = [None]
            if rank == 0:
                ids[0] = eng.comm_unique_id()
            dist.broadcast_object_list(ids, src=0)
            eng.comm_init(ids[0])
        # synthetic MovieLens-shaped tables generated on the device (SURVEY.md §8d): features U[0,1), embeddings N(0, 1/D)
        eng.table_fill(g.TABLE_USER_FEAT, w["U"], w["uP"], seed=3, dist=0, scale=1.0)
        eng.table_fill(g.TABLE_ITEM_FEAT, w["I"], w["cF"], seed=4, dist=0, scale=1.0)
        eng.table_fill(g.TABLE_ITEM_EMB, w["I"], w["D"], seed=5, dist=1, scale=float(1.0 / np.sqrt(w["D"])))
        return eng

    def make_batches(w, B, nb, seed, zipf=None):
        rng = np.random.default_rng(seed + rank)
        from tests.util import make_batch
        return [make_batch(rng, w["U"], w["I"], B, w["S"], pad_frac=0.2, zipf=w["zipf"] if zipf is None else zipf) for _ in range(nb)]

    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def timed_leg(eng, w, B, steps, warmup, profile=False, clocks=True, zipf=None, seed=100, capture=False):
        """K timed steps, inputs resident in HBM, L2 flushed before every step (outside the events).  capture: also
        return step_outputs() of the last timed step, read back after the launch count and before the untimed tail
        trains on; its rows are sampled before the clock sampler starts."""
        host = make_batches(w, B, 4, seed, zipf)
        devb = [tuple(torch.from_numpy(a).to(dev) for a in b) for b in host]
        st = torch.cuda.ExternalStream(eng.stream, device=dev)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]

        def one(i, e=None):
            ur, ir, hist, y = devb[i % len(devb)]
            with torch.cuda.stream(st):
                flush_buf.zero_()                                           # L2 flush (write > L2 capacity)
                if e: e[0].record(st)
                eng.train_step_idx_dev(ur.data_ptr(), ir.data_ptr(), hist.data_ptr(), y.data_ptr(), B)
                if e: e[1].record(st)
        rows = dump_rows(host[(warmup + steps - 1) % len(host)]) if capture else None
        sampler = ClockSampler(local) if (clocks and not profile) else None      # polls from before the warm-up
        for i in range(warmup):
            one(i)
        eng.sync(); torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        l1 = eng.launch_count()
        if profile:
            eng.profile_reset(); eng.profile(True)
        t0 = time.perf_counter(); c0 = time.time()
        for i in range(steps):
            one(warmup + i, ev[i])
        eng.sync(); torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        l2 = eng.launch_count()
        outputs = step_outputs(eng, w, rows) if capture else None
        clk = None
        if sampler:      # untimed tail: the same steps keep the load up until nvidia-smi has had >= 0.3 s to sample it
            k = 0
            # multi-rank steps are collective: every rank must run the same number of tail steps
            ntail = max(8, int(0.35 / max(wall / steps, 1e-4)))
            while (k < ntail) if world > 1 else (time.time() - c0 < 0.3 and k < 400):
                one(k); k += 1
                if k % 8 == 0:
                    eng.sync()
            eng.sync(); torch.cuda.synchronize()
            clk = sampler.stop(c0, time.time())
        if profile:
            eng.profile(False)
        ms = sum(a.elapsed_time(b) for a, b in ev)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        cost = eng.last_cost()
        return dict(ms=ms, wall=wall, clocks=clk, launches=(l2 - l1), host=host, cost=cost, prof=eng.profile_dump() if profile else None,
                    outputs=outputs)

    def rowstats(w, leg):
        """rows a step touches on this rank, and how many of them live on a peer (row % world != rank)"""
        rows = remote = 0
        for ur, ir, hist, y in leg["host"]:
            v = hist >= 0
            rows += int(v.sum()) + int((ir >= 0).sum())
            if world > 1:
                remote += int((v & (hist % world != rank)).sum()) + int(((ir >= 0) & (ir % world != rank)).sum())
        n = len(leg["host"])
        return rows / n, remote / n

    def roofline_of(w, leg, steps, B, traffic_key=None):
        prof = leg["prof"]
        rows, remote = rowstats(w, leg)
        row_bytes = w["D"] * 4
        gbytes = rows * row_bytes + B * (w["S"] + 2) * 4 + B * (w["uP"] + w["cF"]) * 4      # SURVEY §8(d): gather
        sbytes = 2 * rows * row_bytes                                                       # scatter-add = row read-modify-write
        kern = {}
        for name, (ms, n) in prof.items():
            kern[name] = {"ms_per_launch": ms / max(n, 1), "launches_per_step": n / max(steps, 1)}
        fwd = next((k for k in kern if k.startswith("attn_fwd")), None)
        bwd = next((k for k in kern if k.startswith("attn_bwd")), None)
        if fwd:
            kern[fwd].update(algorithmic_bytes=gbytes, gbs=gbytes / (kern[fwd]["ms_per_launch"] * 1e-3) / 1e9)
        if bwd:
            kern[bwd].update(algorithmic_bytes=sbytes, gbs=sbytes / (kern[bwd]["ms_per_launch"] * 1e-3) / 1e9)
        step_ms = sum(v["ms_per_launch"] * v["launches_per_step"] for v in kern.values())
        for v in kern.values():
            v["share_of_step"] = v["ms_per_launch"] * v["launches_per_step"] / step_ms if step_ms else None
        cand = [k for k in (fwd, bwd) if k]
        if not cand:
            return None, kern, None
        dom = max(cand, key=lambda k: kern[k]["ms_per_launch"])
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp) and traffic_key:
            traffic = json.load(open(tp)).get(traffic_key, {}).get(dom)
        pair_ms = sum(kern[k]["ms_per_launch"] for k in cand)
        rl = {"bound": "hbm", "kernel": dom, "achieved": kern[dom]["gbs"], "peak": hbm_peak, "unit": "GB/s",
              "frac": kern[dom]["gbs"] / hbm_peak, "traffic": traffic, "peak_source": peak_src,
              "algorithmic_bytes_per_launch": kern[dom]["algorithmic_bytes"], "ms_per_launch": kern[dom]["ms_per_launch"],
              "fused_pair": {"kernels": cand, "algorithmic_bytes": gbytes + sbytes, "ms": pair_ms,
                             "achieved": (gbytes + sbytes) / (pair_ms * 1e-3) / 1e9,
                             "frac": (gbytes + sbytes) / (pair_ms * 1e-3) / 1e9 / hbm_peak},
              "rows_per_launch": rows,
              "how": "second pass of the same %d steps with every launch bracketed by CUDA events on the engine stream" % steps}
        nv = None
        if world > 1 and fwd and bwd:
            # the sharded step is NVLink bound: every remote row crosses once inbound (forward gather) and once outbound
            # (backward red.add); the HBM fraction above is reported for continuity, the NVLink block is the binding roofline
            rb = remote * row_bytes
            nv = {"remote_rows_per_step": remote, "remote_fraction": remote / max(rows, 1), "bytes_each_way_per_step": rb,
                  "gather_in_GBs": rb / (kern[fwd]["ms_per_launch"] * 1e-3) / 1e9, "red_add_out_GBs": rb / (kern[bwd]["ms_per_launch"] * 1e-3) / 1e9,
                  "nominal_GBs_per_direction": NVLINK_NOMINAL_GBS, "probe_GBs": NVLINK_PROBE_GBS,
                  "frac_of_nominal": {"gather": rb / (kern[fwd]["ms_per_launch"] * 1e-3) / 1e9 / NVLINK_NOMINAL_GBS,
                                      "red_add": rb / (kern[bwd]["ms_per_launch"] * 1e-3) / 1e9 / NVLINK_NOMINAL_GBS},
                  "step_floor_ms_at_probe_rate": rb / 1e6 / NVLINK_PROBE_GBS["gather"] + rb / 1e6 / NVLINK_PROBE_GBS["red_add"],
                  "note": "the two directions are used one after the other (gather, then red.add, separated by the MLP and a barrier): "
                          "per-GPU ceiling = remote bytes / probe rate, each way"}
            rl["note"] = "row-sharded step: the attention kernels wait on NVLink, not HBM — see `nvlink`"
        return rl, kern, nv

    def e2e_legs(eng, w, B, steps):
        """The same metric through the reference-facing host entry points, caller buffers in PAGEABLE host memory
        (plain numpy, as a cgo caller's Go slices would be): (a) ctr_train_keys — recommend.Train over sample keys
        {UserId, ItemId, Timestamp, Label}: 28 B/sample H2D, id maps + ubcache window + training on the device;
        (b) ctr_train_idx — precomputed row ids + history rows: (S+3)*4 B/sample H2D.  Both stage through the internal
        pinned ring; the batch costs are read back D2H before the call returns."""
        out = {}
        rng = np.random.default_rng(200 + rank)
        U, I, S = w["U"], w["I"], w["S"]
        n = B * steps
        # (b) ids
        from tests.util import make_batch
        ur, ir, hist, y = make_batch(rng, U, I, n, S, pad_frac=0.2, zipf=w["zipf"])
        eng.train_idx(ur, ir, hist, y)                                              # warm pass: the ring, the per-call buffers
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        costs = eng.train_idx(ur, ir, hist, y)
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); dt = float(t.item())
        out["idx"] = dict(value=B * world * steps / dt, unit="samples/s", h2d_bytes_per_step=int(B * (S + 3) * 4), d2h_bytes_per_step=8,
                          ms_per_step=1e3 * dt / steps, last_cost=float(costs[-1]), entry="ctr_train_idx", host_memory="pageable (numpy)")
        del hist
        # (a) keys: sparse external ids, per-user behaviour sequences in the device ubcache
        uid = (np.arange(U, dtype=np.int64) * 7 + 3); iid = (np.arange(I, dtype=np.int64) * 5 + 11)
        eng.idmap_build(g.IDMAP_USER, uid); eng.idmap_build(g.IDMAP_ITEM, iid)
        L = 2 * S                                                                   # events per user
        off = (np.arange(U + 1, dtype=np.int64) * L)
        ts = np.tile(np.arange(L, 0, -1, dtype=np.int64) * 1000, U)
        items = (rng.zipf(1.05, U * L) - 1) % I if w["zipf"] else rng.integers(0, I, U * L)
        eng.ubcache_upload(off, ts, items.astype(np.int32))
        su = rng.integers(0, U, n); si = ((rng.zipf(1.05, n) - 1) % I) if w["zipf"] else rng.integers(0, I, n)
        k_user = uid[su]; k_item = iid[si]; k_ts = rng.integers(1000, (L + 1) * 1000, n).astype(np.int64)
        eng.train_keys(k_user, k_item, k_ts, y, epochs=1)                           # warm pass: resident sample arrays of this size
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        eng.train_keys(k_user, k_item, k_ts, y, epochs=0)                           # GetSample only (resolve + compact on the device)
        dt_resolve = time.perf_counter() - t0
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        ep, cost, used = eng.train_keys(k_user, k_item, k_ts, y, epochs=1)
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); dt = float(t.item())
        out["keys"] = dict(value=used * world / dt, unit="samples/s", h2d_bytes_per_step=int(B * 28), d2h_bytes_per_step=8,
                           ms_per_step=1e3 * dt / steps, last_cost=float(cost), entry="ctr_train_keys", host_memory="pageable (numpy)",
                           rows_used=int(used), resolve_ms=1e3 * dt_resolve)
        return out

    def parity_block():
        """N ranks x batch Bp on a row-sharded table == one GPU x batch N*Bp on the whole table (same samples, same
        init, dropout off): batch costs, dense weights after k steps, and the updated table rows.  Rank 0 holds the
        single-GPU reference engine.  Tolerances: both sides scatter with fp32 red.add in arbitrary order."""
        wp = dict(w); wp["I"] = 1_000_003; wp["U"] = 5000
        Bp, k = 2048, 3
        eng_s = build_engine(wp, Bp, placement=1, dropout=0.0)
        rngp = np.random.default_rng(4242)
        from tests.util import make_batch
        glob = [make_batch(rngp, wp["U"], wp["I"], Bp * world, wp["S"], pad_frac=0.2, zipf=True) for _ in range(k)]
        sl = slice(rank * Bp, (rank + 1) * Bp)
        costs = [eng_s.train_step_idx(*(a[sl] for a in b)).cost for b in glob]
        ws = eng_s.get_weights()
        probe_rows = np.unique(np.concatenate([glob[0][2][glob[0][2] >= 0][:4000], glob[0][1][:1000]]))
        # every rank scores the same probe batch through the sharded tables: reads every owner's updated rows
        pr = make_batch(np.random.default_rng(7), wp["U"], wp["I"], Bp, wp["S"], zipf=True)
        eng_s.sync(); dist.barrier()
        p_shard = eng_s.predict_idx(pr[0], pr[1], pr[2])
        dist.barrier()
        res = None
        if rank == 0:
            eng_1 = build_engine(wp, Bp * world, world_=1, rank_=0, dropout=0.0)
            want = [eng_1.train_step_idx(*b).cost for b in glob]
            w1 = eng_1.get_weights()
            cfgp = g.engine.default_config(g.MODEL_DIN_COS, uP=wp["uP"], S=wp["S"], D=wp["D"], cF=wp["cF"], batch=Bp, pred_batch=Bp, device=local, seed=1)
            # score the probe batch on the single-GPU engine's tables (pred_batch = N*Bp >= Bp)
            p_one = eng_1.predict_idx(pr[0], pr[1], pr[2])
            dcost = float(np.max(np.abs(np.array(costs) - np.array(want)) / np.maximum(1.0, np.abs(want))))
            dw = max(float(np.mean(np.abs(a - b) > 2e-4 + 2e-3 * np.abs(b))) for a, b in zip(ws, w1))
            dp = float(np.max(np.abs(p_shard - p_one) / np.maximum(1e-6, np.abs(p_one))))
            ok = bool(dcost <= 2e-4 and dw <= 0.005 and dp <= 2e-3)
            res = {"ok": ok, "what": "%d ranks x batch %d on a row-sharded 1M-row table vs 1 GPU x batch %d, %d SGD steps (Zipf ids, dropout off)" % (world, Bp, Bp * world, k),
                   "max_rel_cost_diff": dcost, "frac_dense_weights_outside_tol": dw, "max_rel_score_diff_after_training": dp,
                   "costs": [float(c) for c in costs], "tolerances": {"cost": 2e-4, "weights": "rtol 2e-3 + atol 2e-4 on >= 99.5 %", "scores": 2e-3}}
            del eng_1
        del eng_s
        torch.cuda.empty_cache()
        return res

    # ------------------------------------------------------------------------------------------------ main line
    B = w["B"]
    eng = build_engine(w, B)
    leg = timed_leg(eng, w, B, args.steps, args.warmup, capture=bool(args.dump_outputs) and rank == 0)
    if leg["outputs"] is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in leg["outputs"].items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    psteps = max(5, min(args.steps, 20))
    prof_leg = timed_leg(eng, w, B, psteps, 1, profile=True)
    rl, kern, nv = roofline_of(w, prof_leg, psteps, B, traffic_key=wname if world == 1 else None)
    value = B * world * args.steps / (leg["ms"] * 1e-3)
    cfg = config_of(args, w, wname, world)
    engine_cfg = dict(table_opt=args.table_opt, gemm=args.gemm, popular_rows="off (uniform ids)" if not w["zipf"] else "rows [0, 32768)",
               placement=("single GPU: the whole table in one HBM (%.1f GB ITEM_EMB + %.1f GB ITEM_FEAT)" % (w["I"] * w["D"] * 4 / 1e9, w["I"] * 56 * 4 / 1e9) if world == 1 else
                          "1 process per GPU; ITEM_EMB / ITEM_FEAT rows sharded row%world; gather and red.add go to the owner's HBM over NVLink peer mappings "
                          "(VMM allocations shared as fds), 2 device-side barriers + 1 NCCL all-reduce (dense gradients) per step" if sharded else
                          "1 process per GPU; ITEM_EMB (%.0f MB) replicated, row + dense gradients all-reduced (NCCL)" % (w["I"] * w["D"] * 4 / 1e6)))
    line = {"metric": "ctr_train_samples_per_sec", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": leg["ms"] / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 (the six GEMMs as error-compensated 3xTF32 on tcgen05, fp32 everything else)", "data": "synthetic",
            "config": cfg, "engine": engine_cfg, "clocks": leg["clocks"], "gpu_launches": int(leg["launches"]), "last_cost": leg["cost"],
            "wall_s_timed_region": leg["wall"], "roofline": rl, "kernels": kern}
    if nv:
        line["nvlink"] = nv
    if rl is not None and w["I"] * w["D"] * 4 / (world if sharded else 1) < 126e6:
        rl["note"] = "table is L2-resident in the timed workload (DRAM traffic << algorithmic bytes): not an HBM reading"
    e2e = e2e_legs(eng, w, B, max(4, min(args.steps, 64)))
    line["e2e"] = {k: e2e["keys"][k] for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step")}
    line["e2e_detail"] = e2e
    if not args.no_side_legs:
        side = {}
        del eng
        torch.cuda.empty_cache()
        # Zipf(1.05) item popularity on the same table (popular-row handling on): hot rows are gathered / updated by every sample
        eng_z = build_engine(w, B, hot=True)
        zl = timed_leg(eng_z, w, B, max(5, args.steps // 4), 3, clocks=False, zipf=True, seed=300)
        side["zipf_ids"] = {"what": "same table, item / history ids drawn Zipf(1.05); rows [0, 32768) handled as popular rows", "value": B * world * max(5, args.steps // 4) / (zl["ms"] * 1e-3),
                            "unit": "samples/s", "ms_per_step": zl["ms"] / max(5, args.steps // 4)}
        del eng_z
        torch.cuda.empty_cache()
        if world > 1 and sharded:
            # BASELINE configs[3] read literally: GLOBAL batch 65536 over the N GPUs (strong-scaling point of the same table)
            Bg = max(256, w["B"] // world)
            eng_g = build_engine(w, Bg)
            ks = max(10, args.steps // 2)
            lg = timed_leg(eng_g, w, Bg, ks, 3, clocks=False, seed=400)
            side["global_batch_%d" % (Bg * world)] = {"what": "configs[3] with the batch read as global: %d samples per GPU and step" % Bg,
                                                     "value": Bg * world * ks / (lg["ms"] * 1e-3), "unit": "samples/s", "ms_per_step": lg["ms"] / ks}
            del eng_g
            torch.cuda.empty_cache()
            side_par = parity_block()
            if rank == 0:
                line["parity"] = side_par
        if world == 1 and wname != "din_ml20m":
            # BASELINE configs[1] (the 7 MB, L2-resident table) on one GPU — kept as a side reading
            w2 = dict(WORKLOADS["din_ml20m"])
            eng2 = build_engine(w2, w2["B"])
            k2 = max(5, args.steps // 2)
            l2_ = timed_leg(eng2, w2, w2["B"], k2, 3, clocks=False, seed=500)
            side["configs1_din_ml20m"] = {"what": w2["note"], "value": w2["B"] * k2 / (l2_["ms"] * 1e-3), "unit": "samples/s", "ms_per_step": l2_["ms"] / k2}
            del eng2
        line["side_legs"] = side
    if rank == 0:
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(w)
        if world > 1 and "parity" in line and line["parity"] and not line["parity"]["ok"]:
            print(json.dumps(line))
            raise SystemExit("parity check failed: %s" % json.dumps(line["parity"]))
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
