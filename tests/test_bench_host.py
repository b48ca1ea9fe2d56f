"""Host-side pieces of bench.py (no GPU): the usable-thread probe, the thread-count picker, a tiny `--impl reference`-style
step through oracle/cpu_fast.c, and what --dump-outputs reads back from an engine."""
import os
import subprocess
import sys

import numpy as np
import pytest

import bench


def test_host_threads_is_within_the_affinity_mask():
    n = bench.host_threads()
    assert 1 <= n <= len(os.sched_getaffinity(0))


def test_pick_threads_keeps_the_fastest_candidate_and_reports_every_timing():
    calls = []

    def step(th):                       # pretend 8 threads are the sweet spot (oversubscription beyond)
        calls.append(th)
        return {64: 0.9, 32: 0.5, 16: 0.3, 8: 0.3}.get(th, 1.0) + (0.0 if th != 16 else -0.05)
    best, tried = bench.pick_threads(step, 64)
    assert best == 16
    assert set(tried) == {"64", "32", "16"} and all(v > 0 for v in tried.values())
    assert calls.count(64) == 2 and calls.count(16) == 2          # one warm + one timed step per candidate


def test_pick_threads_on_a_small_box_only_tries_counts_it_has():
    best, tried = bench.pick_threads(lambda th: 1.0 / th, 6)
    assert best == 6 and set(tried) == {"6", "3", "1"}


def test_cpu_arm_runs_the_fast_oracle_on_the_workload_shape():
    w = dict(bench.WORKLOADS["din_100m"]); w["I"] = 20_000
    state = {}
    v, n, dt, rows = bench.cpu_arm(w, 0.0, 512, 2, min_steps=1, state=state)
    assert n == 1 and v > 0 and rows == 20_000
    v2, n2, _, _ = bench.cpu_arm(w, 0.0, 512, 1, min_steps=2, state=state)      # the trainer is reused across thread counts
    assert n2 == 2 and state["Bc"] == 512


class _TableEngine:
    """numpy stand-in for the read-back entry points step_outputs() calls (gather = the C ABI's row layout)"""

    def __init__(self, w, emb):
        self.w, self.emb = w, emb

    def gather_rows(self, ur, ir, hist):
        w = self.w
        assert (ur == -1).all() and (ir == -1).all() and hist.shape[1] == w["S"]
        ub = np.zeros(hist.shape + (w["D"],), np.float32)
        ub[hist >= 0] = self.emb[hist[hist >= 0]]
        z = lambda n: np.zeros((len(ur), n), np.float32)          # noqa: E731
        return np.concatenate([z(w["uP"]), ub.reshape(len(ur), -1), z(w["D"]), z(w["cF"])], 1)

    def get_weights(self):
        return np.ones((7, 200), np.float32), np.ones((200, 80), np.float32), np.ones((80, 1), np.float32), np.ones(self.w["S"], np.float32)

    def last_cost(self):
        return 0.5


@pytest.mark.parametrize("model", ["din", "youtube"])
def test_step_outputs_are_a_fixed_sample_of_the_rows_the_batch_updated(model):
    w = dict(bench.WORKLOADS["din_100m"], model=model, I=5000, S=7, D=4, uP=3, cF=2)
    rng = np.random.default_rng(0)
    emb = rng.standard_normal((w["I"], w["D"])).astype(np.float32)
    batch = bench.synth_batch(w, rng, 300)
    eng = _TableEngine(w, emb)
    out = bench.step_outputs(eng, w, bench.dump_rows(batch, nrows=500))
    assert set(out) == {"cost", "mlp0", "mlp1", "mlp2", "item_emb_rows"} | ({"att0"} if model == "din" else set())
    assert all(a.dtype == np.float32 for a in out.values()) and out["cost"].tolist() == [0.5]
    row_of = {r.tobytes(): i for i, r in enumerate(emb)}
    got = [row_of[r.tobytes()] for r in out["item_emb_rows"]]
    touched = set(batch[2][batch[2] >= 0].tolist()) | set(batch[1].tolist())
    assert len(got) == 500 and got == sorted(set(got)) and set(got) <= touched
    assert bench.step_outputs(eng, w, bench.dump_rows(batch, nrows=500))["item_emb_rows"].tobytes() == out["item_emb_rows"].tobytes()
    every = bench.step_outputs(eng, w, bench.dump_rows(batch, nrows=10 ** 6))["item_emb_rows"]
    assert sorted(row_of[r.tobytes()] for r in every) == sorted(touched)


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"], ["--workload", "item2vec", "--dump-outputs", "x"],
                                  ["--gpus", "2", "--dump-outputs", "x"], ["--gpus", "8", "--workload", "youtube_10m", "--dump-outputs", "x"]])
def test_bench_refuses_arguments_it_cannot_honour(argv):
    """Refused before any work, with argparse's exit code.  --dump-outputs covers only the engine's CTR step, and not a
    row-sharded item table (more than one GPU, table above 32 MiB), whose rows a local gather cannot read back."""
    r = subprocess.run([sys.executable, bench.__file__] + argv, capture_output=True, text=True, timeout=60)
    assert r.returncode == 2 and "error" in r.stderr
