"""CPU tests of bench.py's contract: the reference arm end to end on a scaled-down graph (it is CPU-only by design), the
byte formulas of SURVEY 8(d) behind `roofline` / `batched.roofline`, and that both arms print the same `config` object."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_reference_arm_prints_the_contract_line(tmp_path):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--scale", "0.004", "--steps", "2",
                        "--warmup", "1", "--gpus", "1", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1                                        # ONE JSON line
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1
    assert d["metric"].startswith("RWR GTEPS") and d["unit"] == "GTEPS" and d["higher_is_better"] is True
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic" and d["dtype"] == "f64"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["gpu_launches"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["unit"] == "GTEPS" and 1 <= cb["cores"] <= 10 and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "GTEPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # the same `config` object as the GPU arm prints for this graph (workload keys only, no model keys)
    cfg = d["config"]
    assert cfg == bench.c2_config(cfg["n_nodes"], cfg["nnz"], 0.004, 1) and cfg["workload"].startswith("C2:")
    assert set(cfg) == {"workload", "n_nodes", "nnz", "scale", "iterations", "top_k", "parallelism", "l2"}
    # the reference's own Model.cs beside the port, where its compiled sources are here
    ri = cb["reference_itself"]
    if ri is not None:
        assert ri["kind"] == "reference" and "error" not in ri and ri["gteps"] > 0
    # --dump-outputs: rank[seed] after Model.run(cpu_iters) of every seed of the last timed step (step 3 of warm-up 1 + 2)
    import oracle as O
    seeds, got = np.load(tmp_path / "seeds.npy"), np.load(tmp_path / "rank_at_seed.npy")
    assert seeds.dtype == got.dtype == np.float64 and len(seeds) == len(got) == cb["cores"]
    links = O.synth_generate(bench.scaled_spec(0.004))
    og = O.OracleGraph(links["node_id"], links["node_type"], links["src"], links["dst"], links["etype"], links["w"])
    assert og.build() == 0
    raw_deg = np.bincount(links["src"], minlength=og.n)
    assert seeds.tolist() == bench.pick_seeds(raw_deg, bench.scaled_spec(0.004)["n_users"], 3 * len(seeds))[-len(seeds):].tolist()
    want = [og.run(int(s), O.widen_float(bench.C_FLOAT), n_iter=2)[0][int(s)] for s in seeds]
    assert np.array_equal(got, want)


def test_other_ranks_of_the_reference_arm_exit_without_work():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--scale", "0.004", "--gpus", "2"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_zero_steps_are_refused():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert p.returncode == 2 and "--steps must be at least 1" in p.stderr


def test_dump_outputs_samples_a_long_rank_vector(tmp_path):
    """Above DUMP_SAMPLE nodes the rank vector is dumped as the same seeded sample of nodes, with their indices, every time."""
    n = bench.DUMP_SAMPLE + 12_345

    class Model:
        def scores(self, slot):
            return np.arange(n) * 0.5

        def topk(self, k):
            return np.arange(k)[None, ::-1] * 3, np.arange(k)[None, ::-1] * 1.5, np.array([k], np.int32)

    outs = []
    for k in range(2):
        bench.dump_outputs(str(tmp_path / f"run{k}"), Model(), 7)
        outs.append({f[:-4]: np.load(tmp_path / f"run{k}" / f) for f in os.listdir(tmp_path / f"run{k}")})
        assert sum(os.path.getsize(tmp_path / f"run{k}" / f) for f in os.listdir(tmp_path / f"run{k}")) <= 64 << 20
    a, b = outs
    assert all(x.dtype == np.float64 and np.array_equal(x, b[name]) for name, x in a.items())
    nodes = a["scores_nodes"]
    assert len(nodes) == bench.DUMP_SAMPLE and np.all(np.diff(nodes) > 0) and nodes[0] >= 0 and nodes[-1] < n
    assert np.array_equal(a["scores"], nodes * 0.5) and a["seed"].tolist() == [7]
    assert a["top10_nodes"].tolist() == list(range(27, -1, -3)) and a["top10_scores"].tolist() == [i * 1.5 for i in range(9, -1, -1)]


@pytest.mark.gpu
def test_dump_outputs_repeat_and_match_the_json_line(tmp_path):
    """--dump-outputs on a scaled-down C2 graph, twice: the same arrays bit for bit (seeded inputs), float64, under 64 MB,
    --steps timed steps in the JSON line, and the dump is the last timed step's seed, rank vector and top-10."""
    runs = []
    for k in range(2):
        out = tmp_path / f"run{k}"
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--scale", "0.004", "--steps", "3", "--warmup", "3",
                            "--no-cpu", "--no-c5", "--batch-seeds", "16", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=900)
        assert p.returncode == 0, p.stderr[-2000:]
        d = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
        assert d["steps"] == 3
        files = sorted(os.listdir(out))
        assert files == ["scores.npy", "scores_nodes.npy", "seed.npy", "top10_nodes.npy", "top10_scores.npy"]
        assert sum(os.path.getsize(out / f) for f in files) <= 64 << 20
        runs.append({f[:-4]: np.load(out / f) for f in files})
    a, b = runs
    for name, x in a.items():
        assert x.dtype == np.float64 and np.array_equal(x.view(np.uint64), b[name].view(np.uint64)), name
    # the seed of the last timed step (warm-up 3 + 3 steps: the sixth bench seed), its whole rank vector at this size and its
    # top-10 against the oracle on the same graph
    import oracle as O
    import recommendersystems_b200 as rs
    spec = bench.scaled_spec(0.004)
    g = rs.Graph.synthetic(spec)
    g.buildGraph()
    seed = int(bench.pick_seeds(g.degrees(raw=True), spec["n_users"], 12)[5])
    links = g.export_links()
    g.close()
    assert a["seed"].tolist() == [seed] and np.array_equal(a["scores_nodes"], np.arange(d["config"]["n_nodes"]))
    og = O.OracleGraph(links["node_id"], links["node_type"], links["src"], links["dst"], links["etype"], links["w"])
    assert og.build() == 0
    want, _ = og.run(seed, O.widen_float(bench.C_FLOAT), n_iter=bench.N_ITER)
    nz = want != 0
    assert np.all(a["scores"][~nz] == 0) and (np.abs(a["scores"][nz] - want[nz]) / want[nz]).max() <= 1e-12
    ids, sc = og.recommend(seed, bench.C_FLOAT, bench.N_ITER, top_n=bench.TOP_K)
    assert a["top10_nodes"].tolist() == ids.tolist() and (np.abs(a["top10_scores"] - sc) / sc).max() <= 1e-12
    og.close()


def test_byte_formulas_of_survey_8d():
    n, nnz = 11_000_000, 205_156_156
    formula, actual = bench.algorithmic_bytes(n, nnz, 8, layout_index=True)
    assert formula == nnz * 12 + 4 * (n + 1) + 16 * n == 2_681_873_876        # the figure VERDICT r1 recomputed
    assert actual == nnz * 4 + 4 * (n + 1) + 16 * n                             # what the index-only layout moves
    assert bench.algorithmic_bytes(n, nnz, 4, layout_index=False) == (nnz * 8 + 4 * (n + 1) + 8 * n,) * 2
    # batched: E (4 + vb) + 4 (N + 1) + 2 N B vb per pass of B seeds; 128 seeds = 16 passes x 20 iterations
    peak = bench.measured_peak_gbs()[0]
    per_pass = nnz * 12 + 4 * (n + 1) + 2 * n * 8 * 8
    assert abs(bench.batched_frac(n, nnz, 8, 8, 128, 1.0) - per_pass * 16 * 20 / 1e9 / peak) < 1e-12
    assert bench.batched_frac(n, nnz, 8, 8, 0, 1.0) == 0.0
    spec = bench.scaled_spec(0.5)
    assert spec["n_users"] == 500_000 and spec["n_like"] == 38_000_000 and bench.scaled_spec(1.0) == bench.C2_SPEC
