"""bench.py prints ONE JSON line with the keys the driver reads, for both arms."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"}


def run(args, timeout):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, capture_output=True,
                         text=True, timeout=timeout)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def test_reference_arm_line():
    from oracle import refshim
    d = run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-seconds", "2"], timeout=200)
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["metric"] == "othello_positions_per_sec_legalgen_step" and d["unit"] == "positions/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None
    cb = d["cpu_baseline"]
    assert cb["kind"] == ("reference" if refshim.available() else "port") and cb["cores"] >= 1 and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "positions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"] == "config3_random_playout"


@pytest.mark.gpu
def test_b200_arm_line():
    d = run(["--steps", "4", "--warmup", "3", "--games", "131072", "--cpu-seconds", "2"], timeout=600)
    assert BASE_KEYS | {"roofline", "cpu_baseline", "clocks", "games_per_s"} <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 4 and d["warmup"] == 3 and d["gpu_launches"] == 4
    assert d["scaling"] == "weak" and d["dtype"] == "u64" and d["data"] == "synthetic"
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and 0 < r["frac"] < 1.2
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["hbm"]["peak"] > 1000
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 131072 * 16 and e["d2h_bytes_per_step"] == 131072 * 2 + 32
    assert e["results_checked"] is True
    assert e["standard_opening"]["value"] > 0 and e["standard_opening"]["h2d_bytes_per_step"] == 0
    assert e["full_results"]["d2h_bytes_per_step"] == 131072 * 20 + 32
    # (chunked launches on rotating streams hide the tail of one launch behind the next: e2e may edge past `value`)
    assert e["value"] <= d["value"] * 1.15
    c4, c5 = d["extra"]["config4"], d["extra"]["config5"]
    assert c4["positions_per_s"] > 0 and c4["children_per_s"] > c4["positions_per_s"]
    assert c5["parity"] == {"allreduced_accumulators_equal_rank0_replay_of_all_game_ids": True,
                            "parameters_identical_on_all_ranks": True}
    assert c5["allreduce_bytes"] == 2560 and len(c5["parameters"]) == 36
    c5t = d["extra"]["config5_table"]                          # the reference's value-table semantics
    assert c5t["iteration_ms"] > 0 and c5t["table_keys"] > 0 and len(c5t["parameters"]) == 36
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] > 0
    assert d["clocks"]["sm_mhz"] is None or d["clocks"]["sm_mhz"] > 500


def _u64(halves):
    return halves[..., 0].astype(np.uint64) | (halves[..., 1].astype(np.uint64) << np.uint64(32))


@pytest.mark.gpu
def test_dump_outputs_are_the_games_of_the_last_timed_step(tmp_path, oracle):
    G, K, W = 8192, 2, 3
    args = ["--steps", str(K), "--warmup", str(W), "--games", str(G), "--no-cpu-baseline", "--no-extra", "--dump-outputs"]
    d = run(args + [str(tmp_path / "a")], timeout=600)
    assert d["steps"] == K and d["gpu_launches"] == K
    run(args + [str(tmp_path / "b")], timeout=600)
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == sorted(p.name for p in (tmp_path / "b").iterdir())
    out, total = {}, 0
    for n in names:
        a = np.load(tmp_path / "a" / n)
        assert a.dtype in (np.float32, np.float64)
        assert np.array_equal(a, np.load(tmp_path / "b" / n))              # same arguments, same outputs
        out[n[:-4]] = a
        total += a.nbytes
    assert total <= 64 << 20
    # step i plays games i*G .. i*G+G-1 of seed 1; the last timed step is i = W+K-1
    gid0 = (W + K - 1) * G
    ref = oracle.playout(1, gid0, G)
    g = out["game_id"].astype(np.int64) - gid0
    assert g.size == G and np.array_equal(g, np.arange(G))
    assert np.array_equal(out["nplies"], ref["nplies"])
    assert np.array_equal(_u64(out["final_black"]), ref["final_black"])
    assert np.array_equal(_u64(out["final_white"]), ref["final_white"])
    tg = out["trajectory_game_id"].astype(np.int64) - gid0
    t = np.arange(ref["black"].shape[0])[:, None]
    pos_ok = t <= ref["nplies"][tg][None, :]
    assert np.array_equal(out["trajectory_black"][..., 0] >= 0, pos_ok)
    assert np.array_equal(_u64(out["trajectory_black"])[pos_ok], ref["black"][:, tg][pos_ok])
    assert np.array_equal(_u64(out["trajectory_white"])[pos_ok], ref["white"][:, tg][pos_ok])
    mv_ok = t[:-1] < ref["nplies"][tg][None, :]
    assert np.array_equal(out["trajectory_move"] >= 0, mv_ok)
    assert np.array_equal(out["trajectory_move"][mv_ok], ref["move"][:, tg][mv_ok])
    # the totals `value` is computed from: plies, disc difference and wins over the games of all K timed steps
    allg = oracle.playout(1, W * G, K * G, trajectory=False)
    nb, nw = np.bitwise_count(allg["final_black"]).astype(np.int64), np.bitwise_count(allg["final_white"]).astype(np.int64)
    want = [allg["nplies"].sum(dtype=np.int64), (nb - nw).sum(), (nb > nw).sum(), (nw > nb).sum()]
    assert out["totals"].tolist() == [float(v) for v in want]
    assert d["value"] == pytest.approx(want[0] / (d["ms_per_step"] * K * 1e-3), rel=1e-9)
