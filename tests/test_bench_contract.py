"""bench.py's driver-facing contract, checked without a GPU: the synthetic matrix is the same for every partition of the
rows (strong scaling compares ONE instance), both arms print the same `config` dict, and the reference arm produces a
well-formed line from the CPU implementation of the path (the unmodified reference functions when `baseline/_ref` is
installed, else the oracle port)."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def _bench():
    argv = sys.argv
    sys.argv = ["bench.py"]
    try:
        spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        sys.argv = argv
    return mod


def test_synthetic_matrix_does_not_depend_on_the_partition():
    b = _bench()
    full = b.host_rows(0, 9000, 37)
    for world in (2, 3, 8):
        per = -(-9000 // world)
        parts = [b.host_rows(min(9000, r * per), min(9000, (r + 1) * per), 37) for r in range(world)]
        assert np.array_equal(full, np.concatenate(parts))
    assert np.array_equal(b.host_rows(100, 5000, 37, np.float32), full[100:5000].astype(np.float32))
    out = np.empty((4096, 37))
    assert b.host_rows(4096, 8192, 37, out=out) is out and np.array_equal(out, full[4096:8192])


def test_both_arms_describe_the_same_config():
    b = _bench()
    sys_argv = sys.argv
    try:
        sys.argv = ["bench.py", "--gpus", "4"]
        ours = b.config_dict(b.parse_args())
        sys.argv = ["bench.py", "--gpus", "4", "--impl", "reference"]
        ref = b.config_dict(b.parse_args())
    finally:
        sys.argv = sys_argv
    assert ours == ref and "37032x6750" in ours["workload"] and "k=10" in ours["workload"]


def test_reference_arm_line(tmp_path):
    env = dict(os.environ, RANK="0", WORLD_SIZE="1", OMP_NUM_THREADS="1")       # as under torchrun: the arm must undo this
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--m", "400", "--n", "500",
                          "--pathways", "12", "--k", "4", "--steps", "2", "--warmup", "1", "--ref-budget-s", "20"],
                         capture_output=True, text=True, timeout=600, env=env, cwd=str(tmp_path))
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads([l for l in res.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["metric"] == "prmf_outer_iterations_per_sec" and line["unit"] == "outer_it/s"
    assert line["higher_is_better"] is True and line["steps"] == 2 and line["warmup"] == 1 and line["value"] > 0
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["value"] == line["value"] and cb["cores"] >= 1 and cb["sample"]
    assert 1 <= cb["inner_steps_per_sample"] <= 10
    assert line["e2e"] == {"value": line["value"], "unit": "outer_it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # ms_per_step is the wall time of a sample, value the rate of a whole outer iteration (10 inner steps + restrict)
    assert line["ms_per_step"] <= line["ms_per_outer_iteration"] * 1.05
    assert os.path.isfile(os.path.join(ROOT, "baseline", "_ref", "bin", "prmf_runner.py")) == (cb["kind"] == "reference")
    # ranks other than 0 exit quietly
    res2 = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--m", "100"],
                          capture_output=True, text=True, timeout=120, env=dict(env, RANK="1", WORLD_SIZE="2"))
    assert res2.returncode == 0 and res2.stdout.strip() == ""


def test_argument_checks():
    for extra in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "d"]):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                             timeout=120)
        assert res.returncode == 2 and "error" in res.stderr, extra


def test_dump_rows_fit_the_budget_and_do_not_depend_on_the_run():
    b = _bench()
    assert b.dump_rows(37032, 10, 1 << 20) is None                     # config 2: all of U
    rows = b.dump_rows(1000000, 128, 20 << 20)                         # config 5: a sample
    assert rows is not None and np.array_equal(rows, b.dump_rows(1000000, 128, 20 << 20))
    assert np.all(np.diff(rows) > 0) and rows[-1] < 1000000
    assert len(rows) * (128 * 8 + 8) + (20 << 20) <= b.DUMP_BYTES < 64 * 10**6
    position, scores = b.restrict_arrays({0: [(2, 0.5), (0, 1.5)], 1: [(1, 1)]}, 2, 3)
    assert position.tolist() == [[2, 0, 1], [0, 1, 0]] and scores.tolist() == [[1.5, 0, 0.5], [0, 1, 0]]


def test_dumped_U_rows_are_the_sampled_rows_of_the_global_U(tmp_path, monkeypatch):
    """A U too large for the dump, sharded over 1, 3 and 8 ranks: rank 0 writes exactly U[U_rows] (rows gathered in
    rank order), whatever the partition."""
    import types
    from prmf_b200.dist import row_block
    b = _bench()
    monkeypatch.setattr(b, "DUMP_BYTES", 40000)
    m, n, k, P = 5000, 7, 3, 4
    U = np.random.default_rng(0).random((m, k))
    V = np.random.default_rng(1).random((n, k))
    last = (np.ones((10, 8)), np.ones((k, P)), np.ones((k, P)), {0: [(1, 2.0)], 1: [(0, 1.0)], 2: [(3, 1.0)]})
    for world in (1, 3, 8):
        out_dir = tmp_path / str(world)
        a = types.SimpleNamespace(m=m, k=k, dump_outputs=str(out_dir))
        pieces = {}

        class Ctx:
            def __init__(self, rank):
                self.rank = rank

            def all_gather_rows(self, local, m_sel):       # ranks 1.. run first; rank 0 collects all pieces
                pieces[self.rank] = local
                if self.rank:
                    return None
                out = np.concatenate([pieces[r] for r in range(world)])
                assert out.shape[0] == m_sel
                return out

        for rank in list(range(1, world)) + [0]:
            lo, hi = row_block(m, world, rank)
            eng = types.SimpleNamespace(get_UV=lambda lo=lo, hi=hi: (U[lo:hi].copy(), V.copy()))
            b.dump_outputs(a, Ctx(rank), eng, lo, hi, last, P)
        rows = np.load(out_dir / "U_rows.npy")
        assert 0 < len(rows) < m and np.array_equal(rows, b.dump_rows(m, k, 10 * 5 * 8 + n * k * 8 + 4 * k * P * 8))
        assert np.array_equal(np.load(out_dir / "U.npy"), U[rows.astype(np.int64)])
        assert np.array_equal(np.load(out_dir / "V.npy"), V)
        assert sum(f.stat().st_size for f in out_dir.iterdir()) < 40000 + 4096


@pytest.mark.gpu
def test_dump_outputs_repeat_bit_for_bit(tmp_path):
    """Two runs with the same arguments dump identical outputs of the last timed step; one more timed step changes them."""
    def run(tag, steps):
        out = tmp_path / tag
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--m", "3000", "--n", "700", "--k", "6",
                              "--pathways", "20", "--steps", str(steps), "--warmup", "1", "--no-parity", "--no-e2e",
                              "--no-converge", "--dump-outputs", str(out)],
                             capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
        assert res.returncode == 0, res.stderr[-2000:]
        line = json.loads([l for l in res.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == steps
        dump = {f[:-4]: np.load(out / f) for f in sorted(os.listdir(out))}
        assert dump["obj_parts"][-1, 4] == line["final_obj"]               # the step the timed loop ended with
        return dump
    a, b, c = run("a", 2), run("b", 2), run("c", 3)
    assert sorted(a) == sorted(["U", "V", "obj_parts", "restrict_position", "restrict_scores", "score_mass",
                                "score_quad_norm"])
    assert a["U"].shape == (3000, 6) and a["V"].shape == (700, 6) and a["obj_parts"].shape == (10, 5)
    assert a["score_mass"].shape == (6, 20) and a["restrict_position"].max() >= 1
    for name in a:
        assert a[name].dtype == np.float64 and np.array_equal(a[name], b[name]), name
    assert not np.array_equal(a["V"], c["V"])
