"""Pin the CPU oracle (oracle/prmf_oracle.py) to the unmodified reference.

(1) against the committed fixtures recorded from the reference (tests/golden/*.npz);
(2) when /root/reference is present (build container), side by side in this process.
"""
import random

import numpy as np
import pytest

from conftest import GOLDEN, GOLDEN_CASES, load_golden
from oracle import prmf_oracle as O

RTOL_OBJ = 1e-10      # per-inner-step objective parts
RTOL_UV = 1e-8        # U / V over the run


def run_oracle(g, **kw):
    meta = g["meta"]
    np.random.seed(meta["seed"]); random.seed(meta["seed"])
    trace = {}
    U, V, od = O.nmf_pathway(g["X"].copy(), [G.copy() for G in g["Gs"]], gamma=meta["gamma_in"],
                             delta=meta["delta_in"], tradeoff=meta["tradeoff"],
                             k_latent=meta["k_latent"], nodelist=g["nodelist"],
                             max_iter=meta["max_iter"], trace=trace, **kw)
    return U, V, od, trace


def check_against_golden(g, U, V, od, trace):
    meta = g["meta"]
    assert trace["sampled"] == meta["sampled"], "sampled pathways differ"
    got = np.array(trace["obj_parts"])
    assert got.shape == g["obj_parts"].shape, "different number of inner steps"
    np.testing.assert_allclose(got, g["obj_parts"], rtol=RTOL_OBJ, atol=1e-12)
    assert len(trace["cands"]) == len(meta["cands"])
    for a, b in zip(trace["cands"], meta["cands"]):
        assert a["kind"] == b["kind"]
        for k, lst in b["data"].items():
            mine = a["data"][int(k)]
            assert [p for p, _ in mine] == [p for p, _ in lst], "candidate lists differ"
            np.testing.assert_allclose([s for _, s in mine], [s for _, s in lst], rtol=1e-10)
    for (Ub, Vb), Ug, Vg in zip(trace["blocks"], g["blocks_U"], g["blocks_V"]):
        np.testing.assert_allclose(Ub, Ug, rtol=RTOL_UV, atol=1e-12)
        np.testing.assert_allclose(Vb, Vg, rtol=RTOL_UV, atol=1e-12)
    np.testing.assert_allclose(U, g["U_final"], rtol=1e-6, atol=1e-10)
    np.testing.assert_allclose(V, g["V_final"], rtol=1e-6, atol=1e-10)
    fm = {int(k): [p for p, _ in v] for k, v in meta["final_map"].items()}
    assert {k: [p for p, _ in v] for k, v in od["latent_to_pathway_data"].items()} == fm
    for key in ("recon", "manifold", "ignore", "fro", "gamma", "delta", "obj"):
        np.testing.assert_allclose(od[key], meta["final"][key], rtol=1e-9)


@pytest.mark.parametrize("case", GOLDEN_CASES)
def test_oracle_matches_reference_fixture(case):
    g = load_golden(case)
    U, V, od, trace = run_oracle(g)
    check_against_golden(g, U, V, od, trace)


def test_stale_reference_golden_gamma_delta():
    """The reference's only golden file pins gamma = 8337.63767 and delta = 0.00020 for the raw test
    instance (test_inferred_nodelist_1_expected_obj.txt; the other lines are stale, SURVEY §0.9)."""
    g = load_golden("test1_raw")
    assert "%.5f" % g["meta"]["final"]["gamma"] == "8337.63767"
    assert "%.5f" % g["meta"]["final"]["delta"] == "0.00020"
    norm_X = np.linalg.norm(g["X"])
    assert "%.5f" % (norm_X / 6) == "8337.63767"


def test_kernel_vectors():
    g = load_golden("kernel_vectors")
    tables = O.PathwayTables(g["Gs"], g["nodelist"])
    V = g["V"]
    K, P = g["score"].shape
    for p in range(P):
        np.testing.assert_allclose(tables.Lns[p].toarray(), g["Ln_dense"][p], rtol=1e-14, atol=0)
    score = np.array([[O.score_match(tables, V[:, k], p) for p in range(P)] for k in range(K)])
    np.testing.assert_allclose(score, g["score"], rtol=1e-13)
    cands = {k: [(p, 1) for p in range(P)] for k in range(K)}
    got = O.restrict(V, tables, cands)
    for k, lst in g["meta"]["restricted"].items():
        assert [p for p, _ in got[int(k)]] == [p for p, _ in lst]
    np.testing.assert_array_equal(O.find_mins(V, tables.Ls), g["find_mins"])


def test_cached_normalized_is_identical():
    g = load_golden("small_tradeoff")
    a = run_oracle(g)
    b = run_oracle(g, cache_normalized=True)
    np.testing.assert_array_equal(a[0], b[0])
    np.testing.assert_array_equal(a[1], b[1])


# ---- side by side with the reference itself (build container only) ---------------------------------
def _ref():
    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
    import ref_shim
    if not ref_shim.reference_available():
        pytest.skip("/root/reference not present on this host")
    return ref_shim


@pytest.mark.parametrize("seed", [0, 1])
def test_oracle_vs_live_reference(seed):
    """The oracle against what the reference returns on two more instances (the weighted one without a tradeoff):
    the fixture `make_golden.py --only-side-by-side` records from the reference, else the reference run here."""
    import contextlib, io, json, os, sys
    sys.path.insert(0, GOLDEN)
    from make_golden_io import side_by_side_instance
    X, nodelist, Gs = side_by_side_instance(seed)
    fixture = os.path.join(GOLDEN, "side_by_side_seed%d.npz" % seed)
    if os.path.exists(fixture):
        z = np.load(fixture, allow_pickle=False)
        Ur, Vr, obj_r, map_r = z["U"], z["V"], float(z["obj"]), json.loads(str(z["final_map"]))
    else:
        ref_shim = _ref()
        R = ref_shim.load_reference()
        ref_shim.reset_globals(R)
        np.random.seed(seed); random.seed(seed)
        with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
            Ur, Vr, odr = R.nmf_pathway(X.copy(), [G.copy() for G in Gs], nodelist=list(nodelist),
                                        k_latent=3, max_iter=300)
        ref_shim.reset_globals(R)
        obj_r = odr["obj"]
        map_r = {str(k): [int(p) for p, _ in v] for k, v in odr["latent_to_pathway_data"].items()}
    np.random.seed(seed); random.seed(seed)
    Uo, Vo, odo = O.nmf_pathway(X.copy(), [G.copy() for G in Gs], nodelist=list(nodelist),
                                k_latent=3, max_iter=300)
    np.testing.assert_allclose(Uo, Ur, rtol=1e-7, atol=1e-12)
    np.testing.assert_allclose(Vo, Vr, rtol=1e-7, atol=1e-12)
    np.testing.assert_allclose(odo["obj"], obj_r, rtol=1e-10)
    assert {str(k): [int(p) for p, _ in v] for k, v in odo["latent_to_pathway_data"].items()} == map_r
