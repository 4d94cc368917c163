"""Shared helpers for the parity tests (test infrastructure; may import the oracle)."""
import contextlib
import io
import random

import numpy as np

from oracle import prmf_oracle as O


def seed_all(seed):
    np.random.seed(seed)
    random.seed(seed)


def oracle_block(X, U, V, Gs, nodelist, active, n_steps, gamma, delta, tradeoff=None):
    """n_steps of the oracle's inner update with a per-step log."""
    tables = O.PathwayTables(Gs, nodelist)
    log = []
    U2, V2, od, g2, d2 = O.update_block(X, U.copy(), V.copy(), tables, active, n_steps, gamma, delta,
                                        tradeoff, log)
    parts = np.array([[d["recon"], d["manifold"], d["ignore"], d["fro"], d["obj"]] for d in log])
    return U2, V2, parts, g2, d2, tables


def run_product(g, **kw):
    """Run prmf_b200.nmf_pathway on a golden-fixture instance with the fixture's seed and arguments."""
    from prmf_b200 import nmf_pathway
    meta = g["meta"]
    seed_all(meta["seed"])
    trace = {"keep_blocks": 3}
    with contextlib.redirect_stdout(io.StringIO()) as out, contextlib.redirect_stderr(io.StringIO()):
        U, V, od = nmf_pathway(g["X"].copy(), [G.copy() for G in g["Gs"]], gamma=meta["gamma_in"],
                               delta=meta["delta_in"], tradeoff=meta["tradeoff"], k_latent=meta["k_latent"],
                               nodelist=list(g["nodelist"]), max_iter=meta["max_iter"], trace=trace, **kw)
    return U, V, od, trace, out.getvalue()


def check_run_against_golden(g, U, V, od, trace, rtol_obj=1e-9, rtol_uv=1e-7):
    """Assignments bit-exact; objective parts / U / V within the stated relative tolerances."""
    meta = g["meta"]
    assert trace["sampled"] == meta["sampled"], "sampled pathways differ from the reference"
    got = np.array(trace["obj_parts"])
    assert got.shape == g["obj_parts"].shape, "different number of inner steps: %s vs %s" % (
        got.shape, g["obj_parts"].shape)
    np.testing.assert_allclose(got, g["obj_parts"], rtol=rtol_obj, atol=1e-11)
    assert len(trace["cands"]) == len(meta["cands"])
    for a, b in zip(trace["cands"], meta["cands"]):
        assert a["kind"] == b["kind"]
        for k, lst in b["data"].items():
            mine = a["data"][int(k)]
            assert [p for p, _ in mine] == [p for p, _ in lst], "candidate lists differ"
            np.testing.assert_allclose([s for _, s in mine], [s for _, s in lst], rtol=1e-9)
    for (Ub, Vb), Ug, Vg in zip(trace["blocks"], g["blocks_U"], g["blocks_V"]):
        np.testing.assert_allclose(Ub, Ug, rtol=rtol_uv, atol=1e-12)
        np.testing.assert_allclose(Vb, Vg, rtol=rtol_uv, atol=1e-12)
    np.testing.assert_allclose(U, g["U_final"], rtol=1e-6, atol=1e-10)
    np.testing.assert_allclose(V, g["V_final"], rtol=1e-6, atol=1e-10)
    fm = {int(k): [p for p, _ in v] for k, v in meta["final_map"].items()}
    assert {k: [p for p, _ in v] for k, v in od["latent_to_pathway_data"].items()} == fm
    for key in ("recon", "manifold", "ignore", "fro", "gamma", "delta", "obj"):
        np.testing.assert_allclose(od[key], meta["final"][key], rtol=1e-8)


def xstream_plan(m, n, k, x_dtype="f64", stages=0, sm_count=148):
    """The launch plan libprmf_b200 gives the two X-stream passes of an m x n handle with k factors on a device with
    `sm_count` SMs (prmf_plan_xstream, no GPU needed).  `stages`: the PRMF_TMA_STAGES override, 0 for none."""
    import ctypes
    from prmf_b200 import _lib
    plan = _lib.XstreamPlan()
    rc = _lib.load().prmf_plan_xstream(m, n, k, _lib.X_DTYPES[x_dtype], sm_count, stages, ctypes.byref(plan))
    assert rc == 0, "prmf_plan_xstream returned %d" % rc
    return plan


def tf32_round(a):
    """Host model of `cvt.rna.tf32.f32` applied to float(a): round to nearest (ties away from zero) to a
    10-bit mantissa.  Returns float64 values that are exactly representable in tf32."""
    b = np.asarray(a, dtype=np.float32).view(np.uint32).astype(np.uint64)
    b = ((b + 0x1000) & 0xFFFFE000).astype(np.uint32)
    return b.view(np.float32).astype(np.float64)
