"""The fp32 storage mode (x_dtype="f32", PRMF_X_F32): X and X^T held as exact fp32 values, streamed through the fp64
DFMA kernels with every element widened before its first use.

An fp32 value widens to fp64 exactly, and the f32 handle runs the same launch plan (panels, chunks, rows per chunk) as an
fp64 handle, so every column runs the same fma chain on the same values in the same order.  Hence the exact oracle of
this file: an f32 handle given X32 must return, bit for bit, what an fp64 handle returns given X32.astype(np.float64),
for single products and whole runs alike.  Every comparison below is np.array_equal or ==, never a tolerance, except
against the reference fixture, which ran on fp64 X.
"""
import contextlib
import io

import numpy as np
import pytest

from conftest import load_golden
from helpers import run_product
from test_sass import _longest_dfma_region, _sass_by_function
from test_xstream_exact import (K_GEN, K_SKINNY, RING_LIMIT, RS, SHAPES, _instance, _run_products, b200,  # noqa: F401
                                default_stages, gen_fg_kt, host_wb)

K_EQ = list(range(1, 11)) + [11, 17, 25, 64, 128]
EQ_SHAPES = [(1, 1), (37, 131), (300, 257), (1025, 1000), (3, 4100), (993, 520), (2049, 33)]


# ---- CPU: the ring plan ---------------------------------------------------------------------------------------
def f32_default_stages(fg):
    """Ring stages of an f32 handle without PRMF_TMA_STAGES (prmf_create_ex): twice the fp64 count."""
    return 2 * default_stages(fg)


def ring_bytes(panel_w, k, stages, elem):
    """Shared memory of a ring of `stages` stages (X rows of `elem` bytes + the W slot + 2 mbarriers per stage)."""
    return stages * (RS * panel_w * elem + host_wb(k)) + 2 * stages * 8


def test_f32_default_ring_fits_and_keeps_the_fp64_bytes_in_flight():
    for k in range(1, 129):
        fg = gen_fg_kt(k)[0] if k > 10 else 1
        panel_w = 1024 // fg                                             # the widest panel
        s32, s64 = f32_default_stages(fg), default_stages(fg)
        assert s32 <= 12, k                                              # inside the PRMF_TMA_STAGES range
        assert ring_bytes(panel_w, k, s32, 4) <= RING_LIMIT, k
        assert s32 * RS * panel_w * 4 >= s64 * RS * panel_w * 8, k       # bytes of X in flight


# ---- CPU: the shipped SASS ------------------------------------------------------------------------------------
def test_f32_stream_kernels_sass():
    funcs = _sass_by_function()
    for k in (6, 10):
        for epi in (0, 1, 2):
            pattern = "skinny_tma_f32_kernelILi%dELi8ELi%dE" % (k, epi)
            names = [n for n in funcs if pattern in n]
            assert len(names) == 1, pattern
            ops = funcs[names[0]]
            assert any(op.startswith("UBLKCP") for op in ops) and any(op.startswith("SYNCS") for op in ops), pattern
            a, b = _longest_dfma_region(ops)
            loop = ops[a:b + 1]
            assert sum(op.startswith("DFMA") for op in loop) >= 8 * 4 * k, pattern
            assert not any(op.startswith(("LDL", "STL")) for op in loop), pattern
    gen = {(kt, fg) for fg, kt in (gen_fg_kt(k) for k in range(11, 129))}
    for kt, fg in gen:
        pattern = "skinny_tma_gen_f32_kernelILi%dELi%dELi8E" % (kt, fg)
        names = [n for n in funcs if pattern in n]
        assert len(names) == 1, pattern
        ops = funcs[names[0]]
        assert any(op.startswith("UBLKCP") for op in ops) and not any(op.startswith(("LDL", "STL")) for op in ops)
    # the fp64 kernels' names do not match the fp32 ones, so the fp64 SASS checks never see them
    assert not [n for n in funcs if "skinny_tma_kernelI" in n and "f32" in n]


# ---- CPU: single rank only ------------------------------------------------------------------------------------
def test_f32_nmf_pathway_refuses_several_ranks_before_any_engine():
    from prmf_b200 import nmf_pathway
    from prmf_b200.dist import DistContext

    def factory(*a, **kw):
        raise AssertionError("an engine was requested")

    X = np.ones((4, 3))
    with pytest.raises(ValueError, match="one rank"):
        nmf_pathway(X, [], nodelist=[0, 1, 2], ctx=DistContext(rank=0, world=2), engine_factory=factory, x_dtype="f32")


# ---- GPU helpers ----------------------------------------------------------------------------------------------
def _engine(m, n, k, x_dtype):
    from prmf_b200 import CudaEngine
    return CudaEngine(m, m, n, k, x_dtype=x_dtype)


def _products(eng):
    return eng.project(), eng.project_t(), eng.normX_sq, eng.residual_sq()


def _assert_same(got, want, what):
    for i, (a, b) in enumerate(zip(got, want)):
        assert np.array_equal(np.asarray(a), np.asarray(b)), "%s: item %d differs" % (what, i)


def _pair_products(X32, U, V):
    """(fp64 handle on the widened X32, f32 handle on X32) products."""
    m, n = X32.shape
    out = []
    for x_dtype, X in (("f64", X32.astype(np.float64)), ("f32", X32)):
        with _engine(m, n, U.shape[1], x_dtype) as eng:
            eng.set_X(X)
            eng.set_UV(U, V)
            out.append(_products(eng))
    return out


# ---- GPU: integer exactness -----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("m,n", SHAPES)
def test_f32_products_integer_exact(b200, m, n):
    """Every skinny_tma_f32_kernel<K,8,0> and every reachable skinny_tma_gen_f32_kernel<KT,FG> against int64."""
    _run_products(m, n, K_SKINNY + K_GEN, x_dtype="f32")


@pytest.mark.gpu
@pytest.mark.parametrize("stages", ["2", "12"])
def test_f32_products_integer_exact_under_stage_overrides(b200, monkeypatch, stages):
    monkeypatch.setenv("PRMF_TMA_STAGES", stages)
    for m, n in SHAPES:
        _run_products(m, n, K_SKINNY + K_GEN, x_dtype="f32", residual=False, label="stages " + stages)


# ---- GPU: bitwise equality with fp64 on the widened matrix ----------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("m,n", EQ_SHAPES)
def test_f32_products_equal_fp64_on_widened_X(b200, m, n):
    for k in K_EQ:
        rng = np.random.Generator(np.random.PCG64(1000 * m + n + k))
        X32 = rng.random((m, n), dtype=np.float32)
        U, V = rng.random((m, k)), rng.random((n, k))
        want, got = _pair_products(X32, U, V)
        _assert_same(got, want, "m=%d n=%d k=%d" % (m, n, k))


def _steps(x_dtype, X, packed, U, V, active, k, tradeoff=None, prefetch_block=False):
    from prmf_b200 import CudaEngine
    m, n = X.shape
    with CudaEngine(m, m, n, k, x_dtype=x_dtype) as eng:
        eng.set_X(X); eng.set_pathways(packed); eng.set_UV(U, V); eng.set_active(active)
        if prefetch_block:
            eng.step_async(5, 2.0, 0.4)
            p1, _, _, tables = eng.block_end(5, want_scores=True, prefetch=True)
            p2, g, d = eng.step(5, 2.0, 0.4)
            parts = (p1, p2, tables[0], tables[1], tables[2], g, d)
        else:
            parts = eng.step(10, 2.0, 0.4, tradeoff=tradeoff)
        return parts, eng.get_UV()


STEP_CASES = [(6, None, {}, False), (25, None, {}, False), (6, 0.5, {}, False), (25, 0.5, {}, False),
              (6, None, {"PRMF_EPI": "0"}, False), (6, None, {"PRMF_DEFER_OBJ": "0"}, False), (6, None, {}, True),
              (25, None, {}, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("k,tradeoff,env,prefetch", STEP_CASES,
                         ids=["k6", "k25", "k6_tradeoff", "k25_tradeoff", "k6_epi0", "k6_defer0", "k6_prefetch",
                              "k25_prefetch"])
def test_f32_inner_steps_equal_fp64_on_widened_X(b200, monkeypatch, k, tradeoff, env, prefetch):
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    X, packed, U, V, active = _instance(300, 1200, k, 9, seed=90 + k)
    X32 = X.astype(np.float32)
    want = _steps("f64", X32.astype(np.float64), packed, U, V, active, k, tradeoff, prefetch)
    got = _steps("f32", X32, packed, U, V, active, k, tradeoff, prefetch)
    _assert_same(list(got[0]) + list(got[1]), list(want[0]) + list(want[1]), "k=%d %s" % (k, env))


@pytest.mark.gpu
def test_f32_nnls_and_pathway_init_equal_fp64_on_widened_X(b200):
    from prmf_b200 import nnls_x, pathway_init, synth
    X, nodelist, Gs = synth.small_instance(m=120, n=400, k_true=3, n_pathways=6, pathway_size=12, seed=7)
    X32 = X.astype(np.float32)
    Xw = X32.astype(np.float64)
    rng = np.random.Generator(np.random.PCG64(8))
    for transpose, rows in ((True, 400), (False, 120)):
        B = rng.random((rows, 5))
        _assert_same(nnls_x(X32, B, transpose=transpose, x_dtype="f32"), nnls_x(Xw, B, transpose=transpose),
                     "nnls_x transpose=%s" % transpose)
    s32, s64 = {}, {}
    got = pathway_init(X32, Gs[:4], nodelist, stats=s32, x_dtype="f32")
    want = pathway_init(Xw, Gs[:4], nodelist, stats=s64)
    _assert_same(got, want, "pathway_init")
    assert s32 == s64
    import torch
    _assert_same(pathway_init(torch.from_numpy(X32).cuda(), Gs[:4], nodelist, x_dtype="f32"), want, "device X32")


@pytest.mark.gpu
def test_f32_whole_run_equals_fp64_on_widened_X(b200):
    g = load_golden("small_planted")
    X32 = g["X"].astype(np.float32)
    runs = []
    for x_dtype, X in (("f64", X32.astype(np.float64)), ("f32", X32)):
        gx = dict(g)
        gx["X"] = X
        runs.append(run_product(gx, x_dtype=x_dtype))
    (U0, V0, od0, tr0, _), (U1, V1, od1, tr1, _) = runs
    assert tr1["sampled"] == tr0["sampled"]
    assert tr1["cands"] == tr0["cands"]
    assert np.array_equal(np.array(tr1["obj_parts"]), np.array(tr0["obj_parts"]))
    assert np.array_equal(U1, U0) and np.array_equal(V1, V0)
    assert od1.keys() == od0.keys()
    for key in od0:
        if isinstance(od0[key], np.ndarray):
            assert np.array_equal(od1[key], od0[key]), key
        else:
            assert od1[key] == od0[key], key


@pytest.mark.gpu
def test_f32_config2_outer_iteration_equals_fp64_on_widened_X(b200):
    """BASELINE config 2's shape (37 032 x 6 750, k = 10): one outer iteration, 10 inner steps + the score tables."""
    from prmf_b200 import pack_pathways, synth
    m, n, k, P = 37032, 6750, 10, 40
    rng = np.random.Generator(np.random.PCG64(2))
    X32 = rng.random((m, n), dtype=np.float32)
    packed = pack_pathways(synth.random_pathway_graphs(rng, n, P), list(range(n)))
    U, V = 3 * (1 - rng.random((m, k))), 3 * (1 - rng.random((n, k)))
    active = [int(rng.integers(0, P)) for _ in range(k)]
    out = []
    for x_dtype, X in (("f64", X32.astype(np.float64)), ("f32", X32)):
        with _engine(m, n, k, x_dtype) as eng:
            eng.set_X(X); eng.set_pathways(packed); eng.set_UV(U, V); eng.set_active(active)
            eng.step_async(10, 2.0, 0.4)
            parts, gam, dl, tables = eng.block_end(10, want_scores=True, prefetch=False)
            out.append([parts, gam, dl, *tables, *eng.get_UV(), eng.normX_sq])
        del X
    _assert_same(out[1], out[0], "config 2")


# ---- GPU: input flavours and pooled buffers -------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k", [6, 25])
def test_f32_input_flavours_store_the_same_matrix(b200, k):
    import torch
    m, n = 37, 131
    rng = np.random.Generator(np.random.PCG64(30 + k))
    X64 = rng.random((m, n)) * 3                                      # not representable in fp32: the store rounds
    X32 = X64.astype(np.float32)
    U, V = rng.random((m, k)), rng.random((n, k))
    with _engine(m, n, k, "f64") as ref:
        ref.set_X(X32.astype(np.float64))
        ref.set_UV(U, V)
        want = _products(ref)
    wide32 = np.full((m, n + 21), np.nan, dtype=np.float32)
    wide32[:, :n] = X32
    wide64 = np.full((m, n + 21), np.nan)
    wide64[:, :n] = X64
    flavours = {"f32 host": X32, "f32 fortran": np.asfortranarray(X32), "f32 host slice": wide32[:, :n],
                "f32 device": torch.from_numpy(X32).cuda(), "f32 device slice": torch.from_numpy(wide32).cuda()[:, :n],
                "f64 host": X64, "f64 fortran": np.asfortranarray(X64), "f64 host slice": wide64[:, :n],
                "f64 device": torch.from_numpy(X64).cuda(), "f64 device slice": torch.from_numpy(wide64).cuda()[:, :n]}
    with _engine(m, n, k, "f32") as eng:
        assert eng.lib.prmf_x_dtype(eng.h) == 2
        eng.set_UV(U, V)
        for name, Xf in flavours.items():
            eng.set_X(Xf)
            _assert_same(_products(eng), want, "%s k=%d" % (name, k))


@pytest.mark.gpu
@pytest.mark.parametrize("m,n,k", [(300, 257, 6), (993, 520, 66)])
def test_f32_pooled_buffers_do_not_leak(b200, m, n, k):
    """A destroyed f32 handle leaves X32, its transposed copy and its arena to the next handle of the same shape."""
    nan = np.full((m, n), np.nan, dtype=np.float32)
    with _engine(m, n, k, "f32") as eng:
        eng.set_X(nan)
        eng.set_UV(np.full((m, k), np.nan), np.full((n, k), np.nan))
        eng.project(); eng.project_t()
    _run_products(m, n, [k], x_dtype="f32", label="after a NaN handle")


# ---- GPU: single rank, and the reference fixture --------------------------------------------------------------
@pytest.mark.gpu
def test_f32_handle_is_single_rank(b200):
    from prmf_b200 import CudaEngine
    from prmf_b200._lib import PrmfLibraryError
    with pytest.raises(PrmfLibraryError, match="single-rank"):
        CudaEngine(10, 20, 16, 4, x_dtype="f32")
    with CudaEngine(10, 10, 16, 4, x_dtype="f32") as eng:
        with pytest.raises(PrmfLibraryError, match="single-rank"):
            eng.attach_comm(0, 2, bytes(128))
        with pytest.raises(PrmfLibraryError, match="single-rank"):
            eng.p2p_attach(0, 2, [bytes(64), bytes(64)])


@pytest.mark.gpu
def test_f32_whole_loop_keeps_the_reference_assignments(b200):
    """small_planted, recorded from the reference on fp64 X: with X rounded to fp32 the sampled pathways and the final
    factor -> pathway map stay the reference's; the rounding may move the convergence test by one outer iteration."""
    g = load_golden("small_planted")
    with contextlib.redirect_stdout(io.StringIO()):
        U, V, od, trace, _ = run_product(g, x_dtype="f32")
    meta = g["meta"]
    common = min(len(trace["sampled"]), len(meta["sampled"]))
    assert abs(len(trace["sampled"]) - len(meta["sampled"])) <= 1
    assert trace["sampled"][:common] == meta["sampled"][:common]
    fm = {int(k): [p for p, _ in v] for k, v in meta["final_map"].items()}
    assert {k: [p for p, _ in v] for k, v in od["latent_to_pathway_data"].items()} == fm
    np.testing.assert_allclose(od["obj"], meta["final"]["obj"], rtol=1e-5)
