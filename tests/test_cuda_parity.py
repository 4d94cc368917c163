"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle and against the fixtures
recorded from the unmodified reference.  Tolerances (fp64): per-inner-step objective parts rel 1e-9,
U/V rel 1e-7 over the first blocks and 1e-6 at return, assignments/candidate lists/iteration counts
identical."""
import numpy as np
import pytest

from conftest import GOLDEN_CASES, load_golden
from helpers import check_run_against_golden, oracle_block, run_product, seed_all

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("case", GOLDEN_CASES)
def test_whole_loop_matches_reference_fixture(case):
    g = load_golden(case)
    U, V, od, trace, _ = run_product(g)
    check_run_against_golden(g, U, V, od, trace)


@pytest.mark.parametrize("case", ["test1_norm", "test2_raw", "small_planted"])
def test_whole_loop_persistent_kernel_matches_reference_fixture(monkeypatch, case):
    """The persistent step kernel (the default of sharded runs; PRMF_BLOCK=1 selects it on one GPU) on the fixtures."""
    monkeypatch.setenv("PRMF_BLOCK", "1")
    g = load_golden(case)
    U, V, od, trace, _ = run_product(g)
    check_run_against_golden(g, U, V, od, trace)


def _instance(m, n, k, P, seed, weighted=False, psize=12):
    from prmf_b200 import synth
    X, nodelist, Gs = synth.small_instance(m=m, n=n, k_true=min(3, P), n_pathways=P, pathway_size=psize,
                                           seed=seed, weighted=weighted)
    rng = np.random.Generator(np.random.PCG64(seed + 100))
    U = 3 * (1 - rng.random((m, k)))
    V = 3 * (1 - rng.random((n, k)))
    active = [int(rng.integers(0, P)) for _ in range(k)]
    return X, nodelist, Gs, U, V, active


@pytest.mark.parametrize("m,n,k,P", [
    (64, 256, 6, 8),       # aligned
    (37, 131, 3, 5),       # odd n, m not a multiple of the row tile
    (5, 33, 1, 3),         # tiny, k = 1
    (130, 1030, 7, 9),     # n just above one gene panel
    (200, 517, 10, 12),    # the benchmark's k
    (96, 300, 12, 6),      # k > 10: two factor tiles
    (70, 210, 17, 6),      # k > 16: pairs-per-thread > 1
    (50, 120, 33, 4),      # larger k: 4 factor groups x 12
    (40, 300, 16, 5),      # one group of 16
    (64, 2100, 64, 6),     # BASELINE config 4's k: 4 groups x 16, several panels
    (33, 150, 100, 4),     # 8 groups, ragged last group
    (24, 140, 128, 3),     # BASELINE config 5's k
    (45, 190, 2, 4),       # k = 2, 4, 5, 8, 9: the fused tails of those K
    (80, 333, 4, 6),
    (51, 260, 5, 7),
    (150, 700, 8, 9),
    (66, 1100, 9, 8),
    (90, 400, 27, 6),      # skinny_tma_gen_kernel<16,2>, tiled tails at 2 columns per thread
    (60, 500, 80, 5),      # skinny_tma_gen_kernel<12,8> with two idle factor groups, tiled tails at 8
])
@pytest.mark.parametrize("weighted", [False, True])
def test_inner_steps_match_oracle(m, n, k, P, weighted):
    from prmf_b200 import nmf_manifold_vec_update
    X, nodelist, Gs, U, V, active = _instance(m, n, k, P, seed=m + n + k, weighted=weighted)
    gamma, delta = 2.5, 0.3
    Uo, Vo, parts_o, _, _, _ = oracle_block(X, U, V, Gs, nodelist, active, 3, gamma, delta)
    import contextlib, io
    with contextlib.redirect_stdout(io.StringIO()) as out:
        Ug, Vg, od = nmf_manifold_vec_update(X, U, V, Gs, active, n_steps=3, gamma=gamma, delta=delta,
                                             nodelist=nodelist)
    np.testing.assert_allclose(Ug, Uo, rtol=1e-10, atol=1e-13)
    np.testing.assert_allclose(Vg, Vo, rtol=1e-10, atol=1e-13)
    lines = out.getvalue().strip().splitlines()
    got_obj = [float(l.split()[1]) for l in lines]
    np.testing.assert_allclose(got_obj, parts_o[:, 4], rtol=1e-10)
    for key, col in (("recon", 0), ("manifold", 1), ("ignore", 2), ("fro", 3), ("obj", 4)):
        np.testing.assert_allclose(od[key], parts_o[-1, col], rtol=1e-9, atol=1e-12)


def test_tradeoff_feedback_matches_oracle():
    from prmf_b200 import nmf_manifold_vec_update
    X, nodelist, Gs, U, V, active = _instance(60, 200, 4, 7, seed=9, weighted=True)
    Uo, Vo, parts_o, g2o, d2o, _ = oracle_block(X, U, V, Gs, nodelist, active, 5, 3.0, 0.2, tradeoff=0.4)
    import contextlib, io
    with contextlib.redirect_stdout(io.StringIO()):
        Ug, Vg, od, g2, d2 = nmf_manifold_vec_update(X, U, V, Gs, active, n_steps=5, gamma=3.0, delta=0.2,
                                                     tradeoff=0.4, nodelist=nodelist)
    np.testing.assert_allclose(Ug, Uo, rtol=1e-9)
    np.testing.assert_allclose(Vg, Vo, rtol=1e-9)
    np.testing.assert_allclose([g2, d2], [g2o, d2o], rtol=1e-9)
    np.testing.assert_allclose(od["obj"], parts_o[-1, 4], rtol=1e-9)


def test_zero_over_zero_and_clamps():
    """U rows of zeros stay zero (0/0 := 1, :422); V is clamped at float32 eps (:442-444)."""
    from prmf_b200 import nmf_manifold_vec_update
    X, nodelist, Gs, U, V, active = _instance(40, 90, 3, 4, seed=4)
    U[3, :] = 0.0
    U[7, 1] = 0.0
    V[5, :] = 0.0
    X[:, 11] = 0.0
    Uo, Vo, parts_o, _, _, _ = oracle_block(X, U, V, Gs, nodelist, active, 2, 1.0, 1.0)
    import contextlib, io
    with contextlib.redirect_stdout(io.StringIO()):
        Ug, Vg, od = nmf_manifold_vec_update(X, U, V, Gs, active, n_steps=2, nodelist=nodelist)
    assert np.all(Ug[3] == 0.0) and np.all(Uo[3] == 0.0)
    eps = np.finfo(np.float32).eps
    assert Vg.min() >= eps
    assert np.all(Vg[:, :][Vo == eps] == eps)
    np.testing.assert_allclose(Ug, Uo, rtol=1e-10, atol=1e-14)
    np.testing.assert_allclose(Vg, Vo, rtol=1e-10, atol=1e-14)


def test_score_tables_match_reference_vectors():
    from prmf_b200 import latent_pathway_tables, find_mins, restrict
    g = load_golden("kernel_vectors")
    mass, qn, qr = latent_pathway_tables(g["V"], g["Gs"], g["nodelist"])
    score = np.sqrt(mass) + (1 - qn)
    np.testing.assert_allclose(score, g["score"], rtol=1e-12)
    np.testing.assert_allclose(qn, g["quad_norm"], rtol=1e-10, atol=1e-14)
    np.testing.assert_allclose(qr, g["quad_raw"], rtol=1e-10, atol=1e-12)
    np.testing.assert_array_equal(find_mins(g["V"], g["Gs"], g["nodelist"]), g["find_mins"])
    K, P = score.shape
    cands = {k: [(p, 1) for p in range(P)] for k in range(K)}
    got = restrict(g["V"], g["Gs"], cands, g["nodelist"])
    for k, lst in g["meta"]["restricted"].items():
        assert [p for p, _ in got[int(k)]] == [p for p, _ in lst]


def test_recon_identity_against_exact_residual():
    """The pass-free identity ||X||^2 - 2<V,X^T U> + <U^T U, V^T V> equals the residual computed by an
    explicit third pass over X."""
    from prmf_b200 import CudaEngine, pack_pathways
    X, nodelist, Gs, U, V, active = _instance(300, 700, 6, 8, seed=21)
    with CudaEngine(300, 300, 700, 6) as eng:
        eng.set_X(X); eng.set_pathways(pack_pathways(Gs, nodelist)); eng.set_UV(U, V); eng.set_active(active)
        parts, _, _ = eng.step(4, 1.0, 1.0)
        exact = eng.residual_sq()
        np.testing.assert_allclose(parts[-1, 7], exact, rtol=1e-11)
        Ug, Vg = eng.get_UV()
        np.testing.assert_allclose(exact, np.linalg.norm(X - Ug @ Vg.T) ** 2, rtol=1e-11)
        np.testing.assert_allclose(eng.normX_sq, np.sum(X * X), rtol=1e-13)


def test_bitwise_deterministic():
    g = load_golden("small_tradeoff")
    a = run_product(g)
    b = run_product(g)
    np.testing.assert_array_equal(a[0], b[0])
    np.testing.assert_array_equal(a[1], b[1])
    assert a[3]["obj_parts"] == b[3]["obj_parts"]


def test_error_behaviour():
    from prmf_b200 import CudaEngine, nmf_pathway, pack_pathways
    from prmf_b200._lib import PrmfLibraryError
    X, nodelist, Gs, U, V, active = _instance(20, 50, 3, 4, seed=2)
    with pytest.raises(ValueError):                     # :656-659
        nmf_pathway(X, Gs, k_latent=3, nodelist=nodelist, U_init=np.ones((19, 3)), quiet=True)
    with pytest.raises(ValueError):
        nmf_pathway(X, Gs, k_latent=3, nodelist=nodelist, V_init=np.ones((50, 2)), quiet=True)
    with CudaEngine(20, 20, 50, 3) as eng:
        with pytest.raises(PrmfLibraryError):           # step before any data
            eng.step(1, 1.0, 1.0)
        eng.set_X(X); eng.set_pathways(pack_pathways(Gs, nodelist)); eng.set_UV(U, V)
        with pytest.raises(PrmfLibraryError):
            eng.set_active([0, 1, 99])                  # pathway id out of range
    with pytest.raises(PrmfLibraryError):
        CudaEngine(10, 10, 10, 500)                     # k too large


def test_full_size_properties():
    """BASELINE config 2 shape (37 032 x 6 750, k=10, 300 pathways): size-independent checks --
    the recon identity against the explicit residual pass, ||X||^2 against numpy, X.V against a
    row sample computed on the host, and the objective decreasing over a 10-step block."""
    from prmf_b200 import CudaEngine, pack_pathways, synth
    m, n, k, P = 37032, 6750, 10, 300
    X, nodelist, Gs = synth.recount2_shape(m, n, P, seed=0)
    rng = np.random.Generator(np.random.PCG64(5))
    U = 3 * (1 - rng.random((m, k))); V = 3 * (1 - rng.random((n, k)))
    packed = pack_pathways(Gs, nodelist)
    active = list(range(k))
    normX = np.linalg.norm(X)
    with CudaEngine(m, m, n, k) as eng:
        eng.set_X(X); eng.set_pathways(packed); eng.set_UV(U, V); eng.set_active(active)
        np.testing.assert_allclose(np.sqrt(eng.normX_sq), normX, rtol=1e-13)
        gamma, delta = normX / k, 10 / normX
        parts, _, _ = eng.step(1, gamma, delta)
        U1, V1 = eng.get_UV()
        rows = rng.integers(0, m, size=64)
        num = X[rows] @ V
        den = U[rows] @ (V.T @ V) + U[rows]
        np.testing.assert_allclose(U1[rows], U[rows] * num / den, rtol=1e-11)
        np.testing.assert_allclose(parts[0, 3], np.sum(U1 * U1), rtol=1e-12)
        parts, _, _ = eng.step(9, gamma, delta)
        np.testing.assert_allclose(parts[-1, 7], eng.residual_sq(), rtol=1e-10)
        assert np.all(np.diff(parts[:, 4]) < 0), "objective should decrease with fixed pathways"


def test_standalone_objective_matches_oracle():
    """nmf_manifold_vec_obj seam (:336-372) on arbitrary U, V (explicit residual pass)."""
    from oracle import prmf_oracle as O
    from prmf_b200 import nmf_manifold_vec_obj
    X, nodelist, Gs, U, V, active = _instance(90, 260, 5, 7, seed=31, weighted=True)
    tables = O.PathwayTables(Gs, nodelist)
    ref = O.objective(X, U, V, tables, active, 3.5, 0.25)
    got = nmf_manifold_vec_obj(X, U, V, Gs, active, gamma=3.5, delta=0.25, nodelist=nodelist)
    for key in ("recon", "manifold", "ignore", "fro", "obj"):
        np.testing.assert_allclose(got[key], ref[key], rtol=1e-12)
    assert list(got) == ["recon", "manifold", "ignore", "fro", "gamma", "delta", "obj"]


@pytest.mark.parametrize("k", [6, 12])          # fused-tail path (k <= 10) and the separate-kernel path
def test_speculative_pass_is_bitwise_neutral(k):
    """prmf_block_end(prefetch=1) starts the next step's X.V pass (and U update) before the host has the score
    tables; U, V, objectives, snapshots and restores must be what they are without it."""
    from prmf_b200 import CudaEngine, pack_pathways
    X, nodelist, Gs, U, V, active = _instance(300, 1200, k, 9, seed=21)
    packed = pack_pathways(Gs, nodelist)
    results = []
    for prefetch in (False, True):
        with CudaEngine(300, 300, 1200, k) as eng:
            eng.set_X(X); eng.set_pathways(packed); eng.set_UV(U, V)
            log = []
            for block in range(3):
                eng.set_active([(a + block) % 9 for a in active])
                eng.step_async(4, 2.0, 0.4)
                parts, _, _, tables = eng.block_end(4, want_scores=True, prefetch=prefetch)
                log.append((parts.copy(), tables[0].copy(), eng.get_UV()))
                if block == 0:
                    eng.snapshot_best()
            after = eng.get_UV()
            eng.restore_best()                       # discards the speculative pass
            best = eng.get_UV()
            eng.set_active(active)
            parts2, _, _ = eng.step(2, 2.0, 0.4)     # and the engine carries on correctly from the restored state
            results.append((log, after, best, parts2, eng.get_UV()))
    a, b = results
    for (pa, ta, uva), (pb, tb, uvb) in zip(a[0], b[0]):
        assert np.array_equal(pa, pb) and np.array_equal(ta, tb)
        assert np.array_equal(uva[0], uvb[0]) and np.array_equal(uva[1], uvb[1])
    for i in (1, 2, 4):
        assert np.array_equal(a[i][0], b[i][0]) and np.array_equal(a[i][1], b[i][1])
    assert np.array_equal(a[3], b[3])
    # the snapshot taken after block 0 is block 0's state
    assert np.array_equal(a[2][0], a[0][0][2][0]) and np.array_equal(a[2][1], a[0][0][2][1])


# ---- the launch-structure switches must not change results ----------------------------------------------
@pytest.mark.parametrize("env", [{"PRMF_EPI": "0"}, {"PRMF_BLOCK": "1"}, {"PRMF_TMA_STAGES": "2"}])
@pytest.mark.parametrize("m,n,k,P", [(200, 517, 10, 12), (1000, 6750, 10, 20), (37, 131, 3, 5)] +
                         [(48, 97 + 10 * k, k, 6) for k in (1, 2, 4, 5, 6, 7, 8, 9)])    # every K of the fused tails
def test_launch_structure_switches(monkeypatch, env, m, n, k, P):
    """PRMF_EPI=0: separate U / V-update launches instead of the fused tails (the path of ranks without rows);
    PRMF_BLOCK=1: the persistent step kernel (the default of sharded runs) on one GPU instead of two fused-tail launches
    per inner step; PRMF_TMA_STAGES=2: the fused-tail X-stream kernels with a ring that wraps every two stages."""
    from prmf_b200 import nmf_manifold_vec_update
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    X, nodelist, Gs, U, V, active = _instance(m, n, k, P, seed=m + n + k, weighted=True)
    Uo, Vo, parts_o, _, _, _ = oracle_block(X, U, V, Gs, nodelist, active, 3, 2.5, 0.3)
    import contextlib, io
    with contextlib.redirect_stdout(io.StringIO()):
        Ug, Vg, od = nmf_manifold_vec_update(X, U, V, Gs, active, n_steps=3, gamma=2.5, delta=0.3, nodelist=nodelist)
    np.testing.assert_allclose(Ug, Uo, rtol=1e-10, atol=1e-13)
    np.testing.assert_allclose(Vg, Vo, rtol=1e-10, atol=1e-13)
    np.testing.assert_allclose(od["obj"], parts_o[-1, 4], rtol=1e-9)


@pytest.mark.parametrize("x_dtype", ["f64", "tf32"])
def test_full_size_properties_config4(x_dtype):
    """BASELINE config 4 shape (37 032 x 6 750, k = 64, 2 000 pathways; stresses the large-k tails and the score
    tables): the same size-independent checks as config 2, plus the k x P tables against the host on a sample of
    (factor, pathway) pairs.  In tf32 mode the tolerances are those of tests/test_tf32.py."""
    from prmf_b200 import CudaEngine, pack_pathways, synth
    from helpers import tf32_round
    m, n, k, P = 37032, 6750, 64, 2000
    X, nodelist, Gs = synth.recount2_shape(m, n, P, seed=0)
    tf32 = x_dtype == "tf32"
    rt = 1e-3 if tf32 else 1e-10
    Xs = tf32_round(X) if tf32 else X                      # the matrix the engine holds
    rng = np.random.Generator(np.random.PCG64(7))
    U = 3 * (1 - rng.random((m, k))); V = 3 * (1 - rng.random((n, k)))
    packed = pack_pathways(Gs, nodelist)
    active = [int(p) for p in rng.integers(0, P, size=k)]
    normX = np.linalg.norm(Xs)
    with CudaEngine(m, m, n, k, x_dtype=x_dtype) as eng:
        eng.set_X(X); eng.set_pathways(packed); eng.set_UV(U, V); eng.set_active(active)
        np.testing.assert_allclose(np.sqrt(eng.normX_sq), normX, rtol=1e-12)
        gamma, delta = normX / k, 10 / normX
        parts, _, _ = eng.step(1, gamma, delta)
        U1, V1 = eng.get_UV()
        rows = rng.integers(0, m, size=48)
        num = Xs[rows] @ V
        den = U[rows] @ (V.T @ V) + U[rows]
        np.testing.assert_allclose(U1[rows], U[rows] * num / den, rtol=max(rt, 1e-10))
        np.testing.assert_allclose(parts[0, 3], np.sum(U1 * U1), rtol=1e-11)
        # genes outside every active pathway: V update without sparse terms (:425-444)
        B = Xs[:, :40].T @ U1
        Vn = V[:40] * B / (V[:40] @ (U1.T @ U1))
        supp = [set(int(g) for g in packed.supports[active[c]]) for c in range(k)]
        free = np.array([[j not in supp[c] for c in range(k)] for j in range(40)])
        np.testing.assert_allclose(V1[:40][free], np.maximum(Vn, 1.1920928955078125e-07)[free], rtol=max(rt, 1e-9))
        parts, g2, d2, (mass, qn, qr) = eng.block_end(0, want_scores=True, prefetch=True)
        parts, _, _ = eng.step(4, gamma, delta)
        np.testing.assert_allclose(parts[-1, 7], eng.residual_sq(), rtol=1e-3 if tf32 else 1e-9)
        assert np.all(np.diff(parts[:, 4]) < 0), "objective should decrease with fixed pathways"
    # score tables of V1 against the host on a sample of pairs (restrict :115-127, force_distinct :232)
    from oracle import prmf_oracle as O
    tables = O.PathwayTables([Gs[p] for p in range(0, P, 97)], nodelist)
    for c in (0, 17, 63):
        v = V1[:, c]
        for q, p in enumerate(range(0, P, 97)):
            score = np.sqrt(mass[c, p]) + 1 - qn[c, p]
            np.testing.assert_allclose(score, O.score_match(tables, v, q), rtol=1e-11)


def test_score_tables_large_and_small_pathways():
    """k x P tables (restrict :115-127, force_distinct :232, find_mins :49) for small and large weighted pathways
    and more factors than warps per block."""
    import networkx as nx
    from oracle import prmf_oracle as O
    from prmf_b200 import latent_pathway_tables
    rng = np.random.Generator(np.random.PCG64(3))
    n, k = 900, 19
    nodelist = ["g%d" % i for i in range(n)]
    Gs = []
    for size in (350, 12, 321, 322, 40):
        genes = rng.choice(n, size=size, replace=False)
        G = nx.Graph()
        G.add_nodes_from(nodelist[g] for g in genes)
        for a, b in zip(genes[:-1], genes[1:]):
            G.add_edge(nodelist[a], nodelist[b], weight=float(rng.random() + 0.5))
        for _ in range(size):
            a, b = rng.choice(genes, size=2, replace=False)
            G.add_edge(nodelist[a], nodelist[b], weight=float(rng.random() + 0.5))
        Gs.append(G)
    V = 3 * (1 - rng.random((n, k)))
    mass, qn, qr = latent_pathway_tables(V, Gs, nodelist)
    tables = O.PathwayTables(Gs, nodelist)
    for c in range(k):
        for p in range(len(Gs)):
            np.testing.assert_allclose(np.sqrt(mass[c, p]) + 1 - qn[c, p], O.score_match(tables, V[:, c], p), rtol=1e-12)
            np.testing.assert_allclose(qr[c, p], tables.Ls[p].dot(V[:, c]).dot(V[:, c]), rtol=1e-11)


# ---- the persistent step kernel (block.cuh) -------------------------------------------------------------
@pytest.mark.parametrize("m,n,k,P", [(300, 1200, 6, 9), (1500, 2100, 10, 12), (37, 131, 3, 5), (700, 523, 10, 9)])
def test_persistent_step_kernel_matches_two_launch_path(monkeypatch, m, n, k, P):
    """One cooperative launch per block of steps (PRMF_BLOCK=1; the default of sharded runs) against the two-launches-per-step path over
    three blocks with the speculative pass on: same objective parts, score tables, U and V to rounding (the two
    differ only in the order the U^T U partials of a share are added)."""
    from prmf_b200 import CudaEngine, pack_pathways
    X, nodelist, Gs, U, V, active = _instance(m, n, k, P, seed=3 * m + k, weighted=True)
    packed = pack_pathways(Gs, nodelist)
    results = []
    for block in ("1", "0"):
        monkeypatch.setenv("PRMF_BLOCK", block)
        with CudaEngine(m, m, n, k) as eng:
            eng.set_X(X); eng.set_pathways(packed); eng.set_UV(U, V)
            log = []
            for blk in range(3):
                eng.set_active([(a + blk) % P for a in active])
                eng.step_async(5, 2.0, 0.4)
                parts, _, _, tables = eng.block_end(5, want_scores=True, prefetch=blk < 2)
                log.append((parts.copy(), tables[0].copy(), tables[1].copy()) + eng.get_UV())
            launches = eng.launch_count
            results.append((log, launches))
    (a, la), (b, lb) = results
    assert la < lb, "the persistent path must launch fewer kernels (%d vs %d)" % (la, lb)
    for x, y in zip(a, b):
        for u, v in zip(x, y):
            np.testing.assert_allclose(u, v, rtol=1e-11, atol=1e-13)


def test_persistent_step_kernel_against_oracle_many_steps(monkeypatch):
    """Ten steps in one launch against the oracle (every step's objective parts)."""
    from prmf_b200 import CudaEngine, pack_pathways
    monkeypatch.setenv("PRMF_BLOCK", "1")
    X, nodelist, Gs, U, V, active = _instance(900, 1300, 10, 14, seed=77, weighted=True)
    Uo, Vo, parts_o, _, _, _ = oracle_block(X, U, V, Gs, nodelist, active, 10, 1.7, 0.6)
    with CudaEngine(900, 900, 1300, 10) as eng:
        eng.set_X(X); eng.set_pathways(pack_pathways(Gs, nodelist)); eng.set_UV(U, V); eng.set_active(active)
        l0 = eng.launch_count
        parts, _, _ = eng.step(10, 1.7, 0.6)
        assert eng.launch_count - l0 <= 3, "10 steps = 1 persistent launch + the deferred objective (+ the active-set build)"
        Ug, Vg = eng.get_UV()
    np.testing.assert_allclose(parts[:, :5], parts_o, rtol=1e-9)
    np.testing.assert_allclose(Ug, Uo, rtol=1e-9, atol=1e-13)
    np.testing.assert_allclose(Vg, Vo, rtol=1e-9, atol=1e-13)


def test_bounded_wait_returns_timeout_instead_of_hanging(monkeypatch):
    """A launch whose thread blocks wait for an arrival that never comes (injected) must end after the deadline with
    PRMF_ERR_TIMEOUT, and the handle must refuse further steps (SURVEY section 5)."""
    from prmf_b200 import CudaEngine, pack_pathways
    from prmf_b200._lib import PrmfLibraryError
    monkeypatch.setenv("PRMF_SPIN_TIMEOUT_MS", "200")
    monkeypatch.setenv("PRMF_BLOCK", "1")
    X, nodelist, Gs, U, V, active = _instance(300, 600, 6, 5, seed=4)
    with CudaEngine(300, 300, 600, 6) as eng:
        eng.set_X(X); eng.set_pathways(pack_pathways(Gs, nodelist)); eng.set_UV(U, V); eng.set_active(active)
        eng.step(2, 1.0, 1.0)
        eng.inject_fault(1)
        import time
        t0 = time.perf_counter()
        with pytest.raises(PrmfLibraryError, match="wait expired"):
            eng.step(2, 1.0, 1.0)
        assert time.perf_counter() - t0 < 20
        with pytest.raises(PrmfLibraryError, match="failed state"):
            eng.step(1, 1.0, 1.0)


def test_score_tables_pathway_larger_than_staging_buffer():
    """A support too large for the shared-memory staging of scores_kernel takes the global-gather branch."""
    import networkx as nx
    from oracle import prmf_oracle as O
    from prmf_b200 import latent_pathway_tables
    rng = np.random.Generator(np.random.PCG64(13))
    n, k = 4000, 10
    nodelist = list(range(n))
    Gs = []
    for size in (2600, 30, 900):
        genes = rng.choice(n, size=size, replace=False)
        G = nx.Graph()
        G.add_nodes_from(int(g) for g in genes)
        for a, b in zip(genes[:-1], genes[1:]):
            G.add_edge(int(a), int(b), weight=float(rng.random() + 0.5))
        for _ in range(2 * size):
            a, b = rng.choice(genes, size=2, replace=False)
            G.add_edge(int(a), int(b), weight=float(rng.random() + 0.5))
        Gs.append(G)
    V = 3 * (1 - rng.random((n, k)))
    mass, qn, qr = latent_pathway_tables(V, Gs, nodelist)
    tables = O.PathwayTables(Gs, nodelist)
    for c in range(k):
        for p in range(len(Gs)):
            np.testing.assert_allclose(np.sqrt(mass[c, p]) + 1 - qn[c, p], O.score_match(tables, V[:, c], p), rtol=1e-12)
            np.testing.assert_allclose(qr[c, p], tables.Ls[p].dot(V[:, c]).dot(V[:, c]), rtol=1e-11)


def test_tight_fit_recon_falls_back_to_the_explicit_residual():
    """Noiseless low-rank X started next to its exact factors: recon^2 is ~1e-12 of ||X||^2, where the identity
    ||X||^2 - 2 sum(V*B) + tr(Gu Gv) has no correct digits left.  The last step of a block (the one the driver's
    convergence test and best-iterate choice read, :745-774) must then carry the explicit residual (:337)."""
    from prmf_b200 import CudaEngine, pack_pathways, synth
    rng = np.random.Generator(np.random.PCG64(8))
    m, n, k = 400, 900, 5
    Ut = rng.gamma(2.0, size=(m, k)); Vt = rng.gamma(2.0, size=(n, k))
    X = Ut @ Vt.T
    nodelist = list(range(n))
    Gs = synth.random_pathway_graphs(rng, n, 6, median_size=12, sigma=0.2, lo=5, hi=20)
    with CudaEngine(m, m, n, k) as eng:
        eng.set_X(X); eng.set_pathways(pack_pathways(Gs, nodelist))
        eng.set_UV(Ut * (1 + 1e-7 * rng.random((m, k))), Vt * (1 + 1e-7 * rng.random((n, k))))
        eng.set_active([0, 1, 2, 3, 4])
        parts, _, _ = eng.step(2, 1e-9, 1e-9)                    # negligible regularisation: the fit stays tight
        U, V = eng.get_UV()
    exact = np.linalg.norm(X - U @ V.T)
    assert exact ** 2 < 1e-8 * np.linalg.norm(X) ** 2, "the instance is not in the cancellation regime"
    np.testing.assert_allclose(parts[-1, 0], exact, rtol=1e-6)
    np.testing.assert_allclose(parts[-1, 4], exact + parts[-1, 5] * parts[-1, 1] + parts[-1, 6] * parts[-1, 2] + parts[-1, 3], rtol=1e-12)
