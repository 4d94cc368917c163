"""Pathway-seeded initialisation on the GPU (prmf_b200.manifold_init): the batched device NNLS against
scipy.optimize.nnls column by column, its error paths, and pathway_init against the reference's per-factor loop
(script/prmf_runner.py:272-334, :1023-1064, restated in tests/init_reference.py)."""
import numpy as np
import pytest

import init_reference as R


def _instance(name):
    rng = np.random.Generator(np.random.PCG64(len(name) * 7919))
    if name == "test1":
        from prmf_b200 import synth
        X, nodelist, Gs = synth.test1_instance()
        return X, [R.pathway_to_vec(X, G, nodelist)[0].ravel() for G in Gs]
    if name == "rank3":
        return rng.random((200, 3)) @ rng.random((3, 150)), []
    m, n = (int(s) for s in name[1:].split("x"))
    return rng.random((m, n)), []


def _rhs(X, seeds, k, transpose, seed):
    """k right-hand sides: the instance's pathway vectors first (A = X^T), then pathway-like and signed vectors."""
    rng = np.random.Generator(np.random.PCG64(seed))
    rows = X.shape[1] if transpose else X.shape[0]
    cols = [s for s in seeds if transpose][:k]
    while len(cols) < k:
        c = len(cols)
        if c % 3 == 2:
            b = rng.standard_normal(rows)                                       # signed: some optima on the boundary
        else:
            b = rng.random(rows) * 0.2
            b[rng.choice(rows, size=max(1, rows // 20), replace=False)] += 1.0  # a bump on a few rows
        cols.append(b / np.linalg.norm(b))
    return np.stack(cols, axis=1)


def _scipy(X, B, transpose):
    import scipy.optimize
    A = X.T if transpose else X
    out = [scipy.optimize.nnls(A, B[:, c]) for c in range(B.shape[1])]
    return np.stack([o[0] for o in out], axis=1), np.array([o[1] for o in out])


def _assert_matches(x, rn, xr, rnr):
    for c in range(x.shape[1]):
        assert set(np.flatnonzero(x[:, c] > 0)) == set(np.flatnonzero(xr[:, c] > 0)), "support of column %d" % c
        scale = np.abs(xr[:, c]).max()
        assert np.abs(x[:, c] - xr[:, c]).max() <= 1e-9 * scale, "column %d" % c
        assert abs(rn[c] - rnr[c]) <= 1e-10 * rnr[c] + 1e-14, "rnorm of column %d" % c     # unit-norm b: exact fits


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 3, 6, 10, 17])
@pytest.mark.parametrize("transpose", [True, False])
@pytest.mark.parametrize("name", ["test1", "u37x129", "u333x517", "u1000x300", "rank3"])
def test_nnls_x_matches_scipy(name, transpose, k):
    from prmf_b200.manifold_init import nnls_x
    X, seeds = _instance(name)
    B = _rhs(X, seeds, k, transpose, seed=k)
    x, rn = nnls_x(X, B, transpose=transpose)
    xr, rnr = _scipy(X, B, transpose)
    assert x.shape == xr.shape and (x >= 0).all()
    _assert_matches(x, rn, xr, rnr)
    x2, rn2 = nnls_x(X, B, transpose=transpose)
    assert np.array_equal(x, x2) and np.array_equal(rn, rn2), "two calls differ"


@pytest.mark.gpu
def test_nnls_x_step_back_and_zero_rhs():
    """A 3 x 3 case worked by hand: column 0 enters first (largest A^T b = 15), column 1 next; the least-squares
    solution on {0, 1} has a negative coefficient for 0, so the step stops at the boundary and drops it, leaving
    x = (0, 11/17, 0) with ||r||^2 = ||b||^2 - 11^2 / 17 = 49 / 17.  b = 0 gives x = 0, ||r|| = 0."""
    from prmf_b200.manifold_init import nnls_x
    A = np.array([[3.0, 2.0, 3.0], [4.0, 3.0, 1.0], [3.0, 2.0, 0.0]])
    b = np.array([0.0, 3.0, 1.0])
    x, rn = nnls_x(A, b, transpose=False)
    np.testing.assert_allclose(x, [0.0, 11.0 / 17.0, 0.0], rtol=1e-14, atol=0)
    assert x[0] == 0.0 and x[2] == 0.0
    np.testing.assert_allclose(rn, np.sqrt(49.0 / 17.0), rtol=1e-14)
    with pytest.raises(RuntimeError, match="Maximum number of iterations reached."):
        nnls_x(A, b, transpose=False, maxiter=2)                # scipy needs 4: two entries, one step back, the last test
    x, _ = nnls_x(A, b, transpose=False, maxiter=4)
    np.testing.assert_allclose(x, [0.0, 11.0 / 17.0, 0.0], rtol=1e-14)
    X = np.random.Generator(np.random.PCG64(3)).random((40, 25))
    for transpose in (True, False):
        B = np.zeros((25 if transpose else 40, 3))
        x, rn = nnls_x(X, B, transpose=transpose)
        assert not x.any() and not rn.any()


@pytest.mark.gpu
def test_nnls_x_iteration_limit_and_capacity():
    import scipy.optimize
    from prmf_b200._lib import PrmfLibraryError
    from prmf_b200.manifold_init import nnls_x
    X = np.random.Generator(np.random.PCG64(4)).random((60, 40))
    b = np.ones(40)
    scipy.optimize.nnls(X.T, b)                                  # needs more than one iteration there as well
    with pytest.raises(RuntimeError, match="Maximum number of iterations reached."):
        scipy.optimize.nnls(X.T, b, maxiter=1)
    with pytest.raises(RuntimeError, match="Maximum number of iterations reached."):
        nnls_x(X, b, transpose=True, maxiter=1)
    # every one of 1100 variables is passive in the solution: more than the 1024 columns the workspace holds
    D = np.diag(np.linspace(1.0, 2.0, 1100))
    with pytest.raises(PrmfLibraryError, match="1024"):
        nnls_x(D, np.ones(1100), transpose=False)


def test_nnls_x_checks_before_the_device():
    """Shapes and finiteness are checked on the host first (runs without a GPU)."""
    from prmf_b200.manifold_init import nnls_x, pathway_init
    X = np.ones((5, 4))
    with pytest.raises(ValueError, match="Incompatible"):
        nnls_x(X, np.ones(5), transpose=True)
    with pytest.raises(ValueError, match="Incompatible"):
        nnls_x(X, np.ones((4, 2)), transpose=False)
    with pytest.raises(ValueError, match="2D"):
        nnls_x(np.ones(5), np.ones(5), transpose=False)
    with pytest.raises(ValueError, match="NaN"):
        nnls_x(X, np.full(4, np.nan), transpose=True)
    bad = X.copy()
    bad[1, 2] = np.inf
    with pytest.raises(ValueError, match="NaN"):
        nnls_x(bad, np.ones(4), transpose=True)
    with pytest.raises(ValueError, match="nodelist"):
        pathway_init(X, [], ["a", "b"])


def _random_pathways(n, count, seed):
    import networkx as nx
    rng = np.random.Generator(np.random.PCG64(seed))
    nodelist = ["g%d" % i for i in range(n)]
    Gs = []
    for _ in range(count):
        G = nx.Graph()
        G.add_nodes_from(nodelist[i] for i in rng.choice(n, size=int(rng.integers(20, 120)), replace=False))
        Gs.append(G)
    return nodelist, Gs


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["test1", "random2000x3000"])
def test_pathway_init_matches_reference_loop(case):
    import random
    import torch
    from prmf_b200 import pathway_init, synth
    if case == "test1":
        X, nodelist, Gs = synth.test1_instance()
        Gs = [Gs[i] for i in (3, 1, 5, 0, 2, 4)]
    else:
        X = np.random.Generator(np.random.PCG64(11)).random((2000, 3000))
        nodelist, Gs = _random_pathways(3000, 10, seed=12)
    Ur, Vr = R.pathway_init(X, Gs, nodelist)
    np_state, py_state = np.random.get_state(), random.getstate()
    U, V = pathway_init(X, Gs, nodelist)
    assert np.array_equal(np.random.get_state()[1], np_state[1]) and random.getstate() == py_state, "RNG consumed"
    assert U.shape == Ur.shape and V.shape == Vr.shape
    assert np.abs(U - Ur).max() <= 1e-9 * np.abs(Ur).max()
    assert np.abs(V - Vr).max() <= 1e-9 * np.abs(Vr).max()
    Ud, Vd = pathway_init(torch.from_numpy(X).cuda(), Gs, nodelist)
    assert np.array_equal(U, Ud) and np.array_equal(V, Vd), "host X and device X differ"


def _kkt(A, b, x):
    """x >= 0, w = A^T (b - A x) <= eps where x = 0 and |w| <= eps where x > 0, eps = 1e-10 max|A^T b|."""
    w = A.T @ (b - A @ x)
    eps = 1e-10 * np.abs(A.T @ b).max()
    assert (x >= 0).all()
    assert (w[x == 0] <= eps).all(), "dual feasibility: %g > %g" % (w[x == 0].max(), eps)
    if (x > 0).any():
        assert np.abs(w[x > 0]).max() <= eps, "stationarity: %g > %g" % (np.abs(w[x > 0]).max(), eps)


@pytest.mark.gpu
def test_init_solves_at_config2_shape_satisfy_kkt():
    """37 032 x 6 750 (config 2), 10 pathways: both batched solves of the init, checked by the KKT conditions."""
    import torch
    from prmf_b200 import synth
    from prmf_b200.manifold_init import nnls_x
    X, nodelist, Gs = synth.recount2_shape(n_pathways=10)
    Xd = torch.from_numpy(X).cuda()
    V0 = np.concatenate([R.pathway_to_vec(X, G, nodelist)[0] for G in Gs], axis=1)
    u, _ = nnls_x(Xd, V0, transpose=True)                       # raises unless every problem converged
    for c in range(u.shape[1]):
        _kkt(X.T, V0[:, c], u[:, c])
    U0 = u / np.linalg.norm(u, axis=0) ** 2
    v, _ = nnls_x(Xd, U0, transpose=False)
    for c in range(v.shape[1]):
        _kkt(X, U0[:, c], v[:, c])
