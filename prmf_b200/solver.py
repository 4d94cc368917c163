"""Host side of the PRMF alternating loop: the reference's control flow, RNG stream and candidate
bookkeeping (script/prmf_runner.py:556-792), with every array operation delegated to the device engine.

Public entry points keep the reference's names and argument meaning:

    nmf_pathway(X, Gs, gamma, delta, tradeoff, k_latent, tol, max_iter, nodelist, modulus,
                U_init, V_init, verbose)                          prmf_runner.py:556
    restrict / force_distinct_lapls / find_mins                    prmf_runner.py:129 / :209 / :37
    nmf_manifold_vec_update / nmf_manifold_vec_obj                 prmf_runner.py:374 / :336

The last two take the packed pathway tables and the list of active pathways instead of the four dicts
of n x n scipy matrices (k_to_W, k_to_D, k_to_L, k_to_feat_inds); see INTEGRATION.md.
"""
import datetime
import math
import sys

import numpy as np

from .dist import DistContext, row_block
from .engine import CudaEngine, attach_collectives
from .pathways import PackedPathways, pack_pathways

PERCENTILE = 19.9                              # prmf_runner.py:159
OBJ_KEYS = ("recon", "manifold", "ignore", "fro", "gamma", "delta", "obj")


def _obj_dict(row):
    """One row of prmf_step's output -> the reference's obj_data dict (:363-371)."""
    return {"recon": float(row[0]), "manifold": float(row[1]), "ignore": float(row[2]),
            "fro": float(row[3]), "gamma": float(row[5]), "delta": float(row[6]), "obj": float(row[4])}


def default_engine_factory(m_local, m_global, n, k, ctx, x_dtype="f64"):
    """One CUDA engine per rank; with more than one rank the engines share an NCCL communicator."""
    device = _rank_device(ctx) if ctx.world > 1 else _current_device()
    eng = CudaEngine(m_local, m_global, n, k, device=device, x_dtype=x_dtype)
    return attach_collectives(eng, ctx)


def _rank_device(ctx):
    """One GPU per rank; ranks beyond the visible devices wrap around (several ranks on one GPU: tests on a one-GPU box)."""
    try:
        import torch
        n = torch.cuda.device_count()
        if n > 0:
            return ctx.local_rank % n
    except ImportError:
        pass
    return ctx.local_rank


def _current_device():
    try:
        import torch
        if torch.cuda.is_available():
            return torch.cuda.current_device()
    except ImportError:
        pass
    return 0


# ----------------------------------------------------------------------------------------------------
# candidate bookkeeping (host)
# ----------------------------------------------------------------------------------------------------
def init_latent_to_pathway_data(k_latent, n_pathways):
    """Every pathway is a candidate of every factor with score 1 (:196-200)."""
    ids, ones = np.arange(n_pathways, dtype=np.int64), np.ones(n_pathways)
    return {k: _CandArrays(ids, ones, [(p, 1) for p in range(n_pathways)]) for k in range(k_latent)}


def count_distinct_pathways(latent_to_pathway_data):
    return min(len(v) for v in latent_to_pathway_data.values())            # :203-207


def _ids_scores(data):
    """Candidate list [(pathway, score), ...] -> (int64 ids, float64 scores)."""
    if isinstance(data, _CandArrays):
        return data.ids, data.scores
    ids = np.fromiter((p for p, _ in data), dtype=np.int64, count=len(data))
    scores = np.fromiter((s for _, s in data), dtype=np.float64, count=len(data))
    return ids, scores


class _CandArrays:
    """The reference's candidate list [(pathway, score), ...] held as two arrays; tuples are made only when
    somebody iterates or indexes (verbose printing, traces, the returned obj_data)."""
    __slots__ = ("ids", "scores", "_fixed")

    def __init__(self, ids, scores, as_list=None):
        self.ids, self.scores, self._fixed = ids, scores, as_list

    def __len__(self):
        return self.ids.shape[0]

    def __iter__(self):
        return iter(self._fixed) if self._fixed is not None else zip(self.ids.tolist(), self.scores)

    def __getitem__(self, i):
        return list(self)[i]

    def __eq__(self, other):
        return list(self) == list(other)

    def __repr__(self):
        return repr(list(self))


def sample_active(latent_to_pathway_data, k_latent):
    """One multinomial draw per factor from the global legacy NumPy RNG, in factor order (:717-730).
    `scipy.stats.multinomial.rvs(1, p)` draws exactly `np.random.multinomial(1, p)` (the last
    probability is implied), and a single-candidate draw consumes no random numbers in either -- so it is
    skipped (its probability is still formed: a zero score must raise as `np.seterr(divide='raise')` does, :22)."""
    active = []
    multinomial = np.random.multinomial
    with np.errstate(divide="raise", invalid="raise"):
        for k in range(k_latent):
            ids, scores = _ids_scores(latent_to_pathway_data[k])
            prob = scores / scores.sum()
            if ids.shape[0] == 1:
                active.append(int(ids[0]))
                continue
            draw = multinomial(1, prob)
            active.append(int(ids[int(draw.argmax())]))
    return active


_Q199 = np.true_divide(PERCENTILE, np.float64(100))


def percentile_19_9(x):
    """`np.percentile(x, 19.9)` for a 1-D float64 array (method 'linear'), without numpy's per-call
    overhead: virtual index (n-1)*q, the two neighbouring order statistics, numpy's `_lerp`.
    tests/test_host_logic.py checks bit-for-bit agreement with np.percentile."""
    n = x.shape[0]
    vi = (n - 1) * _Q199
    lo = int(math.floor(vi))
    hi = min(lo + 1, n - 1)
    g = vi - lo
    part = np.partition(x, (lo, hi))
    a, b = part[lo], part[hi]
    diff = b - a
    if g >= 0.5:
        return b - diff * (1 - g)
    return a + diff * g


def _restrict_numpy(mass, quad_norm, k, ids):
    """One factor of `restrict` in numpy (the expressions prmf_host_restrict evaluates in C)."""
    scores = np.sqrt(mass[k, ids]) + (1 - quad_norm[k, ids])                # :123-125
    keep = np.flatnonzero(scores > percentile_19_9(scores))                 # :171
    return scores, keep


_host_restrict_batch = None


def _restrict_native(mass, quad_norm, todo):
    """All factors of a `restrict` call through libprmf_b200's host helper (plain C++, no CUDA involved): one FFI
    crossing, bit-identical results.  todo: [(k, ids)].  Returns {k: _CandArrays}."""
    global _host_restrict_batch
    if _host_restrict_batch is None:
        from . import _lib
        _host_restrict_batch = _lib.load().prmf_host_restrict_batch
    nf = len(todo)
    factor = np.fromiter((k for k, _ in todo), dtype=np.int32, count=nf)
    off = np.zeros(nf + 1, dtype=np.int64)
    np.cumsum([ids.shape[0] for _, ids in todo], out=off[1:])
    ids_all = np.concatenate([ids for _, ids in todo]).astype(np.int64, copy=False)
    total = int(off[-1])
    kept_ids = np.empty(total, dtype=np.int64)
    kept_scores = np.empty(total)
    kept_off = np.empty(nf + 1, dtype=np.int64)
    rc = _host_restrict_batch(mass.ctypes.data, quad_norm.ctypes.data, mass.shape[1], nf, factor.ctypes.data,
                              ids_all.ctypes.data, off.ctypes.data, _Q199, kept_ids.ctypes.data,
                              kept_scores.ctypes.data, kept_off.ctypes.data)
    if rc == -1000000:
        raise ValueError("prmf_host_restrict_batch: bad arguments")
    if rc < 0:
        k, ids = todo[int(-rc) - 1]
        raise ValueError("restrict: all %d candidate scores of factor %d are equal; the reference's fallback "
                         "(prmf_runner.py:173-183) raises here too" % (len(ids), k))
    bounds = kept_off.tolist()
    return {k: _CandArrays(kept_ids[bounds[f]:bounds[f + 1]], kept_scores[bounds[f]:bounds[f + 1]])
            for f, (k, _) in enumerate(todo)}


def restrict_from_tables(mass, quad_norm, latent_to_pathway_data, native=True):
    """`restrict` (:129-194) given the device tables: score = sqrt(mass) + (1 - quad_norm); keep the
    candidates strictly above the 19.9th percentile (linear interpolation).  `native=False` evaluates the same
    expressions in numpy (the two are bit-identical; tests/test_host_logic.py)."""
    out = {}
    todo = []
    for k in sorted(latent_to_pathway_data):
        data = latent_to_pathway_data[k]
        if len(data) > 1:
            todo.append((k, _ids_scores(data)[0]))
        else:
            out[k] = data
    if not todo:
        return out
    if (native and mass.dtype == np.float64 and quad_norm.dtype == np.float64 and mass.flags.c_contiguous
            and quad_norm.flags.c_contiguous and mass.shape == quad_norm.shape):
        out.update(_restrict_native(mass, quad_norm, todo))
    else:
        for k, ids in todo:
            scores, keep = _restrict_numpy(mass, quad_norm, k, ids)
            if len(keep) == 0:
                # the reference falls into np.random.choice(size=ceil(n*(1-19.9)/100) < 0) and raises
                raise ValueError("restrict: all %d candidate scores of factor %d are equal; the "
                                 "reference's fallback (prmf_runner.py:173-183) raises here too"
                                 % (len(ids), k))
            out[k] = _CandArrays(ids[keep], scores[keep])
    return {k: out[k] for k in sorted(out)}


def force_distinct_from_tables(quad_raw, V, supports, active, latent_to_pathway_data, gamma, delta):
    """`force_distinct_lapls` (:209-258): max-weight matching of factors to remaining candidates with
    weight 1/(gamma * v^T L v + delta * ign).  `ign` is the ignore penalty of the LAST factor only --
    the reference overwrites instead of accumulating (:234-235) -- and is kept that way."""
    import networkx as nx
    ign = 0
    for k2 in sorted(latent_to_pathway_data):
        ign = np.sum(np.power(V[supports[active[k2]], k2] + 1, -1))
    G = nx.Graph()
    for k, data in latent_to_pathway_data.items():
        for p, _ in data:
            denom = gamma * quad_raw[k, p] + delta * ign                    # :237
            G.add_edge("k%d" % k, "l%d" % p, weight=0 if denom == 0 else 1 / denom)
    for a, b in nx.max_weight_matching(G):                                  # :246
        kn, ln = (a, b) if a[0] == "k" else (b, a)
        latent_to_pathway_data[int(kn[1:])] = [(int(ln[1:]), 2)]            # :257
    return latent_to_pathway_data


def find_mins_from_table(quad_raw):
    """`find_mins` (:37-54): argmin_p v_k^T L_p v_k, first minimum wins."""
    return np.argmin(quad_raw, axis=1).astype(np.float64)


# ----------------------------------------------------------------------------------------------------
# inner seams with engine-backed arithmetic
# ----------------------------------------------------------------------------------------------------
def _as_packed(pathways, nodelist, n):
    if isinstance(pathways, PackedPathways):
        return pathways
    if nodelist is None:
        nodelist = list(range(n))
    return pack_pathways(pathways, nodelist)


def nmf_manifold_vec_update(X, U, V, pathways, active, n_steps=10, gamma=1.0, delta=1.0, i=0,
                            verbose=False, norm_X=None, tradeoff=None, nodelist=None, engine=None):
    """`n_steps` multiplicative updates with fixed active pathways (:374-451 / :497-554) on host arrays:
    X, U, V go to the GPU, the steps run there, U and V come back.  Returns (U, V, obj_data) or, with
    `tradeoff`, (U, V, obj_data, gamma, delta) like the reference's two functions."""
    X = np.asarray(X)
    m, n = X.shape
    k = V.shape[1]
    own = engine is None
    eng = engine or CudaEngine(m, m, n, k, device=_current_device())
    try:
        if own:
            eng.set_X(X)
            eng.set_pathways(_as_packed(pathways, nodelist, n))
        eng.set_UV(U, V)
        eng.set_active(active)
        parts, g2, d2 = eng.step(n_steps, gamma, delta, tradeoff)
        for s in range(n_steps):
            print(i + s + 1, float(parts[s, 4]))                            # :447
            if verbose:
                print(_obj_dict(parts[s]))
        U2, V2 = eng.get_UV()
    finally:
        if own:
            eng.close()
    obj_data = _obj_dict(parts[-1])
    if tradeoff is not None:
        return U2, V2, obj_data, g2, d2
    return U2, V2, obj_data


def nmf_manifold_vec_obj(X, U, V, pathways, active, gamma=1, delta=1, nodelist=None, engine=None):
    """Objective parts for host arrays (:336-372): {'recon','manifold','ignore','fro','gamma','delta','obj'}.
    recon is taken by an explicit pass over X, as the reference does."""
    X = np.asarray(X)
    m, n = X.shape
    k = V.shape[1]
    own = engine is None
    eng = engine or CudaEngine(m, m, n, k, device=_current_device())
    try:
        if own:
            eng.set_X(X)
            eng.set_pathways(_as_packed(pathways, nodelist, n))
        eng.set_UV(U, V)
        eng.set_active(active)
        return _obj_dict(eng.objective(gamma, delta))
    finally:
        if own:
            eng.close()


def latent_pathway_tables(V, pathways, nodelist=None, engine=None):
    """(mass, quad_norm, quad_raw), each k x P, for a host V (score/restrict/force_distinct/find_mins)."""
    V = np.asarray(V, dtype=np.float64)
    n, k = V.shape
    own = engine is None
    eng = engine or CudaEngine(0, 0, n, k, device=_current_device())
    try:
        if own:
            eng.set_pathways(_as_packed(pathways, nodelist, n))
        eng.set_UV(None, V)
        return eng.scores()
    finally:
        if own:
            eng.close()


def restrict(V, pathways, latent_to_pathway_data, nodelist=None):
    """Drop-in for `restrict(V, Ls, latent_to_pathway_data, lapl_to_feat_inds)` (:129)."""
    mass, qn, _ = latent_pathway_tables(V, pathways, nodelist)
    return restrict_from_tables(mass, qn, latent_to_pathway_data)


def find_mins(V, pathways, nodelist=None):
    """Drop-in for `find_mins(V, Ls)` (:37)."""
    return find_mins_from_table(latent_pathway_tables(V, pathways, nodelist)[2])


# ----------------------------------------------------------------------------------------------------
# driver
# ----------------------------------------------------------------------------------------------------
def nmf_pathway(X, Gs, gamma=1.0, delta=1.0, tradeoff=None, k_latent=6, tol=1e-3, max_iter=1000,
                nodelist=None, modulus=10, U_init=None, V_init=None, verbose=False, *,
                ctx=None, engine_factory=None, X_is_local=False, m_global=None, trace=None,
                quiet=False, x_dtype="f64"):
    """Pathway-regularised NMF, X ~ U V^T (prmf_runner.py:556-792), on one or more B200s.

    Positional / keyword arguments, return value, stdout lines, RNG consumption and error behaviour are
    the reference's.  Keyword-only extras: `ctx` (a `DistContext`; default: the initialised
    torch.distributed group, else single process), `X_is_local`/`m_global` (X is already this rank's row
    block), `trace` (dict collecting per-iteration diagnostics), `quiet` (suppress the per-step prints),
    `x_dtype` ("f64": parity mode; "f32": X held as exact fp32 values, one rank only, bitwise the "f64" run on
    X.astype(np.float64); "tf32": opt-in tensor-core X streams; see include/prmf_b200.h).
    With several ranks every rank must call this with the same seed and arguments; all return the same
    full U, V and obj_data.
    """
    ctx = ctx or DistContext.current()
    if x_dtype == "f32" and ctx.world > 1:
        raise ValueError('x_dtype="f32" runs on one rank only (this context has %d ranks)' % ctx.world)
    factory = engine_factory or default_engine_factory
    out = (lambda *a: None) if (quiet or ctx.rank != 0) else print
    if nodelist is None:
        raise TypeError("nodelist is required")                             # :663 iterates over it
    X = np.asarray(X) if not hasattr(X, "is_cuda") else X
    if X_is_local:
        m_local, n = X.shape
        if m_global is None:
            raise ValueError("m_global is required with X_is_local")
        m = int(m_global)
        lo, hi = row_block(m, ctx.world, ctx.rank)
        if hi - lo != m_local:
            raise ValueError("local block has %d rows, rank %d of %d owns %d" % (m_local, ctx.rank, ctx.world, hi - lo))
        X_local = X
    else:
        m, n = X.shape
        lo, hi = row_block(m, ctx.world, ctx.rank)
        X_local = X[lo:hi]
    if len(nodelist) != n:
        raise ValueError("nodelist has %d entries, X has %d columns" % (len(nodelist), n))

    eng = factory(hi - lo, m, n, k_latent, ctx) if x_dtype == "f64" else factory(hi - lo, m, n, k_latent, ctx, x_dtype=x_dtype)
    try:
        eng.set_X(X_local)
        norm_X = math.sqrt(eng.normX_sq)                                    # :640
        out("norm(X) = {}".format(norm_X))                                  # :641
        gamma = gamma * norm_X / k_latent                                   # :644
        delta = delta * 10 / norm_X                                         # :645

        # :650-659 -- every rank draws the full U then V from the same global RNG stream
        if U_init is None:
            U_init = 3 * (1 - np.random.rand(m, k_latent))
        if V_init is None:
            V_init = 3 * (1 - np.random.rand(n, k_latent))
        U_init, V_init = np.asarray(U_init), np.asarray(V_init)
        if U_init.shape != (m, k_latent):
            raise ValueError("Invalid U_init with shape {} != (m_obs, k_latent) = {}".format(U_init.shape, (m, k_latent)))
        if V_init.shape != (n, k_latent):
            raise ValueError("Invalid V_init with shape {} != (n_feature, k_latent) = {}".format(V_init.shape, (n, k_latent)))

        # :670-696 -- graphs restricted to the nodelist, packed once for the device
        if isinstance(Gs, PackedPathways):
            packed = Gs
        else:
            packed = pack_pathways(Gs, nodelist)
            if isinstance(Gs, list):
                for gi, G in enumerate(Gs):                                 # the reference mutates Gs too (:671)
                    if hasattr(G, "subgraph"):
                        Gs[gi] = G.subgraph(nodelist)
        eng.set_pathways(packed)
        eng.set_UV(U_init[lo:hi], V_init)

        cands = init_latent_to_pathway_data(k_latent, packed.P)            # :700
        converged, candidates_remain = False, True
        obj, prev_obj = math.inf, math.inf
        obj_data, best_obj_data = {}, {"obj": np.inf}
        have_best = False
        i = 0
        while (i < max_iter) and (candidates_remain or not converged):     # :715
            active = sample_active(cands, k_latent)                        # :717-730
            if verbose:
                out("--------------------------------------------")
                out("Latent/Pathway association at this iteration")
                out("--------------------------------------------")
                for k, p in enumerate(active):
                    out(k, p)
                out("--------------------------------------------")
            eng.set_active(active)
            # :739-742 -- the 10 steps and (while candidates remain) the score tables are enqueued back to
            # back; the host waits once
            # back; the host waits once, and the GPU already streams X for the next block meanwhile
            eng.step_async(modulus, gamma, delta, tradeoff)
            parts, g2, d2, tables = eng.block_end(modulus, want_scores=candidates_remain,
                                                  prefetch=i + modulus < max_iter)
            for s in range(modulus):
                out(i + s + 1, float(parts[s, 4]))                         # :447
                if verbose:
                    out(_obj_dict(parts[s]))
            obj_data = _obj_dict(parts[-1])
            if tradeoff is not None:
                gamma, delta = g2, d2
            i += modulus

            if obj_data["obj"] < best_obj_data["obj"]:                     # :747-750
                eng.snapshot_best()
                best_obj_data = obj_data
                have_best = True

            kind = None
            if candidates_remain:                                          # :754-768
                if count_distinct_pathways(cands) <= k_latent:
                    quad_raw = tables[2]
                    _, V_now = eng.get_UV(want_U=False)
                    cands = force_distinct_from_tables(quad_raw, V_now, packed.supports, active, cands,
                                                       gamma, delta)
                    candidates_remain = False
                    kind = "force"
                else:
                    if ctx.rank == 0:
                        sys.stderr.write("Before restrict: " + str(datetime.datetime.now()) + "\n")
                    cands = restrict_from_tables(tables[0], tables[1], cands)
                    if ctx.rank == 0:
                        sys.stderr.write("After restrict: " + str(datetime.datetime.now()) + "\n")
                    candidates_remain = any(len(v) > 1 for v in cands.values())
                    kind = "restrict"
                if verbose:
                    print_latent_to_pathway_data(cands, out)
            if trace is not None:
                trace.setdefault("sampled", []).append(list(active))
                trace.setdefault("obj_parts", []).extend(parts[:, [0, 1, 2, 3, 4]].tolist())
                trace.setdefault("recon_sq", []).extend(parts[:, 7].tolist())
                if len(trace.setdefault("blocks", [])) < trace.get("keep_blocks", 3):
                    trace["blocks"].append(eng.get_UV())
                if kind:
                    trace.setdefault("cands", []).append({"kind": kind, "data": {k: list(v) for k, v in cands.items()}})

            prev_obj = obj
            obj = obj_data["obj"]
            converged = (abs(obj - prev_obj)) / obj < tol                   # :772-774

        if have_best and best_obj_data["obj"] < obj_data["obj"]:           # :778-782
            out("Local optima at convergence (or after max iterations) is not the best among all iterates; returning best instead")
            eng.restore_best()
            obj_data = best_obj_data
        U_local, V = eng.get_UV()
        ctx.barrier()          # peers may still be reading this rank's exchange buffer
    finally:
        # (no barrier on the error path: a failed rank must surface its exception instead of parking in a
        #  collective while its peers wait for it inside a kernel; their bounded device waits then fail too)
        eng.close()
    U = ctx.all_gather_rows(U_local, m)
    obj_data = dict(obj_data)
    obj_data["latent_to_pathway_data"] = {k: list(v) for k, v in cands.items()}
    return U, V, obj_data


def print_latent_to_pathway_data(latent_to_pathway_data, out=print):
    """Same report as the reference's verbose mode (:67-88)."""
    out("-----------------------------")
    out("Latent to pathway match data:")
    out("-----------------------------")
    for latent_id, pathway_data in latent_to_pathway_data.items():
        out("Latent vector: {}".format(latent_id))
        for pathway_id, score in sorted(pathway_data, key=lambda x: x[1], reverse=True):
            out("  " + "{}\t{}".format(pathway_id, score))
