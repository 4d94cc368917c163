#!/usr/bin/env python
"""Generate the committed golden fixtures by running the UNMODIFIED reference here.

    python tests/golden/make_golden.py            # writes tests/golden/*.npz

Needs `/root/reference` (build container only).  Each fixture records, for one seeded instance, what
the reference's `nmf_pathway` (script/prmf_runner.py:556-792) did: gamma/delta after rescaling, the
pathway sampled for every factor at every outer iteration (:717-730), every inner step's objective
parts (:336-372), the candidate lists after every `restrict` / `force_distinct_lapls` (:129-258), U and V
after the first three 10-step blocks and at return.  Inputs are stored too, so the fixtures do not
depend on regenerating them bit for bit on another host.
"""
import contextlib
import io
import json
import os
import random
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import ref_shim  # noqa: E402
from prmf_b200 import synth  # noqa: E402


def graphs_to_json(Gs):
    out = []
    for G in Gs:
        out.append({
            "nodes": [n for n in G.nodes()],
            "edges": [[u, v, float(d.get("weight", 1))] for u, v, d in G.edges(data=True)],
            "weighted": any("weight" in d for _, _, d in G.edges(data=True)),
        })
    return out


def trace_nmf_pathway(X, Gs, nodelist, k_latent, seed=1, gamma=1.0, delta=1.0, tradeoff=None,
                      max_iter=1000, keep_blocks=3):
    R = ref_shim.load_reference()
    ref_shim.reset_globals(R)
    trace = {"sampled": [], "obj_parts": [], "cands": [], "blocks_U": [], "blocks_V": [],
             "gd": []}
    orig_map, orig_obj = R.map_k_to_lapls, R.nmf_manifold_vec_obj
    orig_restrict, orig_force = R.restrict, R.force_distinct_lapls
    orig_upd, orig_upd_t = R.nmf_manifold_vec_update, R.nmf_manifold_vec_update_tradeoff

    def map_k(k_to_lapl_ind, *a, **kw):
        trace["sampled"].append([int(k_to_lapl_ind[k]) for k in range(k_latent)])
        return orig_map(k_to_lapl_ind, *a, **kw)

    def obj(*a, **kw):
        d = orig_obj(*a, **kw)
        trace["obj_parts"].append([float(d["recon"]), float(d["manifold"]), float(d["ignore"]),
                                   float(d["fro"]), float(d["obj"])])
        trace["gd"].append([float(d["gamma"]), float(d["delta"])])
        return d

    def rec_cands(kind, d):
        trace["cands"].append({"kind": kind, "data": {
            str(k): [[int(p), float(s)] for p, s in v] for k, v in d.items()}})

    def restrict(*a, **kw):
        d = orig_restrict(*a, **kw)
        rec_cands("restrict", d)
        return d

    def force(*a, **kw):
        d = orig_force(*a, **kw)
        rec_cands("force", d)
        return d

    def upd(*a, **kw):
        out = orig_upd(*a, **kw)
        if len(trace["blocks_U"]) < keep_blocks:
            trace["blocks_U"].append(np.array(out[0])); trace["blocks_V"].append(np.array(out[1]))
        return out

    def upd_t(*a, **kw):
        out = orig_upd_t(*a, **kw)
        if len(trace["blocks_U"]) < keep_blocks:
            trace["blocks_U"].append(np.array(out[0])); trace["blocks_V"].append(np.array(out[1]))
        return out

    R.map_k_to_lapls, R.nmf_manifold_vec_obj = map_k, obj
    R.restrict, R.force_distinct_lapls = restrict, force
    R.nmf_manifold_vec_update, R.nmf_manifold_vec_update_tradeoff = upd, upd_t
    try:
        np.random.seed(seed); random.seed(seed)
        Gs_in = [G.copy() for G in Gs]
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(io.StringIO()):
            U, V, obj_data = R.nmf_pathway(X.copy(), Gs_in, nodelist=list(nodelist), gamma=gamma,
                                           delta=delta, tradeoff=tradeoff, k_latent=k_latent,
                                           max_iter=max_iter)
    finally:
        R.map_k_to_lapls, R.nmf_manifold_vec_obj = orig_map, orig_obj
        R.restrict, R.force_distinct_lapls = orig_restrict, orig_force
        R.nmf_manifold_vec_update, R.nmf_manifold_vec_update_tradeoff = orig_upd, orig_upd_t
    final = {k: float(v) for k, v in obj_data.items() if k != "latent_to_pathway_data"}
    final_map = {str(k): [[int(p), float(s)] for p, s in v]
                 for k, v in obj_data["latent_to_pathway_data"].items()}
    stdout_lines = buf.getvalue().splitlines()
    return dict(U=U, V=V, final=final, final_map=final_map, trace=trace, stdout=stdout_lines)


def save_case(name, X, nodelist, Gs, k_latent, **kw):
    res = trace_nmf_pathway(X, Gs, nodelist, k_latent, **kw)
    tr = res["trace"]
    meta = {
        "name": name, "k_latent": k_latent, "seed": kw.get("seed", 1),
        "gamma_in": kw.get("gamma", 1.0), "delta_in": kw.get("delta", 1.0),
        "tradeoff": kw.get("tradeoff", None), "max_iter": kw.get("max_iter", 1000),
        "nodelist": list(nodelist), "graphs": graphs_to_json(Gs),
        "sampled": tr["sampled"], "cands": tr["cands"], "final": res["final"],
        "final_map": res["final_map"], "stdout_head": res["stdout"][:3],
        "n_inner_steps": len(tr["obj_parts"]),
        "versions": {"numpy": np.__version__},
    }
    np.savez_compressed(
        os.path.join(HERE, name + ".npz"),
        X=X, U_final=res["U"], V_final=res["V"],
        obj_parts=np.array(tr["obj_parts"]), gamma_delta=np.array(tr["gd"]),
        blocks_U=np.array(tr["blocks_U"]), blocks_V=np.array(tr["blocks_V"]),
        meta=np.array(json.dumps(meta)))
    print("%-28s steps=%4d obj=%.10g map=%s" % (
        name, len(tr["obj_parts"]), res["final"]["obj"],
        {k: v[0][0] for k, v in res["final_map"].items()}))


def save_kernel_vectors():
    """Known-answer vectors for the pure numpy/scipy seams (SURVEY.md §8c): one call each of
    normalize_laplacian, score_latent_pathway_match_global, restrict, find_mins."""
    import scipy.sparse as sp
    R = ref_shim.load_reference()
    ref_shim.reset_globals(R)
    X, nodelist, Gs = synth.small_instance(m=20, n=120, k_true=3, n_pathways=9, pathway_size=14,
                                           seed=7, weighted=True)
    n = len(nodelist)
    idx = {g: i for i, g in enumerate(nodelist)}
    rng = np.random.Generator(np.random.PCG64(11))
    V = rng.random((n, 4)) + 0.01
    Ls, supports, Lns = [], [], []
    for G in Gs:
        H = G.subgraph(nodelist)
        W = R.nx.adjacency_matrix(H, nodelist=nodelist)
        D = sp.dia_matrix((np.asarray(W.sum(axis=0)), np.array([0])), shape=(n, n))
        L = sp.csr_matrix(D - W)
        supp = [idx[g] for g in H.nodes()]
        Ls.append(L); supports.append(supp)
        Lns.append(R.normalize_laplacian(L, supp))
    R.PATHWAY_TO_SUPPORT = {i: s for i, s in enumerate(supports)}
    R.NORMALIZED_LAPLACIANS = Lns
    P, K = len(Gs), V.shape[1]
    score = np.zeros((K, P)); quad_raw = np.zeros((K, P)); quad_norm = np.zeros((K, P))
    for k in range(K):
        for p in range(P):
            score[k, p] = R.score_latent_pathway_match_global(V[:, k], p)
            quad_raw[k, p] = Ls[p].dot(V[:, k]).dot(V[:, k])
            vu = V[:, k] / np.linalg.norm(V[:, k])
            quad_norm[k, p] = Lns[p].dot(vu).dot(vu)
    cands = R.init_latent_to_pathway_data(K, Ls)
    restricted = R.restrict(V, Ls, cands, R.PATHWAY_TO_SUPPORT)
    # find_mins (:37-54) is dead code in the reference and only works with dense Laplacians
    # (ndarray.dot(sparse) does not dispatch); feed it dense copies.
    mins = R.find_mins(V, [L.toarray() for L in Ls])
    meta = {"nodelist": nodelist, "graphs": graphs_to_json(Gs),
            "restricted": {str(k): [[int(p), float(s)] for p, s in v] for k, v in restricted.items()}}
    np.savez_compressed(os.path.join(HERE, "kernel_vectors.npz"), V=V, score=score,
                        quad_raw=quad_raw, quad_norm=quad_norm, find_mins=mins,
                        Ln_dense=np.array([Ln.toarray() for Ln in Lns]),
                        meta=np.array(json.dumps(meta)))
    ref_shim.reset_globals(R)
    print("kernel_vectors               P=%d K=%d" % (P, K))


def main():
    from sklearn.preprocessing import quantile_transform
    # C1(i): the reference's own test instance, raw (as the stale golden obj.txt was made) ...
    X, nodelist, Gs = synth.test1_instance()
    save_case("test1_raw", X, nodelist, Gs, 6, max_iter=200)
    # ... and quantile-normalised, which is what the shipped CLI does by default (:1019-1020)
    save_case("test1_norm", quantile_transform(X), nodelist, Gs, 6, max_iter=200)
    # test_inferred_nodelist_2: graph-only genes, zero-padded columns
    X2, nodelist2, Gs2 = synth.test1_instance(unmeasured=True)
    save_case("test2_raw", X2, nodelist2, Gs2, 6, max_iter=100)
    # planted small instance with decoys: many restrict rounds, then matching
    X3, nodelist3, Gs3 = synth.small_instance(seed=3)
    save_case("small_planted", X3, nodelist3, Gs3, 4)
    # weighted edges + tradeoff variant (:497-554)
    X4, nodelist4, Gs4 = synth.small_instance(m=40, n=200, k_true=3, n_pathways=12, seed=5,
                                              weighted=True)
    save_case("small_tradeoff", X4, nodelist4, Gs4, 3, tradeoff=0.5, max_iter=120)
    save_bigk()
    save_kernel_vectors()
    save_side_by_side()


def save_bigk():
    """More factors than a 16-wide factor tile (k = 20 over 30 pathways): pins the large-k tails (tiled U / V updates,
    grid-wide Gram fold, separate objective launch) to the reference itself."""
    X5, nodelist5, Gs5 = synth.small_instance(m=120, n=400, k_true=3, n_pathways=30, pathway_size=16, seed=7)
    save_case("small_bigk", X5, nodelist5, Gs5, 20, max_iter=60)


def save_side_by_side():
    """What the reference's `nmf_pathway` returns (U, V, final objective, factor -> pathway map) on the instances of
    tests/test_oracle_golden.py::test_oracle_vs_live_reference: k = 3, max_iter = 300, default gamma / delta."""
    from make_golden_io import side_by_side_instance
    R = ref_shim.load_reference()
    for seed in (0, 1):
        X, nodelist, Gs = side_by_side_instance(seed)
        ref_shim.reset_globals(R)
        np.random.seed(seed); random.seed(seed)
        with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
            U, V, od = R.nmf_pathway(X.copy(), [G.copy() for G in Gs], nodelist=list(nodelist), k_latent=3, max_iter=300)
        fmap = {str(k): [int(p) for p, _ in v] for k, v in od["latent_to_pathway_data"].items()}
        np.savez_compressed(os.path.join(HERE, "side_by_side_seed%d.npz" % seed), U=U, V=V, obj=np.array(float(od["obj"])),
                            final_map=np.array(json.dumps(fmap)))
        print("side_by_side_seed%d          obj=%.10g map=%s" % (seed, od["obj"], fmap))




# ---- CLI golden (appended): run the reference's own main() on the files of its test ------------------
from make_golden_io import write_cli_inputs  # noqa: E402


def save_cli_case():
    import shutil
    import tempfile
    R = ref_shim.load_reference()
    X, nodelist, Gs = synth.test1_instance()
    tmp = tempfile.mkdtemp()
    cwd = os.getcwd()
    try:
        fps = write_cli_inputs(tmp, X, nodelist, Gs)
        os.chdir(tmp)
        rel = [os.path.basename(f) for f in fps]
        init_order = [rel[i] for i in (3, 1, 5, 0, 2, 4)]      # exactly k files: no set-order-dependent sampling
        for tag, extra in (("nonorm", ["--no-normalize"]), ("norm", []),
                           ("init", ["--no-normalize", "--manifolds-init"] + init_order),
                           ("cv", ["--no-normalize", "--cross-validation", "0.2"])):
            ref_shim.reset_globals(R)
            argv = ["prmf_runner.py", "--data", "data.tsv", "--manifolds"] + rel + [
                "--node-attribute", "name", "--nodelist", "nodelist.txt", "--outdir", ".", "--delimiter", "\t",
                "--seed", "1"] + extra
            old = sys.argv
            sys.argv = argv
            try:
                with contextlib.redirect_stdout(io.StringIO()) as out, contextlib.redirect_stderr(io.StringIO()):
                    R.main()
            finally:
                sys.argv = old
            dst = os.path.join(HERE, "cli_test1_" + tag)
            os.makedirs(dst, exist_ok=True)
            for f in ("obj.txt", "U.csv", "V.csv", "init_pathways.txt", "test_error.csv"):
                if os.path.exists(os.path.join(tmp, f)):
                    shutil.move(os.path.join(tmp, f), os.path.join(dst, f))
            with open(os.path.join(dst, "stdout_head.txt"), "w") as fh:
                fh.write("\n".join(out.getvalue().splitlines()[:12]) + "\n")
            print("cli_test1_%-21s %s" % (tag, open(os.path.join(dst, "obj.txt")).read().splitlines()[6]))
    finally:
        os.chdir(cwd)
        shutil.rmtree(tmp)


if __name__ == "__main__" and "--only-bigk" in sys.argv:
    save_bigk()
    sys.exit(0)

if __name__ == "__main__" and "--only-side-by-side" in sys.argv:
    save_side_by_side()
    sys.exit(0)

if __name__ == "__main__":
    if "--cli-only" not in sys.argv:
        main()
    save_cli_case()
